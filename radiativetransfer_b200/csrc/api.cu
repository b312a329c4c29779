// C-ABI of librtb200.so (declared in include/rtb200.h).  No torch types, no CPU fallback.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <algorithm>
#include <string>

#include "portable_math.h"
#include "rtb200_internal.h"
#include "segment_math.cuh"

namespace rtb {

// device evaluation of the portable exp/log (csrc/portable_math.h) for the bit-identity check against the host build
__global__ void portable_math_kernel(const double* __restrict__ x, int64_t n, double* __restrict__ e, double* __restrict__ l) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    e[i] = rtb_pm::pm_exp(x[i]);
    l[i] = rtb_pm::pm_log(x[i]);
  }
}

// the sweeps' FAST exponential (segment_math.cuh: table + short polynomial) for n host values: e^-tau and 1 - e^-tau,
// evaluated as the sweeps do with kappa = tau and the scaled path of a unit length, kExpScale
__global__ void fast_exp_kernel(const double* __restrict__ tau, int64_t n, double* __restrict__ e, double* __restrict__ ome) {
  __shared__ double sT[kExpTableSize];
  if (threadIdx.x < kExpTableSize) sT[threadIdx.x] = kExpTable32[threadIdx.x];
  __syncthreads();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double Ts, p;
    exp_neg_parts32<true>(tau[i], kExpScale, sT, Ts, p);
    e[i] = fma(Ts, p, Ts);
    ome[i] = fma(-Ts, p, 1.0 - Ts);
  }
}

static thread_local char g_cudaErr[512] = "";

void set_cuda_error(const char* what, cudaError_t e, const char* file, int line) {
  snprintf(g_cudaErr, sizeof(g_cudaErr), "%s:%d: %s -> %s", file, line, what, cudaGetErrorString(e));
  if (getenv("RTB200_VERBOSE")) fprintf(stderr, "[rtb200] %s\n", g_cudaErr);
}
const char* last_cuda_error() { return g_cudaErr; }

int ensure_buffer(void** p, size_t* have, size_t need) {
  if (*p && *have >= need) return RTB200_OK;
  if (*p) { cudaFree(*p); *p = nullptr; *have = 0; }
  cudaError_t e = cudaMalloc(p, need);
  if (e != cudaSuccess) {
    set_cuda_error("cudaMalloc", e, __FILE__, __LINE__);
    *p = nullptr;
    return e == cudaErrorMemoryAllocation ? RTB200_ERR_NOMEM : RTB200_ERR_CUDA;
  }
  *have = need;
  return RTB200_OK;
}

static void free_grid(Context& c) {
  amr_release(c);
  point_release(c);
  cudaFree(c.dLevel); cudaFree(c.dHI); cudaFree(c.dHeI); cudaFree(c.dHeII); cudaFree(c.dRho); cudaFree(c.dAbun2);
  cudaFree(c.dKappa); cudaFree(c.tree.child); cudaFree(c.tree.leafX); cudaFree(c.tree.leafY); cudaFree(c.tree.leafZ);
  cudaFree(c.dJ); cudaFree(c.dRates); c.dRates = nullptr;
  cudaFree(c.dKappaT); c.dKappaT = nullptr; c.kappaTBytes = 0;
  cudaFree(c.dEta); c.dEta = nullptr;
  cudaFree(c.dEtaT); c.dEtaT = nullptr; c.etaTBytes = 0;
  cudaFree(c.dSigma); c.dSigma = nullptr;
  release_source_iteration(c);
  c.scatMaxIter = 1; c.scatTol = 0.; c.scatAccel = 0;
  reset_call_results(c);
  cudaFree(c.dDustSigma); c.dDustSigma = nullptr;
  c.dustMode = 0;
  for (int g = 0; g < 3; g++) c.dustBeta[g] = c.dustAlbedo[g] = 0.;
  free_heating(c);
  cudaFree(c.dLogT); c.dLogT = nullptr;
  for (auto& sl : c.pointPool) cudaFree(sl.first);
  c.pointPool.clear();
  c.dLevel = nullptr; c.dHI = c.dHeI = c.dHeII = c.dRho = c.dAbun2 = c.dKappa = c.dJ = nullptr;
  c.tree = DevTree();
  c.uniPlanKey.clear();
  c.amrPlanKey.clear();
  if (c.graphExec) { cudaGraphExecDestroy(c.graphExec); c.graphExec = nullptr; }
}

// Linear octree from the leaf `level` array alone (readCellArray.f90:154-187): nodes 0..n^3-1 are the base cells in
// leaf order (x slowest); every refined node owns 8 consecutive children, x slowest / z fastest
// (the i, j, k loop order of writeCell, equiSources.f90:4053-4059).
static int build_tree(Context& c, const int8_t* level) {
  const int n = c.nx;
  const int64_t nbase = (int64_t)n * n * n;
  c.hChild.assign((size_t)nbase, 0);
  c.hLeafX.resize((size_t)c.nleaf); c.hLeafY.resize((size_t)c.nleaf); c.hLeafZ.resize((size_t)c.nleaf);
  c.maxLevel = 0;
  for (int a = 0; a < 3; a++) c.refinedLayer[a].clear();
  struct Frame { int32_t node; int32_t x, y, z; int8_t lvl; int8_t next; };
  std::vector<Frame> stack;
  int64_t leaf = 0;
  auto mark_refined = [&](int lvl, int x, int y, int z) {
    for (int a = 0; a < 3; a++) {
      if ((int)c.refinedLayer[a].size() <= lvl) c.refinedLayer[a].resize(lvl + 1);
      auto& v = c.refinedLayer[a][lvl];
      if (v.empty()) v.assign((size_t)n << lvl, 0);
      v[a == 0 ? x : (a == 1 ? y : z)] = 1;
    }
  };
  for (int64_t b = 0; b < nbase; b++) {
    int bx = (int)(b / ((int64_t)n * n)), by = (int)((b / n) % n), bz = (int)(b % n);
    stack.clear();
    stack.push_back({(int32_t)b, bx, by, bz, 0, 0});
    while (!stack.empty()) {
      Frame& f = stack.back();
      if (f.next == 0) {
        if (leaf >= c.nleaf) return RTB200_ERR_LEVELS;
        int lv = level[leaf];
        if (lv == f.lvl) {
          c.hChild[f.node] = -(int32_t)(leaf + 1);
          c.hLeafX[leaf] = f.x; c.hLeafY[leaf] = f.y; c.hLeafZ[leaf] = f.z;
          if (lv > c.maxLevel) c.maxLevel = lv;
          leaf++;
          stack.pop_back();
          continue;
        }
        if (lv < f.lvl) return RTB200_ERR_LEVELS;
        if (c.hChild.size() + 8 > (size_t)INT32_MAX) return RTB200_ERR_ARG;
        int32_t first = (int32_t)c.hChild.size();
        c.hChild[f.node] = first;
        c.hChild.resize(c.hChild.size() + 8, 0);
        mark_refined(f.lvl, f.x, f.y, f.z);
      }
      Frame& g = stack.back();  // hChild.resize does not move the stack
      if (g.next == 8) { stack.pop_back(); continue; }
      int q = g.next++;
      Frame ch{c.hChild[g.node] + q, 2 * g.x + (q >> 2), 2 * g.y + ((q >> 1) & 1), 2 * g.z + (q & 1), (int8_t)(g.lvl + 1), 0};
      stack.push_back(ch);
    }
  }
  if (leaf != c.nleaf) return RTB200_ERR_LEVELS;
  c.tree.nnodes = (int64_t)c.hChild.size();
  return RTB200_OK;
}

static int upload(void** dst, const void* src, size_t bytes, size_t padBytes, cudaStream_t s) {
  cudaError_t e = cudaMalloc(dst, bytes + padBytes ? bytes + padBytes : 8);
  if (e != cudaSuccess) { set_cuda_error("cudaMalloc", e, __FILE__, __LINE__); return e == cudaErrorMemoryAllocation ? RTB200_ERR_NOMEM : RTB200_ERR_CUDA; }
  if (src) RTB_CUDA(cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, s));
  else RTB_CUDA(cudaMemsetAsync(*dst, 0, bytes ? bytes : 8, s));
  if (padBytes) RTB_CUDA(cudaMemsetAsync((char*)*dst + bytes, 0, padBytes, s));
  return RTB200_OK;
}

static int resolve_directions(int nAngularLevel, const int32_t* rays, int32_t nrays, std::vector<Direction>& dirs) {
  if (nAngularLevel < 1 || nAngularLevel > 8) return RTB200_ERR_ARG;
  const int64_t total = 12LL << (2 * (nAngularLevel - 1));
  dirs.clear();
  if (!rays || nrays <= 0) {
    if (rays == nullptr && nrays == 0) {
      for (int64_t r = 0; r < total; r++) dirs.push_back(classify_direction(nAngularLevel, r));
    } else if (nrays < 0) {
      return RTB200_ERR_ARG;
    }  // rays != NULL && nrays == 0: empty shard
  } else {
    for (int32_t q = 0; q < nrays; q++) {
      if (rays[q] < 0 || rays[q] >= total) return RTB200_ERR_ARG;
      dirs.push_back(classify_direction(nAngularLevel, rays[q]));
    }
  }
  for (const auto& d : dirs)
    if (d.status) return d.status;
  return RTB200_OK;
}

int run_sweep(Context& c, int nAngularLevel, const double* uvb, const double* beta, const int32_t* rays, int32_t nrays,
              double* dJ, cudaStream_t s, int64_t* nseg, int iter) {
  if (!uvb || !beta || !dJ) return RTB200_ERR_ARG;
  if (c.nleaf == 0) return RTB200_ERR_ARG;
  std::vector<Direction> dirs;
  if (int st = resolve_directions(nAngularLevel, rays, nrays, dirs)) return st;
  RTB_CUDA(cudaSetDevice(c.device));
  // the later sweeps of a source iteration add their counts to the earlier ones
  const int64_t launches0 = iter > 1 ? c.lastLaunches : 0, sweepLaunches0 = iter > 1 ? c.lastSweepLaunches : 0;
  const double bytes0 = iter > 1 ? c.lastAlgBytes : 0.;
  if (iter <= 1) {
    RTB_CUDA(cudaEventRecord(c.evStart, s));
    if (int st = c.dustMode ? launch_compute_opacities_dust(c, beta, s) : launch_compute_opacities(c, beta, s)) return st;
    if (c.dSigma)
      if (int st = launch_add_scattering(c, s)) return st;
  }
  int64_t ns = 0;
  const bool uniformPath = c.uniform && !c.tune.forceAmr;
  int st = uniformPath ? diffuse_uniform(c, nAngularLevel, uvb, dirs, dJ, s, &ns)
                       : diffuse_amr(c, nAngularLevel, uvb, dirs, dJ, s, &ns);
  if (st) return st;
  RTB_CUDA(cudaEventRecord(c.evStop, s));
  if (nseg) *nseg = ns;
  // 72 B per leaf and direction (SURVEY.md 8d), 96 B with the emission coefficients of the 3 groups
  c.lastAlgBytes = bytes0 + (c.sweepEta() ? 96.0 : 72.0) * (double)c.nleaf * (double)dirs.size();
  c.lastLaunches += launches0;
  c.lastSweepLaunches += sweepLaunches0;
  c.statsPending = true;
  c.sweepTimed = uniformPath && !dirs.empty();
  return RTB200_OK;
}

void reset_call_results(Context& c) {
  c.lastScatIter = 0;
  c.lastScatResid = 0.;
  c.dScatResid = nullptr;
  c.lastNgCount = 0;
  c.lastWarm = false;
  c.ngPending = false;
  c.dWarmTaken = nullptr;
  c.heatValid = false;
}

int run_diffuse(Context& c, int nAngularLevel, const double* uvb, const double* beta, const int32_t* rays,
                int32_t nrays, double* dJ, cudaStream_t s, int64_t* nseg) {
  reset_call_results(c);
  int st = RTB200_OK;
  if (!c.scatterSigma()) {
    st = run_sweep(c, nAngularLevel, uvb, beta, rays, nrays, dJ, s, nseg, 0);
  } else if (rays) {   // the J of a direction subset is not the mean intensity the source needs
    c.scatWarm = false;
    return RTB200_ERR_ARG;
  } else {
    st = scatter_solve(c, nAngularLevel, uvb, beta, dJ, s, nseg);
  }
  if (st || !c.dHeat) return st;
  return launch_heating(c, 0, c.nleaf, dJ, c.nleaf, s);
}

// number of entries that are negative, NaN or Inf (the emission check of rtb200_grid_set_emission_device)
__global__ void count_bad_kernel(const double* __restrict__ x, int64_t n, int32_t* bad) {
  int32_t mine = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (!finite_nonneg(x[i])) mine++;
  }
  if (mine) atomicAdd(bad, mine);
}

static bool host_eta_ok(const double* eta, int64_t n) {
  for (int64_t i = 0; i < n; i++)
    if (!finite_nonneg(eta[i])) return false;
  return true;
}

void drop_sweep_plans(Context& c) {
  c.uniPlanKey.clear();
  if (c.graphExec) { cudaGraphExecDestroy(c.graphExec); c.graphExec = nullptr; }
}

int replace_leaf_field(Context& c, double** field, const double* src, bool device, cudaStream_t s) {
  const int64_t n = 3 * c.nleaf;
  const size_t bytes = (size_t)n * sizeof(double);
  if (!device && !host_eta_ok(src, n)) return RTB200_ERR_ARG;
  // the new array goes to a buffer of its own first: a refused array leaves the previous one in place
  double* fresh = nullptr;
  cudaError_t e = cudaMalloc((void**)&fresh, bytes);
  if (e != cudaSuccess) { set_cuda_error("cudaMalloc", e, __FILE__, __LINE__); return e == cudaErrorMemoryAllocation ? RTB200_ERR_NOMEM : RTB200_ERR_CUDA; }
  int st = RTB200_OK;
  if (!device) {
    if (cudaMemcpyAsync(fresh, src, bytes, cudaMemcpyHostToDevice, c.stream) != cudaSuccess ||
        cudaStreamSynchronize(c.stream) != cudaSuccess)
      st = RTB200_ERR_CUDA;
  } else {
    int32_t* dBad = c.dErr + 12;  // scratch word of the 64-byte error block (chemistry uses words 8..11)
    int32_t bad = 0;
    const int blocks = (int)std::min<int64_t>((n + 255) / 256, (int64_t)c.smCount * 8);
    if (cudaMemcpyAsync(fresh, src, bytes, cudaMemcpyDeviceToDevice, s) != cudaSuccess ||
        cudaMemsetAsync(dBad, 0, sizeof(int32_t), s) != cudaSuccess)
      st = RTB200_ERR_CUDA;
    if (!st) {
      count_bad_kernel<<<blocks, 256, 0, s>>>(fresh, n, dBad);
      if (cudaGetLastError() != cudaSuccess || cudaMemcpyAsync(&bad, dBad, sizeof(int32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
          cudaStreamSynchronize(s) != cudaSuccess)
        st = RTB200_ERR_CUDA;
    }
    if (!st && bad) st = RTB200_ERR_ARG;
  }
  if (st) { cudaFree(fresh); return st; }
  cudaFree(*field);
  *field = fresh;
  return RTB200_OK;
}

int set_emission(Context& c, const double* eta, bool device, cudaStream_t s) {
  if (c.nleaf == 0) return RTB200_ERR_ARG;
  RTB_CUDA(cudaSetDevice(c.device));
  // queued sweeps read the current array (as rtb200_grid_update_species)
  RTB_CUDA(cudaDeviceSynchronize());
  if (!eta) {
    cudaFree(c.dEta); c.dEta = nullptr;
    cudaFree(c.dEtaT); c.dEtaT = nullptr; c.etaTBytes = 0;
    drop_sweep_plans(c);   // the sweeps' plans and graphs know whether emission is set
    return RTB200_OK;
  }
  const bool had = c.dEta != nullptr;
  if (int st = replace_leaf_field(c, &c.dEta, eta, device, s)) return st;
  if (!had) drop_sweep_plans(c);
  else if (c.graphExec) { cudaGraphExecDestroy(c.graphExec); c.graphExec = nullptr; }   // the graph holds the pointer
  return RTB200_OK;
}

int context_init(Context& c, int device) {
  c.device = device;
  RTB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  RTB_CUDA(cudaGetDeviceProperties(&prop, device));
  c.smCount = prop.multiProcessorCount;
  c.l2Bytes = (size_t)prop.l2CacheSize;
  if (c.l2Bytes) c.tune.l2BudgetMB = 0.75 * (double)c.l2Bytes / 1048576.0;
  RTB_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
  RTB_CUDA(cudaEventCreate(&c.evStart));
  RTB_CUDA(cudaEventCreate(&c.evStop));
  RTB_CUDA(cudaEventCreate(&c.evSweep0));
  RTB_CUDA(cudaEventCreate(&c.evSweep1));
  RTB_CUDA(cudaMalloc((void**)&c.dErr, 64));
  RTB_CUDA(cudaMemset(c.dErr, 0, 64));
  if (const char* v = getenv("RTB200_SLOTS")) c.tune.slots = atoi(v);
  if (const char* v = getenv("RTB200_GRAPH")) c.tune.useGraph = atoi(v);
  if (const char* v = getenv("RTB200_L2_MB")) c.tune.l2BudgetMB = atof(v);
  return RTB200_OK;
}

void context_destroy(Context& c) {
  cudaSetDevice(c.device);
  cudaDeviceSynchronize();
  free_grid(c);
  cudaFree(c.dChemK);
  cudaFree(c.dMassPart);
  cudaFree(c.dAcc); cudaFree(c.dPlanes); cudaFree(c.dAmrScratch); cudaFree(c.dErr);
  if (c.hPinned) cudaFreeHost(c.hPinned);
  if (c.evStart) cudaEventDestroy(c.evStart);
  if (c.evStop) cudaEventDestroy(c.evStop);
  if (c.evSweep0) cudaEventDestroy(c.evSweep0);
  if (c.evSweep1) cudaEventDestroy(c.evSweep1);
  if (c.stream) cudaStreamDestroy(c.stream);
  c = Context();
}

int device_error(Context& c) {  // status raised by device-side guards of asynchronous calls; clears it
  int32_t err = 0;
  RTB_CUDA(cudaSetDevice(c.device));
  RTB_CUDA(cudaMemcpy(&err, c.dErr, sizeof(err), cudaMemcpyDeviceToHost));
  if (err) cudaMemset(c.dErr, 0, 64);
  return err;
}

int set_math(Context& c, int mode) {
  if (c.mathMode != mode && c.graphExec) { cudaGraphExecDestroy(c.graphExec); c.graphExec = nullptr; }
  c.mathMode = mode;
  return RTB200_OK;
}

int set_tuning(Context& c, const char* key, double value) {
  std::string k(key);
  if (k == "amr_batch") c.tune.amrBatch = (int)value;
  else if (k == "force_amr") c.tune.forceAmr = (int)value;
  else if (k == "amr_slots") c.tune.amrSlots = (int)value;
  else if (k == "amr_thin") c.tune.amrThin = (int)value;
  else if (k == "amr_stream") c.tune.amrStream = (int)value;
  else if (k == "amr_order") c.tune.amrOrder = (int)value;
  else if (k == "amr_min_blocks") c.tune.amrMinBlocks = (int)value;
  else if (k == "slots") c.tune.slots = (int)value;
  else if (k == "graph") c.tune.useGraph = (int)value;
  else if (k == "l2_mb") c.tune.l2BudgetMB = value;
  else if (k == "transpose_z") c.tune.transposeZ = (int)value;
  else if (k == "cells") c.tune.cells = (int)value;
  else if (k == "block_warps") c.tune.blockWarps = (int)value;
  else if (k == "pdl") c.tune.pdl = (int)value;
  else if (k == "dirs_per_task") c.tune.dirsPerTask = (int)value;
  else if (k == "portable_math") c.tune.portableMath = (int)value;
  else if (k == "point_batch") c.tune.pointBatch = (int)value;
  else if (k == "point_min_blocks") c.tune.pointMinBlocks = (int)value;
  else if (k == "point_refill") c.tune.pointRefill = (int)value;
  else if (k == "point_deposit") c.tune.pointDeposit = (int)value;
  else if (k == "point_record_cap") c.tune.pointRecordCap = (long long)value;
  else return RTB200_ERR_ARG;
  c.uniPlanKey.clear();
  if (c.graphExec) { cudaGraphExecDestroy(c.graphExec); c.graphExec = nullptr; }
  return RTB200_OK;
}

int grid_set(Context& c, int nx, int64_t nleaf, const int8_t* level, const double* HI, const double* HeI,
             const double* HeII, const double* rho, const double* abun2, double physicalBoxSize) {
  RTB_CUDA(cudaSetDevice(c.device));
  RTB_CUDA(cudaDeviceSynchronize());
  free_grid(c);
  c.nx = nx; c.nleaf = nleaf; c.boxSize = physicalBoxSize;
  c.hLevel.assign(level, level + nleaf);
  c.uniform = true;
  for (int64_t i = 0; i < nleaf; i++)
    if (level[i] != 0) { c.uniform = false; break; }
  if (c.uniform && nleaf != (int64_t)nx * nx * nx) { c.nleaf = 0; return RTB200_ERR_LEVELS; }
  if (int st = build_tree(c, level)) { c.nleaf = 0; return st; }
  cudaStream_t s = c.stream;
  const size_t nb = (size_t)nleaf * sizeof(double), pad = (size_t)c.padLeaves * sizeof(double);
  int st = upload((void**)&c.dLevel, level, (size_t)nleaf, 0, s);
  if (!st) st = upload((void**)&c.dHI, HI, nb, pad, s);
  if (!st) st = upload((void**)&c.dHeI, HeI, nb, pad, s);
  if (!st) st = upload((void**)&c.dHeII, HeII, nb, pad, s);
  // rho / abun2 are optional (diffuse-only use): without them the point-source and chemistry entry points return
  // RTB200_ERR_ARG instead of working on zero-filled arrays
  if (!st && rho) st = upload((void**)&c.dRho, rho, nb, 0, s);
  if (!st && abun2) st = upload((void**)&c.dAbun2, abun2, nb, 0, s);
  if (!st) st = upload((void**)&c.dKappa, nullptr, 3 * nb, 0, s);
  if (!st) st = upload((void**)&c.dJ, nullptr, 3 * nb, 0, s);
  if (!st) {
    st = upload((void**)&c.tree.child, c.hChild.data(), c.hChild.size() * sizeof(int32_t), 0, s);
    if (!st) st = upload((void**)&c.tree.leafX, c.hLeafX.data(), (size_t)nleaf * sizeof(int32_t), 0, s);
    if (!st) st = upload((void**)&c.tree.leafY, c.hLeafY.data(), (size_t)nleaf * sizeof(int32_t), 0, s);
    if (!st) st = upload((void**)&c.tree.leafZ, c.hLeafZ.data(), (size_t)nleaf * sizeof(int32_t), 0, s);
  }
  if (st) { free_grid(c); c.nleaf = 0; return st; }
  RTB_CUDA(cudaStreamSynchronize(s));
  return RTB200_OK;
}

PointInputs make_point_inputs(int nWave, const double* wavelength, const double* lum, const double* metallicity,
                              double coefSpectrum, const double* aDust, int dust, int maxPixelLevel, int nsrc,
                              const int32_t* srcLeaf, const int32_t* srcWeight) {
  PointInputs in;
  in.nWave = nWave; in.wavelength = wavelength; in.lum = lum; in.metallicity = metallicity;
  in.coefSpectrum = coefSpectrum; in.aDust = aDust; in.dust = dust; in.maxPixelLevel = maxPixelLevel;
  in.nsrc = nsrc; in.srcLeaf = srcLeaf; in.srcWeight = srcWeight;
  return in;
}

void split_diag(const double* d, size_t n, const int* idx, double* rem, double* bnd, double* dust, double* spec,
                int32_t* hpl) {
  for (size_t i = 0; i < n; i++) {
    const double* p = d + i * 320;
    const size_t s = idx ? (size_t)idx[i] : i;
    if (rem) memcpy(rem + s * 7, p, 56);
    if (bnd) memcpy(bnd + s * 7, p + 7, 56);
    if (dust) dust[s] = p[14];
    if (spec) memcpy(spec + s * 300, p + 16, 2400);
    if (hpl) hpl[s] = (int32_t)p[15];
  }
}

}  // namespace rtb

using namespace rtb;

extern "C" {

int rtb200_version(void) { return RTB200_VERSION; }

const char* rtb200_status_string(int status) {
  switch (status) {
    case RTB200_OK: return "ok";
    case RTB200_ERR_PHI: return "error in phi (direction on a quadrant boundary)";
    case RTB200_ERR_THETA: return "error in theta";
    case RTB200_ERR_THETA_OR_PHI: return "error in theta or phi (tie between exit faces)";
    case RTB200_ERR_PATTERN_RANGE: return "Error: ray entry coordinate > 1";
    case RTB200_ERR_TOP_SELECTOR: return "error in xyTop/xzTop/yzTop";
    case RTB200_ERR_RAY_INACTIVE: return "Error: xzRay/yzRay should be active";
    case RTB200_ERR_INTENSITY_GUARD: return "intensity guard: |Iout1+Iout2+Iout3| >= 1e-20 in a refined cell";
    case RTB200_ERR_ANGLE_LARGE: return "angle too large";
    case RTB200_ERR_LEVELS: return "error in levels";
    case RTB200_ERR_CHECKPOINT: return "error in coordinates";
    case RTB200_ERR_IDEPTH: return "error in idepth123";
    case RTB200_ERR_ARG: return "bad argument";
    case RTB200_ERR_CUDA: return last_cuda_error()[0] ? last_cuda_error() : "CUDA error or no CUDA device (no CPU fallback)";
    case RTB200_ERR_NOMEM: return "out of device memory";
    case RTB200_ERR_CHEMISTRY: return "ionisation fraction outside [0,1]";
    default: return "unknown status";
  }
}

int rtb200_create(int device, rtb200_ctx** out) {
  if (!out) return RTB200_ERR_ARG;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_cuda_error("cudaGetDeviceCount", e == cudaSuccess ? cudaErrorNoDevice : e, __FILE__, __LINE__);
    return RTB200_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) return RTB200_ERR_ARG;
  rtb200_ctx* h = new (std::nothrow) rtb200_ctx();
  if (!h) return RTB200_ERR_NOMEM;
  if (int st = context_init(h->c, device)) {   // nothing of a half-built context survives
    context_destroy(h->c);
    delete h;
    return st;
  }
  *out = h;
  return RTB200_OK;
}

int rtb200_destroy(rtb200_ctx* h) {
  if (!h) return RTB200_OK;
  if (h->m) multi_destroy(h->m);
  else context_destroy(h->c);
  delete h;
  return RTB200_OK;
}

int rtb200_set_math(rtb200_ctx* h, int mode) {
  if (!h || (mode != RTB200_MATH_FAST && mode != RTB200_MATH_FAITHFUL)) return RTB200_ERR_ARG;
  if (h->m) return multi_set_math(h->m, mode);
  return set_math(h->c, mode);
}

int rtb200_set_tuning(rtb200_ctx* h, const char* key, double value) {
  if (!h || !key) return RTB200_ERR_ARG;
  if (h->m) return multi_set_tuning(h->m, key, value);
  return set_tuning(h->c, key, value);
}

int rtb200_grid_set(rtb200_ctx* h, int nx, int64_t nleaf, const int8_t* level, const double* HI, const double* HeI,
                    const double* HeII, const double* rho, const double* abun2, double physicalBoxSize) {
  if (!h || nx < 1 || nx > 4096 || !level || !HI || nleaf < (int64_t)nx * nx * nx || nleaf > (int64_t)INT32_MAX)
    return RTB200_ERR_ARG;
  if (h->m) return multi_grid_set(h->m, nx, nleaf, level, HI, HeI, HeII, rho, abun2, physicalBoxSize);
  return grid_set(h->c, nx, nleaf, level, HI, HeI, HeII, rho, abun2, physicalBoxSize);
}

int rtb200_grid_update_species(rtb200_ctx* h, const double* HI, const double* HeI, const double* HeII) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_update_species(h->m, HI, HeI, HeII);
  if (h->c.nleaf == 0) return RTB200_ERR_ARG;
  Context& c = h->c;
  RTB_CUDA(cudaSetDevice(c.device));
  // Work queued by the *_device entry points on the caller's streams (sweeps, chemistry, ray casting) reads and
  // writes the species arrays: it has to be complete before they are overwritten (as rtb200_grid_get_species does).
  RTB_CUDA(cudaDeviceSynchronize());
  const size_t nb = (size_t)c.nleaf * sizeof(double);
  if (HI) RTB_CUDA(cudaMemcpyAsync(c.dHI, HI, nb, cudaMemcpyHostToDevice, c.stream));
  if (HeI) RTB_CUDA(cudaMemcpyAsync(c.dHeI, HeI, nb, cudaMemcpyHostToDevice, c.stream));
  if (HeII) RTB_CUDA(cudaMemcpyAsync(c.dHeII, HeII, nb, cudaMemcpyHostToDevice, c.stream));
  RTB_CUDA(cudaStreamSynchronize(c.stream));
  return RTB200_OK;
}

int rtb200_grid_set_emission(rtb200_ctx* h, const double* eta) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_set_emission(h->m, eta);
  return set_emission(h->c, eta, false, h->c.stream);
}

int rtb200_grid_set_scattering(rtb200_ctx* h, const double* sigma, int32_t maxIterations, double tolerance) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_set_scattering(h->m, sigma, maxIterations, tolerance);
  return set_scattering(h->c, sigma, false, maxIterations, tolerance);
}

int rtb200_grid_set_dust(rtb200_ctx* h, int dustApproximation, const double* betaDust3, const double* albedo3,
                         int32_t maxIterations, double tolerance) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_set_dust(h->m, dustApproximation, betaDust3, albedo3, maxIterations, tolerance);
  return set_dust(h->c, dustApproximation, betaDust3, albedo3, maxIterations, tolerance);
}

int rtb200_last_scattering(rtb200_ctx* h, int32_t* iterations, double* residual) {
  if (!h) return RTB200_ERR_ARG;
  return last_scattering(h->m ? multi_primary(h->m) : h->c, iterations, residual);
}

int rtb200_grid_set_scattering_acceleration(rtb200_ctx* h, int32_t flags) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_set_scattering_acceleration(h->m, flags);
  return set_scattering_acceleration(h->c, flags);
}

int rtb200_grid_set_heating(rtb200_ctx* h, const double* gamma9, const double* width3) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_set_heating(h->m, gamma9, width3);
  return set_heating(h->c, gamma9, width3, h->c.nleaf);
}

int rtb200_last_heating(rtb200_ctx* h, double* heat5) {
  if (!h || !heat5) return RTB200_ERR_ARG;
  if (h->m) return multi_last_heating(h->m, heat5);
  Context& c = h->c;
  if (!c.dHeat || !c.heatValid) return RTB200_ERR_ARG;
  RTB_CUDA(cudaSetDevice(c.device));
  RTB_CUDA(cudaDeviceSynchronize());   // the pass of a *_device call runs on the caller's stream
  RTB_CUDA(cudaMemcpy(heat5, c.dHeat, (size_t)5 * c.nleaf * sizeof(double), cudaMemcpyDeviceToHost));
  return RTB200_OK;
}

int rtb200_heating_device(rtb200_ctx* h, int local, int64_t* offset, int64_t* count, int64_t* stride, double** H_device) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_heating_device(h->m, local, offset, count, stride, H_device);
  if (local != 0 || !h->c.dHeat) return RTB200_ERR_ARG;
  if (offset) *offset = 0;
  if (count) *count = h->c.nleaf;
  if (stride) *stride = h->c.heatStride;
  if (H_device) *H_device = h->c.dHeat;
  return RTB200_OK;
}

int rtb200_last_scattering_acceleration(rtb200_ctx* h, int32_t* extrapolations, int32_t* warmStarted) {
  if (!h) return RTB200_ERR_ARG;
  return last_scattering_acceleration(h->m ? multi_primary(h->m) : h->c, extrapolations, warmStarted);
}

int rtb200_grid_set_emission_device(rtb200_ctx* h, const double* eta_device, void* stream) {
  if (!h || h->m || !eta_device) return RTB200_ERR_ARG;   // a device group takes the host array (slab-wise)
  return set_emission(h->c, eta_device, true, (cudaStream_t)stream);
}

int rtb200_diffuse_device(rtb200_ctx* h, int nAngularLevel, const double* uvb, const double* beta, const int32_t* rays,
                          int32_t nrays, double* J_device, void* stream, int64_t* nseg) {
  if (!h || h->m) return RTB200_ERR_ARG;   // a device group leaves its results in slabs: rtb200_multi_diffuse_resident
  return run_diffuse(h->c, nAngularLevel, uvb, beta, rays, nrays, J_device, (cudaStream_t)stream, nseg);
}

int rtb200_diffuse(rtb200_ctx* h, int nAngularLevel, const double* uvb, const double* beta, const int32_t* rays,
                   int32_t nrays, double* J1, double* J2, double* J3, int64_t* nseg) {
  if (!h || !J1 || !J2 || !J3) return RTB200_ERR_ARG;
  if (h->m) return multi_diffuse_host(h->m, nAngularLevel, uvb, beta, rays, nrays, J1, J2, J3, nseg);
  Context& c = h->c;
  int st = run_diffuse(c, nAngularLevel, uvb, beta, rays, nrays, c.dJ, c.stream, nseg);
  if (st) return st;
  const size_t nb = (size_t)c.nleaf * sizeof(double);
  RTB_CUDA(cudaMemcpyAsync(J1, c.dJ, nb, cudaMemcpyDeviceToHost, c.stream));
  RTB_CUDA(cudaMemcpyAsync(J2, c.dJ + c.nleaf, nb, cudaMemcpyDeviceToHost, c.stream));
  RTB_CUDA(cudaMemcpyAsync(J3, c.dJ + 2 * c.nleaf, nb, cudaMemcpyDeviceToHost, c.stream));
  RTB_CUDA(cudaStreamSynchronize(c.stream));
  int32_t err = 0;
  RTB_CUDA(cudaMemcpy(&err, c.dErr, sizeof(err), cudaMemcpyDeviceToHost));
  if (err) {
    cudaMemset(c.dErr, 0, 64);
    c.scatWarm = false;   // a failed solve is no starting guess
    c.heatValid = false;
    return err;
  }
  return RTB200_OK;
}

int rtb200_diffuse_rates_device(rtb200_ctx* h, const double* J, const double* ksi24, const double* ksi25,
                                const double* ksi26, double* k24, double* k25, double* k26, void* stream) {
  if (!h || h->m || !J || !ksi24 || !ksi25 || !ksi26 || !k24 || !k25 || !k26 || h->c.nleaf == 0) return RTB200_ERR_ARG;
  RTB_CUDA(cudaSetDevice(h->c.device));
  return launch_diffuse_rates(h->c, J, ksi24, ksi25, ksi26, k24, k25, k26, (cudaStream_t)stream);
}

int rtb200_point_device(rtb200_ctx* h, int nWave, const double* wavelength, const double* lum, const double* metallicity,
                        double coefSpectrum, const double* aDust, int dustApproximation, int maxPixelLevel, int32_t nsrc,
                        const int32_t* srcLeaf, const int32_t* srcWeight, double* rates_device, void* stream,
                        double* ndotRemaining, double* ndotBoundary, double* ndotDust, double* ndotSpectrum,
                        int32_t* highestPixelLevel, int64_t* nseg) {
  if (!h || h->m || !rates_device) return RTB200_ERR_ARG;
  PointInputs in = make_point_inputs(nWave, wavelength, lum, metallicity, coefSpectrum, aDust, dustApproximation,
                                     maxPixelLevel, nsrc, srcLeaf, srcWeight);
  const bool wantDiag = ndotRemaining || ndotBoundary || ndotDust || ndotSpectrum || highestPixelLevel;
  std::vector<double> diag(wantDiag ? (size_t)std::max(nsrc, 0) * 320 : 0);
  int st = point_solve(h->c, in, rates_device, wantDiag ? diag.data() : nullptr, nseg, nullptr, 0, nullptr, nullptr,
                       (cudaStream_t)stream);
  if (st) return st;
  if (wantDiag)
    split_diag(diag.data(), (size_t)std::max(nsrc, 0), nullptr, ndotRemaining, ndotBoundary, ndotDust, ndotSpectrum,
               highestPixelLevel);
  return RTB200_OK;
}

static int point_host_call(Context& c, const PointInputs& in, double* const k[6], double* rem, double* bnd, double* dust,
                           double* spec, int32_t* hpl, int64_t* nseg, long long* trace, long long traceCap,
                           long long* traceLen) {
  for (int i = 0; i < 6; i++)
    if (!k[i]) return RTB200_ERR_ARG;
  if (c.nleaf == 0) return RTB200_ERR_ARG;
  RTB_CUDA(cudaSetDevice(c.device));
  const size_t nb = (size_t)c.nleaf * sizeof(double);
  if (!c.dRates) RTB_CUDA(cudaMalloc((void**)&c.dRates, 6 * nb));
  for (int i = 0; i < 6; i++) RTB_CUDA(cudaMemcpyAsync(c.dRates + (size_t)i * c.nleaf, k[i], nb, cudaMemcpyHostToDevice, c.stream));
  std::vector<double> diag((size_t)std::max(in.nsrc, 0) * 320);
  int st = point_solve(c, in, c.dRates, diag.data(), nseg, trace, traceCap, traceLen, nullptr, c.stream);
  if (st) return st;
  for (int i = 0; i < 6; i++) RTB_CUDA(cudaMemcpyAsync(k[i], c.dRates + (size_t)i * c.nleaf, nb, cudaMemcpyDeviceToHost, c.stream));
  RTB_CUDA(cudaStreamSynchronize(c.stream));
  split_diag(diag.data(), (size_t)std::max(in.nsrc, 0), nullptr, rem, bnd, dust, spec, hpl);
  return RTB200_OK;
}

int rtb200_point(rtb200_ctx* h, int nWave, const double* wavelength, const double* lum, const double* metallicity,
                 double coefSpectrum, const double* aDust, int dustApproximation, int maxPixelLevel, int32_t nsrc,
                 const int32_t* srcLeaf, const int32_t* srcWeight, double* krate24, double* krate25, double* krate26,
                 double* crate24, double* crate25, double* crate26, double* ndotRemaining, double* ndotBoundary,
                 double* ndotDust, double* ndotSpectrum, int32_t* highestPixelLevel, int64_t* nseg) {
  if (!h) return RTB200_ERR_ARG;
  PointInputs in = make_point_inputs(nWave, wavelength, lum, metallicity, coefSpectrum, aDust, dustApproximation,
                                     maxPixelLevel, nsrc, srcLeaf, srcWeight);
  double* k[6] = {krate24, krate25, krate26, crate24, crate25, crate26};
  if (h->m)
    return multi_point_host(h->m, in, k, ndotRemaining, ndotBoundary, ndotDust, ndotSpectrum, highestPixelLevel, nseg);
  return point_host_call(h->c, in, k, ndotRemaining, ndotBoundary, ndotDust, ndotSpectrum, highestPixelLevel, nseg,
                         nullptr, 0, nullptr);
}

int rtb200_point_trace(rtb200_ctx* h, int nWave, const double* wavelength, const double* lum, const double* metallicity,
                       double coefSpectrum, const double* aDust, int dustApproximation, int maxPixelLevel, int32_t nsrc,
                       const int32_t* srcLeaf, const int32_t* srcWeight, double* rates6, int64_t* nseg, int64_t* trace,
                       int64_t traceCap, int64_t* traceLen) {
  if (!h || h->m || !rates6 || !trace || traceCap <= 0 || !traceLen) return RTB200_ERR_ARG;
  PointInputs in = make_point_inputs(nWave, wavelength, lum, metallicity, coefSpectrum, aDust, dustApproximation,
                                     maxPixelLevel, nsrc, srcLeaf, srcWeight);
  double* k[6];
  for (int i = 0; i < 6; i++) k[i] = rates6 + (size_t)i * h->c.nleaf;
  long long tl = 0;
  int st = point_host_call(h->c, in, k, nullptr, nullptr, nullptr, nullptr, nullptr, nseg, (long long*)trace, traceCap, &tl);
  *traceLen = tl;
  return st;
}

int rtb200_point_tables(rtb200_ctx* h, int nWave, const double* wavelength, const double* lum, const double* metallicity,
                        double coefSpectrum, const double* aDust, int iMetal, double coefMetal, double* tables) {
  if (!h || !tables || iMetal < 1 || iMetal > 4) return RTB200_ERR_ARG;
  Context& c = h->m ? multi_primary(h->m) : h->c;
  if (c.nleaf == 0) return RTB200_ERR_ARG;
  const int32_t leaf = 0, weight = 0;  // a source of weight 0 casts no rays: only its tables are built
  PointInputs in = make_point_inputs(nWave, wavelength, lum, metallicity, coefSpectrum, aDust, 1, 1, 1, &leaf, &weight);
  in.forceMetal = iMetal; in.forceCoefMetal = coefMetal;
  RTB_CUDA(cudaSetDevice(c.device));
  const size_t nb = (size_t)c.nleaf * sizeof(double);
  if (!c.dRates) RTB_CUDA(cudaMalloc((void**)&c.dRates, 6 * nb));
  return point_solve(c, in, c.dRates, nullptr, nullptr, nullptr, 0, nullptr, tables, c.stream);
}

int rtb200_chemistry_tables(rtb200_ctx* h, int nratec, double logtem0, double logtem9, double dlogtem, const double* k1a,
                            const double* k2a, const double* k3a, const double* k4a, const double* k5a,
                            const double* k6a) {
  if (!h) return RTB200_ERR_ARG;
  const double* k[6] = {k1a, k2a, k3a, k4a, k5a, k6a};
  if (h->m) return multi_chemistry_tables(h->m, nratec, logtem0, logtem9, dlogtem, k);
  return chemistry_set_tables(h->c, nratec, logtem0, logtem9, dlogtem, k);
}

int rtb200_chemistry_temperature(rtb200_ctx* h, const double* tgas) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_chemistry_temperature(h->m, tgas);
  return chemistry_set_temperature(h->c, tgas);
}

int rtb200_chemistry_device(rtb200_ctx* h, const double* rates_device, const double* J_device, const double* ksi,
                            const double* uniform, double* maxChange, void* stream) {
  if (!h || h->m) return RTB200_ERR_ARG;
  return chemistry_run(h->c, rates_device, J_device, ksi, uniform, maxChange, (cudaStream_t)stream);
}

int rtb200_compute_mass(rtb200_ctx* h, double* neutralHydrogenMass, double* totalHydrogenMass, void* stream) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) {  // a device group holds the same species on every device after each step: any member can do the sum
    if (int st = rtb200_multi_sync(h)) return st;
    Context& c = multi_primary(h->m);
    return compute_mass(c, neutralHydrogenMass, totalHydrogenMass, c.stream);
  }
  return compute_mass(h->c, neutralHydrogenMass, totalHydrogenMass, (cudaStream_t)stream);
}

int rtb200_grid_get_species(rtb200_ctx* h, double* HI, double* HeI, double* HeII) {
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_get_species(h->m, HI, HeI, HeII);
  if (h->c.nleaf == 0) return RTB200_ERR_ARG;
  Context& c = h->c;
  RTB_CUDA(cudaSetDevice(c.device));
  RTB_CUDA(cudaDeviceSynchronize());
  const size_t nb = (size_t)c.nleaf * sizeof(double);
  if (HI) RTB_CUDA(cudaMemcpy(HI, c.dHI, nb, cudaMemcpyDeviceToHost));
  if (HeI) RTB_CUDA(cudaMemcpy(HeI, c.dHeI, nb, cudaMemcpyDeviceToHost));
  if (HeII) RTB_CUDA(cudaMemcpy(HeII, c.dHeII, nb, cudaMemcpyDeviceToHost));
  return RTB200_OK;
}

int rtb200_device_error(rtb200_ctx* h) {  // status raised by device-side guards of asynchronous calls
  if (!h) return RTB200_ERR_ARG;
  if (h->m) return multi_device_error(h->m);
  return device_error(h->c);
}

int rtb200_direction(int nAngularLevel, int64_t iray, int32_t* izone, double* phi, double* theta) {
  if (!izone || !phi || !theta || nAngularLevel < 1) return RTB200_ERR_ARG;
  Direction d = classify_direction(nAngularLevel, iray);
  *izone = d.izone; *phi = d.phi; *theta = d.theta;
  return d.status;
}

int rtb200_patterns(int nAngularLevel, int64_t iray, int nx, double* out) {
  if (!out || nx < 1) return RTB200_ERR_ARG;
  Direction d = classify_direction(nAngularLevel, iray);
  if (d.status) return d.status;
  std::vector<RayPattern> pat;
  layer_patterns_level0(d.phi, d.theta, nx, pat);
  for (int i = 0; i < nx; i++) {
    const RayPattern& p = pat[i];
    if (p.status) return p.status;
    double* o = out + 12 * i;
    o[0] = p.xy_x0; o[1] = p.xy_y0; o[2] = p.xy_len;
    o[3] = p.xzActive ? p.xz_x0 : 0.; o[4] = p.xzActive ? p.xz_z0 : 0.; o[5] = p.xzActive ? p.xz_len : 0.;
    o[6] = p.yzActive ? p.yz_y0 : 0.; o[7] = p.yzActive ? p.yz_z0 : 0.; o[8] = p.yzActive ? p.yz_len : 0.;
    o[9] = p.xyTop; o[10] = p.xzTop; o[11] = p.yzTop;
  }
  return RTB200_OK;
}

int rtb200_neighbours(rtb200_ctx* h, int nAngularLevel, int64_t iray, int32_t* nb) {
  if (!h || !nb) return RTB200_ERR_ARG;
  Context& c = h->m ? multi_primary(h->m) : h->c;
  if (c.nleaf == 0) return RTB200_ERR_ARG;
  Direction d = classify_direction(nAngularLevel, iray);
  if (d.status) return d.status;
  RTB_CUDA(cudaSetDevice(c.device));
  return amr_neighbours(c, d, nb);
}

int rtb200_debug_waves(rtb200_ctx* h, int nAngularLevel, int64_t iray, int32_t* waveOfLeaf, int32_t* nwaves) {
  if (!h || !waveOfLeaf) return RTB200_ERR_ARG;
  Context& c = h->m ? multi_primary(h->m) : h->c;
  if (c.nleaf == 0) return RTB200_ERR_ARG;
  Direction d = classify_direction(nAngularLevel, iray);
  if (d.status) return d.status;
  RTB_CUDA(cudaSetDevice(c.device));
  return amr_waves(c, d, waveOfLeaf, nwaves);
}

int rtb200_debug_portable_math(rtb200_ctx* h, int64_t n, const double* x, double* expOut, double* logOut) {
  if (!h || n < 0 || !x || !expOut || !logOut) return RTB200_ERR_ARG;
  if (n == 0) return RTB200_OK;
  Context& c = h->m ? multi_primary(h->m) : h->c;
  RTB_CUDA(cudaSetDevice(c.device));
  double* d = nullptr;
  RTB_CUDA(cudaMalloc((void**)&d, (size_t)3 * n * sizeof(double)));
  cudaError_t e = cudaMemcpyAsync(d, x, (size_t)n * 8, cudaMemcpyHostToDevice, c.stream);
  if (e == cudaSuccess) {
    portable_math_kernel<<<(int)std::min<int64_t>((n + 255) / 256, 4096), 256, 0, c.stream>>>(d, n, d + n, d + 2 * n);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(expOut, d + n, (size_t)n * 8, cudaMemcpyDeviceToHost, c.stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(logOut, d + 2 * n, (size_t)n * 8, cudaMemcpyDeviceToHost, c.stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
  cudaFree(d);
  RTB_CUDA(e);
  return RTB200_OK;
}

int rtb200_debug_fast_exp(rtb200_ctx* h, int64_t n, const double* tau, double* expOut, double* oneMinusOut) {
  if (!h || n < 0 || !tau || !expOut || !oneMinusOut) return RTB200_ERR_ARG;
  if (n == 0) return RTB200_OK;
  Context& c = h->m ? multi_primary(h->m) : h->c;
  RTB_CUDA(cudaSetDevice(c.device));
  double* d = nullptr;
  RTB_CUDA(cudaMalloc((void**)&d, (size_t)3 * n * sizeof(double)));
  cudaError_t e = cudaMemcpyAsync(d, tau, (size_t)n * 8, cudaMemcpyHostToDevice, c.stream);
  if (e == cudaSuccess) {
    fast_exp_kernel<<<(int)std::min<int64_t>((n + 255) / 256, 4096), 256, 0, c.stream>>>(d, n, d + n, d + 2 * n);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(expOut, d + n, (size_t)n * 8, cudaMemcpyDeviceToHost, c.stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(oneMinusOut, d + 2 * n, (size_t)n * 8, cudaMemcpyDeviceToHost, c.stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
  cudaFree(d);
  RTB_CUDA(e);
  return RTB200_OK;
}

int rtb200_last_stats(rtb200_ctx* h, double* ms, double* sweepMs, int64_t* launches, int64_t* sweepLaunches,
                      double* algBytes) {
  if (!h) return RTB200_ERR_ARG;
  Context& c = h->m ? multi_primary(h->m) : h->c;
  if (c.statsPending) {
    RTB_CUDA(cudaSetDevice(c.device));
    RTB_CUDA(cudaEventSynchronize(c.evStop));
    float f = 0;
    RTB_CUDA(cudaEventElapsedTime(&f, c.evStart, c.evStop));
    c.lastMs = f;
    c.lastSweepMs = 0;
    if (c.sweepTimed) {
      RTB_CUDA(cudaEventElapsedTime(&f, c.evSweep0, c.evSweep1));
      c.lastSweepMs = f;
    }
    c.statsPending = false;
  }
  if (ms) *ms = c.lastMs;
  if (sweepMs) *sweepMs = c.lastSweepMs;
  if (sweepLaunches) *sweepLaunches = c.lastSweepLaunches;
  if (launches) *launches = c.lastLaunches;
  if (algBytes) *algBytes = c.lastAlgBytes;
  return RTB200_OK;
}

}  // extern "C"
