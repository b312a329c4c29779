// Isotropic, coherent scattering of the diffuse field by source iteration (DESIGN.md 4.7).
//
// Per leaf and group a scattering coefficient sigma >= 0 (1/cm) joins the extinction, kappa_ext = kappa_abs + sigma,
// and the source: iteration k sweeps with eta_k = eta_th + sigma * J_{k-1} (J_0 = 0), where J is the full Jmean of the
// previous sweep.  The sweeps read one fixed effective-source buffer (Context::dEtaEff), so that the uniform plan and
// its captured graph, the z-major eta copy and the nested grid's opacity records need nothing new: scattering runs the
// EMIT instantiations of the existing sweep kernels.  Between two sweeps one streaming pass (scatter_source_kernel)
// writes the next source, keeps J for the next residual and folds r_k = max |J_k - J_{k-1}| / J_k into a device word.
#include <algorithm>
#include <cmath>
#include <vector>

#include "rtb200_internal.h"

namespace rtb {

// kappa_ext = kappa_abs + sigma, the sum rounded once (the oracle adds sigma last, in the same order)
__global__ void add_scattering_kernel(double* __restrict__ kappa, const double* __restrict__ sigma, int64_t n) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    kappa[i] = __dadd_rn(kappa[i], sigma[i]);
}

// One pass of the source iteration over cnt leaves of the 3 groups:
//   etaOut = eta_th + sigma * J  (two roundings, no FMA, so that numpy repeats it bit for bit)
//   r      = 0 if J == Jprev, +inf if J == 0 != Jprev, else |J - Jprev| / J;  *resid = max(*resid, r)
//   Jprev  = J
// A max is exact, so the residual does not depend on the order of the blocks.  For doubles >= 0 (+inf included) the
// bit pattern orders as the value, which lets atomicMax on the 64-bit word do the fold.
__global__ void scatter_source_kernel(int64_t cnt, const double* __restrict__ J, double* __restrict__ Jprev,
                                      int64_t jStride, const double* __restrict__ sigma, const double* __restrict__ etaTh,
                                      int64_t sStride, double* __restrict__ etaOut, int64_t oStride,
                                      unsigned long long* __restrict__ resid) {
  double r = 0.;
  const int64_t total = 3 * cnt;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = t / cnt, i = t - g * cnt;
    const double j = J[g * jStride + i], jp = Jprev[g * jStride + i];
    const double th = etaTh ? etaTh[g * sStride + i] : 0.;
    etaOut[g * oStride + i] = __dadd_rn(th, __dmul_rn(sigma[g * sStride + i], j));
    Jprev[g * jStride + i] = j;
    const double rk = j == jp ? 0. : (j == 0. ? __longlong_as_double(0x7ff0000000000000LL) : __ddiv_rn(fabs(__dsub_rn(j, jp)), j));
    r = fmax(r, rk);
  }
  unsigned long long b = (unsigned long long)__double_as_longlong(r);
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long v = __shfl_xor_sync(0xffffffffu, b, o);
    b = v > b ? v : b;
  }
  __shared__ unsigned long long warpMax[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) warpMax[warp] = b;
  __syncthreads();
  if (warp == 0) {
    b = lane < (int)(blockDim.x >> 5) ? warpMax[lane] : 0ull;
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long v = __shfl_xor_sync(0xffffffffu, b, o);
      b = v > b ? v : b;
    }
    if (lane == 0 && b) atomicMax(resid, b);
  }
}

int launch_add_scattering(Context& c, cudaStream_t s) {
  const int64_t n = 3 * c.nleaf;
  const int blocks = (int)std::min<int64_t>((n + 255) / 256, (int64_t)c.smCount * 16);
  add_scattering_kernel<<<blocks, 256, 0, s>>>(c.dKappa, c.dSigma, n);
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

int launch_scatter_source(const Context& c, int64_t cnt, const double* J, double* Jprev, int64_t jStride, const double* sigma,
                          const double* etaTh, int64_t sStride, double* etaOut, int64_t oStride, unsigned long long* resid,
                          cudaStream_t s) {
  if (cnt <= 0) return RTB200_OK;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((3 * cnt + 255) / 256, (int64_t)c.smCount * 16));
  scatter_source_kernel<<<blocks, 256, 0, s>>>(cnt, J, Jprev, jStride, sigma, etaTh, sStride, etaOut, oStride, resid);
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

void release_source_iteration(Context& c) {
  last_scattering(c, nullptr, nullptr);   // their words live in the scratch
  last_scattering_acceleration(c, nullptr, nullptr);
  c.dScatResid = nullptr;
  c.dWarmTaken = nullptr;
  c.scatWarm = false;
  free_history(c);
  cudaFree(c.dEtaEff); c.dEtaEff = nullptr;
  cudaFree(c.dScatScratch); c.dScatScratch = nullptr; c.scatScratchBytes = 0;
}

int set_scattering(Context& c, const double* sigma, bool device, int32_t maxIterations, double tolerance) {
  if (c.nleaf == 0) return RTB200_ERR_ARG;
  if (sigma && (maxIterations < 1 || !(tolerance >= 0.) || std::isinf(tolerance))) return RTB200_ERR_ARG;
  if (sigma && c.dDustSigma) return RTB200_ERR_ARG;   // one scattering medium at a time (dust.cu)
  RTB_CUDA(cudaSetDevice(c.device));
  RTB_CUDA(cudaDeviceSynchronize());   // queued sweeps read the current arrays
  if (!sigma) {
    cudaFree(c.dSigma); c.dSigma = nullptr;
    if (!c.dDustSigma) release_source_iteration(c);   // scattering dust keeps the buffers of its source iteration
    drop_sweep_plans(c);
    return RTB200_OK;
  }
  if (!c.dEtaEff) {
    cudaError_t e = cudaMalloc((void**)&c.dEtaEff, (size_t)3 * c.nleaf * sizeof(double));
    if (e != cudaSuccess) {
      c.dEtaEff = nullptr;
      set_cuda_error("cudaMalloc", e, __FILE__, __LINE__);
      return e == cudaErrorMemoryAllocation ? RTB200_ERR_NOMEM : RTB200_ERR_CUDA;
    }
  }
  const bool had = c.dSigma != nullptr;
  if (int st = replace_leaf_field(c, &c.dSigma, sigma, device, c.stream)) {
    if (!had) { cudaFree(c.dEtaEff); c.dEtaEff = nullptr; }
    return st;
  }
  c.scatMaxIter = maxIterations;
  c.scatTol = tolerance;
  drop_sweep_plans(c);   // the sweeps now read dEtaEff
  return RTB200_OK;
}

int last_scattering(Context& c, int32_t* iterations, double* residual) {
  if (c.dScatResid) {
    RTB_CUDA(cudaSetDevice(c.device));
    RTB_CUDA(cudaEventSynchronize(c.evStop));
    std::vector<double> w((size_t)c.nScatResid);
    RTB_CUDA(cudaMemcpy(w.data(), c.dScatResid, w.size() * sizeof(double), cudaMemcpyDeviceToHost));
    c.lastScatResid = *std::max_element(w.begin(), w.end());
    c.dScatResid = nullptr;
  }
  if (iterations) *iterations = c.lastScatIter;
  if (residual) *residual = c.lastScatResid;
  return RTB200_OK;
}

// The source iteration, iterations k = 1, 2, ... of a single context or of one member of a device group
// (p.stageStride > 0).  With the acceleration flags (ng.cu) the warm start takes x_0 from Jprev, which holds the J the
// previous completed solve returned, and Ng extrapolates after every fourth sweep of a cycle; the plain source pass runs
// after every sweep.
//
// Single context, J = the output [3][N], the source pass writes dEtaEff:
//   prologue     warm: [dust opacities] -> source pass from Jprev (J, overwritten by the first sweep, takes its copy of
//                x_0); cold: clear Jprev -> copy (or clear) eta_th into dEtaEff
//   iteration k  sweep -> [Ng, cycle >= 2: Jprev -> hist[cycle - 2]] -> clear the residual word -> source pass ->
//                [tolerance > 0: residual to the host, sync, test] -> [extrapolate: Ng sums, solve + combine]
// Member of a device group, J = its slab Jslab [3][slab], the source pass writes its slice of the stage [3][npad]:
//   prologue     warm flag set: every rank's holding of a stored J to the device and all-gathered -> warm_start_agree
//                (Jprev cleared unless every rank holds one) -> [dust opacities] -> source pass -> share;
//                without the flag as a cold single context
//   iteration k  sweep of the shard, reduced into Jslab -> [hist] -> clear the residual word -> source pass ->
//                [not extrapolating: share] -> [tolerance > 0: residual word to all[rank], all-gather, to the host, sync,
//                max] -> [extrapolate: Ng sums, all-gather of every rank's 5 sums, solve + combine, share]
//   epilogue     [tolerance 0: residual word to all[rank], all-gather]
// "share" is the all-gather of the stage, copied into every rank's dEtaEff.  In a group every branch depends on
// all-gathered data only (the warm start is decided on the devices, the stopping test takes the max over all ranks, the
// Ng solve sums the sums of all ranks), so every rank issues the same collectives and stops after the same k.
int source_iteration(Context& c, const SourcePart& p, const double* beta, cudaStream_t s, int* iters, int64_t* nseg) {
  const bool group = p.stageStride > 0;
  const bool ng = (c.scatAccel & RTB200_SCATTER_NG) != 0;
  const bool held = c.scatWarm;
  c.scatWarm = false;   // Jprev holds a returned J again only when this call completes
  // a group decides on the devices whether x_0 is the stored J, so that a rank that lost its J turns the group cold
  const bool warm = (c.scatAccel & RTB200_SCATTER_WARM_START) && (group || held);
  const int64_t N = c.nleaf;
  const size_t nb = (size_t)3 * p.jStride * sizeof(double);
  // the scratch: the stage | J of the previous iteration | every rank's residual | the residual word | the warm-start word
  const size_t need = (size_t)(3 * p.stageStride + 3 * p.jStride + p.nranks + 2) * sizeof(double);
  if (int st = ensure_buffer((void**)&c.dScatScratch, &c.scatScratchBytes, need)) return st;
  double* stage = c.dScatScratch;
  double* Jprev = stage + 3 * p.stageStride;
  double* all = Jprev + 3 * p.jStride;
  unsigned long long* resid = (unsigned long long*)(all + p.nranks);
  int32_t* warmTaken = (int32_t*)(resid + 1);
  double* etaOut = group ? stage + (size_t)p.rank * p.jStride : c.dEtaEff;
  const int64_t oStride = group ? p.stageStride : N;
  const double* etaTh = c.dEta ? c.dEta + p.off : nullptr;
  double* words = group ? all : (double*)resid;   // the residual words the stopping rule takes the max of
  const int nwords = group ? p.nranks : 1;
  auto source_pass = [&](const double* J, double* Jp) {
    return launch_scatter_source(c, p.cnt, J, Jp, p.jStride, c.scatterSigma() + p.off, etaTh, N, etaOut, oStride, resid, s);
  };
  auto share = [&]() { return group ? p.share_source(stage) : RTB200_OK; };
  auto gather_resid = [&]() -> int {
    if (!group) return RTB200_OK;
    RTB_CUDA(cudaMemcpyAsync(all + p.rank, resid, sizeof(double), cudaMemcpyDeviceToDevice, s));
    return p.allgather(all, 1);
  };
  NgBuffers nbuf{};
  if (ng) {
    if (int st = ng_buffers(c, p.jStride, &nbuf)) return st;
    RTB_CUDA(cudaMemsetAsync(nbuf.count, 0, sizeof(int32_t), s));
  }
  if (warm) {
    if (group) {
      const double h = held ? 1. : 0.;
      RTB_CUDA(cudaMemcpyAsync(all + p.rank, &h, sizeof(double), cudaMemcpyHostToDevice, s));
      if (int st = p.allgather(all, 1)) return st;
      if (int st = launch_warm_start_agree(c, all, p.nranks, Jprev, 3 * p.jStride, warmTaken, s)) return st;
    }
    if (c.dustMode && c.dDustSigma)   // dust computes its sigma from the current species first
      if (int st = launch_compute_opacities_dust(c, beta, s)) return st;
    if (int st = source_pass(Jprev, p.J)) return st;
    if (int st = share()) return st;
  } else {
    // J_0 = 0, eta_1 = eta_th (+ sigma * 0)
    RTB_CUDA(cudaMemsetAsync(Jprev, 0, nb, s));
    if (c.dEta) RTB_CUDA(cudaMemcpyAsync(c.dEtaEff, c.dEta, (size_t)3 * N * sizeof(double), cudaMemcpyDeviceToDevice, s));
    else RTB_CUDA(cudaMemsetAsync(c.dEtaEff, 0, (size_t)3 * N * sizeof(double), s));
  }
  int64_t total = 0;
  int k = 1;
  int cycle = 0;   // sweeps since the call's start or the last attempted extrapolation
  double r = 0.;
  for (;; k++) {
    int64_t ns = 0;
    if (int st = p.sweep(k, &ns)) return st;
    total += ns;
    cycle++;
    const bool extrapolate = ng && cycle == 4 && k < c.scatMaxIter;   // never on the sweep that stops the call
    // Ng keeps y of the cycle's sweeps 1..3: Jprev holds y_{k-1} until the source pass overwrites it
    if (ng && cycle >= 2) RTB_CUDA(cudaMemcpyAsync(nbuf.hist[cycle - 2], Jprev, nb, cudaMemcpyDeviceToDevice, s));
    RTB_CUDA(cudaMemsetAsync(resid, 0, sizeof(unsigned long long), s));
    if (int st = source_pass(p.J, Jprev)) return st;
    if (!extrapolate)
      if (int st = share()) return st;
    c.lastLaunches += 1;
    if (c.scatTol > 0.) {   // the stopping test reads the residual back; tolerance 0 runs on without a host round trip
      if (int st = gather_resid()) return st;
      std::vector<double> v((size_t)nwords);
      RTB_CUDA(cudaMemcpyAsync(v.data(), words, v.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
      RTB_CUDA(cudaStreamSynchronize(s));
      r = *std::max_element(v.begin(), v.end());
      if (r <= c.scatTol) break;
    }
    if (extrapolate) {   // I0..I3 = y_k (J), y_{k-1}, y_{k-2}, y_{k-3}; every rank solves with the sums of all ranks
      if (int st = launch_ng_partials(nbuf, p.cnt, p.J, p.jStride, p.rank, s)) return st;
      if (group)
        if (int st = p.allgather(nbuf.sums, 5)) return st;
      if (int st = launch_ng_apply(c, nbuf, p.nranks, p.cnt, p.J, Jprev, p.jStride, c.scatterSigma() + p.off, etaTh, N,
                                   etaOut, oStride, s))
        return st;
      if (int st = share()) return st;
      c.lastLaunches += 4;
      cycle = 0;
    }
    if (k == c.scatMaxIter) break;
  }
  if (c.scatTol == 0.)   // read by rtb200_last_scattering: no host round trip in the call
    if (int st = gather_resid()) return st;
  RTB_CUDA(cudaEventRecord(c.evStop, s));   // device time of the whole call, source passes included
  if (nseg) *nseg = total;
  c.lastScatIter = k;
  c.lastScatResid = r;
  c.dScatResid = c.scatTol == 0. ? words : nullptr;
  c.nScatResid = nwords;
  // a group's warm-start decision and the Ng count stay on the device: rtb200_last_scattering_acceleration reads them
  c.lastWarm = warm && !group;
  c.dWarmTaken = warm && group ? warmTaken : nullptr;
  c.ngPending = ng;
  c.scatWarm = true;   // the source pass left y_k in Jprev
  *iters = k;
  return RTB200_OK;
}

// the source iteration of a single context over all directions of nAngularLevel, into dJ (J_k, the last iteration's)
int scatter_solve(Context& c, int nAngularLevel, const double* uvb, const double* beta, double* dJ, cudaStream_t s,
                  int64_t* nseg) {
  if (!uvb || !beta || !dJ || c.nleaf == 0) return RTB200_ERR_ARG;
  RTB_CUDA(cudaSetDevice(c.device));
  SourcePart p;
  p.cnt = p.jStride = c.nleaf;
  p.J = dJ;
  p.sweep = [&](int k, int64_t* ns) { return run_sweep(c, nAngularLevel, uvb, beta, nullptr, 0, dJ, s, ns, k); };
  int iters = 0;
  return source_iteration(c, p, beta, s, &iters, nseg);
}

}  // namespace rtb
