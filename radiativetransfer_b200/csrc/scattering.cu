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

int set_scattering(Context& c, const double* sigma, bool device, int32_t maxIterations, double tolerance) {
  if (c.nleaf == 0) return RTB200_ERR_ARG;
  if (sigma && (maxIterations < 1 || !(tolerance >= 0.) || std::isinf(tolerance))) return RTB200_ERR_ARG;
  if (sigma && c.dDustSigma) return RTB200_ERR_ARG;   // one scattering medium at a time (dust.cu)
  RTB_CUDA(cudaSetDevice(c.device));
  RTB_CUDA(cudaDeviceSynchronize());   // queued sweeps read the current arrays
  if (!sigma) {
    cudaFree(c.dSigma); c.dSigma = nullptr;
    if (!c.dDustSigma) {   // scattering dust keeps the buffers of its source iteration
      release_acceleration(c);
      cudaFree(c.dEtaEff); c.dEtaEff = nullptr;
      cudaFree(c.dScatScratch); c.dScatScratch = nullptr; c.scatScratchBytes = 0;
    }
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
  if (c.scatResidPending) {
    RTB_CUDA(cudaSetDevice(c.device));
    RTB_CUDA(cudaEventSynchronize(c.evStop));
    RTB_CUDA(cudaMemcpy(&c.lastScatResid, c.dScatScratch + 3 * c.nleaf, sizeof(double), cudaMemcpyDeviceToHost));
    c.scatResidPending = false;
  }
  if (iterations) *iterations = c.lastScatIter;
  if (residual) *residual = c.lastScatResid;
  return RTB200_OK;
}

// Source iteration of a single context over all directions of nAngularLevel, into dJ (J_k, the last iteration's).  With
// the acceleration flags (ng.cu): the warm start takes x_0 from Jprev, which holds the J the previous completed solve
// returned, and Ng extrapolates after every fourth sweep of a cycle; the plain source pass runs after every sweep.
int scatter_solve(Context& c, int nAngularLevel, const double* uvb, const double* beta, double* dJ, cudaStream_t s,
                  int64_t* nseg) {
  if (!uvb || !beta || !dJ || c.nleaf == 0) return RTB200_ERR_ARG;
  const bool warm = (c.scatAccel & RTB200_SCATTER_WARM_START) && c.scatWarm;
  const bool ng = (c.scatAccel & RTB200_SCATTER_NG) != 0;
  c.scatWarm = false;   // Jprev holds a returned J again only when this call completes
  RTB_CUDA(cudaSetDevice(c.device));
  const int64_t N = c.nleaf;
  // [3][N] J of the previous iteration, then the residual word
  if (int st = ensure_buffer((void**)&c.dScatScratch, &c.scatScratchBytes, (size_t)(3 * N + 1) * sizeof(double))) return st;
  double* Jprev = c.dScatScratch;
  unsigned long long* resid = (unsigned long long*)(c.dScatScratch + 3 * N);
  NgBuffers nb{};
  if (ng) {
    if (int st = ng_buffers(c, N, &nb)) return st;
    RTB_CUDA(cudaMemsetAsync(nb.count, 0, sizeof(int32_t), s));
  }
  if (warm) {
    // eta_1 = eta_th + sigma * x_0 by the source pass (dJ, overwritten by the first sweep, takes its copy of x_0); dust
    // computes its sigma from the current species first
    if (c.dustMode && c.dDustSigma)
      if (int st = launch_compute_opacities_dust(c, beta, s)) return st;
    if (int st = launch_scatter_source(c, N, Jprev, dJ, N, c.scatterSigma(), c.dEta, N, c.dEtaEff, N, resid, s)) return st;
  } else {
    // J_0 = 0, eta_1 = eta_th (+ sigma * 0)
    RTB_CUDA(cudaMemsetAsync(Jprev, 0, (size_t)3 * N * sizeof(double), s));
    if (c.dEta) RTB_CUDA(cudaMemcpyAsync(c.dEtaEff, c.dEta, (size_t)3 * N * sizeof(double), cudaMemcpyDeviceToDevice, s));
    else RTB_CUDA(cudaMemsetAsync(c.dEtaEff, 0, (size_t)3 * N * sizeof(double), s));
  }
  int64_t total = 0;
  int k = 0;
  int cycle = 0;   // sweeps since the call's start or the last attempted extrapolation
  double r = 0.;
  for (k = 1; k <= c.scatMaxIter; k++) {
    int64_t ns = 0;
    if (int st = run_sweep(c, nAngularLevel, uvb, beta, nullptr, 0, dJ, s, &ns, k)) return st;
    total += ns;
    cycle++;
    // Ng keeps y of the cycle's sweeps 1..3: Jprev holds y_{k-1} until the source pass overwrites it
    if (ng && cycle >= 2)
      RTB_CUDA(cudaMemcpyAsync(nb.hist[cycle - 2], Jprev, (size_t)3 * N * sizeof(double), cudaMemcpyDeviceToDevice, s));
    RTB_CUDA(cudaMemsetAsync(resid, 0, sizeof(unsigned long long), s));
    if (int st = launch_scatter_source(c, N, dJ, Jprev, N, c.scatterSigma(), c.dEta, N, c.dEtaEff, N, resid, s)) return st;
    c.lastLaunches += 1;
    if (c.scatTol > 0.) {   // the stopping test reads the residual back; tolerance 0 runs on without a host round trip
      RTB_CUDA(cudaMemcpyAsync(&r, resid, sizeof(double), cudaMemcpyDeviceToHost, s));
      RTB_CUDA(cudaStreamSynchronize(s));
      if (r <= c.scatTol) break;
    }
    if (ng && cycle == 4 && k < c.scatMaxIter) {   // I0..I3 = y_k (dJ), y_{k-1}, y_{k-2}, y_{k-3}
      if (int st = launch_ng_partials(nb, N, dJ, N, 0, s)) return st;
      if (int st = launch_ng_apply(c, nb, 1, N, dJ, Jprev, N, c.scatterSigma(), c.dEta, N, c.dEtaEff, N, s)) return st;
      c.lastLaunches += 4;
      cycle = 0;
    }
  }
  if (k > c.scatMaxIter) k = c.scatMaxIter;
  RTB_CUDA(cudaEventRecord(c.evStop, s));   // device time of the whole call, source passes included
  if (nseg) *nseg = total;
  c.lastScatIter = k;
  c.lastScatResid = r;
  c.scatResidPending = c.scatTol == 0.;     // rtb200_last_scattering reads it once the call's work is done
  c.lastWarm = warm;
  c.ngPending = ng;                         // rtb200_last_scattering_acceleration reads the count likewise
  c.scatWarm = true;                        // the source pass left y_k in Jprev
  return RTB200_OK;
}

}  // namespace rtb
