// Acceleration of the source iteration of scattering.cu (DESIGN.md 4.9): a warm start from the J of the previous call
// and Ng extrapolation of order 2 (Auer 1987, in the form of Olson, Auer & Buchler 1986).
//
// An extrapolation is three small steps that never leave the device: a streaming pass over the four latest sweep outputs
// writes per-block partials of five sums, one block adds them in block order (a device group all-gathers the ranks' sums
// and every rank adds them in rank order), and one thread solves the 2x2 system and writes {1 - a - b, a, b, apply}.
// A last streaming pass then forms x = max(0, (1-a-b) I0 + a I1 + b I2), the next source eta_th + sigma * x and keeps x
// for the next residual; when the step is skipped it writes nothing, which leaves the plain source pass's result.
// Every sum runs over a fixed grid in a fixed order, so the results are bit-identical from run to run.
#include <algorithm>
#include <cmath>

#include "rtb200_internal.h"

namespace rtb {

namespace {

constexpr int kNgThreads = 256;
constexpr int64_t kNgPart = 0, kNgSums = kNgPart + 5 * kNgBlocks, kNgCoef = kNgSums + 5 * kNgMaxRanks,
                  kNgCount = kNgCoef + 4, kNgHist = kNgCount + 4;   // offsets in doubles (the history 64-byte aligned)

}  // namespace

// five sums over t < 3 cnt of the weighted differences of I0..I3 (entry (g, i) at g * jStride + i), one partial per
// block: grid-stride partial sums per thread, then a fixed tree in shared memory
__global__ void __launch_bounds__(kNgThreads) ng_partials_kernel(int64_t cnt, const double* __restrict__ I0,
                                                                 const double* __restrict__ I1,
                                                                 const double* __restrict__ I2,
                                                                 const double* __restrict__ I3, int64_t jStride,
                                                                 double* __restrict__ part) {
  double s0 = 0., s1 = 0., s2 = 0., s3 = 0., s4 = 0.;
  const int64_t total = 3 * cnt;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = t / cnt, i = t - g * cnt, e = g * jStride + i;
    const double i0 = I0[e], i1 = I1[e], i2 = I2[e], i3 = I3[e];
    const double w = i0 > 0. ? 1. / i0 : 0.;
    const double d0 = (i0 - i1) * w, d1 = (i1 - i2) * w, d2 = (i2 - i3) * w;
    const double q1 = d0 - d1, q2 = d0 - d2;
    s0 += q1 * q1; s1 += q1 * q2; s2 += q2 * q2; s3 += d0 * q1; s4 += d0 * q2;
  }
  __shared__ double sh[5][kNgThreads];
  const int x = threadIdx.x;
  sh[0][x] = s0; sh[1][x] = s1; sh[2][x] = s2; sh[3][x] = s3; sh[4][x] = s4;
  __syncthreads();
  for (int h = kNgThreads / 2; h > 0; h >>= 1) {
    if (x < h)
      for (int k = 0; k < 5; k++) sh[k][x] += sh[k][x + h];
    __syncthreads();
  }
  if (x < 5) part[(int64_t)blockIdx.x * 5 + x] = sh[x][0];
}

// the block partials in block order: this rank's five sums
__global__ void ng_rank_sum_kernel(const double* __restrict__ part, double* __restrict__ sums) {
  const int k = threadIdx.x;
  if (k >= 5) return;
  double a = 0.;
  for (int b = 0; b < kNgBlocks; b++) a += part[b * 5 + k];
  sums[k] = a;
}

// the ranks' sums in rank order, the 2x2 solve and the decision (one thread)
__global__ void ng_solve_kernel(const double* __restrict__ sums, int nranks, double* __restrict__ coef,
                                int32_t* __restrict__ count) {
  double s[5] = {0., 0., 0., 0., 0.};
  for (int r = 0; r < nranks; r++)
    for (int k = 0; k < 5; k++) s[k] += sums[r * 5 + k];
  const double A11 = s[0], A12 = s[1], A22 = s[2], c1 = s[3], c2 = s[4];
  const double det = A11 * A22 - A12 * A12;
  const double a = (c1 * A22 - c2 * A12) / det, b = (c2 * A11 - c1 * A12) / det;
  const bool apply = det > 1e-14 * A11 * A22 && isfinite(a) && isfinite(b);
  coef[0] = apply ? 1. - a - b : 1.;
  coef[1] = apply ? a : 0.;
  coef[2] = apply ? b : 0.;
  coef[3] = apply ? 1. : 0.;
  if (apply) *count += 1;
}

// x = max(0, (1-a-b) I0 + a I1 + b I2) (no FMA), Jprev = x, etaOut = eta_th + sigma * x as scatter_source_kernel does;
// nothing when the step is skipped
__global__ void ng_combine_kernel(int64_t cnt, const double* __restrict__ I0, const double* __restrict__ I1,
                                  const double* __restrict__ I2, double* __restrict__ Jprev, int64_t jStride,
                                  const double* __restrict__ sigma, const double* __restrict__ etaTh, int64_t sStride,
                                  double* __restrict__ etaOut, int64_t oStride, const double* __restrict__ coef) {
  if (coef[3] == 0.) return;
  const double c0 = coef[0], a = coef[1], b = coef[2];
  const int64_t total = 3 * cnt;
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = t / cnt, i = t - g * cnt, e = g * jStride + i;
    const double v = __dadd_rn(__dadd_rn(__dmul_rn(c0, I0[e]), __dmul_rn(a, I1[e])), __dmul_rn(b, I2[e]));
    const double xk = v > 0. ? v : 0.;   // NaN -> 0 as well: the sweeps need sources >= 0
    Jprev[e] = xk;
    const double th = etaTh ? etaTh[g * sStride + i] : 0.;
    etaOut[g * oStride + i] = __dadd_rn(th, __dmul_rn(sigma[g * sStride + i], xk));
  }
}

// warm start of a device group: x_0 is the stored Jprev only where every rank holds one (flags[r] != 0 for all ranks),
// else 0, so that all ranks start alike; *used records the decision
__global__ void warm_start_agree_kernel(const double* __restrict__ flags, int nranks, double* __restrict__ Jprev,
                                        int64_t n, int32_t* __restrict__ used) {
  bool all = true;
  for (int r = 0; r < nranks; r++) all = all && flags[r] != 0.;
  if (blockIdx.x == 0 && threadIdx.x == 0) *used = all ? 1 : 0;
  if (all) return;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) Jprev[i] = 0.;
}

int launch_warm_start_agree(const Context& c, const double* flags, int nranks, double* Jprev, int64_t n, int32_t* used,
                            cudaStream_t s) {
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)c.smCount * 16));
  warm_start_agree_kernel<<<blocks, 256, 0, s>>>(flags, nranks, Jprev, n, used);
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

int ng_buffers(Context& c, int64_t stride, NgBuffers* b) {
  const size_t need = (size_t)(kNgHist + 9 * stride) * sizeof(double);
  if (int st = ensure_buffer((void**)&c.dNg, &c.ngBytes, need)) return st;
  b->part = c.dNg + kNgPart;
  b->sums = c.dNg + kNgSums;
  b->coef = c.dNg + kNgCoef;
  b->count = (int32_t*)(c.dNg + kNgCount);
  for (int j = 0; j < 3; j++) b->hist[j] = c.dNg + kNgHist + (int64_t)j * 3 * stride;
  return RTB200_OK;
}

int launch_ng_partials(const NgBuffers& b, int64_t cnt, const double* I0, int64_t jStride, int rank, cudaStream_t s) {
  // I1..I3 = y_{k-1}, y_{k-2}, y_{k-3}: the history of the cycle's sweeps 3, 2, 1
  ng_partials_kernel<<<kNgBlocks, kNgThreads, 0, s>>>(cnt, I0, b.hist[2], b.hist[1], b.hist[0],
                                                      jStride, b.part);
  RTB_CUDA(cudaGetLastError());
  ng_rank_sum_kernel<<<1, 32, 0, s>>>(b.part, b.sums + 5 * rank);
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

int launch_ng_apply(const Context& c, const NgBuffers& b, int nranks, int64_t cnt, const double* I0, double* Jprev,
                    int64_t jStride, const double* sigma, const double* etaTh, int64_t sStride, double* etaOut,
                    int64_t oStride, cudaStream_t s) {
  ng_solve_kernel<<<1, 1, 0, s>>>(b.sums, nranks, b.coef, b.count);
  RTB_CUDA(cudaGetLastError());
  if (cnt <= 0) return RTB200_OK;
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((3 * cnt + 255) / 256, (int64_t)c.smCount * 16));
  ng_combine_kernel<<<blocks, 256, 0, s>>>(cnt, I0, b.hist[2], b.hist[1], Jprev, jStride, sigma, etaTh, sStride, etaOut,
                                           oStride, b.coef);
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

void free_history(Context& c) {
  if (c.ngPending) {
    if (cudaMemcpy(&c.lastNgCount, c.dNg + kNgCount, sizeof(int32_t), cudaMemcpyDeviceToHost) != cudaSuccess) c.lastNgCount = 0;
    c.ngPending = false;
  }
  cudaFree(c.dNg); c.dNg = nullptr; c.ngBytes = 0;
}

int set_scattering_acceleration(Context& c, int32_t flags) {
  if (c.nleaf == 0 || (flags & ~(RTB200_SCATTER_NG | RTB200_SCATTER_WARM_START))) return RTB200_ERR_ARG;
  RTB_CUDA(cudaSetDevice(c.device));
  RTB_CUDA(cudaDeviceSynchronize());   // queued solves read the flags' buffers
  if (!(flags & RTB200_SCATTER_NG)) free_history(c);
  c.scatAccel = flags;
  return RTB200_OK;
}

int last_scattering_acceleration(Context& c, int32_t* extrapolations, int32_t* warmStarted) {
  if (c.ngPending) {
    RTB_CUDA(cudaSetDevice(c.device));
    RTB_CUDA(cudaEventSynchronize(c.evStop));
    RTB_CUDA(cudaMemcpy(&c.lastNgCount, c.dNg + kNgCount, sizeof(int32_t), cudaMemcpyDeviceToHost));
    c.ngPending = false;
  }
  if (c.dWarmTaken) {   // device group: the ranks decided the warm start on the devices
    RTB_CUDA(cudaSetDevice(c.device));
    RTB_CUDA(cudaEventSynchronize(c.evStop));
    int32_t used = 0;
    RTB_CUDA(cudaMemcpy(&used, c.dWarmTaken, sizeof(int32_t), cudaMemcpyDeviceToHost));
    c.lastWarm = used != 0;
    c.dWarmTaken = nullptr;
  }
  if (extrapolations) *extrapolations = c.lastNgCount;
  if (warmStarted) *warmStarted = c.lastWarm ? 1 : 0;
  return RTB200_OK;
}

}  // namespace rtb
