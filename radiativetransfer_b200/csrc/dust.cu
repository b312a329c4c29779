// Dust in the diffuse sweep (DESIGN.md 4.8): the dust model of the point-source path as an opacity of the diffuse field.
//
// Per leaf and group the dust opacity kd_g follows the current species of every call (mode 1 is proportional to HI,
// which chemistry changes between the calls without a host round trip), so it is computed on the device together with
// the gas opacities, in one streaming pass that replaces compute_opacities_kernel while dust is set.  A dust albedo > 0
// routes albedo * kd_g into the source iteration of scattering.cu: the pass writes it into Context::dDustSigma, which the
// source iteration reads as its sigma (Context::scatterSigma).  Nothing downstream changes: the sweeps read dKappa.
#include <algorithm>
#include <cmath>

#include "rtb200_internal.h"

namespace rtb {

struct DustParams {
  double b0, b3, b4, b6, b7, b8;   // gas cross-sections, as compute_opacities_kernel takes them
  double bd[3];                    // band-mean dust cross-sections [cm^2 per H]
  double al[3];                    // albedos
  int mode;                        // 1: dust column from HI, 2: from rho
};

// kappa_g = kappa_abs,g + kd_g (the gas sequence of compute_opacities_kernel, then kd added and rounded once) and, with
// sigmaSrc, sigmaSrc_g = albedo_g * kd_g.  Every step rounded on its own (no FMA), so that numpy repeats it bit for bit:
//   mode 1: kd = ((HI * bd) * abun2) / 0.2f,   mode 2: kd = (((((0.76f * rho) / m_H) * bd) * abun2) / 0.2f
__global__ void compute_opacities_dust_kernel(const double* __restrict__ HI, const double* __restrict__ HeI,
                                              const double* __restrict__ HeII, const double* __restrict__ rho,
                                              const double* __restrict__ abun2, double* __restrict__ kappa,
                                              double* __restrict__ sigmaSrc, int64_t n, DustParams p) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double h = HI[i], he1 = HeI[i], he2 = HeII[i], a = abun2[i];
    const double col = p.mode == 1 ? h : __ddiv_rn(__dmul_rn((double)0.76f, rho[i]), (double)1.6726231e-24f);
    double kd[3];
    for (int g = 0; g < 3; g++) kd[g] = __ddiv_rn(__dmul_rn(__dmul_rn(col, p.bd[g]), a), (double)0.2f);
    kappa[i] = __dadd_rn(__dmul_rn(h, p.b0), kd[0]);
    kappa[n + i] = __dadd_rn(__dadd_rn(__dmul_rn(h, p.b3), __dmul_rn(he1, p.b4)), kd[1]);
    kappa[2 * n + i] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(h, p.b6), __dmul_rn(he1, p.b7)), __dmul_rn(he2, p.b8)), kd[2]);
    if (sigmaSrc)
      for (int g = 0; g < 3; g++) sigmaSrc[g * n + i] = __dmul_rn(p.al[g], kd[g]);
  }
}

int launch_compute_opacities_dust(Context& c, const double* beta, cudaStream_t s) {
  DustParams p;
  p.b0 = beta[0]; p.b3 = beta[3]; p.b4 = beta[4]; p.b6 = beta[6]; p.b7 = beta[7]; p.b8 = beta[8];
  for (int g = 0; g < 3; g++) { p.bd[g] = c.dustBeta[g]; p.al[g] = c.dustAlbedo[g]; }
  p.mode = c.dustMode;
  const int blocks = (int)std::min<int64_t>((c.nleaf + 255) / 256, (int64_t)c.smCount * 16);
  compute_opacities_dust_kernel<<<blocks, 256, 0, s>>>(c.dHI, c.dHeI, c.dHeII, c.dRho, c.dAbun2, c.dKappa, c.dDustSigma,
                                                       c.nleaf, p);
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

static bool scatters(const double* albedo) { return albedo[0] > 0. || albedo[1] > 0. || albedo[2] > 0.; }

bool dust_args_ok(int mode, const double* betaDust, const double* albedo, int32_t maxIterations, double tolerance) {
  if (mode < 0 || mode > 2) return false;
  if (mode == 0) return true;
  if (!betaDust || !albedo) return false;
  for (int g = 0; g < 3; g++) {
    if (!(betaDust[g] >= 0. && betaDust[g] <= 1.7976931348623157e308)) return false;   // negative, NaN, Inf
    if (!(albedo[g] >= 0. && albedo[g] <= 1.)) return false;
  }
  if (scatters(albedo) && (maxIterations < 1 || !(tolerance >= 0.) || std::isinf(tolerance))) return false;
  return true;
}

int set_dust(Context& c, int mode, const double* betaDust, const double* albedo, int32_t maxIterations, double tolerance) {
  if (c.nleaf == 0 || !dust_args_ok(mode, betaDust, albedo, maxIterations, tolerance)) return RTB200_ERR_ARG;
  if ((mode == 1 && !c.dAbun2) || (mode == 2 && (!c.dRho || !c.dAbun2))) return RTB200_ERR_ARG;
  const bool scatter = mode != 0 && scatters(albedo);
  if (scatter && c.dSigma) return RTB200_ERR_ARG;   // one scattering medium at a time
  RTB_CUDA(cudaSetDevice(c.device));
  RTB_CUDA(cudaDeviceSynchronize());   // queued sweeps read the current state
  const double* eta0 = c.sweepEta();
  if (scatter) {   // the buffers of the source iteration first: a failed allocation leaves the previous state
    const size_t nb = (size_t)3 * c.nleaf * sizeof(double);
    const bool newEff = !c.dEtaEff, newSig = !c.dDustSigma;
    cudaError_t e = cudaSuccess;
    if (newEff) e = cudaMalloc((void**)&c.dEtaEff, nb);
    if (e == cudaSuccess && newSig) e = cudaMalloc((void**)&c.dDustSigma, nb);
    if (e != cudaSuccess) {
      if (newEff) { cudaFree(c.dEtaEff); c.dEtaEff = nullptr; }
      if (newSig) { cudaFree(c.dDustSigma); c.dDustSigma = nullptr; }
      set_cuda_error("cudaMalloc", e, __FILE__, __LINE__);
      return e == cudaErrorMemoryAllocation ? RTB200_ERR_NOMEM : RTB200_ERR_CUDA;
    }
    c.scatMaxIter = maxIterations;
    c.scatTol = tolerance;
  } else if (c.dDustSigma) {   // dust stops scattering: the source iteration's buffers go unless a per-leaf sigma needs them
    cudaFree(c.dDustSigma); c.dDustSigma = nullptr;
    cudaFree(c.dEtaEff); c.dEtaEff = nullptr;
    cudaFree(c.dScatScratch); c.dScatScratch = nullptr; c.scatScratchBytes = 0;
  }
  c.dustMode = mode;
  for (int g = 0; g < 3; g++) {
    c.dustBeta[g] = mode ? betaDust[g] : 0.;
    c.dustAlbedo[g] = mode ? albedo[g] : 0.;
  }
  if (c.sweepEta() != eta0) drop_sweep_plans(c);   // the uniform plan and graph know which source the sweeps read
  return RTB200_OK;
}

}  // namespace rtb
