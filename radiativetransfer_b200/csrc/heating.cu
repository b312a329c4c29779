// Photo-heating and dust absorption of the diffuse field per leaf (DESIGN.md 4.10).
//
// While heating is set, every diffuse call ends with one streaming pass over the J it returns (after the source
// iteration of a scattering solve; after the reduction in a device group).  Per leaf, with t_g = 4 pi J_g:
//   f 0..2  Gamma_s = ((t_1 gamma[1][s]) + (t_2 gamma[2][s])) + (t_3 gamma[3][s])          [erg/s per absorber]
//   f 3     H_gas   = ((HI Gamma_HI) + (HeI Gamma_HeI)) + (HeII Gamma_HeII)                  [erg/s/cm^3]
//   f 4     H_dust  = (u_1 + u_2) + u_3,  u_g = ((1 - albedo_g) kd_g) (t_g W_g)              [erg/s/cm^3]
// every operation rounded on its own (no FMA), so that numpy repeats the pass bit for bit (tests/heating_oracle.py).
// kd_g is dust_kd of dust_model.cuh, the opacity the sweep ran with.  One kernel serves every route, so a single context
// and a device group give the same bits for the same J.  The pass is separate from the sweep's merge, the nested-grid
// writes and the peer reduction: ~100 B per leaf against the sweep's 72 B per leaf and direction.
#include <algorithm>

#include "dust_model.cuh"
#include "rtb200_internal.h"

namespace rtb {

struct HeatParams {
  double gam[9];   // [group][gammaHI, gammaHeI, gammaHeII]
  double W[3];     // band widths [Hz]
  double bd[3];    // dust cross-sections of rtb200_grid_set_dust
  double al[3];    // dust albedos
  int mode;        // dust mode, 0 = no dust
};

__global__ void heating_kernel(int64_t cnt, const double* __restrict__ J, int64_t jStride, const double* __restrict__ HI,
                               const double* __restrict__ HeI, const double* __restrict__ HeII,
                               const double* __restrict__ rho, const double* __restrict__ abun2, double* __restrict__ H,
                               int64_t hStride, HeatParams p) {
  const double fourPi = 4. * kPi;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x) {
    double t[3];
    for (int g = 0; g < 3; g++) t[g] = __dmul_rn(fourPi, J[g * jStride + i]);
    double G[3];
    for (int s = 0; s < 3; s++)
      G[s] = __dadd_rn(__dadd_rn(__dmul_rn(t[0], p.gam[s]), __dmul_rn(t[1], p.gam[3 + s])), __dmul_rn(t[2], p.gam[6 + s]));
    const double h = HI[i];
    const double gas = __dadd_rn(__dadd_rn(__dmul_rn(h, G[0]), __dmul_rn(HeI[i], G[1])), __dmul_rn(HeII[i], G[2]));
    double dust = 0.;
    if (p.mode) {
      const double col = dust_column(p.mode, h, rho, i), a = abun2[i];
      double u[3];
      for (int g = 0; g < 3; g++)
        u[g] = __dmul_rn(__dmul_rn(__dsub_rn(1., p.al[g]), dust_kd(col, p.bd[g], a)), __dmul_rn(t[g], p.W[g]));
      dust = __dadd_rn(__dadd_rn(u[0], u[1]), u[2]);
    }
    for (int s = 0; s < 3; s++) H[s * hStride + i] = G[s];
    H[3 * hStride + i] = gas;
    H[4 * hStride + i] = dust;
  }
}

bool heating_args_ok(const double* gamma9, const double* width3) {
  if (!gamma9 || !width3) return false;
  for (int k = 0; k < 9; k++)
    if (!finite_nonneg(gamma9[k])) return false;
  for (int g = 0; g < 3; g++)
    if (!finite_nonneg(width3[g])) return false;
  return true;
}

void free_heating(Context& c) {
  cudaFree(c.dHeat);
  c.dHeat = nullptr;
  c.heatStride = 0;
  c.heatValid = false;
  for (int k = 0; k < 9; k++) c.heatGamma[k] = 0.;
  for (int g = 0; g < 3; g++) c.heatWidth[g] = 0.;
}

int set_heating(Context& c, const double* gamma9, const double* width3, int64_t stride) {
  if (c.nleaf == 0 || stride < 1 || (gamma9 && !heating_args_ok(gamma9, width3))) return RTB200_ERR_ARG;
  RTB_CUDA(cudaSetDevice(c.device));
  RTB_CUDA(cudaDeviceSynchronize());   // queued passes write the current buffer
  if (!gamma9) {
    free_heating(c);
    return RTB200_OK;
  }
  if (!c.dHeat || c.heatStride != stride) {   // a failed allocation leaves the previous state
    double* fresh = nullptr;
    const size_t bytes = (size_t)5 * stride * sizeof(double);
    cudaError_t e = cudaMalloc((void**)&fresh, bytes);
    if (e == cudaSuccess) e = cudaMemset(fresh, 0, bytes);
    if (e != cudaSuccess) {
      cudaFree(fresh);
      set_cuda_error("cudaMalloc", e, __FILE__, __LINE__);
      return e == cudaErrorMemoryAllocation ? RTB200_ERR_NOMEM : RTB200_ERR_CUDA;
    }
    cudaFree(c.dHeat);
    c.dHeat = fresh;
    c.heatStride = stride;
  }
  for (int k = 0; k < 9; k++) c.heatGamma[k] = gamma9[k];
  for (int g = 0; g < 3; g++) c.heatWidth[g] = width3[g];
  c.heatValid = false;
  return RTB200_OK;
}

int launch_heating(Context& c, int64_t off, int64_t cnt, const double* J, int64_t jStride, cudaStream_t s) {
  HeatParams p;
  for (int k = 0; k < 9; k++) p.gam[k] = c.heatGamma[k];
  for (int g = 0; g < 3; g++) {
    p.W[g] = c.heatWidth[g];
    p.bd[g] = c.dustBeta[g];
    p.al[g] = c.dustAlbedo[g];
  }
  p.mode = c.dustMode;
  if (cnt > 0) {
    const int blocks = (int)std::min<int64_t>((cnt + 255) / 256, (int64_t)c.smCount * 16);
    heating_kernel<<<blocks, 256, 0, s>>>(cnt, J, jStride, c.dHI + off, c.dHeI + off, c.dHeII + off,
                                          c.dRho ? c.dRho + off : nullptr, c.dAbun2 ? c.dAbun2 + off : nullptr, c.dHeat,
                                          c.heatStride, p);
    RTB_CUDA(cudaGetLastError());
    c.lastLaunches += 1;
  }
  RTB_CUDA(cudaEventRecord(c.evStop, s));   // the call's device time includes the pass
  c.heatValid = true;
  return RTB200_OK;
}

}  // namespace rtb
