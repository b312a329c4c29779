// The dust opacity of a leaf in the diffuse field (DESIGN.md 4.8), shared by the opacity pass (dust.cu) and the heating
// pass (heating.cu), so that the dust absorption the heating pass reports is the opacity the sweep ran with.  Every step
// is rounded on its own (no FMA), so that numpy repeats it bit for bit:
//   mode 1: kd = ((HI * bd) * abun2) / 0.2f,   mode 2: kd = (((((0.76f * rho) / m_H) * bd) * abun2) / 0.2f
#pragma once
#include <cstdint>

namespace rtb {

// the dust column of leaf i: HI in mode 1, 0.76f * rho / m_H in mode 2 (rho is read in mode 2 only)
__device__ __forceinline__ double dust_column(int mode, double HI, const double* __restrict__ rho, int64_t i) {
  return mode == 1 ? HI : __ddiv_rn(__dmul_rn((double)0.76f, rho[i]), (double)1.6726231e-24f);
}

// kd of one group from the column, the band-mean cross-section bd [cm^2 per H] and the leaf's abun2
__device__ __forceinline__ double dust_kd(double col, double bd, double abun2) {
  return __ddiv_rn(__dmul_rn(__dmul_rn(col, bd), abun2), (double)0.2f);
}

}  // namespace rtb
