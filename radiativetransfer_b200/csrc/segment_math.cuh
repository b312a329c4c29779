// Per-segment arithmetic of the diffuse sweep (fp64, no tensor cores: the update is a chain of scalar
// exponentials, not a contraction).
//
// Reference (transportRoutinesModule.f90:651-698 and :1036-1054, identical inline copy equiSources.f90:1611-1643):
//     tau  = kappa * dpath;  Iout = Iin * exp(-tau)
//     Jseg = (Iin - Iout) / log(Iin / Iout)   if Iout < Iin,   else 0.5 * (Iin + Iout)
// FAITHFUL mode evaluates exactly that sequence (CUDA libm exp/log, IEEE division).
// FAST mode uses log(Iin/Iout) == tau, i.e. Jseg = Iin * (1 - exp(-tau)) / tau, with (1 - exp(-tau)) obtained
// without cancellation from the same polynomial that yields exp(-tau): one exponential and no log / division per
// segment.  The two differ by the rounding noise of the reference formula, ~1.1e-16 / tau relative.
#pragma once
#include <cuda_runtime.h>

namespace rtb {

// exp(-tau) = 2^(-k/16) * exp(-r),  k = round(tau * 16/ln2),  r = tau - k*ln2/16,  |r| <= ln2/32:
// a 16-entry table of 2^(-j/16) (one row of shared memory: any set of lanes reads it without bank conflicts), an
// exponent-field subtraction for 2^-(k>>4) and a degree-7 polynomial.  13-15 FP64 instructions instead of ~20 for a
// table-free evaluation; the sweep is bound by the FP64 pipe, so this is where its time goes.
// Constants sit in constant memory so that the DFMAs read them from the constant bank / uniform registers.
static __constant__ double kExpC[16] = {
    -1.98412698412698412698e-04,  // [0] -1/7!
    1.38888888888888888889e-03,   // [1]  1/6!
    -8.33333333333333333333e-03,  // [2] -1/5!
    4.16666666666666666667e-02,   // [3]  1/4!
    -1.66666666666666666667e-01,  // [4] -1/3!
    0.5,                          // [5]
    -1.0,                         // [6]
    23.083120654223414,           // [7]  16/ln2
    6755399441055744.0,           // [8]  1.5 * 2^52: adding it rounds to nearest integer
    -0.0433216979727149,          // [9]  -ln2/16, high part (27 trailing zero bits: k*hi is exact)
    -8.12281680868118e-10,        // [10] -ln2/16, low part
    707.0,                        // [11] clamp: keeps 2^-(k>>4) * 2^(-j/16) a normal number
    0., 0., 0., 0.};
static __constant__ double kExpTable[16] = {
    1.00000000000000000000e+00, 9.57603280698573700036e-01, 9.17004043204671215328e-01, 8.78126080186649726755e-01,
    8.40896415253714502036e-01, 8.05245165974627141736e-01, 7.71105412703970372057e-01, 7.38413072969749673113e-01,
    7.07106781186547572737e-01, 6.77127773468446325644e-01, 6.48419777325504820276e-01, 6.20928906036742001007e-01,
    5.94603557501360513449e-01, 5.69394317378345782288e-01, 5.45253866332628844837e-01, 5.22136891213706877402e-01};

// Straight-line code on purpose: a rare-case branch here would end the basic block and keep the compiler from
// interleaving the (independent) exponentials of the three frequency groups and of the 1..3 segments, which is where
// the instruction-level parallelism of the sweep comes from.  tau is clamped at 707: exp(-tau) below 2^-1020 is
// returned as ~2^-1020 (it only ever multiplies an intensity, and such products are far below anything physical).
// Returns Ts = 2^(-k/16) and p = exp(-r) - 1, so that  exp(-tau) = Ts + Ts*p  and  1 - exp(-tau) = (1 - Ts) - Ts*p
// (1 - Ts is exact, and for k == 0 the latter is exactly -p: no cancellation for small tau).
template <bool GUARD = true>
__device__ __forceinline__ void exp_neg_parts(double tau, const double* __restrict__ T, double& Ts, double& p) {
  // tau >= 0 (kappa >= 0, path > 0): clamp at 707 with ONE integer min on the high word instead of an FP64 compare
  // and two selects (0x40861800'00000000 = 707.0; the low word stays, so the clamped value lies in [707, 707.0005)).
  // GUARD = false: the caller knows tau <= 64 for the whole warp (see sweep_cell_kernel) and skips the clamp.
  if (GUARD) tau = __hiloint2double(min(__double2hiint(tau), 0x40861800), __double2loint(tau));
  double t = fma(tau, kExpC[7], kExpC[8]);
  int k = __double2loint(t);
  double fn = t - kExpC[8];
  double r = fma(fn, kExpC[9], tau);
  r = fma(fn, kExpC[10], r);
  double q = kExpC[0];
#pragma unroll
  for (int i = 1; i <= 6; i++) q = fma(q, r, kExpC[i]);
  p = q * r;
  double Tj = T[k & 15];
  Ts = __hiloint2double(__double2hiint(Tj) - ((k >> 4) << 20), __double2loint(Tj));
}

// The sweeps' exponential (round 2).  The uniform sweep runs into the board's power cap, so its time follows the fp64
// instruction count: a larger table shortens the polynomial.  64 entries: |r| <= ln2/128 = 0.0054, p = e^-r - 1 through
// r^4 -- 3 of the 12 FP64 instructions less per exponential.  Truncation: |dp / p| <= r^4 / 120 = 7.2e-12, i.e. 3.9e-14
// of e^-tau per segment, < 2e-11 after the 512 segments of the longest ray, and 7.2e-12 of a segment's contribution to
// J: two orders of magnitude inside the 1e-9 that FAST arithmetic is held to (measured FAST vs FAITHFUL on the full
// 256^3 x 192 solve: 4.1e-10, unchanged -- that difference is the reference formula's own rounding noise).
// Measured at 256^3 on one box, 20 solves back to back under the power cap: 16 entries / r^7 53.8 ms, 32 / r^5
// 50.7 ms, 64 / r^4 49.8 ms (the 4-way bank conflicts of the larger table cost less than the DFMA saves).
// (The point-source kernels keep the 16-entry / r^7 version above: their deposits are differences of exponentials.)
constexpr int kExpTableSize = 64;   // |r| <= ln2/128, polynomial through r^4
static __constant__ double kExpC32[12] = {
    0., 4.16666666666666666667e-02, -1.66666666666666666667e-01, 0.5, -1.0,
    92.33248261689366,            // [5]  64/ln2
    6755399441055744.0,
    -0.010830424493178725,        // [7]  -ln2/64 hi
    -2.030704202170295e-10,       // [8]  -ln2/64 lo
    0., 0., 0.};
constexpr int kExpDeg = 3;
constexpr int kExpShift = 6;
static __constant__ double kExpTable32[64] = {
    1.00000000000000000000e+00, 9.89228013193975463935e-01, 9.78572062087700089705e-01, 9.68030896746147173637e-01,
    9.57603280698573700036e-01, 9.47287990793482803653e-01, 9.37083817055149981279e-01, 9.26989562541692735387e-01,
    9.17004043204671215328e-01, 9.07126087750199427973e-01, 8.97354537501553584100e-01, 8.87688246263260594127e-01,
    8.78126080186649726755e-01, 8.68666917636853108675e-01, 8.59309649061238967072e-01, 8.50053176859261738763e-01,
    8.40896415253714502036e-01, 8.31838290163368188068e-01, 8.22877739076982472888e-01, 8.14013710928673916989e-01,
    8.05245165974627141736e-01, 7.96571075671133499441e-01, 7.87990422553943248296e-01, 7.79502200118918464611e-01,
    7.71105412703970372057e-01, 7.62799075372269208550e-01, 7.54582213796711420706e-01, 7.46453864145632417504e-01,
    7.38413072969749673113e-01, 7.30458897090323522328e-01, 7.22590403488523325137e-01, 7.14806669195985011633e-01,
    7.07106781186547572737e-01, 6.99489836269155618176e-01, 6.91954940981916011289e-01, 6.84501211487295257996e-01,
    6.77127773468446325644e-01, 6.69833762026651458044e-01, 6.62618321579870661608e-01, 6.55480605762382206869e-01,
    6.48419777325504820276e-01, 6.41435008039389131795e-01, 6.34525478595866609943e-01, 6.27690378512345548145e-01,
    6.20928906036742001007e-01, 6.14240268053435012341e-01, 6.07623679990234477621e-01, 6.01078365726351537823e-01,
    5.94603557501360513449e-01, 5.88198495825140610371e-01, 5.81862429388788737761e-01, 5.75594614976491336655e-01,
    5.69394317378345782288e-01, 5.63260809304120924068e-01, 5.57193371297946216103e-01, 5.51191291653920445448e-01,
    5.45253866332628844837e-01, 5.39380398878559930154e-01, 5.33570200338411848584e-01, 5.27822589180278578525e-01,
    5.22136891213706877402e-01, 5.16512439510614207450e-01, 5.10948574327058313571e-01, 5.05444643025850237628e-01};

template <bool GUARD = true>
__device__ __forceinline__ void exp_neg_parts32(double tau, const double* __restrict__ T, double& Ts, double& p) {
  if (GUARD) tau = __hiloint2double(min(__double2hiint(tau), 0x40861800), __double2loint(tau));
  double t = fma(tau, kExpC32[5], kExpC32[6]);
  int k = __double2loint(t);
  double fn = t - kExpC32[6];
  double r = fma(fn, kExpC32[7], tau);
  r = fma(fn, kExpC32[8], r);
  double q = kExpC32[4 - kExpDeg];
#pragma unroll
  for (int i = 5 - kExpDeg; i <= 4; i++) q = fma(q, r, kExpC32[i]);
  p = q * r;
  double Tj = T[k & (kExpTableSize - 1)];
  Ts = __hiloint2double(__double2hiint(Tj) - ((k >> kExpShift) << 20), __double2loint(Tj));
}

// FAST-mode segment: Iout = Iin e^-tau and the segment's contribution to the cell's mean intensity,
//   J_seg * weight/nseg = Iin (1 - e^-tau) / (kappa d) * wn = [Iin (1 - e^-tau)] * cs * (2^-200 / kappa),
// cs = 2^200 wn / d a per-(layer, direction, segment) constant from the host and 2^-200/kappa a per-cell constant that
// the caller applies ONCE per layer to the sum A over all directions and segments (the power of two keeps every
// intermediate far from the subnormal range, including the kappa -> 0 limit).  With Ts = 2^(-k/16), p = e^-r - 1:
//   X = Iin Ts,  Iout = X + X p,  Iin (1 - e^-tau) = (Iin - X) - X p      (Iin - X is exact for k = 0: no cancellation)
// 5 FP64 instructions after the exponential's 12, instead of 8.
// GUARD = false (tau <= 64 for every segment of the warp): no clamp, and no test for Iout underflowing to 0 -- with
// tau <= 64 that can only happen where Iin < 5e-324 e^64 = 3e-296, i.e. where the segment's contribution to Jmean
// (< Iin) is itself below every tolerance floor (the parity tests compare with a floor of 1e-290).
template <bool GUARD = true>
__device__ __forceinline__ double segment_fast(double Iin, double tau, double cs, const double* __restrict__ T, double& A) {
  double Ts, p;
  exp_neg_parts32<GUARD>(tau, T, Ts, p);
  const double X = Iin * Ts;
  const double Iout = fma(X, p, X);
  const double Z = fma(-X, p, Iin - X);
  // Iout == 0 (underflow): the reference gets (Iin - 0)/log(Iin/0) = 0.  Integer test + predicated DFMA.
  if (!GUARD || ((__double2hiint(Iout) << 1) | __double2loint(Iout)) != 0) A = fma(Z, cs, A);
  return Iout;
}

template <bool GUARD = true>
__device__ __forceinline__ double attenuate_fast(double Iin, double tau, const double* __restrict__ T) {
  double Ts, p;
  exp_neg_parts32<GUARD>(tau, T, Ts, p);
  const double X = Iin * Ts;
  return fma(X, p, X);
}

struct SegResult {
  double Iout, J;
};

// FAITHFUL-mode segment: the reference's operation sequence (CUDA libm exp / log, IEEE arithmetic, no contraction)
__device__ __forceinline__ SegResult segment_faithful(double Iin, double kappa, double dpath) {
  SegResult r;
  double tau = __dmul_rn(kappa, dpath);
  double a = exp(-tau);
  r.Iout = __dmul_rn(Iin, a);
  if (r.Iout < Iin) r.J = __ddiv_rn(__dsub_rn(Iin, r.Iout), log(__ddiv_rn(Iin, r.Iout)));
  else r.J = __dmul_rn(0.5, __dadd_rn(Iin, r.Iout));
  return r;
}

// ---- emission (DESIGN.md 4.6) -------------------------------------------------------------------------------------
// A segment of an emitting leaf (coefficient eta >= 0, units of uvb per cm) adds to the attenuated intensity
//   Iout = Iin e^-tau + eta t,   t = (1 - e^-tau) / kappa  if tau > (double)1.e-10f  else dpath
// (the reference's nemi slot with nemi = eta dpath, transportRoutinesModule.f90:673-678), and to its mean intensity
//   J_seg = L(Iin) + eta dpath phi(tau),   phi(tau) = (tau - 1 + e^-tau) / tau^2,  phi(0) = 1/2,
// L = what the mode computes for pure attenuation: the exact path average of Iin e^-kappa s + eta (1 - e^-kappa s) / kappa.
// Below kPhiSeries phi is its series (through tau^6: truncation < 3e-20), above it (tau - (1 - e^-tau)) / tau^2 from the
// exponential pieces the mode already has (relative rounding ~2e-16 / tau <= 2e-14).  An opacity of exactly 0 (or the
// FAST floor) gives exactly t = dpath and phi = 1/2.
constexpr double kPhiSeries = 1e-2;
__device__ __forceinline__ double emission_phi(double tau, double ome) {
  double s = fma(tau, 1. / 40320., -1. / 5040.);
  s = fma(s, tau, 1. / 720.);
  s = fma(s, tau, -1. / 120.);
  s = fma(s, tau, 1. / 24.);
  s = fma(s, tau, -1. / 6.);
  s = fma(s, tau, 0.5);
  return tau < kPhiSeries ? s : (tau - ome) / (tau * tau);
}
__device__ __forceinline__ double emission_t(double tau, double ome, double invk, double dpath) {
  return tau > (double)1.e-10f ? ome * invk : dpath;
}

// FAST-mode segment with emission: as segment_fast, plus E += phi(tau) * dw (dw = dpath * weight / nseg; the caller
// adds eta * E to the cell's sum once per layer) and the emitted part of Iout.  invk = 1 / kappa (kappa floored).
template <bool GUARD = true>
__device__ __forceinline__ double segment_fast_emit(double Iin, double tau, double cs, const double* __restrict__ T, double& A,
                                                    double eta, double invk, double d, double dw, double& E) {
  double Ts, p;
  exp_neg_parts32<GUARD>(tau, T, Ts, p);
  const double X = Iin * Ts;
  const double Iatt = fma(X, p, X);
  const double Z = fma(-X, p, Iin - X);
  if (!GUARD || ((__double2hiint(Iatt) << 1) | __double2loint(Iatt)) != 0) A = fma(Z, cs, A);
  const double ome = fma(-Ts, p, 1.0 - Ts);
  E = fma(emission_phi(tau, ome), dw, E);
  return fma(eta, emission_t(tau, ome, invk, d), Iatt);
}

// the outgoing intensity alone, bit for bit what segment_fast_emit returns for the same arguments
template <bool GUARD = true>
__device__ __forceinline__ double attenuate_fast_emit(double Iin, double tau, const double* __restrict__ T, double eta,
                                                      double invk, double d) {
  double Ts, p;
  exp_neg_parts32<GUARD>(tau, T, Ts, p);
  const double X = Iin * Ts;
  const double Iatt = fma(X, p, X);
  const double ome = fma(-Ts, p, 1.0 - Ts);
  return fma(eta, emission_t(tau, ome, invk, d), Iatt);
}

// FAITHFUL-mode segment with emission: L is segment_faithful's operation sequence on the attenuated part, the eta
// terms are one FMA each, so eta = 0 reproduces segment_faithful bit for bit
__device__ __forceinline__ SegResult segment_faithful_emit(double Iin, double kappa, double dpath, double eta) {
  SegResult r;
  const double tau = __dmul_rn(kappa, dpath);
  const double a = exp(-tau);
  const double Iatt = __dmul_rn(Iin, a);
  double L;
  if (Iatt < Iin) L = __ddiv_rn(__dsub_rn(Iin, Iatt), log(__ddiv_rn(Iin, Iatt)));
  else L = __dmul_rn(0.5, __dadd_rn(Iin, Iatt));
  const double ome = __dsub_rn(1.0, a);
  const double t = tau > (double)1.e-10f ? __ddiv_rn(ome, kappa) : dpath;
  double phi = 0.5;
  if (tau >= kPhiSeries) phi = __ddiv_rn(__dsub_rn(tau, ome), __dmul_rn(tau, tau));
  else phi = emission_phi(tau, ome);
  r.Iout = fma(eta, t, Iatt);
  r.J = fma(__dmul_rn(eta, dpath), phi, L);
  return r;
}
// the outgoing intensity alone (the recomputed upstream cell of the uniform sweep)
__device__ __forceinline__ double attenuate_faithful_emit(double Iin, double kappa, double dpath, double eta) {
  const double tau = __dmul_rn(kappa, dpath);
  const double a = exp(-tau);
  const double ome = __dsub_rn(1.0, a);
  const double t = tau > (double)1.e-10f ? __ddiv_rn(ome, kappa) : dpath;
  return fma(eta, t, __dmul_rn(Iin, a));
}

}  // namespace rtb
