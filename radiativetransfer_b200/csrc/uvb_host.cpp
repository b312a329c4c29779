// UV-background tables of the diffuse path (host side, a few hundred libm calls, once per run):
//   * band amplitudes uvb1..3 and the effective slopes alpha(3)      equiSources.f90:198-246, powerSpectrumIndex :4985-5043
//   * group cross-sections beta24..31, rate weights ksi24..31 and heating weights gammaHI/HeI/HeII of the three
//     frequency groups                                               uvbBetaTable.f90:31-296
//   * band-mean dust cross-sections of the groups with the same weights (an extension, DESIGN.md 4.8)
// They are what computeOpacities (equiSources.f90:4956-4983) and the diffuse photo-rates (:3546-3553) consume, i.e.
// the `beta[9]` / `ksi*` arguments of rtb200_diffuse* and rtb200_chemistry_device.
// Every Fortran real literal without a d-exponent is single precision and is widened where it meets a double; integer
// powers are repeated products; sums run in the reference's bin order.  Compiled with -ffp-contract=off.
#include <cmath>
#include <vector>

#include "../../include/rtb200.h"
#include "point_host.h"

namespace rtb {
namespace {

inline double w(float x) { return (double)x; }   // a single-precision literal widened to double
const double kNu[3] = {w(13.598f), w(24.587f), w(54.418f)};   // definitionsModule.f90:30-35: nu1, nu2, nu3 [eV]
const double kPiF = w(3.141592654f);                          // definitionsModule.f90:8
const double kEvToErg = 1.60217646e-12;                       // :36 (a true double)
const double kEvToHz = kEvToErg / w(6.6260693e-27f);          // :38 with hp of :15

inline double sq(double x) { return x * x; }
inline double cube(double x) { return x * x * x; }
inline double quart(double x) { const double y = x * x; return y * y; }

// hydrogen-like threshold cross-section (uvbBetaTable.f90:35-55): s0 (E0/E)^4 exp(4 - 4 atan(d)/d) / (1 - exp(-2 pi/d))
double hydrogenic(double s0, double e0, double e) {
  if (!(e > e0)) return 0.;
  const double d = std::sqrt(e / e0 - 1);
  return s0 * quart(e0 / e) * std::exp(4.0 - 4.0 * std::atan(d) / d) / (1 - std::exp(-2.0 * kPiF / d));
}

// the eight photo cross-sections of one energy bin in the order 24 (HI), 25 (HeII), 26 (HeI), 27 (H-), 28 (H2+),
// 29 (H2), 30 (H2+ -> 2H+), 31 (H2 Lyman-Werner): uvbBetaTable.f90:35-101
void cross_sections(double e, double s[8]) {
  s[0] = hydrogenic(w(6.3e-18f), kNu[0], e);
  s[1] = hydrogenic(w(1.58e-18f), kNu[2], e);
  s[2] = 0.;
  if (e > kNu[1]) {
    const double r = e / kNu[1];
    s[2] = w(7.42e-18f) * (w(1.66f) * std::pow(r, w(-2.05f)) - w(0.66f) * std::pow(r, w(-3.05f)));
  }
  const double e27 = w(0.755f), e28a = w(2.65f), e28b = w(11.27f), e28c = w(21.0f), e29a = w(15.42f), e29b = w(16.5f),
               e29c = w(17.7f), e30a = w(30.0f), e30b = w(70.0f);
  s[3] = e > e27 ? w(2.11e-16f) * std::pow(e - e27, 1.5) / cube(e) : 0.;
  if (e > e28a && e <= e28b) s[4] = std::pow(10.0, w(-40.97f) + w(6.03f) * e - w(0.504f) * sq(e) + w(1.387e-2f) * cube(e));
  else if (e > e28b && e < e28c) s[4] = std::pow(10.0, w(-30.26f) + w(2.79f) * e - w(0.184f) * sq(e) + w(3.535e-3f) * cube(e));
  else s[4] = 0.;
  if (e > e29a && e <= e29b) s[5] = w(6.2e-18f) * e - w(9.4e-17f);
  else if (e > e29b && e <= e29c) s[5] = w(1.4e-18f) * e - w(1.48e-17f);
  else if (e > e29c) s[5] = w(2.5e-14f) * std::pow(e, w(-2.71f));
  else s[5] = 0.;
  s[6] = (e >= e30a && e < e30b)
             ? std::pow(10.0, w(-16.926f) - w(4.528e-2f) * e + w(2.238e-4f) * sq(e) + w(4.245e-7f) * cube(e)) : 0.;
  s[7] = (e > e28b && e < kNu[0]) ? w(3.71e-18f) : 0.;
}

// band integral of a power law of slope a and amplitude u between nug and nugplus (or to infinity), as
// powerSpectrumIndex writes it (equiSources.f90:5000-5013)
double band(double u, double a, double ratio, bool bound) {
  return bound ? u / (a - 1.) * (1. - std::pow(ratio, a - 1.)) : u / (a - 1.);
}
bool opposite_signs(double a, double b) { return (a > 0. && b < 0.) || (a < 0. && b > 0.); }

// slope of the single power law whose band integral equals that of the two components (regula falsi with the
// reference's bracket and stopping rule, equiSources.f90:5006-5040)
int effective_slope(double u1, double a1, double u2, double a2, double nug, double nugplus, bool bound, double* total,
                    double* slope) {
  const double ratio = nug / nugplus;
  const double u = u1 + u2;
  const double target = band(u1, a1, ratio, bound) + band(u2, a2, ratio, bound);
  double lo = w(1.1f) * a1 - w(0.1f) * a2, hi = w(1.1f) * a2 - w(0.1f) * a1;
  double flo = band(u, lo, ratio, bound) - target, fhi = band(u, hi, ratio, bound) - target;
  if (!opposite_signs(flo, fhi)) return RTB200_ERR_ARG;   // 'wrong sign' ... stop (:5016-5019)
  double prev = lo, cur = hi;
  while (std::fabs(cur - prev) >= w(1e-8f)) {
    prev = cur;
    cur = (lo * std::fabs(fhi) + hi * std::fabs(flo)) / (std::fabs(flo) + std::fabs(fhi));
    const double fc = band(u, cur, ratio, bound) - target;
    if (opposite_signs(fc, flo)) { hi = cur; fhi = fc; }
    else { lo = cur; flo = fc; }
  }
  *total = u;
  *slope = cur;
  return RTB200_OK;
}

// the frequency groups' bins (uvbBetaTable.f90:171-257): [nu_g, nu_g+1] for groups 1, 2, from nu_3 on for group 3
bool in_band(int g, double freq) { return g < 2 ? (freq >= kNu[g] && freq <= kNu[g + 1]) : freq >= kNu[2]; }

// band integral of (e / nu_g)^-alpha_g in units of nu_g, the normalisation of beta24 (:259-293)
void band_shapes(const double* alpha, double shape[3]) {
  shape[0] = (1. - std::pow(kNu[1] / kNu[0], 1. - alpha[0])) / (alpha[0] - 1.);
  shape[1] = (1. - std::pow(kNu[2] / kNu[1], 1. - alpha[1])) / (alpha[1] - 1.);
  shape[2] = 1. / (alpha[2] - 1.);
}

}  // namespace
}  // namespace rtb

using namespace rtb;

extern "C" {

int rtb200_uvb_amplitudes(double currentRedshift, double uvbCoefficient, double* uvb, double* alpha) {
  if (!uvb || !alpha) return RTB200_ERR_ARG;
  const double z = currentRedshift;
  const double aQ = w(1.8f), aS = w(5.f);                         // alphaQuasar, alphaStellar (equiSources.f90:61-62)
  // Abel & Haehnelt 99 / Paschos 02 / Razoumov 02 components, equiSources.f90:198-225
  const double damp = 1. + quart(7. / (1. + z));
  const double stellar99 = 1. / damp * std::exp(-cube(z / 4.));
  const double pascal02 = w(0.0188f) * std::exp(-sq(z - 0.5) / (1. + w(0.0625f) * std::pow(z + w(2.09f), w(2.075f)))) *
                          std::pow(1. + z, w(3.35f));
  const double s1 = 0.5 * (std::tanh((z - w(4.2f)) * 1.5) + 1.);
  const double stellar02 = (1. - s1) * stellar99 + s1 * pascal02;
  const double quasar02 = 10. / damp * std::exp(-cube(z / 2.5));
  const double gaussian = std::exp(-sq((z - 4.5) / 2.)) * w(0.3f);
  const double newQuasar = gaussian * stellar02 + (1. - gaussian) * quasar02;
  double newStellar = (1. - gaussian) * stellar02 + gaussian * quasar02;
  const double s2 = 0.5 * (std::tanh((z - 14.) * 0.5) + 1.);
  newStellar = s2 * 0. + (1. - s2) * newStellar;
  // band amplitudes of the two components (:236-242; contributionStellar = contributionQuasar = 1)
  double st[3], qs[3];
  st[0] = newStellar * 1.e-21 * 1. * uvbCoefficient;
  qs[0] = newQuasar * 1.e-21 * 1. * uvbCoefficient;
  for (int g = 1; g < 3; g++) {
    st[g] = st[g - 1] * std::pow(kNu[g] / kNu[g - 1], -aS);
    qs[g] = qs[g - 1] * std::pow(kNu[g] / kNu[g - 1], -aQ);
  }
  for (int g = 0; g < 3; g++) {                                     // :244-246
    const bool bound = g < 2;
    if (int e = effective_slope(st[g], aS, qs[g], aQ, kNu[g], bound ? kNu[g + 1] : kNu[g], bound, &uvb[g], &alpha[g]))
      return e;
  }
  return RTB200_OK;
}

int rtb200_uvb_beta_table(int nfreq, double freqdel, const double* alpha, double* table57) {
  if (nfreq < 2 || !alpha || !table57) return RTB200_ERR_ARG;
  std::vector<double> e((size_t)nfreq), sig((size_t)nfreq * 8);
  for (int i = 0; i < nfreq; i++) {
    e[i] = std::pow(10.0, (double)i * freqdel);                     // uvbBetaTable.f90:33
    cross_sections(e[i], &sig[(size_t)i * 8]);
  }
  for (int i = 0; i < 57; i++) table57[i] = 0.;
  for (int i = 1; i < nfreq; i++) {                                 // :171-257 (do i = 2, nfreq)
    const double freq = e[i], dnu = e[i] - e[i - 1];
    const double* s = &sig[(size_t)i * 8];
    for (int g = 0; g < 3; g++) {
      if (!in_band(g, freq)) continue;
      double* G = table57 + 19 * g;
      const double dt = std::pow(freq / kNu[g], -alpha[g]) * dnu;
      const double dtE = dt * kEvToHz / (freq * kEvToErg);
      for (int k = 0; k < 8; k++) {
        G[k] = G[k] + dt * s[k];
        G[8 + k] = G[8 + k] + dtE * s[k];
      }
      // heating weights: HI in every group, HeI from group 2, HeII in group 3 (:199, :225-226, :252-254)
      G[16] = G[16] + dtE * (freq - kNu[0]) * kEvToErg * s[0];
      if (g >= 1) G[17] = G[17] + dtE * (freq - kNu[1]) * kEvToErg * s[2];
      if (g == 2) G[18] = G[18] + dtE * (freq - kNu[2]) * kEvToErg * s[1];
    }
  }
  double shape[3];
  band_shapes(alpha, shape);
  for (int g = 0; g < 3; g++) {                                     // :259-293
    const double energyShape = shape[g] * kNu[g];
    for (int k = 0; k < 8; k++) table57[19 * g + k] = table57[19 * g + k] / energyShape;
  }
  return RTB200_OK;
}

int rtb200_uvb_dust_beta(int nfreq, double freqdel, const double* alpha, const double* aDust, double* betaDust3) {
  if (nfreq < 2 || !alpha || !aDust || !betaDust3) return RTB200_ERR_ARG;
  const double clight = w(2.99792458e10f);
  double G[3] = {0., 0., 0.};
  double prev = 1.;                                                 // e_0 = 10^0
  for (int i = 1; i < nfreq; i++) {                                 // the bins and weights of beta24 above
    const double freq = std::pow(10.0, (double)i * freqdel), dnu = freq - prev;
    prev = freq;
    // the dust cross-section as point_frequency_tables evaluates it: wavelength in A, the fit in micron
    const double lambda = clight / (freq * kEvToHz) * w(1.e8f);
    const double sD = smc_dust_sigma(lambda / w(1.e4f), aDust) * w(1.e-22f);
    for (int g = 0; g < 3; g++) {
      if (!in_band(g, freq)) continue;
      const double dt = std::pow(freq / kNu[g], -alpha[g]) * dnu;
      G[g] = G[g] + dt * sD;
    }
  }
  double shape[3];
  band_shapes(alpha, shape);
  for (int g = 0; g < 3; g++) betaDust3[g] = G[g] / (shape[g] * kNu[g]);
  return RTB200_OK;
}

int rtb200_uvb_background(double currentRedshift, double uvbCoefficient, int nfreq, double freqdel, double* uvb,
                          double* alpha, double* beta, double* ksi24, double* ksi25, double* ksi26, double* table57) {
  double a[3], u[3], t[57];
  if (int st = rtb200_uvb_amplitudes(currentRedshift, uvbCoefficient, u, a)) return st;
  if (int st = rtb200_uvb_beta_table(nfreq, freqdel, a, t)) return st;
  for (int g = 0; g < 3; g++) {
    if (uvb) uvb[g] = u[g];
    if (alpha) alpha[g] = a[g];
    if (beta) {   // [group][beta24, beta26, beta25]: the order computeOpacities reads them (equiSources.f90:4974-4977)
      beta[3 * g] = t[19 * g]; beta[3 * g + 1] = t[19 * g + 2]; beta[3 * g + 2] = t[19 * g + 1];
    }
    if (ksi24) ksi24[g] = t[19 * g + 8];
  }
  if (ksi25) ksi25[0] = t[38 + 9];                                  // group3%ksi25 (:3550)
  if (ksi26) { ksi26[0] = t[19 + 10]; ksi26[1] = t[38 + 10]; }      // group2%ksi26, group3%ksi26 (:3552-3553)
  if (table57)
    for (int i = 0; i < 57; i++) table57[i] = t[i];
  return RTB200_OK;
}

}  // extern "C"
