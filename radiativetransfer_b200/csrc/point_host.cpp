// Host-side tables of the point-source path (glibc libm, no FMA contraction, the reference's single-precision
// literals): frequency grid and cross-section ratios, dust cross-section, per-source photon spectrum, split radii,
// HEALPix pixel directions.  Replaces stellarBetaTable.f90:31-152, stellarPopulationModule.f90:7-50,
// dustModule.f90:30-73, equiSources.f90:304-309 and the pixel-angle cache of equiSources.f90:1301-1318, 3294-3314.
// Everything here is O(400) or O(16380) work per call; the 400 x 11^4 table sums and the ray march run on the GPU.
#include "point_host.h"

#include <algorithm>
#include <cmath>

#include "geometry.h"

namespace rtb {

static const double kHp = (double)6.6260693e-27f, kClight = (double)2.99792458e10f, kAngstrom = (double)1.e-8f;
static const double kEvToErg = 1.60217646e-12, kEvToHz = kEvToErg / kHp;
static const double kNu[3] = {(double)13.598f, (double)24.587f, (double)54.418f};  // HI, HeI, HeII thresholds [eV]

double smc_dust_sigma(double lambdaMicron, const double* a) {  // dustModule.f90:36-50, 7-term fit
  double sum = 0;
  for (int t = 0; t < 7; t++) {
    const double* row = a + 5 * t;
    double x = lambdaMicron / row[0];
    sum = sum + row[1] / (std::pow(x, row[3]) + std::pow(x, -row[4]) + row[2]);
  }
  return (double)1.1f * sum * (double)0.9210340372f;
}

static inline double sq2(double x) { double y = x * x; return y * y; }

static double sigma_hydrogenic(double nu, double thr, double s0) {  // stellarBetaTable.f90:31-49
  double dum = std::sqrt(nu / thr - 1);
  return s0 * sq2(thr / nu) * std::exp(4.0 - 4.0 * std::atan(dum) / dum) / (1 - std::exp(-2.0 * kPi / dum));
}

static double sigma_hei(double nu) {  // stellarBetaTable.f90:51-60
  const double t = kNu[1];
  return (double)7.42e-18f * ((double)1.66f * std::pow(nu / t, (double)(-2.05f)) - (double)0.66f * std::pow(nu / t, (double)(-3.05f)));
}

void point_frequency_tables(const double* aDust, PointFreq& F) {
  const double freqdel = (double)0.02f;
  for (int i = 0; i < kNfreq; i++) {
    double nu = std::pow(10.0, (double)i * freqdel);
    F.nu[i] = nu;
    double lambda = kClight / (nu * kEvToHz) * (double)1.e8f;
    double sD = smc_dust_sigma(lambda / (double)1.e4f, aDust) * (double)1.e-22f;
    double s24 = nu > kNu[0] ? sigma_hydrogenic(nu, kNu[0], (double)6.3e-18f) : 0.;
    double s25 = nu > kNu[2] ? sigma_hydrogenic(nu, kNu[2], (double)1.58e-18f) : 0.;
    double s26 = nu > kNu[1] ? sigma_hei(nu) : 0.;
    // the ratios the table loop multiplies the depth grid with (stellarBetaTable.f90:246-250)
    F.r24[i] = s24 / (double)6.3e-18f;
    F.r26[i] = s26 / (double)7.42e-18f;
    F.r25[i] = s25 / (double)1.58e-18f;
    F.rD[i] = sD / (double)5.4116737e-22f;
  }
  const double lo = kNu[0], hi = 10. * kNu[0];
  for (int e = 0; e < kNenergy; e++) {  // stellarBetaTable.f90:119-152
    double freq = lo * std::exp((double)((float)e / (float)(kNenergy - 1)) * (std::log(hi) - std::log(lo)));
    double lambda = kClight / (freq * kEvToHz) * (double)1.e8f;
    double sD = smc_dust_sigma(lambda / (double)1.e4f, aDust) * (double)1.e-22f;
    double s24 = freq > kNu[0] ? sigma_hydrogenic(freq, kNu[0], (double)6.3e-18f) : (freq == kNu[0] ? (double)6.3e-18f : 0.);
    double s25 = freq > kNu[2] ? sigma_hydrogenic(freq, kNu[2], (double)1.58e-18f) : 0.;
    double s26 = freq > kNu[1] ? sigma_hei(freq) : 0.;
    // startNewLongRay divides by the threshold cross-sections again (equiSources.f90:3216-3219)
    F.out24[e] = s24 / (double)6.30e-18f;
    F.out26[e] = s26 / (double)7.42e-18f;
    F.out25[e] = s25 / (double)1.58e-18f;
    F.outD[e] = sD / (double)5.4116737e-22f;
  }
}

// photons per second in frequency bin i (i = 1..399; bin 0 is unused): stellarBetaTable.f90:224-229 with the
// tri-linear spectrum lookup of stellarPopulationModule.f90:7-50
void point_source_spectrum(const PointFreq& F, int nWave, const double* wavelength, const double* lum,
                           double coefSpectrum, int iMetal, double coefMetal, double* dtmp) {
  dtmp[0] = 0.;
  for (int i = 1; i < kNfreq; i++) {
    const double freq = F.nu[i], dnu = F.nu[i] - F.nu[i - 1];
    const double wl = kClight / (freq * kEvToHz);
    // 0-based index of the bracket's lower edge: the reference scans `while (wl > wavelength(w+1)) w++` from the
    // first entry; the table ascends, so that is the first entry from the second on that is not below wl
    int w = (int)(std::lower_bound(wavelength + 1, wavelength + nWave, wl) - (wavelength + 1));
    if (w > nWave - 2) w = nWave - 2;   // (the reference would run off the table)
    double cw = (wl - wavelength[w]) / (wavelength[w + 1] - wavelength[w]);
    cw = std::fmin(std::fmax(0., cw), 1.);
    auto L = [&](int m, int t, int k) { return lum[((size_t)m * 2 + t) * nWave + k]; };
    const int m = iMetal - 1;
    double a = coefSpectrum * ((1. - cw) * L(m, 1, w) + cw * 1. * L(m, 1, w + 1)) +
               (1. - coefSpectrum) * ((1. - cw) * L(m, 0, w) + cw * L(m, 0, w + 1));
    double b = coefSpectrum * ((1. - cw) * L(m + 1, 1, w) + cw * 1. * L(m + 1, 1, w + 1)) +
               (1. - coefSpectrum) * ((1. - cw) * L(m + 1, 0, w) + cw * L(m + 1, 0, w + 1));
    double sp = (1. - coefMetal) * a + coefMetal * b;
    double fh = freq * kEvToHz;
    double lnu = std::pow(10., sp) / kAngstrom * kClight / (fh * fh);
    dtmp[i] = lnu / (freq * kEvToErg) * dnu * kEvToHz;
  }
}

// metallicity bracket of a source's host cell (equiSources.f90:1282-1293)
void point_metal_bracket(double abun2, const double* metallicity, int* iMetal, double* coefMetal) {
  double t = abun2 > (double)1.e-20f ? std::log10(abun2) : -20.;
  int m = 1;
  while (t > metallicity[m]) {
    m++;
    if (m + 1 == 5) break;
  }
  double c = (t - metallicity[m - 1]) / (metallicity[m] - metallicity[m - 1]);
  *iMetal = m;
  *coefMetal = std::fmin(std::fmax(0., c), 1.);
}

void point_split_radii(double* rmax /* [31], index = pixel level */) {  // equiSources.f90:304-309
  rmax[0] = 0.;
  for (int ir = 1; ir <= 30; ir++) {
    float v = std::sqrt(3.f) * (std::sqrt(0.5f * std::pow(4.f, (float)(ir - 1)) - 1.f / 12.f) + 0.5f);
    rmax[ir] = (double)v / 2.;
  }
}

// unit vectors of every HEALPix pixel of levels 1..maxLevel, nested order, level L starting at 12*(4^(L-1)-1)/3
int point_pixel_directions(int maxLevel, std::vector<double>& dirs /* [npix][3]: prox, proy, proz */) {
  int64_t total = 0;
  for (int L = 1; L <= maxLevel; L++) total += 12LL << (2 * (L - 1));
  dirs.resize((size_t)total * 3);
  int64_t o = 0;
  for (int L = 1; L <= maxLevel; L++) {
    const int64_t np = 12LL << (2 * (L - 1));
    for (int64_t p = 0; p < np; p++, o++) {
      double phi, theta;
      int st = healpix_center(1 << (L - 1), p, &phi, &theta);
      if (st) return st;
      dirs[3 * o] = std::cos(phi) * std::cos(theta);      // equiSources.f90:2440-2442
      dirs[3 * o + 1] = std::sin(phi) * std::cos(theta);
      dirs[3 * o + 2] = std::sin(theta);
    }
  }
  return 0;
}

}  // namespace rtb
