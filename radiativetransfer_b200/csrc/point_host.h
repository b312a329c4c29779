// Host-side tables of the point-source path (see point_host.cpp).
#pragma once
#include <cstdint>
#include <vector>

namespace rtb {

constexpr int kNfreq = 400;    // nfbins (definitionsModule.f90:239)
constexpr int kNenergy = 300;  // nenergy (definitionsModule.f90:291)
constexpr int kNdepth = 10;    // ndepth1..3, ndepthDust (definitionsModule.f90:72)
constexpr int kTableEntries = 11 * 11 * 11 * 11;

struct PointFreq {
  double nu[kNfreq];                                        // bin energies [eV]
  double r24[kNfreq], r26[kNfreq], r25[kNfreq], rD[kNfreq]; // sigma(nu) / sigma(threshold)
  double out24[kNenergy], out26[kNenergy], out25[kNenergy], outD[kNenergy];  // same ratios on the 300 output energies
};

// dust cross-section of the 7-term extinction fit a[7][5] at lambdaMicron, in units of 1e-22 cm^2 (dustModule.f90:36-50)
double smc_dust_sigma(double lambdaMicron, const double* a);
void point_frequency_tables(const double* aDust, PointFreq& F);
void point_source_spectrum(const PointFreq& F, int nWave, const double* wavelength, const double* lum,
                           double coefSpectrum, int iMetal, double coefMetal, double* dtmp);
void point_metal_bracket(double abun2, const double* metallicity, int* iMetal, double* coefMetal);
void point_split_radii(double* rmax);
int point_pixel_directions(int maxLevel, std::vector<double>& dirs);

}  // namespace rtb
