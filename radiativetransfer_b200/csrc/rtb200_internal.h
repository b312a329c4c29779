// Internal declarations shared by the C-ABI (api.cu) and the kernel translation units.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <functional>
#include <string>
#include <vector>

#include "../../include/rtb200.h"
#include "geometry.h"

namespace rtb {

#define RTB_CUDA(call)                                                              \
  do {                                                                              \
    cudaError_t e_ = (call);                                                        \
    if (e_ != cudaSuccess) {                                                        \
      rtb::set_cuda_error(#call, e_, __FILE__, __LINE__);                           \
      return RTB200_ERR_CUDA;                                                       \
    }                                                                               \
  } while (0)

void set_cuda_error(const char* what, cudaError_t e, const char* file, int line);
const char* last_cuda_error();

// ------------------------------------------------------------------------------------------------
// Device tables of the uniform-grid sweep
// ------------------------------------------------------------------------------------------------
// One layer of one direction, in CHAIN order: a characteristic entering the layer through the bottom face
// crosses 1..3 cells (segments 0,1,2) before it leaves through the top (SURVEY.md appendix A).
//   kind 0: xy                      kind 1: xy -> yz            kind 2: xy -> yz -> xz
//   kind 3: xy -> xz                kind 4: xy -> xz -> yz
// The second segment of kinds 1,2 (a yz ray) is fed by the cell at k-1, of kinds 3,4 (an xz ray) by the cell at
// j-1; the third segment by the other one.
struct LayerSeg {
  double d[3];     // path length [cm]: cellSize * len (a FAST launch of the plain uniform sweep reads d * kExpScale
                   // in non-thin layers: diffuse_uniform.cu, fill_step_segs)
  double cs[3];    // fast mode: 2^200 * (weight / nseg) / d   (segment_math.cuh, segment_fast)
  double dmax;     // longest segment of the layer [cm] (fast mode: decides whether the overflow guards can be skipped)
  double w;        // weight          (faithful mode divides by nseg first, transportRoutinesModule.f90:953)
  int32_t kind;
  int32_t nseg;
  int32_t thin;    // an active segment is shorter than 1e-2 cell: evaluate this layer with the reference's operation sequence
  int32_t pad;
};
static_assert(sizeof(LayerSeg) == 80, "LayerSeg layout");

constexpr int kMaxDirPerTask = 8;   // (12 = one task per zone at nAngularLevel = 3 measured no faster: r02f, fewer and longer blocks)

// One task = up to kMaxDirPerTask directions of one zone (same index rotation), swept together layer by layer so
// that kappa is read once and J is accumulated in registers across the directions.
struct UniTaskHost {
  int64_t origin = 0, si = 0, sj = 0, sk = 0;  // leaf index = origin + i*si + j*sj + k*sk (0-based rotated indices)
  int ndir = 0;
  int izone = 0;
  int laneIsK = 1;       // 1: threadIdx.x runs along rotated k, 0: along rotated j
  int slot = 0;          // J accumulator / stream this task uses
  int firstInSlot = 0;   // 1: overwrite the accumulator instead of adding
  int planeFirst = 0;    // index of the task's first direction in the plane buffers
  int transposed = 0;    // 1: this task reads kappa / writes its accumulator in the z-major layout (see diffuse_uniform.cu)
  std::vector<LayerSeg> seg;  // [n layers][kMaxDirPerTask]
};

struct Tuning {
  int slots = 0;         // uniform sweep: zone tasks per launch, each with its own J accumulator (0 = 40, the most a launch takes)
  int useGraph = 1;
  int forceAmr = 0;      // route uniform grids through the general (AMR) path as well (cross-check)
  int amrSlots = 1;      // nested grids: per-item arrays indexed by the leaf's position in the wave order (1) or by leaf number (0)
  int amrMinBlocks = 0;  // nested grids, FAST arithmetic: blocks of 128 threads per SM the wave kernel's register cap allows (8: 64,
                         // 6: 80 registers; 0 = 6 for small waves, 8 for large ones)
  int amrStream = -1;    // nested grids, 2:1 balanced: the whole sweep as one launch ordered by the records' sign epoch (1), one launch
                         // per wave (0), or by the size of the waves (-1)
  int amrOrder = -1;     // nested grids, waves of the sweep: centre-sum key (0), depth in the dependency graph (1), or the key on
                         // 2:1-balanced grids and the depth elsewhere (-1)
  int amrThin = 1;       // nested grids, FAST arithmetic: thin layers use the reference's operation sequence (1)
  int amrBatch = 0;      // directions per AMR batch (0 = as many as fit in half of the free memory)
  double l2BudgetMB = 96.0;
  int pdl = 1;           // uniform sweep: programmatic dependent launch of layer l+1 on layer l (its prologue overlaps the tail)
  int blockWarps = 0;    // uniform sweep: warps per block: 8, 4, 2, or 0 = chosen from the number of blocks per launch
  int cells = 0;         // uniform sweep, FAST arithmetic: cells of a layer per thread (2: two rows per warp, see
                         // sweep_cell2_kernel; 0 = 2 from n = 192 on, where it measured 1-2% faster, else 1: 6% faster at 128^3)
  int transposeZ = 1;    // uniform sweep: zones sweeping along the contiguous axis use a z-major copy of kappa / J
  int dirsPerTask = 0;   // directions of one zone swept together (0 = kMaxDirPerTask)
  int portableMath = 1;  // point path, FAITHFUL mode: exp/log from portable_math.h (bit-identical on host and device)
  int pointDeposit = 2;  // point path: 0 = fp64 RED.ADD into the rate fields, 1 = atomic-free: (leaf, deposit) records,
                         // radix sort by (leaf, ray, segment), one thread per cell adds its run (deterministic order),
                         // 2 = planned: as 1, but the sort is done once per (grid, sources) and every later pass writes
                         // its deposits to their cached leaf-ordered slots (falls back to 1 with dust)
  long long pointRecordCap = 0;  // upper limit of the record buffer of mode 1 (0 = 60% of the free memory)
  int pointRefill = 0;   // point path, last pixel level: 1 = lanes take further rays from a per-source queue (fuller warps but
  int pointMinBlocks = 5;  // point march kernel (FAST, RED deposition): blocks of 128 threads per SM the register cap allows (5: 96 registers)
                         // incoherent gathers: measured slower, DESIGN.md 4.3)
  int pointBatch = 0;    // sources per batch of the point path (0 = as many as fit in half of the free memory)
};

// inputs of the point-source pass (equiSources.f90:1256-1370); none of the reference's data files ship with it, so
// the population-synthesis spectra and the dust fit parameters are arguments
struct PointInputs {
  int nWave = 0;
  const double* wavelength = nullptr;   // [nWave] cm, increasing
  const double* lum = nullptr;          // [5][2][nWave] log10(erg/s/A): metallicity x (iSpectrum, iSpectrum+1)
  const double* metallicity = nullptr;  // [5] log10 Z
  double coefSpectrum = 0;
  const double* aDust = nullptr;        // [7][5]
  int dust = 0, maxPixelLevel = 6, nsrc = 0;
  const int32_t* srcLeaf = nullptr;
  const int32_t* srcWeight = nullptr;
  int forceMetal = 0;                   // != 0: use (forceMetal, forceCoefMetal) instead of the host cell's bracket
  double forceCoefMetal = 0;
};

// ------------------------------------------------------------------------------------------------
// AMR tables
// ------------------------------------------------------------------------------------------------
struct DevTree {
  int32_t* child = nullptr;      // [nnodes] >=0: first of 8 children (x slowest, z fastest); <0: -(leaf+1)
  int32_t* leafX = nullptr;      // [nleaf] integer coordinates at the leaf's own level
  int32_t* leafY = nullptr;
  int32_t* leafZ = nullptr;
  int64_t nnodes = 0;
};

struct Context {
  int device = 0;
  int mathMode = RTB200_MATH_FAST;
  Tuning tune;
  cudaStream_t stream = nullptr;  // internal stream for host-buffer calls
  cudaEvent_t evStart = nullptr, evStop = nullptr, evSweep0 = nullptr, evSweep1 = nullptr;
  int smCount = 148;
  size_t l2Bytes = 0;

  // grid
  int nx = 0;
  int64_t nleaf = 0;
  int maxLevel = 0;
  double boxSize = 0;
  bool uniform = true;
  std::vector<int8_t> hLevel;
  int64_t padLeaves = 0;      // extra entries allocated behind every species array (multi-GPU: slabs of equal size)
  int8_t* dLevel = nullptr;
  double *dHI = nullptr, *dHeI = nullptr, *dHeII = nullptr, *dRho = nullptr, *dAbun2 = nullptr;
  // chemistry (solveRateEquations): rate-coefficient tables and log(tgas) per leaf
  double* dChemK = nullptr;  // [6][nratec]
  int chemNratec = 0;
  double chemLogtem0 = 0, chemLogtem9 = 0, chemDlogtem = 0;
  double* dLogT = nullptr;   // [nleaf]
  double* dMassPart = nullptr;  // computeMass partial sums
  double* dKappa = nullptr;  // [3][nleaf]
  double* dKappaT = nullptr; // [3][nleaf] z-major copy (index (z*n + x)*n + y) for the uniform sweep, lazily allocated
  size_t kappaTBytes = 0;
  // emission coefficient per leaf and frequency group (rtb200_grid_set_emission): [3][nleaf], nullptr = no emission
  double* dEta = nullptr;
  double* dEtaT = nullptr;   // z-major copy of dEta for the uniform sweep (like dKappaT), lazily allocated
  size_t etaTBytes = 0;
  // isotropic scattering (rtb200_grid_set_scattering, scattering.cu): sigma [3][nleaf], nullptr = no scattering.  While
  // it is set the sweeps read dEtaEff = eta_th + sigma * J of the previous iteration, one fixed buffer, so that the
  // uniform plan and the captured graph stay valid across the iterations and the calls
  double* dSigma = nullptr;
  double* dEtaEff = nullptr;
  double* dScatScratch = nullptr;   // scratch of the source iteration, laid out by source_scratch (lazily allocated)
  size_t scatScratchBytes = 0;
  int32_t scatMaxIter = 1;
  double scatTol = 0;
  int32_t lastScatIter = 0;         // sweeps and last residual of the latest diffuse call
  double lastScatResid = 0;
  // tolerance 0: the residual is still on the device, as the max of these words (the context's own residual word, or
  // every rank's in a device group), read by last_scattering
  const double* dScatResid = nullptr;
  int nScatResid = 0;
  // acceleration of the source iteration (rtb200_grid_set_scattering_acceleration, ng.cu): RTB200_SCATTER_* flags
  int32_t scatAccel = 0;
  bool scatWarm = false;            // the J of the previous iteration (Jprev) is the J the latest completed solve returned
  double* dNg = nullptr;            // Ng history and sums (ng_buffers), allocated while the NG flag is set and a solve runs
  size_t ngBytes = 0;
  int32_t lastNgCount = 0;          // extrapolations applied by the latest diffuse call (on the device while ngPending)
  bool lastWarm = false, ngPending = false;
  const int32_t* dWarmTaken = nullptr;   // device group: the device's word saying whether the latest call started warm
  // dust (rtb200_grid_set_dust, dust.cu): mode 0 = none.  compute_opacities_dust_kernel adds kd to the opacities of every
  // call and, while an albedo is > 0, writes the scattering source albedo * kd into dDustSigma [3][nleaf]
  int dustMode = 0;
  double dustBeta[3] = {0, 0, 0}, dustAlbedo[3] = {0, 0, 0};
  double* dDustSigma = nullptr;     // allocated while dust scatters
  // the scattering coefficient of the source iteration: the per-leaf sigma or the dust's (nullptr: no scattering)
  const double* scatterSigma() const { return dSigma ? dSigma : dDustSigma; }
  // the source the sweeps read: the effective one while the context scatters, else the emission (nullptr: none)
  const double* sweepEta() const { return scatterSigma() ? dEtaEff : dEta; }
  // photo-heating and dust absorption (rtb200_grid_set_heating, heating.cu): while dHeat is set, every diffuse call ends
  // with one pass over the J it returns into dHeat [5][heatStride] (nleaf, or the slab of a device-group member)
  double heatGamma[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};   // [group][gammaHI, gammaHeI, gammaHeII]
  double heatWidth[3] = {0, 0, 0};                    // band widths [Hz]
  double* dHeat = nullptr;
  int64_t heatStride = 0;
  bool heatValid = false;   // dHeat holds the fields of a diffuse call that completed since the setting or the grid changed
  int uniStdSlots = 0;      // slots [0, uniStdSlots) are in leaf order, the rest z-major
  DevTree tree;
  std::vector<int32_t> hChild;               // host copy of the linear octree
  std::vector<int32_t> hLeafX, hLeafY, hLeafZ;
  // per physical axis and level: which layers contain a refined cell (pattern sub-tree exists there)
  std::vector<std::vector<uint8_t>> refinedLayer[3];

  // scratch owned by the diffuse paths (sized lazily, reused across calls)
  double* dJ = nullptr;        // [3][nleaf] result buffer for the host-pointer API
  double* dRates = nullptr;    // [6][nleaf] rate buffer of the host-pointer point-source API (lazy)
  // scratch of the point-source path, kept between calls (request i of a call reuses slot i; freed with the grid)
  std::vector<std::pair<void*, size_t>> pointPool;
  std::vector<double> pointDirs;   // HEALPix pixel directions of levels 1..pointDirsLevel (host copy)
  int pointDirsLevel = 0;
  void* pointPlan = nullptr; // point_source.cu: cached ray geometry of the planned deposition (point_release frees it)
  void* amrState = nullptr;  // diffuse_amr.cu: wave plan, pattern tables and batch buffers of this context (amr_release frees it)
  double* dAcc = nullptr;      // slot accumulators
  size_t accBytes = 0;
  double* dPlanes = nullptr;   // ping-pong top-exit planes
  size_t planeBytes = 0;
  void* dAmrScratch = nullptr;
  size_t amrScratchBytes = 0;
  int32_t* dErr = nullptr;     // device error flag
  double* hPinned = nullptr;   // pinned staging for host-pointer results
  size_t pinnedBytes = 0;

  // graph cache for the uniform sweep
  cudaGraphExec_t graphExec = nullptr;
  std::string graphKey;
  // cached plan of the uniform sweep (pattern tables, zone tasks): valid while uniPlanKey matches
  std::string uniPlanKey;
  int uniSlots = 0;
  std::vector<UniTaskHost> uniTasks;
  int64_t uniNseg = 0, uniLaunches = 0;
  int uniResidentWarps[5] = {0, 0, 0, 0, 0};  // resident warps per SM of each uniform sweep kernel (diffuse_uniform.cu)
  std::string amrPlanKey;
  bool statsPending = false, sweepTimed = false;

  // stats of the last call
  double lastMs = 0, lastSweepMs = 0;
  int64_t lastSweepLaunches = 0;
  int64_t lastLaunches = 0;
  double lastAlgBytes = 0;
};

// an entry of a per-leaf field the library accepts (emission, sigma, dust cross-sections): >= 0 and finite
__host__ __device__ inline bool finite_nonneg(double v) { return v >= 0. && v <= 1.7976931348623157e308; }

int ensure_buffer(void** p, size_t* have, size_t need);
int context_init(Context& c, int device);
void context_destroy(Context& c);
int grid_set(Context& c, int nx, int64_t nleaf, const int8_t* level, const double* HI, const double* HeI, const double* HeII,
             const double* rho, const double* abun2, double physicalBoxSize);
int set_tuning(Context& c, const char* key, double value);
// emission: eta = host [3][nleaf] (nullptr clears), or a device array on stream s (device = true); negative, NaN or
// Inf entries are refused with RTB200_ERR_ARG and leave the previous emission in place
int set_emission(Context& c, const double* eta, bool device, cudaStream_t s);
// per-leaf field of the 3 groups, [3][nleaf] on the host or (device = true) on the device on stream s: checked (>= 0,
// finite) and copied into a fresh buffer that replaces *field only on success (set_emission, set_scattering)
int replace_leaf_field(Context& c, double** field, const double* src, bool device, cudaStream_t s);
// forget the uniform plan and the captured graph (they know which source the sweeps read)
void drop_sweep_plans(Context& c);
// scattering: sigma = host [3][nleaf] (nullptr clears), or a device array (device = true, device groups) on c.stream
int set_scattering(Context& c, const double* sigma, bool device, int32_t maxIterations, double tolerance);
// the diffuse call: one sweep, or the source iteration while scattering is set (a direction subset is refused then)
int run_diffuse(Context& c, int nAngularLevel, const double* uvb, const double* beta, const int32_t* rays, int32_t nrays,
                double* dJ, cudaStream_t s, int64_t* nseg);
// forget the scattering results of the previous diffuse call (every diffuse call starts with it)
void reset_call_results(Context& c);
// one sweep of the given directions with the context's current source.  iter <= 1: opacities first (+ sigma while
// scattering is set) and the call's timing starts; iter > 1: stats add up to the earlier sweeps of the call
int run_sweep(Context& c, int nAngularLevel, const double* uvb, const double* beta, const int32_t* rays, int32_t nrays,
              double* dJ, cudaStream_t s, int64_t* nseg, int iter);
// scattering.cu: source iteration of a single context over the full direction set
int scatter_solve(Context& c, int nAngularLevel, const double* uvb, const double* beta, double* dJ, cudaStream_t s,
                  int64_t* nseg);
// The part of the grid a context iterates and the exchanges around it: the whole grid for a single context (stageStride
// 0, hooks empty), a slab for a member of a device group.  source_iteration (scattering.cu) is the one loop for both.
struct SourcePart {
  int rank = 0, nranks = 1;
  int64_t off = 0, cnt = 0;      // leaves [off, off + cnt): sigma and eta_th are read at + off
  double* J = nullptr;           // y_k after sweep(k), [3][jStride]; Jprev and the Ng history use the same stride
  int64_t jStride = 0;
  std::function<int(int k, int64_t* ns)> sweep;   // sweep k with the current dEtaEff, its result in J
  // a member of a device group: the source pass writes this rank's slice (at rank * jStride) of a stage [3][stageStride]
  // instead of dEtaEff, share_source all-gathers the stage into every rank's dEtaEff, and allgather gathers every
  // rank's n words at words + n * rank into every rank's words, in place
  int64_t stageStride = 0;
  std::function<int(double* stage)> share_source;
  std::function<int(double* words, int n)> allgather;
};
int source_iteration(Context& c, const SourcePart& p, const double* beta, cudaStream_t s, int* iters, int64_t* nseg);
// frees dEtaEff, the scratch and the Ng history and drops the stored J; results the latest call left on the device are
// read first (scattering cleared, grid replaced)
void release_source_iteration(Context& c);
// eta_out[g * oStride + i] = eta_th + sigma * J, Jprev = J and the residual max |J - Jprev| / J folded into *resid (the
// bits of a non-negative double) for i < cnt, g < 3; J and Jprev with stride jStride, sigma / eta_th (may be nullptr)
// with stride sStride
int launch_scatter_source(const Context& c, int64_t cnt, const double* J, double* Jprev, int64_t jStride, const double* sigma,
                          const double* etaTh, int64_t sStride, double* etaOut, int64_t oStride, unsigned long long* resid,
                          cudaStream_t s);
int launch_add_scattering(Context& c, cudaStream_t s);
// dust.cu: dust (mode 0 clears; albedo may make it scatter) and the opacities with dust, in place of
// launch_compute_opacities while a mode is set
int set_dust(Context& c, int mode, const double* betaDust, const double* albedo, int32_t maxIterations, double tolerance);
// the argument checks of set_dust that need no context (the device group runs them once for all members)
bool dust_args_ok(int mode, const double* betaDust, const double* albedo, int32_t maxIterations, double tolerance);
int launch_compute_opacities_dust(Context& c, const double* beta, cudaStream_t s);
int last_scattering(Context& c, int32_t* iterations, double* residual);
// heating.cu: the heating setting (gamma9 = nullptr clears; stride = entries per field of dHeat) and its pass
bool heating_args_ok(const double* gamma9, const double* width3);
int set_heating(Context& c, const double* gamma9, const double* width3, int64_t stride);
void free_heating(Context& c);
// the heating pass over leaves [off, off + cnt) into dHeat [f * heatStride + i - off], from J [g * jStride + i - off]
// and the species at + off; counted in the call's launches and device time
int launch_heating(Context& c, int64_t off, int64_t cnt, const double* J, int64_t jStride, cudaStream_t s);

// ng.cu: acceleration of the source iteration (DESIGN.md 4.9)
constexpr int kNgBlocks = 1024;    // fixed grid of the partial-sum pass: its sums do not depend on the device
constexpr int kNgMaxRanks = 64;
// views into Context::dNg for fields of `stride` entries per group: hist[j] = y of sweep j + 1 of the current cycle of
// four, the block partials [kNgBlocks][5], every rank's five sums [kNgMaxRanks][5], coef = {1 - a - b, a, b, apply}
// and the count of applied extrapolations
struct NgBuffers {
  double* hist[3];
  double* part;
  double* sums;
  double* coef;
  int32_t* count;
};
int ng_buffers(Context& c, int64_t stride, NgBuffers* b);
int set_scattering_acceleration(Context& c, int32_t flags);
void free_history(Context& c);   // frees the Ng history (a count the latest call left on the device is read first)
// the five sums of this rank's cnt entries of I0..I3 (stride jStride) into b.sums[5 * rank ..]
int launch_ng_partials(const NgBuffers& b, int64_t cnt, const double* I0, int64_t jStride, int rank, cudaStream_t s);
// from the sums of nranks ranks: a, b and the decision; when it applies, x = max(0, (1-a-b) I0 + a I1 + b I2) into
// Jprev and eta_th + sigma * x into etaOut (strides as launch_scatter_source), else nothing changes
int launch_ng_apply(const Context& c, const NgBuffers& b, int nranks, int64_t cnt, const double* I0, double* Jprev,
                    int64_t jStride, const double* sigma, const double* etaTh, int64_t sStride, double* etaOut,
                    int64_t oStride, cudaStream_t s);
int last_scattering_acceleration(Context& c, int32_t* extrapolations, int32_t* warmStarted);
// device group, warm start: *used = 1 if flags[r] != 0 for every r < nranks, else Jprev[0 .. n) = 0 and *used = 0
int launch_warm_start_agree(const Context& c, const double* flags, int nranks, double* Jprev, int64_t n, int32_t* used,
                            cudaStream_t s);

// kernels / launchers --------------------------------------------------------------------------------
int launch_compute_opacities(Context& c, const double* beta, cudaStream_t s);
int diffuse_uniform(Context& c, int nAngularLevel, const double* uvb, const std::vector<Direction>& dirs,
                    double* dJout, cudaStream_t s, int64_t* nseg);
int diffuse_amr(Context& c, int nAngularLevel, const double* uvb, const std::vector<Direction>& dirs,
                double* dJout, cudaStream_t s, int64_t* nseg);
int amr_neighbours(Context& c, const Direction& d, int32_t* nbHost);
int amr_waves(Context& c, const Direction& d, int32_t* waveOfLeaf, int32_t* nwaves);
void amr_release(Context& c);
void point_release(Context& c);
int launch_diffuse_rates(Context& c, const double* J, const double* ksi24, const double* ksi25, const double* ksi26,
                         double* k24, double* k25, double* k26, cudaStream_t s);

int chemistry_set_tables(Context& c, int nratec, double logtem0, double logtem9, double dlogtem, const double* const k[6]);
int chemistry_set_temperature(Context& c, const double* tgas);
int compute_mass(Context& c, double* neutralHydrogenMass, double* totalHydrogenMass, cudaStream_t s);
int chemistry_run(Context& c, const double* dRates, const double* dJ, const double* ksi, const double* uniform,
                  double* maxChange, cudaStream_t s);
// the same pass over leaves [first, first + count) only, with the rate / J arrays given as slabs: element (field f,
// leaf c) at rates[f * rStride + c - first] and J[g * jStride + c - first]   (multi-GPU: every rank solves its slab)
int chemistry_run_slab(Context& c, int64_t first, int64_t count, const double* dRates, int64_t rStride, const double* dJ,
                       int64_t jStride, const double* ksi, const double* uniform, cudaStream_t s);

// point sources: dRates = device [6][nleaf] (krate24, krate25, krate26, crate24, crate25, crate26), accumulated;
// hDiag = host [nsrc][320] (remaining[7], boundary[7], dust, pad, spectrum[300]) or NULL
int point_solve(Context& c, const PointInputs& in, double* dRates, double* hDiag, int64_t* nseg, long long* hTrace,
                long long traceCap, long long* traceLen, double* hRawTables, cudaStream_t s);
PointInputs make_point_inputs(int nWave, const double* wavelength, const double* lum, const double* metallicity,
                              double coefSpectrum, const double* aDust, int dust, int maxPixelLevel, int nsrc,
                              const int32_t* srcLeaf, const int32_t* srcWeight);
// hDiag records of n sources into the caller's per-source arrays (any may be NULL): record i belongs to source
// idx[i], or to source i without idx
void split_diag(const double* d, size_t n, const int* idx, double* rem, double* bnd, double* dust, double* spec,
                int32_t* hpl);

int set_math(Context& c, int mode);
int device_error(Context& c);

// ---- multi-GPU (multi.cu) -----------------------------------------------------------------------------------------
struct Multi;
void multi_destroy(Multi* m);
Context& multi_primary(Multi* m);
int multi_set_math(Multi* m, int mode);
int multi_set_tuning(Multi* m, const char* key, double value);
int multi_grid_set(Multi* m, int nx, int64_t nleaf, const int8_t* level, const double* HI, const double* HeI,
                   const double* HeII, const double* rho, const double* abun2, double physicalBoxSize);
int multi_update_species(Multi* m, const double* HI, const double* HeI, const double* HeII);
int multi_set_emission(Multi* m, const double* eta);
int multi_set_scattering(Multi* m, const double* sigma, int32_t maxIterations, double tolerance);
int multi_set_scattering_acceleration(Multi* m, int32_t flags);
int multi_set_dust(Multi* m, int mode, const double* betaDust, const double* albedo, int32_t maxIterations, double tolerance);
int multi_set_heating(Multi* m, const double* gamma9, const double* width3);
int multi_last_heating(Multi* m, double* heat5);
int multi_heating_device(Multi* m, int local, int64_t* offset, int64_t* count, int64_t* stride, double** H);
int multi_get_species(Multi* m, double* HI, double* HeI, double* HeII);
int multi_diffuse_host(Multi* m, int nAngularLevel, const double* uvb, const double* beta, const int32_t* rays,
                       int32_t nrays, double* J1, double* J2, double* J3, int64_t* nseg);
int multi_point_host(Multi* m, const PointInputs& in, double* const k[6], double* rem, double* bnd, double* dust,
                     double* spec, int32_t* hpl, int64_t* nseg);
int multi_chemistry_tables(Multi* m, int nratec, double logtem0, double logtem9, double dlogtem, const double* const k[6]);
int multi_chemistry_temperature(Multi* m, const double* tgas);
int multi_device_error(Multi* m);

}  // namespace rtb

// the opaque handle of the C-ABI: one context (rtb200_create) or a group of them (rtb200_create_multi / _rank)
struct rtb200_ctx {
  rtb::Context c;            // single-GPU handle; unused when m != nullptr
  rtb::Multi* m = nullptr;
};
