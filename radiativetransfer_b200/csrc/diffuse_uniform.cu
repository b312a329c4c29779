// Diffuse sweep on a uniform (single-level) grid: replaces the direction loop of equiSources.f90:1389-1806 for
// grids without refinement (configs 2 and 4 of BASELINE.json).
//
// Formulation (DESIGN.md "uniform sweep"):
//  * All directions of one zone share the index rotation (rotateIndicesModule.f90), so they are swept TOGETHER,
//    layer by layer along the zone's sweep axis: one thread owns one cell of the layer, reads kappa1..3 once,
//    loops over the zone's directions and adds all their contributions to J in registers -> one J update per
//    cell per zone instead of one per direction.
//  * Within a layer every cell carries the same 1..3 segments (its "pattern"); a characteristic that leaves a
//    cell sideways continues in the k+1 and/or j+1 neighbour of the SAME layer.  Along the lane axis that hand-over
//    is a warp shuffle of the neighbour lane's own result (a warp covers 31 positions + 1 recomputed halo, and the
//    positions of a layer run end to end across rows and warps: lane_position); along the row axis the thread
//    recomputes what the (b-1) cell emits from the previous layer's plane value and that cell's kappa.  No
//    shared-memory exchange, no barrier in the loop, no inter-block communication.
//  * The only inter-layer state is the intensity leaving each cell through its top face: one padded plane of
//    3 doubles per cell per direction ([row][column][group]), ping-ponged in global memory.
//  * One launch per layer covers every zone task of the batch (gridDim.z); each task owns a private J accumulator
//    ("slot"), so no atomics and a fixed summation order.  Final kernels sum the slot accumulators into J.
//  * Zones that sweep along the contiguous axis of the leaf order read a z-major copy of kappa and accumulate in
//    that layout (transpose_kappa_kernel / merge_transposed_kernel) so that their lanes stay coalesced.
//  * Layer kernels: sweep_cell_kernel (one cell per thread, FAST or FAITHFUL), sweep_cell2_kernel (two cells per
//    thread, FAST) and sweep_cell_emit_kernel (one cell per thread, with emission); launch_cells picks one per launch.

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>

#include "rtb200_internal.h"
#include "segment_math.cuh"

namespace rtb {

__global__ void compute_opacities_kernel(const double* __restrict__ HI, const double* __restrict__ HeI,
                                         const double* __restrict__ HeII, double* __restrict__ kappa, int64_t n,
                                         double b0, double b3, double b4, double b6, double b7, double b8) {
  // equiSources.f90:4974-4977, same association order, no FMA contraction
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double h = HI[i], he1 = HeI[i], he2 = HeII[i];
    kappa[i] = __dmul_rn(h, b0);
    kappa[n + i] = __dadd_rn(__dmul_rn(h, b3), __dmul_rn(he1, b4));
    kappa[2 * n + i] = __dadd_rn(__dadd_rn(__dmul_rn(h, b6), __dmul_rn(he1, b7)), __dmul_rn(he2, b8));
  }
}

int launch_compute_opacities(Context& c, const double* beta, cudaStream_t s) {
  int blocks = std::min<int64_t>((c.nleaf + 255) / 256, (int64_t)c.smCount * 16);
  compute_opacities_kernel<<<blocks, 256, 0, s>>>(c.dHI, c.dHeI, c.dHeII, c.dKappa, c.nleaf, beta[0], beta[3], beta[4],
                                                  beta[6], beta[7], beta[8]);
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

// ---------------------------------------------------------------------------------------------------------
// one layer step of one zone
//
// thread = one cell of the layer; it loops over the zone's directions, keeping kappa (own cell and the three
// upstream neighbours of the layer) and the J sum in registers.  A segment fed by a same-layer neighbour needs that
// neighbour's outgoing intensity, which is a pure function of the previous layer's top-exit plane and of kappa:
// the thread RECOMPUTES it (one or two extra exponentials, bit-identical to what the neighbour's own thread
// computes) instead of waiting for it.  Threads are independent: no shared memory, no halo, no barrier.
// The per-step tables travel as a __grid_constant__ kernel parameter, i.e. they are read from the constant bank.
// ---------------------------------------------------------------------------------------------------------
struct StepParams {
  LayerSeg P[kMaxDirPerTask];
  const double* planeIn;   // this task's planes of the previous layer  [ndir][n+1][n+1][3 groups] (padded, see below)
  double* planeOut;
  double* acc;             // slot accumulator [3][N]
  const double* kappa;     // [3][N] in the layout the task's strides refer to (leaf order or z-major)
  int32_t origin;          // leaf index of rotated (step, 0, 0)
  int32_t sj, sk;
  int32_t ndir, laneIsK, firstInSlot, n;
  int32_t anyThin;         // a direction of this layer is thin (LayerSeg::thin)
};

// Planes carry one extra row and column on the upstream side (index -1) that permanently hold the boundary
// intensity, and the plane read by the first layer is filled with it: together with kappa = 0 for out-of-domain
// neighbours (exp(-0) = 1 exactly) this makes "no neighbour -> uvb" (transportRoutinesModule.f90:594-597) fall out
// of the same arithmetic as an interior cell, with no per-direction edge test.
__global__ void fill_planes_kernel(double* __restrict__ planes, int64_t perGroup, int64_t total, double u0, double u1,
                                   double u2) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    int g = (int)(i % 3);  // the three frequency groups of a cell are adjacent: [direction][row][column][group]
    planes[i] = g == 0 ? u0 : (g == 1 ? u1 : u2);
  }
}

// One direction of one cell, straight-line for a given segment count and chain order.
//   NSEG: 1..3 segments.  SECL: the second segment is fed by the neighbour along the LANE axis (cell a-1, same row)
//   and the third by the neighbour along the ROW axis (cell b-1, same lane); !SECL: the other way round.
// Lane-axis hand-over = warp shuffle of the neighbour lane's own result; row-axis hand-over = recompute of what the
// (b-1) cell emits from the previous layer's plane value `upR` and its kappa `kR` (bit-identical to that cell's own
// arithmetic).  Every lane of the warp must call this (shuffles), including the halo lane and out-of-domain lanes.
//
// FAST arithmetic (segment_math.cuh: segment_fast): A[g] collects Iin (1 - e^-tau) cs over all segments and
// directions of the layer; the caller multiplies by 2^-200 / kappa once per layer.
// Emission (EMIT, DESIGN.md 4.6): the cell's and the (b-1) cell's emission coefficients and 1 / kappa ride along in Em;
// every segment also adds phi(tau) dpath weight / nseg to E[g], which the caller multiplies by eta once per layer.
struct Em {
  double eta[3], etaR[3];    // own cell, (b-1) cell (0 outside the domain)
  double invk[3], invkR[3];  // FAST arithmetic: 1 / kappa with kappa floored as in the segment
};

// `d` is the layer table's path: the scaled path d * kExpScale for the plain sweep, the path itself for the emissive one
// (emission needs tau = kappa d; the scaled path is formed here, as the same product the host forms for the plain
// sweep, so that eta = 0 reproduces it bit for bit).  See fill_step_segs.
template <bool GUARD, bool EMIT>
__device__ __forceinline__ double seg_fast(double Iin, double kap, double d, double cs, const double* __restrict__ T,
                                           double& A, double eta, double invk, double dw, double& E) {
  if (EMIT) return segment_fast_emit<GUARD>(Iin, kap, d * kExpScale, cs, T, A, eta, invk, d, dw, E);
  return segment_fast<GUARD>(Iin, kap, d, cs, T, A);
}
template <bool GUARD, bool EMIT>
__device__ __forceinline__ double att_fast(double Iin, double kap, double d, const double* __restrict__ T, double eta,
                                           double invk) {
  if (EMIT) return attenuate_fast_emit<GUARD>(Iin, kap, d * kExpScale, T, eta, invk, d);
  return attenuate_fast<GUARD>(Iin, kap, d, T);
}

template <int NSEG, bool SECL, bool GUARD, bool EMIT = false>
__device__ __forceinline__ void direction_fast(const LayerSeg& P, const double (&cur)[3], const double (&upR)[3],
                                               const double (&kap)[3], const double (&kR)[3], double (&I)[3],
                                               double (&A)[3], const double* __restrict__ T, const Em& em,
                                               double (&E)[3]) {
  const unsigned full = 0xffffffffu;
  const double wn = EMIT ? P.w * (1.0 / NSEG) : 0.;
#pragma unroll
  for (int g = 0; g < 3; g++) {
    const double I1 = seg_fast<GUARD, EMIT>(cur[g], kap[g], P.d[0], P.cs[0], T, A[g], em.eta[g], em.invk[g], P.d[0] * wn, E[g]);
    I[g] = I1;
    if (NSEG >= 2) {
      double rup = 0.;  // xy-segment output of the (b-1) cell
      if (!SECL || NSEG == 3) rup = att_fast<GUARD, EMIT>(upR[g], kR[g], P.d[0], T, em.etaR[g], em.invkR[g]);
      const double in2 = SECL ? __shfl_up_sync(full, I1, 1) : rup;
      const double I2 = seg_fast<GUARD, EMIT>(in2, kap[g], P.d[1], P.cs[1], T, A[g], em.eta[g], em.invk[g], P.d[1] * wn, E[g]);
      I[g] = I2;
      if (NSEG == 3) {
        double in3;
        if (SECL) {
          // third segment from the (b-1) cell's SECOND segment, which was fed by the (b-1, a-1) cell's xy segment
          const double x = __shfl_up_sync(full, rup, 1);
          in3 = att_fast<GUARD, EMIT>(x, kR[g], P.d[1], T, em.etaR[g], em.invkR[g]);
        } else {
          in3 = __shfl_up_sync(full, I2, 1);  // the (a-1) cell's second segment
        }
        I[g] = seg_fast<GUARD, EMIT>(in3, kap[g], P.d[2], P.cs[2], T, A[g], em.eta[g], em.invk[g], P.d[2] * wn, E[g]);
      }
    }
  }
}

// The reference's own operation sequence (RTB200_MATH_FAITHFUL, and the thin layers of FAST mode): adds
// (sum of the segments' J) / nseg * weight to acc (transportRoutinesModule.f90:953-955).
template <bool EMIT>
__device__ __forceinline__ SegResult seg_faithful(double Iin, double kap, double d, double eta) {
  if (EMIT) return segment_faithful_emit(Iin, kap, d, eta);
  return segment_faithful(Iin, kap, d);
}
template <bool EMIT>
__device__ __forceinline__ double att_faithful(double Iin, double kap, double d, double eta) {
  if (EMIT) return attenuate_faithful_emit(Iin, kap, d, eta);
  return __dmul_rn(Iin, exp(-__dmul_rn(kap, d)));
}

template <int NSEG, bool SECL, bool EMIT = false>
__device__ __forceinline__ void direction_faithful(const LayerSeg& P, const double (&cur)[3], const double (&upR)[3],
                                                   const double (&kap)[3], const double (&kR)[3], double (&I)[3],
                                                   double (&acc)[3], const double (&eta)[3], const double (&etaR)[3]) {
  const unsigned full = 0xffffffffu;
#pragma unroll
  for (int g = 0; g < 3; g++) {
    SegResult r1 = seg_faithful<EMIT>(cur[g], kap[g], P.d[0], eta[g]);
    double Jsum = r1.J;
    I[g] = r1.Iout;
    if (NSEG >= 2) {
      double rup = 0.;
      if (!SECL || NSEG == 3) rup = att_faithful<EMIT>(upR[g], kR[g], P.d[0], etaR[g]);
      const double in2 = SECL ? __shfl_up_sync(full, r1.Iout, 1) : rup;
      SegResult r2 = seg_faithful<EMIT>(in2, kap[g], P.d[1], eta[g]);
      I[g] = r2.Iout;
      double J3 = 0.;
      if (NSEG == 3) {
        double in3;
        if (SECL) {
          const double x = __shfl_up_sync(full, rup, 1);
          in3 = att_faithful<EMIT>(x, kR[g], P.d[1], etaR[g]);
        } else {
          in3 = __shfl_up_sync(full, r2.Iout, 1);
        }
        SegResult r3 = seg_faithful<EMIT>(in3, kap[g], P.d[2], eta[g]);
        I[g] = r3.Iout;
        J3 = r3.J;
      }
      // the reference sums the segments in the order xy, xz, yz (transportRoutinesModule.f90:698,818,941);
      // P.kind <= 2 <=> the second segment is the yz ray
      const bool yzSecond = P.kind <= 2;
      const double Jxz = yzSecond ? J3 : r2.J, Jyz = yzSecond ? r2.J : J3;
      Jsum = r1.J;
      if (NSEG == 3 || !yzSecond) Jsum = __dadd_rn(Jsum, Jxz);
      if (NSEG == 3 || yzSecond) Jsum = __dadd_rn(Jsum, Jyz);
    }
    acc[g] = __dadd_rn(acc[g], __dmul_rn(__ddiv_rn(Jsum, (double)NSEG), P.w));
  }
}

// dispatch on the layer's chain kind (warp-uniform).  kmax = the largest opacity this thread multiplies a path with.
// If kmax * (longest segment of the layer) <= 64 for every lane of the warp, the overflow guards of segment_fast are
// dropped (4 fewer instructions per segment update); `thick` warps take the guarded instantiation.
template <bool GUARD, bool EMIT>
__device__ __forceinline__ void direction_kinds_fast(const LayerSeg& P, bool secL, const double (&cur)[3],
                                                     const double (&upR)[3], const double (&kap)[3],
                                                     const double (&kR)[3], double (&I)[3], double (&A)[3],
                                                     const double* __restrict__ T, const Em& em, double (&E)[3]) {
  const int kind = P.kind;
  if (kind == 0) direction_fast<1, true, GUARD, EMIT>(P, cur, upR, kap, kR, I, A, T, em, E);
  else if (kind == 1 || kind == 3) {
    if (secL) direction_fast<2, true, GUARD, EMIT>(P, cur, upR, kap, kR, I, A, T, em, E);
    else direction_fast<2, false, GUARD, EMIT>(P, cur, upR, kap, kR, I, A, T, em, E);
  } else {
    if (secL) direction_fast<3, true, GUARD, EMIT>(P, cur, upR, kap, kR, I, A, T, em, E);
    else direction_fast<3, false, GUARD, EMIT>(P, cur, upR, kap, kR, I, A, T, em, E);
  }
}

template <bool EMIT>
__device__ __forceinline__ void direction_dispatch_fast(const LayerSeg& P, bool secL, double kmax, const double (&cur)[3],
                                                        const double (&upR)[3], const double (&kap)[3],
                                                        const double (&kR)[3], double (&I)[3], double (&A)[3],
                                                        const double* __restrict__ T, const Em& em, double (&E)[3]) {
  if (__any_sync(0xffffffffu, kmax * P.dmax > 64.)) direction_kinds_fast<true, EMIT>(P, secL, cur, upR, kap, kR, I, A, T, em, E);
  else direction_kinds_fast<false, EMIT>(P, secL, cur, upR, kap, kR, I, A, T, em, E);
}

// By value: the rare faithful branch must not force the fast path's per-direction arrays into local memory.
struct Tri {
  double v[3];
};
struct FaithOut {
  Tri I, acc;
};
template <bool EMIT>
__device__ __forceinline__ FaithOut direction_faithful_kinds(double d0, double d1, double d2, double w, int kind, bool secL,
                                                             const Tri& cur_, const Tri& upR_, const Tri& kap_,
                                                             const Tri& kR_, const Tri& acc_, const Tri& eta_,
                                                             const Tri& etaR_) {
  LayerSeg P;
  P.d[0] = d0; P.d[1] = d1; P.d[2] = d2; P.w = w; P.kind = kind;
  double cur[3] = {cur_.v[0], cur_.v[1], cur_.v[2]}, upR[3] = {upR_.v[0], upR_.v[1], upR_.v[2]};
  double kap[3] = {kap_.v[0], kap_.v[1], kap_.v[2]}, kR[3] = {kR_.v[0], kR_.v[1], kR_.v[2]};
  double acc[3] = {acc_.v[0], acc_.v[1], acc_.v[2]}, I[3] = {0., 0., 0.};
  double eta[3] = {eta_.v[0], eta_.v[1], eta_.v[2]}, etaR[3] = {etaR_.v[0], etaR_.v[1], etaR_.v[2]};
  if (kind == 0) direction_faithful<1, true, EMIT>(P, cur, upR, kap, kR, I, acc, eta, etaR);
  else if (kind == 1 || kind == 3) {
    if (secL) direction_faithful<2, true, EMIT>(P, cur, upR, kap, kR, I, acc, eta, etaR);
    else direction_faithful<2, false, EMIT>(P, cur, upR, kap, kR, I, acc, eta, etaR);
  } else {
    if (secL) direction_faithful<3, true, EMIT>(P, cur, upR, kap, kR, I, acc, eta, etaR);
    else direction_faithful<3, false, EMIT>(P, cur, upR, kap, kR, I, acc, eta, etaR);
  }
  FaithOut o;
#pragma unroll
  for (int g = 0; g < 3; g++) { o.I.v[g] = I[g]; o.acc.v[g] = acc[g]; }
  return o;
}
__device__ __forceinline__ FaithOut direction_call_faithful(double d0, double d1, double d2, double w, int kind,
                                                            bool secL, Tri cur_, Tri upR_, Tri kap_, Tri kR_, Tri acc_) {
  const Tri zero = {{0., 0., 0.}};
  return direction_faithful_kinds<false>(d0, d1, d2, w, kind, secL, cur_, upR_, kap_, kR_, acc_, zero, zero);
}
__device__ __forceinline__ FaithOut direction_call_faithful_emit(double d0, double d1, double d2, double w, int kind,
                                                                 bool secL, Tri cur_, Tri upR_, Tri kap_, Tri kR_,
                                                                 Tri acc_, Tri eta_, Tri etaR_) {
  return direction_faithful_kinds<true>(d0, d1, d2, w, kind, secL, cur_, upR_, kap_, kR_, acc_, eta_, etaR_);
}
template <bool EMIT = false>
__device__ __forceinline__ void direction_dispatch_faithful(const LayerSeg& P, bool secL, const double (&cur)[3],
                                                            const double (&upR)[3], const double (&kap)[3],
                                                            const double (&kR)[3], double (&I)[3], double (&acc)[3],
                                                            const double* eta = nullptr, const double* etaR = nullptr) {
  const FaithOut o =
      EMIT ? direction_call_faithful_emit(P.d[0], P.d[1], P.d[2], P.w, P.kind, secL, Tri{{cur[0], cur[1], cur[2]}},
                                          Tri{{upR[0], upR[1], upR[2]}}, Tri{{kap[0], kap[1], kap[2]}},
                                          Tri{{kR[0], kR[1], kR[2]}}, Tri{{acc[0], acc[1], acc[2]}},
                                          Tri{{eta[0], eta[1], eta[2]}}, Tri{{etaR[0], etaR[1], etaR[2]}})
           : direction_call_faithful(P.d[0], P.d[1], P.d[2], P.w, P.kind, secL, Tri{{cur[0], cur[1], cur[2]}},
                                     Tri{{upR[0], upR[1], upR[2]}}, Tri{{kap[0], kap[1], kap[2]}},
                                     Tri{{kR[0], kR[1], kR[2]}}, Tri{{acc[0], acc[1], acc[2]}});
#pragma unroll
  for (int g = 0; g < 3; g++) { I[g] = o.I.v[g]; acc[g] = o.acc.v[g]; }
}

__device__ __forceinline__ void prefetch_l1(const double* p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }

constexpr double kKappaFloor = 1e-100;  // FAST mode: kappa = 0 is evaluated as this (every formula takes its limit)
constexpr double kTwoM200 = 6.223015277861141707e-61;  // 2^-200

// Lanes and cells.  Per task and layer the positions q = 0 .. R (n+1) - 1 run over R rows (row pairs for two-cell
// threads) of n + 1 columns: row r = q / (n+1), column a = q mod (n+1) - 1, where a = -1 is the pad column (plane
// value = boundary intensity, kappa = 0: "no neighbour").  Warp w, lane L takes q = 31 w + L, so the positions run end
// to end across rows and warps and no lane idles past a row's end:
//  * lane 0 is a halo: it recomputes the position that lane 31 of warp w - 1 writes, or a pad;
//  * the writers are lanes 1..31 at a real cell (a >= 0);
//  * lanes past the last position evaluate the last row's pad and only take part in the shuffles.
// Invariant that makes this correct without a per-lane select after a shuffle: every value a lane takes from lane - 1
// is of depth 1 -- the neighbour's xy-segment output (a1 / b1 / I1) or its recomputed (b-1) output (rup, or a2 / I2
// fed by rup), each a function of the neighbour's OWN plane values and opacities only, never of a shuffled value.  So
// a halo or pad lane whose own shuffled inputs are garbage (the end of the previous row, or a pad in mid-warp at the
// start of a row) still hands over exactly what the cell to its right needs.  The per-cell arithmetic and the
// summation order do not depend on where a cell sits in a warp; only the warp-wide guard vote does, and the guarded
// and unguarded exponentials agree bit for bit where the vote lets a warp skip the guard (segment_math.cuh).
struct LanePos {
  int a, r;       // column (-1 = pad) and row (pair) of this lane's position
  bool warpLive;  // warp-uniform: the warp holds at least one writer
};
__device__ __forceinline__ LanePos lane_position(int rows, int np1) {
  const int P = rows * np1;                                   // positions per task and layer
  const int w = blockIdx.x * blockDim.y + threadIdx.y;
  LanePos lp;
  lp.warpLive = 31 * w < P - 1;
  int q = 31 * w + (int)threadIdx.x;
  if (q >= P) q = P - np1;                                    // past the end: the last row's pad
  lp.r = q / np1;
  lp.a = q - lp.r * np1 - 1;
  return lp;
}
// warps per task and layer (host side of lane_position)
static inline int warps_per_layer(int n, int rows) { return (rows * (n + 1) - 2) / 31 + 1; }

constexpr int kMaxBatch = 40;  // tasks per launch: 40 x 728 B of parameters (the limit is 32764 B since CUDA 12.1)
struct BatchParams {
  StepParams t[kMaxBatch];
};
static_assert(sizeof(BatchParams) + 64 <= 32764, "kernel parameter space");

// gridDim.z tasks (zones) per launch, all at the same layer index: one launch per layer keeps the device full
// (thousands of blocks) instead of many small concurrent kernels.
// A layer whose pattern has a very short segment (a corner clip, len < 1e-2 cell; 1.7% of the (direction, layer)
// pairs) is evaluated with the reference's own operation sequence even in FAST mode: there tau is tiny and the
// rounding noise of the reference's (Iin-Iout)/log(Iin/Iout), ~1.1e-16/tau, would otherwise show up as a parity
// difference.  That branch is warp-uniform (P.thin is a per-layer table entry).
// Emission (DESIGN.md 4.6): the emission coefficients of every task, in the layout of its kappa (leaf order or z-major)
struct EtaParams {
  const double* eta[kMaxBatch];
};

template <bool FAITHFUL, bool EMIT>
__device__ __forceinline__ void sweep_cell_body(const BatchParams& bp, const double* __restrict__ etaTask, int N, int n,
                                                int np1, int npl3) {
  // n, np1 = n + 1 and npl3 = 3 (n+1)^2 are the same for every task: as top-level parameters they are constant-bank
  // operands instead of values re-derived from the task table for every direction
  const StepParams& sp = bp.t[blockIdx.z];
  const double* __restrict__ kappa = sp.kappa;
  __shared__ double sT[kExpTableSize];
  // Programmatic dependent launch (set_tuning "pdl"): the next layer's grid may start as soon as every block of this
  // one is running, do its own prologue (table, indices, opacities -- nothing a sweep kernel writes) and then wait at
  // griddepcontrol.wait below until this grid has completed and flushed.  Both instructions are no-ops for a grid
  // launched without the attribute.
  asm volatile("griddepcontrol.launch_dependents;");
  if (threadIdx.y * 32 + threadIdx.x < kExpTableSize) sT[threadIdx.y * 32 + threadIdx.x] = kExpTable32[threadIdx.y * 32 + threadIdx.x];
  __syncthreads();
  const LanePos lp = lane_position(n, np1);
  if (!lp.warpLive) return;                                    // warp-uniform
  const int a = lp.a, b = lp.r;
  const bool cell = a >= 0;                                    // a real cell (not the pad column)
  const bool writer = cell && threadIdx.x >= 1;
  const int laneIsK = sp.laneIsK;
  const int sA = laneIsK ? sp.sk : sp.sj, sB = laneIsK ? sp.sj : sp.sk;
  const int leaf = sp.origin + a * sA + b * sB;
  double kap[3], kapF[3], kR[3];
#pragma unroll
  for (int g = 0; g < 3; g++) {
    const double* kg = kappa + (int64_t)g * N + leaf;
    kapF[g] = cell ? kg[0] : 0.;
    kR[g] = (cell && b > 0) ? kg[-sB] : 0.;                    // kappa = 0 outside: exp(-0) = 1 exactly
    kap[g] = kapF[g] > 0. ? kapF[g] : kKappaFloor;
  }
  const double kmax = fmax(fmax(fmax(kap[0], kap[1]), fmax(kap[2], kR[0])), fmax(kR[1], kR[2]));
  double A[3] = {0., 0., 0.}, acc[3] = {0., 0., 0.};
  Em em;
  double E[3] = {0., 0., 0.};
  if (EMIT) {
#pragma unroll
    for (int g = 0; g < 3; g++) {
      const double* eg = etaTask + (int64_t)g * N + leaf;
      em.eta[g] = cell ? eg[0] : 0.;
      em.etaR[g] = (cell && b > 0) ? eg[-sB] : 0.;                // the pad row and column emit nothing
      em.invk[g] = FAITHFUL ? 0. : 1.0 / kap[g];
      em.invkR[g] = FAITHFUL ? 0. : 1.0 / (kR[g] > 0. ? kR[g] : kKappaFloor);   // as the (b-1) cell's own thread
    }
  }
  const int pidx = (b + 1) * np1 + a + 1;
  const int ndir = sp.ndir;
  const int dstride = npl3;                                    // one direction's plane (3 groups per cell)
  const int up = 3 * np1;                                      // one row up
  const double* pin = sp.planeIn + 3 * pidx;
  double* pout = sp.planeOut + 3 * pidx;
  asm volatile("griddepcontrol.wait;" ::: "memory");           // the previous layer's planes and accumulators
  for (int q = 0; q < ndir; q++, pin += dstride, pout += dstride) {
    const LayerSeg& P = sp.P[q];
    const int kind = P.kind;
    // Pull the NEXT direction's plane values towards L1 with prefetch instructions: they hold no destination
    // register (at 64 registers per thread a register prefetch is spilled at once, and the spill store then waits
    // for the load -- 35% of all stall samples in the r01 profile).
    if (q + 1 < ndir) {
      prefetch_l1(pin + dstride);
      prefetch_l1(pin + dstride - up);
    }
    double cur[3], upR[3] = {0., 0., 0.}, I[3];
#pragma unroll
    for (int g = 0; g < 3; g++) cur[g] = pin[g];
    // kinds 1,2: second segment fed from k-1, third (kind 2) from j-1; kinds 3,4 the other way round
    const bool secL = (kind <= 2) == (laneIsK != 0);
    if (kind == 2 || kind == 4 || (kind != 0 && !secL)) {
#pragma unroll
      for (int g = 0; g < 3; g++) upR[g] = pin[g - up];
    }
    if (FAITHFUL || P.thin) direction_dispatch_faithful<EMIT>(P, secL, cur, upR, kapF, kR, I, acc, em.eta, em.etaR);
    else direction_dispatch_fast<EMIT>(P, secL, kmax, cur, upR, kap, kR, I, A, sT, em, E);
    if (writer) {
#pragma unroll
      for (int g = 0; g < 3; g++) pout[g] = I[g];
    }
  }
  if (writer) {
#pragma unroll
    for (int g = 0; g < 3; g++) {
      if (!FAITHFUL) acc[g] = fma(A[g], kTwoM200 / kap[g], acc[g]);
      if (EMIT && !FAITHFUL) acc[g] = fma(em.eta[g], E[g], acc[g]);
      double* p = sp.acc + (int64_t)g * N + leaf;
      *p = sp.firstInSlot ? acc[g] : __dadd_rn(*p, acc[g]);
    }
  }
}

// register budget: FAST arithmetic 4 blocks of 256 threads per SM (64 registers; 2 or 3 blocks measured slower,
// DESIGN.md 4.2), FAITHFUL 2
template <bool FAITHFUL>
__global__ void __launch_bounds__(256, FAITHFUL ? 2 : 4)
sweep_cell_kernel(const __grid_constant__ BatchParams bp, int N, int n, int np1, int npl3) {
  sweep_cell_body<FAITHFUL, false>(bp, nullptr, N, n, np1, npl3);
}

// the emissive sweep: one cell per thread, 2 blocks of 256 threads per SM (the emission terms need registers)
template <bool FAITHFUL>
__global__ void __launch_bounds__(256, 2)
sweep_cell_emit_kernel(const __grid_constant__ BatchParams bp, int N, int n, int np1, int npl3,
                       const __grid_constant__ EtaParams ep) {
  sweep_cell_body<FAITHFUL, true>(bp, ep.eta[blockIdx.z], N, n, np1, npl3);
}

// ---------------------------------------------------------------------------------------------------------
// Two cells per thread (FAST arithmetic; set_tuning "cells" = 2, the default): a thread owns the cells (a, b0) and
// (a, b0 + 1) of the layer, b0 even.  What the upper cell needs from the row below it -- the previous layer's plane
// value of (a, b0) and the intensity the lower cell hands over along the row axis -- is already in the thread's
// registers: no recomputed (b-1) segment and no second plane load for the upper cell, and the per-direction
// bookkeeping (table reads, kind dispatch, pointer updates, prefetches) is paid once per two cells.  The arithmetic
// of every cell is unchanged: the handed-over value is bit for bit what the single-cell kernel recomputes.
//   r01 ncu of the single-cell kernel: 318 warp instructions per direction, 194 of them not FP64 (issue-bound).
// ---------------------------------------------------------------------------------------------------------
template <int NSEG, bool SECL, bool GUARD>
__device__ __forceinline__ void direction_fast2(const LayerSeg& P, const double (&cur0)[3], const double (&cur1)[3],
                                                const double (&upR)[3], const double (&kap0)[3], const double (&kap1)[3],
                                                const double (&kR)[3], double (&I0)[3], double (&I1)[3], double (&A0)[3],
                                                double (&A1)[3], const double* __restrict__ T) {
  const unsigned full = 0xffffffffu;
#pragma unroll
  for (int g = 0; g < 3; g++) {
    const double a1 = segment_fast<GUARD>(cur0[g], kap0[g], P.d[0], P.cs[0], T, A0[g]);
    const double b1 = segment_fast<GUARD>(cur1[g], kap1[g], P.d[0], P.cs[0], T, A1[g]);
    I0[g] = a1; I1[g] = b1;
    if (NSEG >= 2) {
      double rup = 0.;  // xy-segment output of the (b0 - 1) cell, recomputed (lower cell only)
      if (!SECL || NSEG == 3) rup = attenuate_fast<GUARD>(upR[g], kR[g], P.d[0], T);
      const double a_in2 = SECL ? __shfl_up_sync(full, a1, 1) : rup;
      const double b_in2 = SECL ? __shfl_up_sync(full, b1, 1) : a1;   // the lower cell's own xy output
      const double a2 = segment_fast<GUARD>(a_in2, kap0[g], P.d[1], P.cs[1], T, A0[g]);
      const double b2 = segment_fast<GUARD>(b_in2, kap1[g], P.d[1], P.cs[1], T, A1[g]);
      I0[g] = a2; I1[g] = b2;
      if (NSEG == 3) {
        double a_in3, b_in3;
        if (SECL) {
          const double x = __shfl_up_sync(full, rup, 1);
          a_in3 = attenuate_fast<GUARD>(x, kR[g], P.d[1], T);
          b_in3 = a2;                                                 // the lower cell's second segment
        } else {
          a_in3 = __shfl_up_sync(full, a2, 1);
          b_in3 = __shfl_up_sync(full, b2, 1);
        }
        I0[g] = segment_fast<GUARD>(a_in3, kap0[g], P.d[2], P.cs[2], T, A0[g]);
        I1[g] = segment_fast<GUARD>(b_in3, kap1[g], P.d[2], P.cs[2], T, A1[g]);
      }
    }
  }
}

template <bool GUARD>
__device__ __forceinline__ void direction_kinds_fast2(const LayerSeg& P, bool secL, const double (&cur0)[3],
                                                      const double (&cur1)[3], const double (&upR)[3],
                                                      const double (&kap0)[3], const double (&kap1)[3],
                                                      const double (&kR)[3], double (&I0)[3], double (&I1)[3],
                                                      double (&A0)[3], double (&A1)[3], const double* __restrict__ T) {
  const int kind = P.kind;
  if (kind == 0) direction_fast2<1, true, GUARD>(P, cur0, cur1, upR, kap0, kap1, kR, I0, I1, A0, A1, T);
  else if (kind == 1 || kind == 3) {
    if (secL) direction_fast2<2, true, GUARD>(P, cur0, cur1, upR, kap0, kap1, kR, I0, I1, A0, A1, T);
    else direction_fast2<2, false, GUARD>(P, cur0, cur1, upR, kap0, kap1, kR, I0, I1, A0, A1, T);
  } else {
    if (secL) direction_fast2<3, true, GUARD>(P, cur0, cur1, upR, kap0, kap1, kR, I0, I1, A0, A1, T);
    else direction_fast2<3, false, GUARD>(P, cur0, cur1, upR, kap0, kap1, kR, I0, I1, A0, A1, T);
  }
}

// The thin layers of the two-cell kernel (P.thin: 0.2% of the direction-layers): the reference's operation sequence,
// cell by cell, on the unfloored opacities; the upper cell takes the lower one as its (b-1) cell exactly as the
// single-cell kernel does.  Returns the two cells' sums.  Out of line and reloading what it needs, so that none of its
// state is live in the FAST loop.
struct FaithOut2 {
  Tri acc0, acc1;
};
__device__ __noinline__ FaithOut2 thin_pass2(const StepParams& sp, int pidx, int up, int up1, int dstride,
                                             const double* __restrict__ kg, int N, int sB, bool cell0, bool cell1,
                                             bool hasR, bool writer0, bool writer1) {
  double kF0[3], kF1[3], kR[3], acc0[3] = {0., 0., 0.}, acc1[3] = {0., 0., 0.};
#pragma unroll
  for (int g = 0; g < 3; g++) {
    const double* k = kg + (int64_t)g * N;
    kF0[g] = cell0 ? k[0] : 0.;
    kF1[g] = cell1 ? k[sB] : 0.;
    kR[g] = hasR ? k[-sB] : 0.;
  }
  const double* pin = sp.planeIn + 3 * pidx;
  double* pout = sp.planeOut + 3 * pidx;
  for (int q = 0; q < sp.ndir; q++, pin += dstride, pout += dstride) {
    const LayerSeg& P = sp.P[q];
    if (!P.thin) continue;
    const int kind = P.kind;
    double cur0[3], cur1[3], upR[3] = {0., 0., 0.}, I0[3], I1[3];
#pragma unroll
    for (int g = 0; g < 3; g++) { cur0[g] = pin[g]; cur1[g] = pin[g + up1]; }
    const bool secL = (kind <= 2) == (sp.laneIsK != 0);
    if (kind == 2 || kind == 4 || (kind != 0 && !secL)) {
#pragma unroll
      for (int g = 0; g < 3; g++) upR[g] = pin[g - up];
    }
    direction_dispatch_faithful(P, secL, cur0, upR, kF0, kR, I0, acc0);
    direction_dispatch_faithful(P, secL, cur1, cur0, kF1, kF0, I1, acc1);
    if (writer0) {
#pragma unroll
      for (int g = 0; g < 3; g++) pout[g] = I0[g];
    }
    if (writer1) {
#pragma unroll
      for (int g = 0; g < 3; g++) pout[g + up] = I1[g];
    }
  }
  FaithOut2 o;
#pragma unroll
  for (int g = 0; g < 3; g++) { o.acc0.v[g] = acc0[g]; o.acc1.v[g] = acc1[g]; }
  return o;
}

// Positions are row pairs (see lane_position): a lane holds the cell (a, b0) and the one above it.  Register budget: 6
// blocks of 128 threads per SM (80 registers): 24 resident warps per SM instead of 16 at 124 registers, for a kernel
// that is latency-bound (dependent FP64 and shuffle chains; DESIGN.md 4.1, 4.2: 5 blocks at 96 registers gained nothing).  The few spill slots ptxas uses hold
// loop-invariant values: stored before the direction loop, one 4-byte reload per direction, the rest around the call
// of thin_pass2 -- none inside the segment arithmetic.
// The thin layers (P.thin) are swept in a second pass over the directions, after the FAST ones: their sums and the
// FAST sums A0/A1 are separate until the final fma, and every direction has its own plane, so the order of the two
// passes changes no bit.
constexpr int kCell2Warps = 4;  // warps per block at most
__global__ void __launch_bounds__(32 * kCell2Warps, 6)
sweep_cell2_kernel(const __grid_constant__ BatchParams bp, int N, int n, int np1, int npl3) {
  const StepParams& sp = bp.t[blockIdx.z];
  const double* __restrict__ kappa = sp.kappa;
  __shared__ double sT[kExpTableSize];
  asm volatile("griddepcontrol.launch_dependents;");
  if (threadIdx.y * 32 + threadIdx.x < kExpTableSize) sT[threadIdx.y * 32 + threadIdx.x] = kExpTable32[threadIdx.y * 32 + threadIdx.x];
  __syncthreads();
  const LanePos lp = lane_position((n + 1) / 2, np1);
  if (!lp.warpLive) return;                                    // warp-uniform
  const int a = lp.a, b0 = 2 * lp.r;
  const bool row1 = b0 + 1 < n;                                // the upper row exists (not in the last pair of odd n)
  const bool cell0 = a >= 0, cell1 = cell0 && row1;
  const bool writer0 = cell0 && threadIdx.x >= 1, writer1 = writer0 && row1;
  const int laneIsK = sp.laneIsK;
  const int sA = laneIsK ? sp.sk : sp.sj, sB = laneIsK ? sp.sj : sp.sk;
  const int leaf0 = sp.origin + a * sA + b0 * sB;
  double kap0[3], kap1[3], kR[3];
#pragma unroll
  for (int g = 0; g < 3; g++) {
    const double* kg = kappa + (int64_t)g * N + leaf0;
    const double kF0 = cell0 ? kg[0] : 0., kF1 = cell1 ? kg[sB] : 0.;
    kR[g] = (cell0 && b0 > 0) ? kg[-sB] : 0.;                  // kappa = 0 outside: exp(-0) = 1 exactly
    kap0[g] = kF0 > 0. ? kF0 : kKappaFloor;
    kap1[g] = kF1 > 0. ? kF1 : kKappaFloor;
  }
  const double kmax = fmax(fmax(fmax(fmax(kap0[0], kap0[1]), fmax(kap0[2], kR[0])), fmax(kR[1], kR[2])),
                           fmax(fmax(kap1[0], kap1[1]), kap1[2]));
  double A0[3] = {0., 0., 0.}, A1[3] = {0., 0., 0.};
  const int pidx = (b0 + 1) * np1 + a + 1;
  const int ndir = sp.ndir;
  const int dstride = npl3;
  const int up = 3 * np1;                                      // one row up in the plane
  const int up1 = row1 ? up : 0;                               // the upper row's plane values (stay in bounds without it)
  const double* pin = sp.planeIn + 3 * pidx;
  double* pout = sp.planeOut + 3 * pidx;
  asm volatile("griddepcontrol.wait;" ::: "memory");
  for (int q = 0; q < ndir; q++, pin += dstride, pout += dstride) {
    const LayerSeg& P = sp.P[q];
    const int kind = P.kind;
    if (q + 1 < ndir) {
      prefetch_l1(pin + dstride);
      prefetch_l1(pin + dstride + up1);
      prefetch_l1(pin + dstride - up);
    }
    if (P.thin) continue;                                      // second pass
    double cur0[3], cur1[3], upR[3] = {0., 0., 0.}, I0[3], I1[3];
#pragma unroll
    for (int g = 0; g < 3; g++) { cur0[g] = pin[g]; cur1[g] = pin[g + up1]; }
    const bool secL = (kind <= 2) == (laneIsK != 0);
    if (kind == 2 || kind == 4 || (kind != 0 && !secL)) {
#pragma unroll
      for (int g = 0; g < 3; g++) upR[g] = pin[g - up];
    }
    if (__any_sync(0xffffffffu, kmax * P.dmax > 64.))
      direction_kinds_fast2<true>(P, secL, cur0, cur1, upR, kap0, kap1, kR, I0, I1, A0, A1, sT);
    else
      direction_kinds_fast2<false>(P, secL, cur0, cur1, upR, kap0, kap1, kR, I0, I1, A0, A1, sT);
    if (writer0) {
#pragma unroll
      for (int g = 0; g < 3; g++) pout[g] = I0[g];
    }
    if (writer1) {
#pragma unroll
      for (int g = 0; g < 3; g++) pout[g + up] = I1[g];
    }
  }
  FaithOut2 acc = {};
  if (sp.anyThin)
    acc = thin_pass2(sp, pidx, up, up1, dstride, kappa + leaf0, N, sB, cell0, cell1, cell0 && b0 > 0, writer0, writer1);
  if (writer0) {
#pragma unroll
    for (int g = 0; g < 3; g++) {
      const double v = fma(A0[g], kTwoM200 / kap0[g], acc.acc0.v[g]);
      double* p = sp.acc + (int64_t)g * N + leaf0;
      *p = sp.firstInSlot ? v : __dadd_rn(*p, v);
    }
  }
  if (writer1) {
#pragma unroll
    for (int g = 0; g < 3; g++) {
      const double v = fma(A1[g], kTwoM200 / kap1[g], acc.acc1.v[g]);
      double* p = sp.acc + (int64_t)g * N + leaf0 + sB;
      *p = sp.firstInSlot ? v : __dadd_rn(*p, v);
    }
  }
}

// z-major layout.  A zone whose sweep axis is the contiguous (z) axis of the leaf order has its lanes run along y:
// every lane of a kappa load or accumulator store would touch its own 32-byte sector (measured: those 8 zones take 1.7x
// the time of the others).  Such tasks read a z-major copy of kappa, index (z*n + x)*n + y, and write their accumulator
// in the same layout, so that lanes are contiguous again; the final merge transposes those slots back through a
// shared-memory tile.
__global__ void transpose_kappa_kernel(const double* __restrict__ kap, double* __restrict__ kapT, int n) {
  __shared__ double tile[32][33];
  const int x = blockIdx.z % n, g = blockIdx.z / n;
  const int64_t N = (int64_t)n * n * n;
  const int z0 = blockIdx.x * 32, y0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) {   // read leaf order: z contiguous
    const int y = y0 + r, z = z0 + threadIdx.x;
    if (y < n && z < n) tile[r][threadIdx.x] = kap[g * N + ((int64_t)x * n + y) * n + z];
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {   // write z-major: y contiguous
    const int z = z0 + r, y = y0 + threadIdx.x;
    if (y < n && z < n) kapT[g * N + ((int64_t)z * n + x) * n + y] = tile[threadIdx.x][r];
  }
}

// J += sum of the z-major slots [first, first + count), transposed back to leaf order
__global__ void merge_transposed_kernel(const double* __restrict__ acc, int first, int count, int n,
                                        double* __restrict__ J) {
  __shared__ double tile[32][33];
  const int x = blockIdx.z % n, g = blockIdx.z / n;
  const int64_t N = (int64_t)n * n * n, total = 3 * N;
  const int z0 = blockIdx.x * 32, y0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int z = z0 + r, y = y0 + threadIdx.x;
    if (y < n && z < n) {
      const int64_t i = g * N + ((int64_t)z * n + x) * n + y;
      double s = acc[(int64_t)first * total + i];
      for (int k = 1; k < count; k++) s = __dadd_rn(s, acc[(int64_t)(first + k) * total + i]);
      tile[r][threadIdx.x] = s;
    }
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += 8) {
    const int y = y0 + r, z = z0 + threadIdx.x;
    if (y < n && z < n) {
      double* p = J + g * N + ((int64_t)x * n + y) * n + z;
      *p = __dadd_rn(*p, tile[threadIdx.x][r]);
    }
  }
}

// sum of the slot accumulators -> J (fixed order: slot 0, 1, ...)
__global__ void merge_slots_kernel(const double* __restrict__ acc, int nslots, int64_t total, double* __restrict__ J) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    double s = acc[i];
    for (int k = 1; k < nslots; k++) s = __dadd_rn(s, acc[(int64_t)k * total + i]);
    J[i] = s;
  }
}

__global__ void diffuse_rates_kernel(const double* __restrict__ J, int64_t n, double fourPi, double a0, double a1,
                                     double a2, double b3, double c2, double c3, double* k24, double* k25, double* k26) {
  // equiSources.f90:3546-3553
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    double t1 = fourPi * J[i], t2 = fourPi * J[n + i], t3 = fourPi * J[2 * n + i];
    k24[i] = k24[i] + t1 * a0 + t2 * a1 + t3 * a2;
    k25[i] = k25[i] + t3 * b3;
    k26[i] = k26[i] + t2 * c2 + t3 * c3;
  }
}

int launch_diffuse_rates(Context& c, const double* J, const double* ksi24, const double* ksi25, const double* ksi26,
                         double* k24, double* k25, double* k26, cudaStream_t s) {
  int blocks = std::min<int64_t>((c.nleaf + 255) / 256, (int64_t)c.smCount * 16);
  diffuse_rates_kernel<<<blocks, 256, 0, s>>>(J, c.nleaf, 4. * kPi, ksi24[0], ksi24[1], ksi24[2], ksi25[0], ksi26[0],
                                              ksi26[1], k24, k25, k26);
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

// ---------------------------------------------------------------------------------------------------------
// host side: plan + launch
// ---------------------------------------------------------------------------------------------------------
// FAST mode evaluates a layer with the reference's own operation sequence when one of its segments is shorter than
// this (in cells).  Every segment of a cell enters Jmean with weight 1/(nseg * ndirections) whatever its length
// (transportRoutinesModule.f90:953-955), and the reference formula's rounding noise is ~1.1e-16 / tau_segment, so a
// segment disturbs a cell's Jmean by ~1.1e-16 / (576 tau_segment) where all directions contribute alike, and by up to
// ~1.1e-16 / (3 tau_segment) where a single direction dominates (cells shadowed from most sides).  Measured at 128^3
// (tau_cell >= 1e-3): threshold 1e-4 leaves a worst cell at 1.03e-9 between FAST and FAITHFUL, 1e-3 at ~1e-10.
// 0.2% of the (direction, layer) pairs take this branch.
constexpr double kThinLen = 1e-3;

// The layer table a launch reads.  The plan holds the paths d; the FAST layers of the plain sweep read the scaled path
// d * kExpScale that their exponential takes (segment_math.cuh, exp_neg_parts32), in the same slots.  Thin layers
// (the reference's operation sequence), FAITHFUL mode and the emissive sweep read d.
static void fill_step_segs(LayerSeg* P, const LayerSeg* plan, int ndir, bool scaled) {
  for (int q = 0; q < ndir; q++) {
    P[q] = plan[q];
    if (scaled && !P[q].thin)
      for (int s = 0; s < 3; s++) P[q].d[s] = plan[q].d[s] * kExpScale;
  }
}

static LayerSeg make_layer_seg(const RayPattern& p, double cellSize, double weight) {
  LayerSeg L;
  std::memset(&L, 0, sizeof(L));
  double len[3] = {p.xy_len, 0., 0.};
  int kind = 0;
  if (p.xyTop == 1) kind = 0;
  else if (p.yzTop == 1) {  // xy leaves through x = 1 -> yz ray next door
    kind = p.xzActive ? 2 : 1;
    len[1] = p.yz_len;
    len[2] = p.xzActive ? p.xz_len : 0.;
  } else {                  // xy leaves through y = 1 -> xz ray next door
    kind = p.yzActive ? 4 : 3;
    len[1] = p.xz_len;
    len[2] = p.yzActive ? p.yz_len : 0.;
  }
  L.kind = kind;
  L.nseg = 1 + (kind != 0) + (kind == 2 || kind == 4);
  for (int s = 0; s < 3; s++) {
    L.d[s] = cellSize * len[s];
  }
  L.w = weight;
  const double wn = weight / (double)L.nseg;
  L.dmax = std::max(L.d[0], std::max(L.d[1], L.d[2]));
  for (int s = 0; s < 3; s++) L.cs[s] = L.d[s] > 0. ? 1.6069380442589903e60 * wn / L.d[s] : 0.;  // 2^200 wn / d
  L.thin = 0;
  for (int sg = 0; sg < L.nseg; sg++)
    if (len[sg] < kThinLen) L.thin = 1;
  return L;
}


// `warps` = warps per block (8, 4 or 2): small direction shards (multi-GPU ranks) put only a few hundred 8-warp blocks on
// the device per layer, 1.5 "waves" of which cost as much as 2; smaller blocks spread the same warps evenly over the SMs
template <class Kernel, class... Extra>
static cudaError_t launch_layer(Kernel kern, dim3 grid, cudaStream_t s, bool pdl, const BatchParams& bp, int N, int n,
                                int warps, const Extra&... extra) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(32, warps);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, bp, N, n, n + 1, 3 * (n + 1) * (n + 1), extra...);
}

// The layer kernels, the largest block each takes (warps), and how many of its warps an SM holds at that block size --
// from the occupancy calculator, once per context, so that the wave arithmetic below follows the register budgets.
enum SweepKernel { kCell1, kCell1Faithful, kCell2, kEmit, kEmitFaithful };
static int max_block_warps(int k) { return k == kCell2 ? kCell2Warps : 8; }
static cudaError_t resident_warps(Context& c, int k, int* out) {
  int& w = c.uniResidentWarps[k];
  if (w == 0) {
    const int warps = max_block_warps(k), threads = 32 * warps;
    int blocks = 0;
    cudaError_t e = cudaSuccess;
    switch (k) {
      case kCell1: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, sweep_cell_kernel<false>, threads, 0); break;
      case kCell1Faithful: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, sweep_cell_kernel<true>, threads, 0); break;
      case kCell2: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, sweep_cell2_kernel, threads, 0); break;
      case kEmit: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, sweep_cell_emit_kernel<false>, threads, 0); break;
      default: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, sweep_cell_emit_kernel<true>, threads, 0); break;
    }
    if (e != cudaSuccess) return e;
    w = std::max(1, blocks) * warps;
  }
  *out = w;
  return cudaSuccess;
}

// `pdl`: programmatic dependent launch on the previous launch of the stream (only for a layer whose predecessor in
// the stream is the previous layer's sweep kernel)
// `ep` != nullptr: the emissive sweep (sweep_cell_emit_kernel: one cell per thread)
// `warps` (set_tuning "block_warps"): 8, 4 or 2, at most the kernel's largest block; anything else = automatic
static cudaError_t launch_cells(Context& c, bool faithful, bool pdl, dim3 grid, cudaStream_t s, const BatchParams& bp,
                                int N, int n, int cells, int warps, const EtaParams* ep = nullptr) {
  // automatic: two cells per thread pay (1-2%) when the launch has many zone tasks; a small direction shard (3 zone
  // tasks on each of 8 GPUs) is 1.3 waves of two-cell threads but fills the device evenly with one-cell threads
  // (measured on the shards of an 8-GPU run: 7.03 against 7.21 ms mean, 7.31 against 7.93 ms for the slowest rank)
  if (cells == 0) cells = (n >= 192 && grid.z >= 6) ? 2 : 1;
  if (faithful || ep) cells = 1;
  const int k = ep ? (faithful ? kEmitFaithful : kEmit) : faithful ? kCell1Faithful : cells == 2 ? kCell2 : kCell1;
  const int wpl = warps_per_layer(n, cells == 2 ? (n + 1) / 2 : n);   // warps per task and layer
  if (warps != 8 && warps != 4 && warps != 2) {
    // automatic: the largest block that still gives the device ~6 blocks per resident 8 warps
    int resident = 0;
    if (cudaError_t e = resident_warps(c, k, &resident)) return e;
    const long long slots = (long long)c.smCount * resident / 8;
    warps = max_block_warps(k);
    while (warps > 2 && (long long)((wpl + warps - 1) / warps) * grid.z < 6 * slots) warps /= 2;
  }
  warps = std::min(warps, max_block_warps(k));
  grid.x = (unsigned)((wpl + warps - 1) / warps);
  grid.y = 1;
  switch (k) {
    case kEmitFaithful: return launch_layer(sweep_cell_emit_kernel<true>, grid, s, pdl, bp, N, n, warps, *ep);
    case kEmit: return launch_layer(sweep_cell_emit_kernel<false>, grid, s, pdl, bp, N, n, warps, *ep);
    case kCell1Faithful: return launch_layer(sweep_cell_kernel<true>, grid, s, pdl, bp, N, n, warps);
    case kCell2: return launch_layer(sweep_cell2_kernel, grid, s, pdl, bp, N, n, warps);
    default: return launch_layer(sweep_cell_kernel<false>, grid, s, pdl, bp, N, n, warps);
  }
}

int diffuse_uniform(Context& c, int nAngularLevel, const double* uvb, const std::vector<Direction>& dirs,
                    double* dJout, cudaStream_t s, int64_t* nsegOut) {
  const int n = c.nx;
  const int64_t N = c.nleaf, nn = (int64_t)n * n, npl = (int64_t)(n + 1) * (n + 1);
  const int ndir = (int)dirs.size();
  const int64_t nraysTotal = 12LL << (2 * (nAngularLevel - 1));
  const double weight = (double)(1.f / (float)nraysTotal);  // equiSources.f90:1386 (single-precision division)
  const double cellSize = c.boxSize / (double)n;             // equiSources.f90:1570
  const double* etaSrc = c.sweepEta();                       // emission or the scattering source (scattering.cu)
  const bool emit = etaSrc != nullptr;

  // ---- plan: pattern tables and zone tasks.  Depends only on the grid size and the direction list, so it is
  //      cached across the outer transport<->chemistry iterations. ----
  std::string planKey;
  {
    char buf[128];
    snprintf(buf, sizeof(buf), "%d:%a:%d:%d:%d:%d:%d:%d:", n, c.boxSize, nAngularLevel, c.tune.slots, c.tune.dirsPerTask,
             c.tune.transposeZ, (int)emit, c.tune.blockWarps);
    planKey = buf;
    for (const auto& d : dirs) { snprintf(buf, sizeof(buf), "%lld,", (long long)d.iray); planKey += buf; }
  }
  if (planKey != c.uniPlanKey) {
    c.uniTasks.clear();
    std::vector<RayPattern> pat;
    int64_t nseg = 0;
    int planeCursor = 0;
    // Directions per task.  Every task contributes (n/31)*(n/8) blocks per layer launch whatever its direction
    // count, so a shard with few zones (multi-GPU runs) fills the device better when its zones are cut into smaller
    // pieces: pick the piece size that minimises (waves of resident blocks) x (block time ~ directions + fixed part).
    int dpt = std::max(1, std::min(c.tune.dirsPerTask > 0 ? c.tune.dirsPerTask : kMaxDirPerTask, kMaxDirPerTask));
    if (c.tune.dirsPerTask <= 0) {
      int perZone[25] = {0};
      for (int d = 0; d < ndir; d++) perZone[dirs[d].izone]++;
      // in units of one-cell threads in 8-warp blocks (the shard shapes this choice serves run one-cell threads)
      int resident = 0;
      RTB_CUDA(resident_warps(c, kCell1, &resident));
      const int64_t bpt = (warps_per_layer(n, n) + 7) / 8;
      const int64_t cap = (int64_t)c.smCount * resident / 8;   // resident 8-warp blocks
      double best = 1e300;
      for (int d = kMaxDirPerTask; d >= 2; d--) {
        int64_t T = 0;
        int maxPiece = 0;
        for (int z = 1; z <= 24; z++)
          if (perZone[z]) {
            const int pieces = (perZone[z] + d - 1) / d;
            T += pieces;
            maxPiece = std::max(maxPiece, (perZone[z] + pieces - 1) / pieces);
          }
        if (T == 0 || T > kMaxBatch) continue;
        // with the block size chosen per launch (block_warps = 0) a partly filled last wave costs its share only
        const double fill = (double)(T * bpt) / (double)cap;
        const double waves = c.tune.blockWarps == 0 ? std::max(1.0, fill) : std::ceil(fill);
        const double cost = waves * (maxPiece + 1.5);
        if (cost < best * 0.97) { best = cost; dpt = d; }   // prefer larger pieces unless clearly better
      }
    }
    for (int z = 1; z <= 24; z++) {
      std::vector<int> mine;
      for (int d = 0; d < ndir; d++)
        if (dirs[d].izone == z) mine.push_back(d);
      if (mine.empty()) continue;
      const int pieces = ((int)mine.size() + dpt - 1) / dpt;
      size_t o = 0;
      for (int pc = 0; pc < pieces; pc++) {
        const size_t cnt = (mine.size() - o + (pieces - pc) - 1) / (pieces - pc);  // balanced split
        UniTaskHost T;
        ZoneStrides zs = zone_strides(z, n);
        T.origin = zs.origin; T.si = zs.stride[0]; T.sj = zs.stride[1]; T.sk = zs.stride[2];
        T.izone = z;
        T.ndir = (int)cnt;
        T.planeFirst = planeCursor;
        planeCursor += T.ndir;
        int64_t aj = T.sj < 0 ? -T.sj : T.sj, ak = T.sk < 0 ? -T.sk : T.sk;
        T.laneIsK = ak <= aj;
        T.seg.assign((size_t)n * kMaxDirPerTask, LayerSeg());
        for (int q = 0; q < T.ndir; q++) {
          const Direction& dd = dirs[mine[o + q]];
          if (dd.status) return dd.status;
          layer_patterns_level0(dd.phi, dd.theta, n, pat);
          for (int i = 0; i < n; i++) {
            if (pat[i].status) return pat[i].status;
            LayerSeg L = make_layer_seg(pat[i], cellSize, weight);
            T.seg[(size_t)i * kMaxDirPerTask + q] = L;
            nseg += (int64_t)L.nseg * nn;
          }
        }
        o += cnt;
        c.uniTasks.push_back(std::move(T));
      }
    }
    const int ntask = (int)c.uniTasks.size();
    // slots = zone tasks per launch, each with a private J accumulator; batch b = tasks [b*slots, (b+1)*slots)
    int slots = c.tune.slots > 0 ? c.tune.slots : kMaxBatch;
    slots = std::min(std::max(1, std::min(slots, ntask)), kMaxBatch);
    std::vector<int> seen(slots, 0);
    for (int t = 0; t < ntask; t++) c.uniTasks[t].slot = t % slots;
    c.uniStdSlots = slots;
    if (c.tune.transposeZ && ntask <= slots && n >= 32) {
      // every task owns its slot: tasks sweeping along the contiguous axis switch to the z-major layout (see
      // transpose_kappa_kernel) and are moved behind the others so that their slots form one range
      std::stable_partition(c.uniTasks.begin(), c.uniTasks.end(), [](const UniTaskHost& T) { return T.si != 1 && T.si != -1; });
      int nStd = 0;
      for (int t = 0; t < ntask; t++) {
        UniTaskHost& T = c.uniTasks[t];
        T.slot = t;
        if (T.si != 1 && T.si != -1) { nStd++; continue; }
        const int64_t physT[3] = {n, 1, (int64_t)n * n};
        ZoneStrides zs = zone_strides_layout(T.izone, n, physT);
        T.origin = zs.origin; T.si = zs.stride[0]; T.sj = zs.stride[1]; T.sk = zs.stride[2];
        const int64_t aj = T.sj < 0 ? -T.sj : T.sj, ak = T.sk < 0 ? -T.sk : T.sk;
        T.laneIsK = ak <= aj;
        T.transposed = 1;
      }
      c.uniStdSlots = nStd;
      if (nStd < ntask) {
        if (int st = ensure_buffer((void**)&c.dKappaT, &c.kappaTBytes, (size_t)3 * N * sizeof(double))) return st;
        if (emit)
          if (int st = ensure_buffer((void**)&c.dEtaT, &c.etaTBytes, (size_t)3 * N * sizeof(double))) return st;
      }
    }
    for (int t = 0; t < ntask; t++) {  // first task of a slot (in issue order) overwrites the accumulator
      c.uniTasks[t].firstInSlot = !seen[c.uniTasks[t].slot];
      seen[c.uniTasks[t].slot] = 1;
    }
    if (int st = ensure_buffer((void**)&c.dAcc, &c.accBytes, (size_t)slots * 3 * N * sizeof(double))) return st;
    if (int st = ensure_buffer((void**)&c.dPlanes, &c.planeBytes, (size_t)2 * std::max(ndir, 1) * 3 * npl * sizeof(double))) return st;
    c.uniPlanKey = planKey;
    c.uniSlots = slots;
    c.uniNseg = nseg;
    if (c.graphExec) { cudaGraphExecDestroy(c.graphExec); c.graphExec = nullptr; }
  }
  const int ntask = (int)c.uniTasks.size(), slots = c.uniSlots;
  if (nsegOut) *nsegOut = c.uniNseg;
  if (ntask == 0) {
    RTB_CUDA(cudaMemsetAsync(dJout, 0, 3 * N * sizeof(double), s));
    c.lastSweepLaunches = 0;
    c.lastLaunches = 1;
    return RTB200_OK;
  }

  if (int st = ensure_buffer((void**)&c.dAcc, &c.accBytes, (size_t)c.uniSlots * 3 * N * sizeof(double))) return st;
  if (int st = ensure_buffer((void**)&c.dPlanes, &c.planeBytes, (size_t)2 * std::max(ndir, 1) * 3 * npl * sizeof(double))) return st;
  dim3 grid(1, 1, 1);                                        // launch_cells sizes x; z = tasks of the batch
  double* planeA = c.dPlanes;
  double* planeB = c.dPlanes + (size_t)ndir * 3 * npl;
  const bool faithful = c.mathMode == RTB200_MATH_FAITHFUL;
  int64_t nLaunched = 1;

  // Every task (zone) is a chain of n layer steps.  The tasks of a batch advance one layer per launch, each into its own
  // accumulator slot; the batches run one after the other, so task t shares slot t % slots with the tasks of the
  // earlier batches.
  auto issue = [&](cudaStream_t st) -> int {
    if (c.uniStdSlots < (int)c.uniTasks.size() && c.uniStdSlots < c.uniSlots) {
      dim3 tg((n + 31) / 32, (n + 31) / 32, 3 * n);
      transpose_kappa_kernel<<<tg, dim3(32, 8), 0, st>>>(c.dKappa, c.dKappaT, n);
      if (emit) transpose_kappa_kernel<<<tg, dim3(32, 8), 0, st>>>(etaSrc, c.dEtaT, n);
    }
    {  // both plane buffers start as "boundary intensity everywhere": first-layer input and the permanent pads
      const int64_t total = (int64_t)2 * ndir * 3 * npl;
      int blocks = (int)std::min<int64_t>((total + 255) / 256, (int64_t)c.smCount * 16);
      fill_planes_kernel<<<blocks, 256, 0, st>>>(c.dPlanes, npl, total, uvb[0], uvb[1], uvb[2]);
    }
    // fill one task's parameters for one layer
    auto fill = [&](StepParams& sp, const UniTaskHost& T, int step, int first) -> int {
      sp.acc = c.dAcc + (size_t)T.slot * 3 * N;
      sp.kappa = T.transposed ? c.dKappaT : c.dKappa;
      sp.sj = (int32_t)T.sj; sp.sk = (int32_t)T.sk;
      sp.laneIsK = T.laneIsK; sp.n = n;
      sp.planeIn = ((step & 1) ? planeA : planeB) + (size_t)T.planeFirst * 3 * npl;
      sp.planeOut = ((step & 1) ? planeB : planeA) + (size_t)T.planeFirst * 3 * npl;
      sp.origin = (int32_t)(T.origin + step * T.si);
      fill_step_segs(sp.P, &T.seg[(size_t)step * kMaxDirPerTask], T.ndir, !faithful && !emit);
      sp.anyThin = 0;
      for (int q = 0; q < T.ndir; q++) sp.anyThin |= sp.P[q].thin;
      sp.ndir = T.ndir;
      sp.firstInSlot = first;
      return T.ndir;
    };
    static thread_local BatchParams bp;
    static thread_local EtaParams ep;
    const EtaParams* epp = emit ? &ep : nullptr;
    auto etaOf = [&](const UniTaskHost& T) -> const double* { return T.transposed ? c.dEtaT : etaSrc; };
    for (int base = 0; base < ntask; base += slots) {
      const int nb = std::min(slots, ntask - base);
      for (int step = 0; step < n; step++) {
        for (int z = 0; z < nb; z++) {
          const UniTaskHost& T = c.uniTasks[base + z];
          fill(bp.t[z], T, step, T.firstInSlot);  // every layer touches its own cells once per task
          ep.eta[z] = etaOf(T);
        }
        dim3 gz = grid;
        gz.z = nb;
        RTB_CUDA(launch_cells(c, faithful, c.tune.pdl && step > 0, gz, st, bp, (int)N, n, c.tune.cells, c.tune.blockWarps, epp));
        nLaunched++;
      }
    }
    return RTB200_OK;
  };
  RTB_CUDA(cudaEventRecord(c.evSweep0, s));
  if (c.tune.useGraph) {
    // The launch sequence depends only on the plan, the mode and the buffers: capture once, replay afterwards.
    char key[256];
    snprintf(key, sizeof(key), "u:%d:%d:%d:%d:%p:%p:%p:%a:%a:%a:%p:%p", n, ntask, slots,
             (int)faithful * 64 + 10000 * c.tune.pdl + 100000 * c.tune.cells + 1000000 * c.tune.blockWarps,
             (void*)c.dAcc, (void*)c.dPlanes, (void*)c.dKappa, uvb[0], uvb[1], uvb[2], (const void*)etaSrc, (void*)c.dEtaT);
    if (!c.graphExec || c.graphKey != key) {
      if (c.graphExec) { cudaGraphExecDestroy(c.graphExec); c.graphExec = nullptr; }
      cudaGraph_t graph;
      // capture on the internal stream (the caller's stream may be the legacy default stream, which cannot capture)
      RTB_CUDA(cudaStreamBeginCapture(c.stream, cudaStreamCaptureModeThreadLocal));
      int ist = issue(c.stream);
      cudaError_t ce = cudaStreamEndCapture(c.stream, &graph);
      if (ist) return ist;
      RTB_CUDA(ce);
      RTB_CUDA(cudaGraphInstantiate(&c.graphExec, graph, 0));
      cudaGraphDestroy(graph);
      c.graphKey = key;
    }
    RTB_CUDA(cudaGraphLaunch(c.graphExec, s));
  } else {
    if (int ist = issue(s)) return ist;
  }
  RTB_CUDA(cudaEventRecord(c.evSweep1, s));
  {
    const int nStd = std::min(c.uniStdSlots, slots);
    int blocks = std::min<int64_t>((3 * N + 255) / 256, (int64_t)c.smCount * 16);
    if (nStd > 0) merge_slots_kernel<<<blocks, 256, 0, s>>>(c.dAcc, nStd, 3 * N, dJout);
    else RTB_CUDA(cudaMemsetAsync(dJout, 0, 3 * N * sizeof(double), s));
    if (nStd < slots) {
      dim3 tg((n + 31) / 32, (n + 31) / 32, 3 * n);
      merge_transposed_kernel<<<tg, dim3(32, 8), 0, s>>>(c.dAcc, nStd, slots - nStd, n, dJout);
    }
  }
  RTB_CUDA(cudaGetLastError());
  if (nLaunched > 1) c.uniLaunches = nLaunched;  // a replayed graph issues what was captured
  c.lastSweepLaunches = c.uniLaunches;
  c.lastLaunches = c.uniLaunches + 2;  // + compute_opacities + merge
  return RTB200_OK;
}

}  // namespace rtb
