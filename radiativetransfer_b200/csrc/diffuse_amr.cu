// Diffuse sweep on refined (AMR) grids: replaces, per direction, the reference's three passes over the octree --
// pattern assignment (setRaysRefined, transportRoutinesModule.f90:121-218), neighbour threading
// (localizeCellFindNeighbours / findNeighbours / get??Neighbour, :264-558) and transport (:560-963 plus the inline
// base-cell copy equiSources.f90:1580-1788).
//
//  * Patterns depend only on (direction, level, fine layer index along the sweep axis): full tables per level are
//    built on the host (geometry.cpp) -- level L has n*2^L entries, entry 2i / 2i+1 derived from entry i of level
//    L-1 exactly as setRaysRefined derives the lower / upper sub-layer.
//  * Neighbour threading is integer arithmetic on the leaf's rotated coordinates (walk up while the cell sits on the
//    low face of its parent, step to the sibling / base neighbour, descend the linear octree with the `.le.0.5`
//    tests on the exactly halved/doubled entry point).  One thread per (leaf, direction).
//  * Transport order: the reference visits leaves in rotated i/j/k order so that upstream leaves are finished.  Here
//    leaves are grouped in waves; all leaves a leaf reads from lie in earlier waves.  On 2:1-balanced grids the wave
//    is the sum of the leaf's centre coordinates in rotated space, which increases strictly along every dependency
//    edge when neighbouring leaves differ by at most one level; on any other octree it is the leaf's depth in the
//    dependency graph (build_waves).  One launch per wave for all directions of the batch, or one launch for the
//    whole batch whose work items wait for the records they read (amr_stream_kernel).  (tuning amr_order = 0: the
//    round-1 scheme for unbalanced grids -- centre-sum waves, a leaf whose upstream leaf has not been published yet
//    is put on a deferred list that is retried after every 16th wave.)
//  * Items are stored DIRECTION-fastest: the directions of a batch are grouped by zone (up to 8 per group: same index
//    rotation, hence the same upstream leaves away from refinement boundaries), 8 adjacent lanes of a warp work on
//    the 8 directions of one leaf, and the per-item arrays are [group][leaf][8]: what a warp gathers for a leaf --
//    neighbour records, upstream intensities -- is contiguous, and per-leaf data (opacity, pattern index) is read
//    once per 8 lanes.  (A wave is a diagonal plane of the grid: leaf-fastest items shared no sectors at all.)
//  * Per-item arrays are indexed by the leaf's POSITION IN THE WAVE ORDER ("slot"), not by its leaf number: a wave
//    writes one contiguous stretch of neighbour records and intensities, and what it reads -- the records of its
//    upstream leaves, which lie one to three waves back and are ordered the same way -- is close to a stream as well
//    (leaf-indexed records put every leaf of a diagonal wave in its own 256-byte island).  Intensity records are 24
//    bytes (three frequency groups, no pad).
//  * J has a fixed summation order and no atomics: the 8 directions of a group are added by a butterfly, every
//    (group, leaf) writes its sum once into a per-group array, and the groups are added to the result one after the
//    other in group order (independent of how the groups are batched).  On grids that violate the 2:1 balance, where
//    items may be deferred, every item stores its own contribution and the same fixed order is applied afterwards.
//    Everything else is the reference's arithmetic (segment_math.cuh), incl. the coarse-neighbour averaging fallback
//    (transportRoutinesModule.f90:612-634) and the intensity guard (:680-688).
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <thread>

#include "rtb200_internal.h"
#include "segment_math.cuh"

namespace rtb {

struct alignas(32) DevPattern {   // subset of RayPattern the device needs, 128 B = four 32-byte sectors
  // first two sectors: all the sweep reads
  double dpath[3];       // cellSize(level) * len per ray (xy, yz, xz = ray id 0, 1, 2), multiplied on the host
  int8_t top[3];         // xyTop, yzTop, xzTop: which ray (1 xy, 2 yz, 3 xz) leaves through the top / x=1 / y=1 face
  int8_t active[3];      // xy (always), yz, xz
  int8_t level;          // refinement level of the table
  int8_t thin;           // bit r: active ray r is shorter than 1e-3 cell -- FAST arithmetic evaluates THAT segment with the
                         // reference's operation sequence (same rule and reason as the uniform sweep, diffuse_uniform.cu)
  double cs[3];          // FAST arithmetic: weight / (number of active rays * dpath), see amr_transport_leaf
  double pad1;
  // neighbour threading only
  double e0[3], e1[3];   // entry point of each ray on its face: xy (x0,y0), yz (y0,z0), xz (x0,z0)
  double pad2[2];
};
static_assert(sizeof(DevPattern) == 128, "DevPattern is four sectors");

// What the sweep reads of the patterns, for the (up to) 8 directions of a group side by side: the 8 lanes of a leaf
// (same group = same zone = same table index) read 64 contiguous bytes per field, not 8 structs 128 bytes apart
// (the pattern gathers were ~60% of the sweep's L1 sector requests).
struct alignas(32) GroupPattern {
  double dpath[3][8];
  double cs[3][8];
  int32_t flags[8];      // level | thin << 8
};
static_assert(sizeof(GroupPattern) == 416, "13 sectors");

struct AmrDir {          // one direction of the batch
  int8_t src[3], refl[3];  // zone map: physical component c takes rotated index src[c], reflected if refl[c]
  int8_t inv[3];           // rotated axis r is physical component inv[r]
  int8_t combo;            // reflection combination 0..7 -> wave order
  int8_t patRow;           // row of patIdx[6][N] this direction reads: sweep axis (0..2), +3 if that axis is reflected
  int32_t patBase;         // offset of this direction's pattern tables
  int32_t group, lane;     // where the direction's items live: group of the batch, lane 0..7 inside it
  double w;                // weight
};
static_assert(sizeof(AmrDir) == 32, "one sector per direction");
constexpr int kGroup = 8;  // directions per group (a zone has 8 at nAngularLevel = 3)

struct AmrParams {
  const int32_t* child;
  const int32_t *lx, *ly, *lz;
  const int8_t* level;
  const double* kappa;     // [3][N]
  const DevPattern* pats;
  const GroupPattern* gpats; // [group][perDir]
  int32_t perDir;
  const int32_t* levelOff; // [maxLevel+2] offsets of the per-level tables inside one direction's block
  const AmrDir* dirs;
  const int2* groups;      // [ngroups] (first direction of the batch, number of directions <= 8)
  int32_t* nb;             // debugging export only: [ndir][3][N] upstream leaf per ray (xy, yz, xz): -1 boundary, -2 inactive
  uint8_t* code;           // debugging export only: [ndir][3][N] what to read from the upstream leaf
  int32_t* nbc;            // [group][slot][8][4] the same packed for the sweep: upstream SLOT << 3 | code (or -1 / -2) per ray, 16 B per item
  const int32_t* patIdx;   // [6][N] levelOff[level] + coordinate along physical axis a (a = 0..2), then reflected (3..5)
  const double* kappaA;    // [N][6] leaf-major: opacity of the 3 groups, then 1 / max(opacity, floor) (FAST arithmetic);
                           // [N][9] with the emission coefficients of the 3 groups behind them when emission is set
  double* JA;              // [N][3] running sum over the groups, leaf-major, un-interleaved into J at the end
  double* JS;              // balanced grids: [group][N][4] sum over the 8 directions of a group per leaf (one sector)
  double* JI;              // unbalanced grids: [group][slot][8][3] contribution of every item
  double* Iout;            // [group][3 rays][slot][3][8]: the three frequency groups of a (direction, ray, leaf), 8 lanes side by side
  uint8_t* done;           // [group][slot][8]
  const int32_t* slotOf[8];  // per reflection combination: position of every leaf in the wave order
  const int32_t* sorted[8];  // ... and its inverse
  const int32_t* patIdxS;    // streamed sweep: [8 combos][3 axes][N] patIdx in wave order (slot) per reflection combination
  const double* kappaS;      // streamed sweep: [8 combos][N][6 or 9] kappaA in wave order
  uint64_t epochSign;        // streamed sweep: sign bit this sweep's intensity records carry (0 or 1 << 63), see amr_stream_kernel
  int32_t* abortFlag;        // streamed sweep: set by the first poll that gave up, ends every other poll
  int noThin;                // experiments: FAST arithmetic on thin layers as well
  int slotIsLeaf;            // tuning "amr_slots" = 0: per-item arrays indexed by leaf number instead (the round-1 layout)
  double* J;               // [3][N]
  int32_t* err;
  int64_t N;
  int n, maxLevel;
  double u0, u1, u2, cellSize0;
};

// codes: 0,1,2 = take that ray of the neighbour; 3 = 0.5*(xz+xy); 4 = 0.5*(yz+xy); 5 = xy (fallback, no side ray)
__device__ __forceinline__ void rotated_coords(const AmrDir& D, int nL, int px, int py, int pz, int (&r)[3]) {
  const int p[3] = {px, py, pz};
#pragma unroll
  for (int c = 0; c < 3; c++) r[D.src[c]] = D.refl[c] ? nL - 1 - p[c] : p[c];
}

__device__ __forceinline__ void physical_coords(const AmrDir& D, int nL, const int (&r)[3], int (&p)[3]) {
#pragma unroll
  for (int c = 0; c < 3; c++) p[c] = D.refl[c] ? nL - 1 - r[D.src[c]] : r[D.src[c]];
}

// node of the cell with physical coordinates p at level l
__device__ __forceinline__ int node_at(const int32_t* __restrict__ child, int n, int l, const int (&p)[3]) {
  int node = ((p[0] >> l) * n + (p[1] >> l)) * n + (p[2] >> l);
  for (int t = l - 1; t >= 0; t--) node = child[node] + (((p[0] >> t) & 1) << 2) + (((p[1] >> t) & 1) << 1) + ((p[2] >> t) & 1);
  return node;
}

// item (direction lane of a group, slot of the leaf in the group's wave order) -> index into the [group][N][8] arrays
__device__ __forceinline__ int64_t item_index(const AmrParams& P, int group, int lane, int64_t slot) {
  return ((int64_t)group * P.N + slot) * kGroup + lane;
}

// block = 16 leaves x 8 direction lanes, blockIdx.y = group
__global__ void amr_neighbour_kernel(AmrParams P, int ngroups) {
  const int64_t leaf = blockIdx.x * (int64_t)(blockDim.x / kGroup) + threadIdx.x / kGroup;
  const int gi = blockIdx.y, lane = threadIdx.x % kGroup;
  if (leaf >= P.N || gi >= ngroups) return;
  const int2 grp = P.groups[gi];
  if (lane >= grp.y) return;
  const int d = grp.x + lane;
  const AmrDir D = P.dirs[d];
  const int L = P.level[leaf];
  const int nL = P.n << L;
  int r[3];
  rotated_coords(D, nL, P.lx[leaf], P.ly[leaf], P.lz[leaf], r);
  const DevPattern& pat = P.pats[D.patBase + P.levelOff[L] + r[0]];
  // ray id: 0 xy (upstream across the low-i face), 1 yz (low-k face), 2 xz (low-j face)
  for (int ray = 0; ray < 3; ray++) {
    int32_t result = -2;
    uint8_t code = 0;
    if (pat.active[ray]) {
      // face point (a, b): xy -> (x, y), yz -> (y, z), xz -> (x, z); x follows rotated k, y follows j, z follows i
      double a = pat.e0[ray], b = pat.e1[ray];
      const int lead = ray == 0 ? 0 : (ray == 1 ? 2 : 1);            // rotated axis the ray came across
      const int axA = ray == 0 ? 2 : (ray == 1 ? 1 : 2);             // rotated axis of coordinate a
      const int axB = ray == 0 ? 1 : 0;                              // rotated axis of coordinate b
      result = -1;
      for (int l = L; l >= 0; l--) {
        const int sh = L - l;
        int anc[3] = {r[0] >> sh, r[1] >> sh, r[2] >> sh};
        const int idx = l == 0 ? anc[lead] : (anc[lead] & 1);       // 0-based index on the lead axis
        if (idx > 0) {
          anc[lead] -= 1;
          int p[3];
          physical_coords(D, P.n << l, anc, p);
          int node = node_at(P.child, P.n, l, p);
          int lvl = l;
          while (P.child[node] >= 0) {                               // get??Neighbour: descend with .le.0.5
            const int ia = a <= 0.5 ? 0 : 1, ib = b <= 0.5 ? 0 : 1;
            int cr[3];
            cr[lead] = 1;                                            // the child touching our face (index 2)
            cr[axA] = ia;
            cr[axB] = ib;
            int cp[3];
#pragma unroll
            for (int c = 0; c < 3; c++) cp[c] = D.refl[c] ? 1 - cr[D.src[c]] : cr[D.src[c]];
            node = P.child[node] + (cp[0] << 2) + (cp[1] << 1) + cp[2];
            a = ia ? 2. * a - 1. : 2. * a;
            b = ib ? 2. * b - 1. : 2. * b;
            lvl++;
          }
          result = -P.child[node] - 1;
          // selector: the neighbour's xyTop / yzTop / xzTop (transportRoutinesModule.f90:598-634)
          const int nbL = P.level[result];
          int nr[3];
          rotated_coords(D, P.n << nbL, P.lx[result], P.ly[result], P.lz[result], nr);
          const DevPattern& np = P.pats[D.patBase + P.levelOff[nbL] + nr[0]];
          const int sel = np.top[ray];
          if (sel >= 1) {
            code = (uint8_t)(sel - 1);
            if (ray != 0 && !np.active[sel - 1]) atomicMax(P.err, RTB200_ERR_RAY_INACTIVE);
          } else {
            // selector 0 is only legal when reading a coarser neighbour from a refined leaf
            if (L == 0 || L <= nbL) atomicMax(P.err, RTB200_ERR_TOP_SELECTOR);
            code = np.active[2] ? 3 : (np.active[1] ? 4 : 5);
          }
          (void)lvl;
          break;
        }
        // on the low face of the parent: rescale the face point to the parent's units
        const int ca = l == 0 ? (anc[axA] == 0 ? 0 : 1) : (anc[axA] & 1);
        const int cb = l == 0 ? (anc[axB] == 0 ? 0 : 1) : (anc[axB] & 1);
        a = ca ? a / 2. + 0.5 : a / 2.;
        b = cb ? b / 2. + 0.5 : b / 2.;
      }
    }
    if (P.nb) {
      P.nb[((int64_t)d * 3 + ray) * P.N + leaf] = result;
      P.code[((int64_t)d * 3 + ray) * P.N + leaf] = code;
    }
    if (P.nbc) {
      const int32_t* so = P.slotOf[D.combo];
      const int64_t mySlot = P.slotIsLeaf ? leaf : so[leaf];
      const int32_t nbSlot = result >= 0 ? (P.slotIsLeaf ? result : so[result]) : result;
      P.nbc[item_index(P, gi, lane, mySlot) * 4 + ray] = result >= 0 ? ((nbSlot << 3) | code) : result;
    }
  }
}

// leaf-major copies for the sweep's gathers
constexpr double kAmrKappaFloor = 1e-100;  // FAST arithmetic: kappa = 0 is evaluated as this (every formula takes its limit)
// record length of the per-leaf inputs: opacity, 1 / opacity [, emission coefficient]
template <bool EMIT>
__host__ __device__ constexpr int kappa_record() { return EMIT ? 9 : 6; }

template <bool EMIT = false>
__global__ void interleave_kappa_kernel(const double* __restrict__ in, double* __restrict__ out, int64_t N,
                                        const double* __restrict__ eta = nullptr) {
  constexpr int R = kappa_record<EMIT>();
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < 3 * N; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t leaf = i / 3;
    const int g = (int)(i - 3 * leaf);
    const double k = in[g * N + leaf];
    out[leaf * R + g] = k;
    out[leaf * R + 3 + g] = 1.0 / (k > 0. ? k : kAmrKappaFloor);
    if (EMIT) out[leaf * R + 6 + g] = eta[g * N + leaf];
  }
}
__global__ void deinterleave3_kernel(const double* __restrict__ in, double* __restrict__ out, int64_t N) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < 3 * N; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = i / N, leaf = i - g * N;
    out[i] = in[leaf * 3 + g];
  }
}

// streamed sweep: the same per-leaf inputs in wave order, one copy per reflection combination
template <bool EMIT = false>
__global__ void kappa_slots_kernel(const double* __restrict__ in, double* __restrict__ out, AmrParams P,
                                   const double* __restrict__ eta = nullptr) {
  constexpr int R = kappa_record<EMIT>();
  const int64_t N = P.N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < 8 * N; i += (int64_t)gridDim.x * blockDim.x) {
    const int combo = (int)(i / N);
    const int64_t slot = i - combo * N, leaf = P.sorted[combo][slot];
#pragma unroll
    for (int g = 0; g < 3; g++) {
      const double k = in[g * N + leaf];
      out[i * R + g] = k;
      out[i * R + 3 + g] = 1.0 / (k > 0. ? k : kAmrKappaFloor);
      if (EMIT) out[i * R + 6 + g] = eta[g * N + leaf];
    }
  }
}
__global__ void patidx_slots_kernel(const int32_t* __restrict__ patIdx, int32_t* __restrict__ out, AmrParams P) {
  const int64_t N = P.N;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < 24 * N; i += (int64_t)gridDim.x * blockDim.x) {
    const int ca = (int)(i / N), combo = ca / 3, a = ca - 3 * combo;
    const int64_t leaf = P.sorted[combo][i - (int64_t)ca * N];
    out[i] = patIdx[(int64_t)(((combo >> a) & 1) ? 3 + a : a) * N + leaf];
  }
}

// one (leaf, direction): returns false if an upstream leaf is not published yet.  CHECK = false: the grid is 2:1
// balanced, the wave order alone guarantees that every upstream leaf was finished by an earlier launch, so the
// per-leaf `done` flags (three dependent gathers, two fences and a store per item) are not needed.
//
// The item is latency-bound (ncu r01b: 28 of 36 stall cycles per issue are long-scoreboard), so every gather is
// issued before the arithmetic starts: the packed neighbour record first, then -- independent of each other --
// opacity, pattern and the three upstream intensities.  Iout records are 32 bytes (3 groups + pad) per (direction,
// ray, leaf): one sector per upstream read, and only the active rays of a leaf are written.
// word g of the record lies at + g * kGroup: the 8 lanes of a leaf read / write 64 contiguous bytes (two full sectors)
// per frequency group, instead of every third word of 192 bytes
__device__ __forceinline__ int64_t iout_record(const AmrParams& P, int group, int lane, int ray, int64_t slot) {
  return (((int64_t)group * 3 + ray) * P.N + slot) * (3 * kGroup) + lane;
}

__device__ __forceinline__ uint64_t ld_relaxed_u64(const double* p) {
  uint64_t v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// MODE 0: the record was written by an earlier launch.  1: possibly by another block of this launch, guarded by the
// `done` flags: read through L2.  2 (streamed sweep): written by an earlier work item of THIS launch, and valid once
// its sign bit is the sweep's (`first` = the words of a first attempt issued earlier, so that a thread's gathers overlap)
template <int MODE>
__device__ __forceinline__ void load_record(const AmrParams& P, const double* p, double (&v)[3]) {
  if (MODE == 1) {
    v[0] = __ldcg(p); v[1] = __ldcg(p + kGroup); v[2] = __ldcg(p + 2 * kGroup);
  } else if (MODE == 0) {
    v[0] = __ldg(p); v[1] = __ldg(p + kGroup); v[2] = __ldg(p + 2 * kGroup);
  } else {
    uint64_t a = ld_relaxed_u64(p), b = ld_relaxed_u64(p + kGroup), c = ld_relaxed_u64(p + 2 * kGroup);
    unsigned spins = 0;
    // every word validates itself (a 64-bit store is indivisible), so no fence and no ordering between the words
    while ((((a ^ P.epochSign) | (b ^ P.epochSign) | (c ^ P.epochSign)) >> 63) != 0) {
      __nanosleep(100);
      if ((++spins & 63) == 0) {
        if (*(volatile int32_t*)P.abortFlag) break;
        if (spins > (1u << 20)) { atomicExch(P.abortFlag, 1); atomicMax(P.err, RTB200_ERR_CUDA); break; }
      }
      a = ld_relaxed_u64(p); b = ld_relaxed_u64(p + kGroup); c = ld_relaxed_u64(p + 2 * kGroup);
    }
    const uint64_t m = ~(1ull << 63);
    v[0] = __longlong_as_double((long long)(a & m)); v[1] = __longlong_as_double((long long)(b & m));
    v[2] = __longlong_as_double((long long)(c & m));
  }
}

// one segment (three frequency groups) with the reference's operation sequence: the thin segments of FAST arithmetic,
// out of line so that the libm exp / log and the two divisions cost the common path no registers
struct ThinSeg {
  double out[3], J[3];
};
__device__ __noinline__ ThinSeg amr_thin_segment(double i0, double i1, double i2, double k0, double k1, double k2, double dpath) {
  ThinSeg o;
  const double Iin[3] = {i0, i1, i2}, kap[3] = {k0, k1, k2};
  for (int g = 0; g < 3; g++) {
    const SegResult sr = segment_faithful(Iin[g], kap[g], dpath);
    o.out[g] = sr.Iout;
    o.J[g] = sr.J;
  }
  return o;
}
// the same with emission (segment_faithful_emit)
__device__ __noinline__ ThinSeg amr_thin_segment_emit(double i0, double i1, double i2, double k0, double k1, double k2,
                                                      double dpath, double e0, double e1, double e2) {
  ThinSeg o;
  const double Iin[3] = {i0, i1, i2}, kap[3] = {k0, k1, k2}, eta[3] = {e0, e1, e2};
  for (int g = 0; g < 3; g++) {
    const SegResult sr = segment_faithful_emit(Iin[g], kap[g], dpath, eta[g]);
    o.out[g] = sr.Iout;
    o.J[g] = sr.J;
  }
  return o;
}

// Jc = this direction's contribution to the leaf's mean intensity (the caller adds it up)
// EMIT: emission (DESIGN.md 4.6), the coefficients are words 6..8 of the opacity record
template <bool FAITHFUL, int MODE, bool EMIT = false>
__device__ __forceinline__ bool amr_transport_leaf(const AmrParams& P, const AmrDir& D, int gi, int lane, int64_t leaf,
                                                   int64_t slot, double (&Jc)[3], const double* __restrict__ sT) {
  const int64_t item = item_index(P, gi, lane, slot);
  int32_t nbl[3];
  int cd[3];
  {
    const int4 q = *reinterpret_cast<const int4*>(P.nbc + item * 4);
    const int32_t v[3] = {q.x, q.y, q.z};
#pragma unroll
    for (int ray = 0; ray < 3; ray++) {
      nbl[ray] = v[ray] >= 0 ? (v[ray] >> 3) : v[ray];
      cd[ray] = v[ray] & 7;
    }
  }
  constexpr bool CHECK = MODE == 1;
  if (CHECK) {
    asm volatile("griddepcontrol.wait;" ::: "memory");             // the flags are written by the launches before
    const volatile uint8_t* done = P.done;
#pragma unroll
    for (int ray = 0; ray < 3; ray++)
      if (nbl[ray] >= 0 && !done[item_index(P, gi, lane, nbl[ray])]) return false;
    __threadfence();
  }
  // ---- gathers -----------------------------------------------------------------------------------------------
  // pattern of the leaf's (level, layer along the sweep axis): one gather of a precomputed index
  // (streamed sweep: from the copies in wave order -- no leaf number, nothing to wait for but the neighbour record)
  const int32_t pidx = MODE == 2 ? __ldg(P.patIdxS + ((int64_t)D.combo * 3 + D.patRow % 3) * P.N + slot)
                                 : P.patIdx[(int64_t)D.patRow * P.N + leaf];
  constexpr int R = kappa_record<EMIT>();
  const double* kA = MODE == 2 ? P.kappaS + ((int64_t)D.combo * P.N + slot) * R : P.kappaA + leaf * R;
  double kap[3], invk[3], eta[3];
#pragma unroll
  for (int g = 0; g < 3; g++) {
    kap[g] = kA[g];
    invk[g] = FAITHFUL ? 0. : kA[3 + g];
    eta[g] = EMIT ? kA[6 + g] : 0.;
  }
  // Programmatic dependent launch: everything above is geometry or per-sweep input; the upstream intensities below
  // come from the waves before this one (no-op for a grid launched without the attribute)
  if (MODE == 0) asm volatile("griddepcontrol.wait;" ::: "memory");
  double Iin[3][3];
#pragma unroll
  for (int ray = 0; ray < 3; ray++) {
    Iin[ray][0] = P.u0; Iin[ray][1] = P.u1; Iin[ray][2] = P.u2;      // no upstream leaf: the background
    if (nbl[ray] >= 0) {
      // codes 0..2: that ray of the neighbour; 3, 4: mean with its xy ray (below); 5: its xy ray
      const int c = cd[ray];
      load_record<MODE>(P, P.Iout + iout_record(P, gi, lane, c <= 2 ? c : 0, nbl[ray]), Iin[ray]);
    }
  }
  const GroupPattern& pat = P.gpats[(int64_t)gi * P.perDir + pidx];
  const int patFlags = pat.flags[lane];
  const int L = patFlags & 0xff;
  double dpath[3];
#pragma unroll
  for (int ray = 0; ray < 3; ray++) dpath[ray] = pat.dpath[ray][lane];     // cellSize(level) * len (:583, 651)
  // coarse-neighbour averaging fallback (transportRoutinesModule.f90:612-634): rare, a second record
#pragma unroll
  for (int ray = 0; ray < 3; ray++) {
    if (nbl[ray] >= 0 && (cd[ray] == 3 || cd[ray] == 4)) {
      double side[3];
      load_record<MODE>(P, P.Iout + iout_record(P, gi, lane, cd[ray] == 3 ? 2 : 1, nbl[ray]), side);
#pragma unroll
      for (int g = 0; g < 3; g++) Iin[ray][g] = __dmul_rn(0.5, __dadd_rn(side[g], Iin[ray][g]));
    }
  }
  // ---- arithmetic --------------------------------------------------------------------------------------------
  // FAITHFUL: the reference's sequence per segment, J = (sum of the segments' J) / (number of segments) * weight.
  // FAST (segment_math.cuh, as the uniform sweep): J_seg weight / nseg = Iin (1 - e^-tau) / (kappa dpath) * weight / nseg
  //   = [Iin (1 - e^-tau)] * cs / kappa with cs = weight / (nseg dpath) from the host tables and 1 / kappa per leaf:
  //   one table exponential and no division per segment.
  double Jm[3] = {0., 0., 0.};
  double xy[3] = {0., 0., 0.};
  int imean = 0;
  const int thinMask = (!FAITHFUL && !P.noThin) ? (patFlags >> 8) : 0;
  const double kapRaw[3] = {kap[0], kap[1], kap[2]};
  double Jthin[3] = {0., 0., 0.};   // thin segments: sum of the reference-formula segment means (divided by nseg, times w below)
  double E[3] = {0., 0., 0.};       // emission, FAST arithmetic: sum of phi(tau) dpath w / nseg (times eta below)
  const int nact = 1 + (nbl[1] != -2) + (nbl[2] != -2);
  const double wn = EMIT && !FAITHFUL ? D.w * (nact == 1 ? 1.0 : (nact == 2 ? 0.5 : 1.0 / 3.0)) : 0.;
  if (!FAITHFUL) {
#pragma unroll
    for (int g = 0; g < 3; g++) kap[g] = kap[g] > 0. ? kap[g] : kAmrKappaFloor;
  }
  // the reference processes xy, then xz, then yz
  const int order[3] = {0, 2, 1};
#pragma unroll
  for (int q = 0; q < 3; q++) {
    const int ray = order[q];
    if (nbl[ray] == -2) continue;                                    // inactive ray: nobody reads its record
    double out[3];
    if (FAITHFUL) {
#pragma unroll
      for (int g = 0; g < 3; g++) {
        SegResult sr = EMIT ? segment_faithful_emit(Iin[ray][g], kap[g], dpath[ray], eta[g])
                            : segment_faithful(Iin[ray][g], kap[g], dpath[ray]);
        out[g] = sr.Iout;
        Jm[g] = __dadd_rn(Jm[g], sr.J);
      }
    } else if (thinMask & (1 << ray)) {
      const ThinSeg t =
          EMIT ? amr_thin_segment_emit(Iin[ray][0], Iin[ray][1], Iin[ray][2], kapRaw[0], kapRaw[1], kapRaw[2], dpath[ray],
                                       eta[0], eta[1], eta[2])
               : amr_thin_segment(Iin[ray][0], Iin[ray][1], Iin[ray][2], kapRaw[0], kapRaw[1], kapRaw[2], dpath[ray]);
#pragma unroll
      for (int g = 0; g < 3; g++) { out[g] = t.out[g]; Jthin[g] = __dadd_rn(Jthin[g], t.J[g]); }
    } else {
      const double cs = pat.cs[ray][lane];
      const double ds = dpath[ray] * kExpScale;   // the exponential's scaled path, once for the three groups
#pragma unroll
      for (int g = 0; g < 3; g++)
        out[g] = EMIT ? segment_fast_emit<true>(Iin[ray][g], kap[g], ds, cs, sT, Jm[g], eta[g], invk[g], dpath[ray],
                                                dpath[ray] * wn, E[g])
                      : segment_fast<true>(Iin[ray][g], kap[g], ds, cs, sT, Jm[g]);
    }
    if (ray == 0) { xy[0] = out[0]; xy[1] = out[1]; xy[2] = out[2]; }
    imean++;
    double* mine = P.Iout + iout_record(P, gi, lane, ray, slot);
    if (MODE == 2) {   // intensities are >= 0: the sign bit is free to say which sweep wrote the record
#pragma unroll
      for (int g = 0; g < 3; g++)
        __stcg(reinterpret_cast<unsigned long long*>(mine) + g * kGroup,
               (unsigned long long)((uint64_t)__double_as_longlong(out[g]) & ~(1ull << 63)) | P.epochSign);
    } else {
      mine[0] = out[0]; mine[kGroup] = out[1]; mine[2 * kGroup] = out[2];
    }
  }
  if (L > 0) {  // refined path only: guard on the xy ray's sum (transportRoutinesModule.f90:680,803,926)
    const double tmp = __dadd_rn(__dadd_rn(xy[0], xy[1]), xy[2]);
    if (!(tmp < 1.e-20 && tmp > -1.e-20)) atomicMax(P.err, RTB200_ERR_INTENSITY_GUARD);
  }
#pragma unroll
  for (int g = 0; g < 3; g++) {
    if (FAITHFUL) Jc[g] = __dmul_rn(__ddiv_rn(Jm[g], (double)imean), D.w);
    else {
      Jc[g] = Jm[g] * invk[g];
      if (thinMask) Jc[g] += __dmul_rn(__ddiv_rn(Jthin[g], (double)imean), D.w);   // the thin segments' share of sum(J) / nseg * w
      if (EMIT) Jc[g] = fma(eta[g], E[g], Jc[g]);
    }
  }
  if (CHECK) {
    __threadfence();
    ((volatile uint8_t*)P.done)[item] = 1;
  }
  return true;
}

struct WaveParams {
  const int32_t* sorted[8];   // leaves ordered by wave key, per reflection combination
  int32_t begin[8], count[8]; // this wave's range in each order
  int64_t* deferred;          // list of (d << 32 | leaf) that could not run
  int32_t* deferredCount;
  int64_t deferredCap;
};

// block = 16 leaves of the wave x 8 direction lanes; blockIdx.y = group of the batch
template <bool FAITHFUL, bool CHECK, int MINB = 8, bool EMIT = false>
__global__ void __launch_bounds__(128, MINB) amr_wave_kernel(AmrParams P, WaveParams Wp, int ngroups) {
  __shared__ double sT[kExpTableSize];
  asm volatile("griddepcontrol.launch_dependents;");               // the next wave may start its prologue early
  if (!FAITHFUL) {
    if (threadIdx.x < kExpTableSize) sT[threadIdx.x] = kExpTable32[threadIdx.x];
    __syncthreads();
  }
  const int gi = blockIdx.y;
  const int2 grp = P.groups[gi];
  const int lane = threadIdx.x % kGroup;
  const int combo = P.dirs[grp.x].combo;                         // the same for the whole group (one zone)
  const int i = blockIdx.x * (blockDim.x / kGroup) + threadIdx.x / kGroup;
  const bool have = i < Wp.count[combo];                         // uniform over the 8 lanes of a leaf
  const bool mine = have && lane < grp.y;
  double Jc[3] = {0., 0., 0.};
  int64_t leaf = 0;
  int64_t slot = Wp.begin[combo] + i;
  if (have) leaf = Wp.sorted[combo][slot];
  if (P.slotIsLeaf) slot = leaf;
  bool deferred = false;
  if (mine) {
    const int d = grp.x + lane;
    if (!amr_transport_leaf<FAITHFUL, CHECK ? 1 : 0, EMIT>(P, P.dirs[d], gi, lane, leaf, slot, Jc, sT)) {
      deferred = true;
      int q = atomicAdd(Wp.deferredCount, 1);
      if (q < Wp.deferredCap) Wp.deferred[q] = ((int64_t)d << 32) | slot;
      else atomicMax(P.err, RTB200_ERR_NOMEM);
    }
  }
  if (CHECK) {
    // items may finish later (retry kernel): every item keeps its own contribution, added up in fixed order afterwards
    if (have && !deferred) {
      double* q = P.JI + item_index(P, gi, lane, slot) * 3;
      q[0] = Jc[0]; q[1] = Jc[1]; q[2] = Jc[2];                     // lanes without a direction store zeros
    }
    return;
  }
  // the 8 directions of the leaf: butterfly sum (fixed order), one store per (group, leaf)
  double v[3];
#pragma unroll
  for (int g = 0; g < 3; g++) {
    v[g] = Jc[g];
    v[g] = __dadd_rn(v[g], __shfl_xor_sync(0xffffffffu, v[g], 1));
    v[g] = __dadd_rn(v[g], __shfl_xor_sync(0xffffffffu, v[g], 2));
    v[g] = __dadd_rn(v[g], __shfl_xor_sync(0xffffffffu, v[g], 4));
  }
  if (have && lane == 0) {
    double* q = P.JS + ((int64_t)gi * P.N + leaf) * 4;
    *reinterpret_cast<double2*>(q) = make_double2(v[0], v[1]);
    q[2] = v[2];
  }
}

// Streamed sweep (2:1-balanced grids): the whole batch in ONE launch.  The per-wave launches above are latency-bound
// -- a diagonal wave of a 64^3 + 3 levels grid holds ~20K items and takes ~20 us whatever its size, 573 times per
// sweep.  Here resident blocks take work items -- 16 leaves of one wave and group, in wave order -- from a counter, and
// an item simply waits for the upstream intensity records it reads: a record is valid once its three words carry the
// sweep's sign bit (intensities are >= 0, so the sign is free; sweeps alternate it, and every sweep rewrites every
// record that is ever read, so at the start of a sweep all of them carry the other sign).  Work is handed out in wave
// order and a record's writer lies in an earlier wave, so the oldest unfinished item never waits: no deadlock, no
// co-residency requirement, no flags, no fences.  The arithmetic and every summation order are those of the wave
// kernel: results are bit-identical.
struct StreamParams {
  const int2* items;        // (group | leaves << 8, first slot): 1..16 consecutive slots of one wave in the group's order
  int32_t nitems;
  int32_t* counter;         // zero at launch
};

constexpr int kStreamDirs = 192;   // directions of a batch the streamed kernel keeps in shared memory

// Every WARP is a worker of its own (4 leaves x 8 direction lanes = a quarter of a work item): no block barrier couples
// fast and slow leaves.  Lane 0 runs three quarters ahead with the work counter and two ahead with the item record
// (a small per-warp ring in shared memory).  (Prefetching the next quarter's neighbour record, opacities and pattern
// index into L1 was tried: 6% more instructions, no gain -- the kernel is bound by instruction issue at ~24 warps per
// SM, ncu profiles/r02k2_*: IPC 1.75, 1130 warp instructions per quarter, not by the latency of those loads.  Also
// tried: register caps for 5 / 6 / 8 blocks per SM (8.15 / 8.15 / 8.65 ms at 64^3 + 3 levels), and completing the
// partly written 32-byte sectors of the record rows of leaves with inactive lanes so that L2 evicts whole sectors
// (8.56 against 8.37 ms: the extra stores cost more than the avoided fills); the pause between two polls of a missing
// record, 40 ns to 3 us (8.13 ms +- 0.02 throughout, profiles/r02y_amr_stream_poll_interval_*: waiting warps are not what
// limits the kernel); and issuing the first attempt at all three upstream records before examining any (8.22 ms).)
template <bool FAITHFUL, int MINB, bool EMIT = false>
__global__ void __launch_bounds__(128, MINB) amr_stream_kernel(AmrParams P, StreamParams Q, int ndirs, int ngroups) {
  __shared__ double sT[kExpTableSize];
  __shared__ AmrDir sDirs[kStreamDirs];
  __shared__ int2 sGroups[kStreamDirs / kGroup * 2];
  __shared__ int4 sRing[4][4];       // per warp: (group | leaves << 8, first slot, quarter, valid)
  if (threadIdx.x < kExpTableSize) sT[threadIdx.x] = kExpTable32[threadIdx.x];
  if (threadIdx.x < ngroups) sGroups[threadIdx.x] = P.groups[threadIdx.x];
  for (int q = threadIdx.x; q < ndirs * 4; q += blockDim.x)    // 32-byte records, 8 bytes at a time
    reinterpret_cast<double*>(sDirs)[q] = __ldg(reinterpret_cast<const double*>(P.dirs) + q);
  __syncthreads();
  const int w = threadIdx.x >> 5, l32 = threadIdx.x & 31;
  const int lane = l32 % kGroup, li = l32 / kGroup;
  const int total = Q.nitems * 4;
  int cB = 0;
  if (l32 == 0) {
    for (int k = 0; k < 2; k++) {
      const int c = atomicAdd(Q.counter, 1);
      int4 r = make_int4(0, 0, 0, 0);
      if (c < total) { const int2 e = __ldg(Q.items + (c >> 2)); r = make_int4(e.x, e.y, c & 3, 1); }
      sRing[w][k] = r;
    }
    cB = atomicAdd(Q.counter, 1);
  }
  __syncwarp();
  for (int k = 0;; k++) {
    int2 eB = make_int2(0, 0);
    int cA = 0;
    if (l32 == 0) {                          // issued now, consumed after this quarter's work
      if (cB < total) eB = __ldg(Q.items + (cB >> 2));
      cA = atomicAdd(Q.counter, 1);
    }
    const int4 cur = sRing[w][k & 3];
    if (!cur.w) break;
    const int gi = cur.x & 0xff, count = cur.x >> 8, i = cur.z * 4 + li;
    const int2 grp = sGroups[gi];
    const bool have = i < count, mine = have && lane < grp.y;
    const int64_t slot = cur.y + i;
    double Jc[3] = {0., 0., 0.};
    if (mine) amr_transport_leaf<FAITHFUL, 2, EMIT>(P, sDirs[grp.x + lane], gi, lane, 0, slot, Jc, sT);
    __syncwarp();
    double v[3];
#pragma unroll
    for (int g = 0; g < 3; g++) {
      v[g] = Jc[g];
      v[g] = __dadd_rn(v[g], __shfl_xor_sync(0xffffffffu, v[g], 1));
      v[g] = __dadd_rn(v[g], __shfl_xor_sync(0xffffffffu, v[g], 2));
      v[g] = __dadd_rn(v[g], __shfl_xor_sync(0xffffffffu, v[g], 4));
    }
    if (have && lane == 0) {                 // per (group, SLOT): the merge looks the leaf's slot up
      double* q = P.JS + ((int64_t)gi * P.N + slot) * 4;
      *reinterpret_cast<double2*>(q) = make_double2(v[0], v[1]);
      q[2] = v[2];
    }
    if (l32 == 0) {
      sRing[w][(k + 2) & 3] = cB < total ? make_int4(eB.x, eB.y, cB & 3, 1) : make_int4(0, 0, 0, 0);
      cB = cA;
    }
    __syncwarp();
  }
}

template <bool FAITHFUL, bool EMIT = false>
__global__ void amr_retry_kernel(AmrParams P, const int64_t* in, const int32_t* inCount, int64_t* out, int32_t* outCount,
                                 int64_t cap) {
  __shared__ double sT[kExpTableSize];
  if (!FAITHFUL) {
    if (threadIdx.x < kExpTableSize) sT[threadIdx.x] = kExpTable32[threadIdx.x];
    __syncthreads();
  }
  const int n = min((int64_t)*inCount, cap);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int64_t item = in[i];
    const int d = (int)(item >> 32);
    const int64_t slot = item & 0xffffffffLL;
    const int64_t leaf = P.slotIsLeaf ? slot : P.sorted[P.dirs[d].combo][slot];
    double Jc[3];
    if (!amr_transport_leaf<FAITHFUL, 1, EMIT>(P, P.dirs[d], P.dirs[d].group, P.dirs[d].lane, leaf, slot, Jc, sT)) {
      int q = atomicAdd(outCount, 1);
      if (q < cap) out[q] = item;
    } else {
      double* q = P.JI + item_index(P, P.dirs[d].group, P.dirs[d].lane, slot) * 3;
      q[0] = Jc[0]; q[1] = Jc[1]; q[2] = Jc[2];
    }
  }
}

// JA[leaf] += the batch's groups, one after the other in group order (thread = leaf): the summation order of a leaf is
// group 0, 1, 2, ... of the whole call whatever the batching.  ITEMS: the per-item contributions of the unbalanced
// path, the 8 lanes added in the butterfly's order ((0+1)+(2+3))+((4+5)+(6+7)).
template <bool ITEMS, bool BYSLOT = false>
__global__ void amr_merge_kernel(AmrParams P, int ngroups) {
  for (int64_t leaf = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; leaf < P.N; leaf += (int64_t)gridDim.x * blockDim.x) {
    double s[3] = {P.JA[leaf * 3], P.JA[leaf * 3 + 1], P.JA[leaf * 3 + 2]};
    for (int gi = 0; gi < ngroups; gi++) {
      if (ITEMS) {
        const int combo = P.dirs[P.groups[gi].x].combo;
        const double* q = P.JI + item_index(P, gi, 0, P.slotIsLeaf ? leaf : P.slotOf[combo][leaf]) * 3;
#pragma unroll
        for (int g = 0; g < 3; g++) {
          const double a = __dadd_rn(__dadd_rn(q[g], q[3 + g]), __dadd_rn(q[6 + g], q[9 + g]));
          const double b = __dadd_rn(__dadd_rn(q[12 + g], q[15 + g]), __dadd_rn(q[18 + g], q[21 + g]));
          s[g] = __dadd_rn(s[g], __dadd_rn(a, b));
        }
      } else {
        const double* q = P.JS + ((int64_t)gi * P.N + (BYSLOT ? P.slotOf[P.dirs[P.groups[gi].x].combo][leaf] : leaf)) * 4;
        const double2 ab = *reinterpret_cast<const double2*>(q);
        s[0] = __dadd_rn(s[0], ab.x); s[1] = __dadd_rn(s[1], ab.y); s[2] = __dadd_rn(s[2], q[2]);
      }
    }
    P.JA[leaf * 3] = s[0]; P.JA[leaf * 3 + 1] = s[1]; P.JA[leaf * 3 + 2] = s[2];
  }
}

// ---------------------------------------------------------------------------------------------------------
// host
// ---------------------------------------------------------------------------------------------------------
static DevPattern to_dev(const RayPattern& p, double cellSize, int level, double weight) {
  DevPattern q;
  std::memset(&q, 0, sizeof(q));
  const double len[3] = {p.xy_len, p.yz_len, p.xz_len};
  q.level = (int8_t)level;
  for (int r = 0; r < 3; r++) q.dpath[r] = cellSize * len[r];
  q.e0[0] = p.xy_x0; q.e1[0] = p.xy_y0;
  q.e0[1] = p.yz_y0; q.e1[1] = p.yz_z0;
  q.e0[2] = p.xz_x0; q.e1[2] = p.xz_z0;
  q.top[0] = p.xyTop; q.top[1] = p.yzTop; q.top[2] = p.xzTop;
  q.active[0] = 1; q.active[1] = p.yzActive; q.active[2] = p.xzActive;
  const int nseg = 1 + (p.yzActive ? 1 : 0) + (p.xzActive ? 1 : 0);
  for (int r = 0; r < 3; r++)
    if (q.active[r] && len[r] < 1e-3) q.thin |= (int8_t)(1 << r);
  for (int r = 0; r < 3; r++) q.cs[r] = q.active[r] && q.dpath[r] > 0. ? weight / ((double)nseg * q.dpath[r]) : 0.;
  return q;
}

struct AmrPlan {
  bool balanced = false;              // face neighbours differ by at most one level
  std::vector<int32_t> sorted[8];
  std::vector<int32_t> waveStart[8];  // [nkeys + 1]
  int nkeys = 0;
  int32_t* dSorted[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int32_t* dSlotOf[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // inverse of dSorted
  int32_t* dPatIdx = nullptr;         // [6][N], see AmrParams
  int32_t* dPatIdxS = nullptr;        // [8][3][N] the same in wave order (streamed sweep), built on first use
};

// leaf that contains the finest-level cell p (physical coordinates at level Lmax)
static int32_t leaf_at_finest(const Context& c, const int (&p)[3]) {
  const int n = c.nx, Lmax = c.maxLevel;
  int node = ((p[0] >> Lmax) * n + (p[1] >> Lmax)) * n + (p[2] >> Lmax);
  for (int t = Lmax - 1; c.hChild[node] >= 0; t--)
    node = c.hChild[node] + (((p[0] >> t) & 1) << 2) + (((p[1] >> t) & 1) << 1) + ((p[2] >> t) & 1);
  return -(c.hChild[node] + 1);
}

// Waves of the sweep, per reflection combination: `sorted` = leaves ordered by wave, `waveStart` = first position of
// every wave.  All leaves a leaf reads from -- its neighbours across the three low faces in reflected coordinates --
// must lie in earlier waves.
//  * 2:1-balanced grids: wave = sum over the axes of the leaf centre in half-finest-cell units, which increases strictly
//    along every dependency when face neighbours differ by at most one level (see header comment).
//  * any other octree (`byDepth`): no linear function of position and size orders every face pair (a coarse leaf
//    next to leaves two or more levels finer breaks the centre sum either way), so the wave is the leaf's DEPTH in
//    the dependency graph, 1 + max over its upstream face neighbours.  It is computed in one pass over the leaves in
//    Morton order of the reflected coordinates -- the order in which the reference itself visits the tree, and a
//    topological order of the dependencies for ANY octree (a leaf and its upstream face neighbour sit in two children
//    of their lowest common ancestor that differ only in the bit of the crossed axis).  A neighbour of the same size
//    or coarser is looked up and its depth pulled; finer neighbours were visited before and have pushed theirs.
static void build_waves(Context& c, AmrPlan& plan, bool byDepth) {
  const int Lmax = c.maxLevel;
  const int64_t N = c.nleaf;
  const int span = (c.nx << Lmax) * 2;  // centre coordinate range per axis
  const int fine = c.nx << Lmax;        // finest cells per axis
  std::vector<std::vector<int32_t>> keys(8);
  int maxKey[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  auto one_combo = [&](int combo) {
    std::vector<int32_t>& key = keys[combo];
    key.resize((size_t)N);
    if (!byDepth) {
      for (int64_t l = 0; l < N; l++) {
        const int L = c.hLevel[l];
        const int sc = 1 << (Lmax - L);
        const int nL = c.nx << L;
        const int p[3] = {c.hLeafX[l], c.hLeafY[l], c.hLeafZ[l]};
        int k = 0;
        for (int a = 0; a < 3; a++) {
          const int r = (combo >> a) & 1 ? nL - 1 - p[a] : p[a];
          k += (2 * r + 1) * sc;
        }
        key[l] = k;
      }
      return;
    }
    // reflected low corner at the finest level, Morton code of it
    std::vector<uint64_t> morton((size_t)N);
    std::vector<int32_t> order((size_t)N), cand((size_t)N, 0);
    std::vector<int32_t>& depth = key;
    auto rlo = [&](int64_t l, int (&r)[3], int& sz) {
      const int L = c.hLevel[l];
      sz = 1 << (Lmax - L);
      const int p[3] = {c.hLeafX[l] * sz, c.hLeafY[l] * sz, c.hLeafZ[l] * sz};
      for (int a = 0; a < 3; a++) r[a] = (combo >> a) & 1 ? fine - sz - p[a] : p[a];
    };
    for (int64_t l = 0; l < N; l++) {
      int r[3], sz;
      rlo(l, r, sz);
      uint64_t m = 0;
      for (int b = 0; b < 21; b++)
        m |= ((uint64_t)((r[0] >> b) & 1) << (3 * b + 2)) | ((uint64_t)((r[1] >> b) & 1) << (3 * b + 1)) |
             ((uint64_t)((r[2] >> b) & 1) << (3 * b));
      morton[(size_t)l] = m;
      order[(size_t)l] = (int32_t)l;
    }
    std::sort(order.begin(), order.end(), [&](int32_t x, int32_t y) { return morton[(size_t)x] < morton[(size_t)y]; });
    auto physical = [&](const int (&r)[3], int (&p)[3]) {   // reflected finest cell -> physical finest cell
      for (int a = 0; a < 3; a++) p[a] = (combo >> a) & 1 ? fine - 1 - r[a] : r[a];
    };
    int top = 0;
    for (int64_t i = 0; i < N; i++) {
      const int32_t l = order[(size_t)i];
      int r[3], sz;
      rlo(l, r, sz);
      int d = cand[(size_t)l];
      for (int a = 0; a < 3; a++) {          // upstream: the leaf behind the low face, if it is not finer
        if (r[a] == 0) continue;
        int q[3] = {r[0], r[1], r[2]}, p[3];
        q[a] = r[a] - 1;
        physical(q, p);
        const int32_t u = leaf_at_finest(c, p);
        if (c.hLevel[u] <= c.hLevel[l]) d = std::max(d, depth[(size_t)u] + 1);
      }
      depth[(size_t)l] = d;
      top = std::max(top, d);
      for (int a = 0; a < 3; a++) {          // downstream: a coarser leaf behind the high face learns about this one
        if (r[a] + sz >= fine) continue;
        int q[3] = {r[0], r[1], r[2]}, p[3];
        q[a] = r[a] + sz;
        physical(q, p);
        const int32_t dn = leaf_at_finest(c, p);
        if (c.hLevel[dn] < c.hLevel[l]) cand[(size_t)dn] = std::max(cand[(size_t)dn], d + 1);
      }
    }
    maxKey[combo] = top;
  };
  if (byDepth && N > 100000) {   // the eight passes are independent: one host thread each
    std::vector<std::thread> th;
    for (int combo = 0; combo < 8; combo++) th.emplace_back(one_combo, combo);
    for (auto& t : th) t.join();
  } else {
    for (int combo = 0; combo < 8; combo++) one_combo(combo);
  }
  int nkeys = 3 * span + 1;
  if (byDepth) {
    nkeys = 1;
    for (int combo = 0; combo < 8; combo++) nkeys = std::max(nkeys, maxKey[combo] + 1);
  }
  plan.nkeys = nkeys;
  for (int combo = 0; combo < 8; combo++) {
    const std::vector<int32_t>& k = keys[combo];
    std::vector<int32_t>& start = plan.waveStart[combo];
    start.assign(plan.nkeys + 1, 0);
    for (int64_t l = 0; l < N; l++) start[k[l] + 1]++;
    for (int w = 0; w < plan.nkeys; w++) start[w + 1] += start[w];
    std::vector<int32_t> cursor(start.begin(), start.end() - 1);
    plan.sorted[combo].resize((size_t)N);
    for (int64_t l = 0; l < N; l++) plan.sorted[combo][cursor[k[l]]++] = (int32_t)l;
  }
}

// level of the leaf that contains the cell with coordinates p at level l (the leaf may be coarser than l)
static int leaf_level_at(const Context& c, int l, const int (&p)[3]) {
  const int n = c.nx;
  int node = ((p[0] >> l) * n + (p[1] >> l)) * n + (p[2] >> l);
  for (int t = l - 1; t >= 0; t--) {
    if (c.hChild[node] < 0) return l - 1 - t;
    node = c.hChild[node] + (((p[0] >> t) & 1) << 2) + (((p[1] >> t) & 1) << 1) + ((p[2] >> t) & 1);
  }
  return l;
}

static bool grid_is_balanced(const Context& c) {
  for (int64_t leaf = 0; leaf < c.nleaf; leaf++) {
    const int L = c.hLevel[leaf];
    if (L < 2) continue;  // a face neighbour cannot be two levels coarser
    const int nL = c.nx << L;
    for (int f = 0; f < 6; f++) {
      int p[3] = {c.hLeafX[leaf], c.hLeafY[leaf], c.hLeafZ[leaf]};
      p[f >> 1] += (f & 1) ? 1 : -1;
      if (p[f >> 1] < 0 || p[f >> 1] >= nL) continue;
      if (leaf_level_at(c, L, p) < L - 1) return false;
    }
  }
  return true;
}

struct DirTables {
  std::vector<DevPattern> pats;
  std::vector<AmrDir> dirs;           // sorted by zone
  std::vector<int2> groups;           // (first direction, count <= kGroup): consecutive directions of one zone
  std::vector<int32_t> levelOff;
  int perDir = 0;
};

// device buffers of one batch of directions (kept across calls while the sizes fit)
struct AmrBuffers {
  DevPattern* pats = nullptr;
  GroupPattern* gpats = nullptr;
  std::string uploadKey;        // tables + group range whose patterns / directions / groups the device copies hold
  AmrDir* dirs = nullptr;
  int2* groups = nullptr;
  int32_t* levelOff = nullptr;
  int32_t* nb = nullptr;
  uint8_t* code = nullptr;
  int32_t* nbc = nullptr;
  double* kappaA = nullptr;
  double* kappaS = nullptr;     // streamed sweep: [8][N][kappaSRecord]
  int kappaSRecord = 0;
  double* JA = nullptr;
  double* JS = nullptr;
  double* JI = nullptr;
  double* Iout = nullptr;
  uint8_t* done = nullptr;
  int64_t* defA = nullptr;
  int64_t* defB = nullptr;
  int32_t* defCount = nullptr;  // [2]
  int2* items = nullptr;        // streamed sweep: work list of the batch (see StreamParams)
  size_t itemsCap = 0;
  int32_t nitems = 0;
  std::string itemsKey;         // tables + group range the list was built for
  std::string epochKey;         // tables whose records all carry the sign of sweep `epoch` (empty: unknown, re-initialise)
  uint64_t epoch = 0;
  std::string sizeKey;
  int batch = 0, batchNdir = 0;   // batch size (in groups) chosen when the buffers were allocated, and for how many directions
  int batchTune = 0;              // ... under which "amr_batch" setting
  int64_t batchN = 0;             // ... and leaf count
  std::string nbKey;              // grid + direction list whose neighbour tables (nb, code, nbc) the buffers hold
  void release() {
    cudaFree(pats); cudaFree(gpats); cudaFree(dirs); cudaFree(groups); cudaFree(levelOff); cudaFree(nb); cudaFree(code); cudaFree(Iout); cudaFree(done);
    cudaFree(nbc); cudaFree(kappaA); cudaFree(kappaS); cudaFree(JA); cudaFree(JS); cudaFree(JI);
    cudaFree(defA); cudaFree(defB); cudaFree(defCount); cudaFree(items);
    *this = AmrBuffers();
  }
};

struct AmrState {
  AmrPlan plan;
  std::string key;
  DirTables tables;       // per-direction pattern tables of the last call (depend on the grid and the direction list)
  std::string tablesKey;
  AmrBuffers buffers;
};
// the nested-grid state lives in its context (opaque there: rtb200_internal.h only knows the pointer)
static AmrState* state_of(Context& c) {
  if (!c.amrState) c.amrState = new AmrState();
  return static_cast<AmrState*>(c.amrState);
}
void amr_release(Context& c) {
  AmrState* S = static_cast<AmrState*>(c.amrState);
  if (!S) return;
  for (int k = 0; k < 8; k++) { cudaFree(S->plan.dSorted[k]); cudaFree(S->plan.dSlotOf[k]); }
  cudaFree(S->plan.dPatIdx);
  cudaFree(S->plan.dPatIdxS);
  S->buffers.release();
  delete S;
  c.amrState = nullptr;
}

static int ensure_plan(Context& c, AmrState& S) {
  char buf[64];
  snprintf(buf, sizeof(buf), "%p:%lld:%d:%d", (void*)c.tree.child, (long long)c.nleaf, c.maxLevel, c.tune.amrOrder);
  if (S.key == buf) return RTB200_OK;
  for (int k = 0; k < 8; k++) {
    cudaFree(S.plan.dSorted[k]); S.plan.dSorted[k] = nullptr;
    cudaFree(S.plan.dSlotOf[k]); S.plan.dSlotOf[k] = nullptr;
  }
  // `balanced` from here on means "the wave order alone guarantees finished upstream leaves": true for the centre-sum
  // waves of a 2:1-balanced grid and for the depth waves of any other grid; the per-leaf `done` flags and the deferred
  // list remain for tuning "amr_order" = 0 (centre-sum waves whatever the grid: the round-1 scheme, for comparison)
  const bool geomBalanced = grid_is_balanced(c);
  const bool byDepth = c.tune.amrOrder > 0 || (c.tune.amrOrder < 0 && !geomBalanced);
  build_waves(c, S.plan, byDepth);
  S.plan.balanced = geomBalanced || byDepth;
  S.tablesKey.clear();
  {
    std::vector<int32_t> levelOff(c.maxLevel + 2, 0);
    for (int L = 0; L <= c.maxLevel; L++) levelOff[L + 1] = levelOff[L] + (c.nx << L);
    std::vector<int32_t> idx((size_t)6 * c.nleaf);
    for (int64_t l = 0; l < c.nleaf; l++) {
      const int L = c.hLevel[l], nL = c.nx << L;
      const int p[3] = {c.hLeafX[l], c.hLeafY[l], c.hLeafZ[l]};
      for (int a = 0; a < 3; a++) {
        idx[(size_t)a * c.nleaf + l] = levelOff[L] + p[a];
        idx[(size_t)(3 + a) * c.nleaf + l] = levelOff[L] + nL - 1 - p[a];
      }
    }
    cudaFree(S.plan.dPatIdxS); S.plan.dPatIdxS = nullptr;
    cudaFree(S.plan.dPatIdx);
    RTB_CUDA(cudaMalloc((void**)&S.plan.dPatIdx, idx.size() * sizeof(int32_t)));
    RTB_CUDA(cudaMemcpy(S.plan.dPatIdx, idx.data(), idx.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  std::vector<int32_t> inv((size_t)c.nleaf);
  for (int k = 0; k < 8; k++) {
    RTB_CUDA(cudaMalloc((void**)&S.plan.dSorted[k], (size_t)c.nleaf * sizeof(int32_t)));
    RTB_CUDA(cudaMemcpy(S.plan.dSorted[k], S.plan.sorted[k].data(), (size_t)c.nleaf * sizeof(int32_t), cudaMemcpyHostToDevice));
    for (int64_t q = 0; q < c.nleaf; q++) inv[(size_t)S.plan.sorted[k][(size_t)q]] = (int32_t)q;
    RTB_CUDA(cudaMalloc((void**)&S.plan.dSlotOf[k], (size_t)c.nleaf * sizeof(int32_t)));
    RTB_CUDA(cudaMemcpy(S.plan.dSlotOf[k], inv.data(), (size_t)c.nleaf * sizeof(int32_t), cudaMemcpyHostToDevice));
  }
  S.key = buf;
  return RTB200_OK;
}

static int build_dir_tables(Context& c, int nAngularLevel, const std::vector<Direction>& dirs, DirTables& T) {
  const int Lmax = c.maxLevel, n = c.nx;
  const int64_t nraysTotal = 12LL << (2 * (nAngularLevel - 1));
  const double weight = (double)(1.f / (float)nraysTotal);
  T.levelOff.assign(Lmax + 2, 0);
  for (int L = 0; L <= Lmax; L++) T.levelOff[L + 1] = T.levelOff[L] + (n << L);
  T.perDir = T.levelOff[Lmax + 1];
  T.pats.resize((size_t)T.perDir * dirs.size());
  T.dirs.resize(dirs.size());
  // directions of one zone next to each other (stable), cut into groups of at most kGroup
  std::vector<int> order(dirs.size());
  for (size_t d = 0; d < dirs.size(); d++) order[d] = (int)d;
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return dirs[a].izone < dirs[b].izone; });
  T.groups.clear();
  for (size_t d = 0; d < dirs.size(); d++) {
    if (d == 0 || dirs[order[d]].izone != dirs[order[d - 1]].izone || T.groups.back().y == kGroup)
      T.groups.push_back(make_int2((int)d, 0));
    T.groups.back().y++;
  }
  std::vector<RayPattern> cur, next;
  for (size_t d = 0; d < dirs.size(); d++) {
    const Direction& dd = dirs[order[d]];
    if (dd.status) return dd.status;
    ZoneMap m = zone_map(dd.izone);
    AmrDir& A = T.dirs[d];
    int combo = 0;
    for (int cc = 0; cc < 3; cc++) {
      A.src[cc] = m.src[cc]; A.refl[cc] = m.refl[cc];
      A.inv[m.src[cc]] = (int8_t)cc;
      if (m.refl[cc]) combo |= 1 << cc;
    }
    A.combo = (int8_t)combo;
    A.patRow = (int8_t)(A.inv[0] + (A.refl[A.inv[0]] ? 3 : 0));
    A.patBase = (int32_t)(d * T.perDir);
    A.w = weight;
    // which physical axis is the sweep axis, and is it reflected: decides which sub-layers exist in the reference
    const int sweepAxis = A.inv[0];
    layer_patterns_level0(dd.phi, dd.theta, n, cur);
    for (int L = 0; L <= Lmax; L++) {
      const int nL = n << L;
      for (int i = 0; i < nL; i++) {
        const RayPattern& p = cur[i];
        if (p.status) {
          // the reference only builds the patterns of layers that hold cells: level 0 always, deeper levels where a
          // cell of the layer above is refined
          bool needed = (L == 0);
          if (L > 0) {
            const int pi = i >> 1;
            const int phys = A.refl[sweepAxis] ? (n << (L - 1)) - 1 - pi : pi;
            const auto& v = c.refinedLayer[sweepAxis];
            needed = (int)v.size() > L - 1 && !v[L - 1].empty() && v[L - 1][phys];
          }
          if (needed) return p.status;
        }
        T.pats[(size_t)A.patBase + T.levelOff[L] + i] = to_dev(p, (c.boxSize / (double)c.nx) / (double)(1 << L), L, weight);
      }
      if (L < Lmax) {
        layer_patterns_refine(dd.phi, dd.theta, cur, next);
        cur.swap(next);
      }
    }
  }
  return RTB200_OK;
}

// ngroups groups of kGroup item lanes each; debugNb: also the per-direction nb / code arrays of the debugging export
static int alloc_batch(AmrBuffers& B, const DirTables& T, int64_t N, int ngroups, int64_t defCap, bool debugNb,
                       bool balanced) {
  const size_t slots = (size_t)ngroups * kGroup;
  RTB_CUDA(cudaMalloc((void**)&B.pats, (size_t)T.perDir * slots * sizeof(DevPattern)));
  RTB_CUDA(cudaMalloc((void**)&B.gpats, (size_t)T.perDir * ngroups * sizeof(GroupPattern)));
  RTB_CUDA(cudaMalloc((void**)&B.dirs, slots * sizeof(AmrDir)));
  RTB_CUDA(cudaMalloc((void**)&B.groups, (size_t)ngroups * sizeof(int2)));
  RTB_CUDA(cudaMalloc((void**)&B.levelOff, T.levelOff.size() * sizeof(int32_t)));
  if (debugNb) {
    RTB_CUDA(cudaMalloc((void**)&B.nb, slots * 3 * N * sizeof(int32_t)));
    RTB_CUDA(cudaMalloc((void**)&B.code, slots * 3 * N));
    return RTB200_OK;
  }
  RTB_CUDA(cudaMalloc((void**)&B.nbc, slots * 4 * N * sizeof(int32_t)));
  RTB_CUDA(cudaMalloc((void**)&B.kappaA, (size_t)9 * N * sizeof(double)));   // room for the emission coefficients
  RTB_CUDA(cudaMalloc((void**)&B.JA, (size_t)3 * N * sizeof(double)));
  if (balanced) RTB_CUDA(cudaMalloc((void**)&B.JS, (size_t)ngroups * N * 4 * sizeof(double)));
  else RTB_CUDA(cudaMalloc((void**)&B.JI, slots * N * 3 * sizeof(double)));
  RTB_CUDA(cudaMalloc((void**)&B.Iout, slots * N * 9 * sizeof(double)));
  RTB_CUDA(cudaMalloc((void**)&B.done, slots * N));
  RTB_CUDA(cudaMalloc((void**)&B.defA, (size_t)defCap * sizeof(int64_t)));
  RTB_CUDA(cudaMalloc((void**)&B.defB, (size_t)defCap * sizeof(int64_t)));
  RTB_CUDA(cudaMalloc((void**)&B.defCount, 2 * sizeof(int32_t)));
  return RTB200_OK;
}

// groups per batch
static int choose_batch(Context& c, int ngroups) {
  size_t freeB = 0, totalB = 0;
  cudaMemGetInfo(&freeB, &totalB);
  const double perGroup = (double)kGroup * ((double)c.nleaf * (9 * 8 + 16 + 1 + 24) + 1e6);
  int nb = (int)std::max(1.0, std::min((double)ngroups, 0.5 * (double)freeB / perGroup));
  if (c.tune.amrBatch > 0) nb = std::min(nb, std::max(1, c.tune.amrBatch / kGroup));   // the knob counts directions
  return nb;
}

// groups [g0, g0 + ng) of the tables
template <bool EMIT>
static int run_batch(Context& c, AmrState& S, const DirTables& T, int g0, int ng, const double* uvb, double* dJ,
                     cudaStream_t s, bool faithful, AmrBuffers& B, int64_t defCap, int64_t* launches) {
  const int64_t N = c.nleaf;
  const int d0 = T.groups[g0].x;
  const int nd = T.groups[g0 + ng - 1].x + T.groups[g0 + ng - 1].y - d0;
  std::vector<AmrDir> dl(T.dirs.begin() + d0, T.dirs.begin() + d0 + nd);
  std::vector<int2> gl(T.groups.begin() + g0, T.groups.begin() + g0 + ng);
  for (int g = 0; g < ng; g++) {
    gl[g].x -= d0;
    for (int k = 0; k < gl[g].y; k++) {
      AmrDir& A = dl[gl[g].x + k];
      A.patBase = (gl[g].x + k) * T.perDir;
      A.group = g;
      A.lane = k;
    }
  }
  char ub[64];
  snprintf(ub, sizeof(ub), "|%d:%d", g0, ng);
  const std::string ukey = S.tablesKey + ub;
  if (B.uploadKey != ukey || S.tablesKey.empty()) {
    // tables of the batch: a function of the grid and the direction list, kept across the outer iterations
    std::vector<GroupPattern> gp((size_t)ng * T.perDir);
    std::memset(gp.data(), 0, gp.size() * sizeof(GroupPattern));
    for (int g = 0; g < ng; g++)
      for (int k = 0; k < gl[g].y; k++) {
        const DevPattern* src = T.pats.data() + (size_t)(d0 + gl[g].x + k) * T.perDir;
        for (int i = 0; i < T.perDir; i++) {
          GroupPattern& q = gp[(size_t)g * T.perDir + i];
          for (int r = 0; r < 3; r++) { q.dpath[r][k] = src[i].dpath[r]; q.cs[r][k] = src[i].cs[r]; }
          q.flags[k] = (int32_t)(uint8_t)src[i].level | ((int32_t)(uint8_t)src[i].thin << 8);
        }
      }
    RTB_CUDA(cudaMemcpyAsync(B.pats, T.pats.data() + (size_t)d0 * T.perDir, (size_t)T.perDir * nd * sizeof(DevPattern),
                             cudaMemcpyHostToDevice, s));
    RTB_CUDA(cudaMemcpyAsync(B.gpats, gp.data(), gp.size() * sizeof(GroupPattern), cudaMemcpyHostToDevice, s));
    RTB_CUDA(cudaMemcpyAsync(B.dirs, dl.data(), (size_t)nd * sizeof(AmrDir), cudaMemcpyHostToDevice, s));
    RTB_CUDA(cudaMemcpyAsync(B.groups, gl.data(), (size_t)ng * sizeof(int2), cudaMemcpyHostToDevice, s));
    RTB_CUDA(cudaMemcpyAsync(B.levelOff, T.levelOff.data(), T.levelOff.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
    RTB_CUDA(cudaStreamSynchronize(s));  // the sources are locals
    B.uploadKey = ukey;
  }
  if (!S.plan.balanced) RTB_CUDA(cudaMemsetAsync(B.done, 0, (size_t)ng * kGroup * N, s));
  RTB_CUDA(cudaMemsetAsync(B.defCount, 0, 2 * sizeof(int32_t), s));
  AmrParams P;
  P.child = c.tree.child; P.lx = c.tree.leafX; P.ly = c.tree.leafY; P.lz = c.tree.leafZ; P.level = c.dLevel;
  P.kappa = c.dKappa; P.pats = B.pats; P.gpats = B.gpats; P.perDir = T.perDir; P.levelOff = B.levelOff; P.dirs = B.dirs; P.nb = nullptr; P.code = nullptr;
  P.groups = B.groups;
  P.Iout = B.Iout; P.done = B.done; P.J = dJ; P.err = c.dErr; P.N = N; P.n = c.nx; P.maxLevel = c.maxLevel;
  P.nbc = B.nbc; P.patIdx = S.plan.dPatIdx; P.kappaA = B.kappaA; P.JA = B.JA; P.JS = B.JS; P.JI = B.JI;
  for (int k = 0; k < 8; k++) { P.slotOf[k] = S.plan.dSlotOf[k]; P.sorted[k] = S.plan.dSorted[k]; }
  P.slotIsLeaf = c.tune.amrSlots == 0; P.noThin = c.tune.amrThin == 0;
  P.epochSign = 0; P.abortFlag = B.defCount + 1; P.patIdxS = nullptr; P.kappaS = nullptr;
  P.u0 = uvb[0]; P.u1 = uvb[1]; P.u2 = uvb[2];
  P.cellSize0 = c.boxSize / (double)c.nx;  // equiSources.f90:1570
  // neighbour threading is geometry only (grid + directions): when one batch holds every direction of the call, the
  // tables stay valid across the outer transport <-> chemistry iterations
  const bool wholeCall = g0 == 0 && ng == (int)T.groups.size();
  if (!(wholeCall && !S.tablesKey.empty() && B.nbKey == S.tablesKey)) {
    dim3 grid((unsigned)((N + 15) / 16), ng);
    amr_neighbour_kernel<<<grid, 128, 0, s>>>(P, ng);
    (*launches)++;
    B.nbKey = wholeCall ? S.tablesKey : std::string();
  }
  // One launch for the whole batch, or one per wave?  Measured (profiles/r02k_*): 64^3 + 3 levels (21K leaf-groups per
  // wave) 8.45 against 9.15 ms, 128^3 + 2 levels (87K per wave) 49.1 against 43.9 ms -- the streamed path saves the
  // launch hand-overs of small waves and pays for its wave-ordered opacity copies and the merge's slot look-up.
  int nonEmpty = 0;
  for (int w = 0; w < S.plan.nkeys; w++)
    for (int k = 0; k < 8; k++)
      if (S.plan.waveStart[k][w + 1] > S.plan.waveStart[k][w]) { nonEmpty++; break; }
  const double perWave = (double)N * ng / std::max(1, nonEmpty);
  const bool smallWaves = perWave < 40000.;
  const bool wantStream = c.tune.amrStream > 0 || (c.tune.amrStream < 0 && smallWaves);
  if (S.plan.balanced && wantStream && !P.slotIsLeaf && nd <= kStreamDirs && ng <= kStreamDirs / kGroup * 2) {
    // ---- one launch for the whole batch (amr_stream_kernel) ----
    char kb[64];
    snprintf(kb, sizeof(kb), "|%d:%d", g0, ng);
    const std::string ikey = S.tablesKey + kb;
    if (B.itemsKey != ikey) {
      std::vector<int2> items;
      for (int w = 0; w < S.plan.nkeys; w++)
        for (int g = 0; g < ng; g++) {
          const int combo = dl[gl[g].x].combo;
          const int begin = S.plan.waveStart[combo][w], cnt = S.plan.waveStart[combo][w + 1] - begin;
          for (int off = 0; off < cnt; off += 16) items.push_back(make_int2(g | (std::min(16, cnt - off) << 8), begin + off));
        }
      if (items.size() > B.itemsCap) {
        cudaFree(B.items);
        B.items = nullptr; B.itemsCap = 0;
        RTB_CUDA(cudaMalloc((void**)&B.items, items.size() * sizeof(int2)));
        B.itemsCap = items.size();
      }
      RTB_CUDA(cudaMemcpyAsync(B.items, items.data(), items.size() * sizeof(int2), cudaMemcpyHostToDevice, s));
      RTB_CUDA(cudaStreamSynchronize(s));
      B.nitems = (int32_t)items.size();
      B.itemsKey = ikey;
    }
    // sign epoch of the intensity records: alternates from sweep to sweep while the same records are rewritten
    if (wholeCall && !S.tablesKey.empty() && B.epochKey == S.tablesKey) B.epoch++;
    else {
      RTB_CUDA(cudaMemsetAsync(B.Iout, 0, (size_t)ng * kGroup * N * 9 * sizeof(double), s));   // sign 0 everywhere
      B.epoch = 1;
      B.epochKey = wholeCall ? S.tablesKey : std::string();
    }
    P.epochSign = (B.epoch & 1) ? (1ull << 63) : 0ull;
    P.abortFlag = B.defCount + 1;
    // per-leaf inputs in wave order: pattern indices once per grid, opacities every sweep
    const int cb = (int)std::min<int64_t>((8 * N + 255) / 256, (int64_t)c.smCount * 16);
    if (!S.plan.dPatIdxS) {
      RTB_CUDA(cudaMalloc((void**)&S.plan.dPatIdxS, (size_t)24 * N * sizeof(int32_t)));
      patidx_slots_kernel<<<cb, 256, 0, s>>>(S.plan.dPatIdx, S.plan.dPatIdxS, P);
      (*launches)++;
    }
    constexpr int R = kappa_record<EMIT>();
    if (B.kappaS && B.kappaSRecord < R) { cudaFree(B.kappaS); B.kappaS = nullptr; }
    if (!B.kappaS) {
      RTB_CUDA(cudaMalloc((void**)&B.kappaS, (size_t)8 * N * R * sizeof(double)));
      B.kappaSRecord = R;
    }
    kappa_slots_kernel<EMIT><<<cb, 256, 0, s>>>(c.dKappa, B.kappaS, P, c.sweepEta());
    (*launches)++;
    P.patIdxS = S.plan.dPatIdxS; P.kappaS = B.kappaS;
    StreamParams Q;
    Q.items = B.items; Q.nitems = B.nitems; Q.counter = B.defCount;
    int perSm = 0;
    if (faithful) {
      RTB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, amr_stream_kernel<true, 4, EMIT>, 128, 0));
      amr_stream_kernel<true, 4, EMIT><<<std::min(perSm * c.smCount, (int)B.nitems), 128, 0, s>>>(P, Q, nd, ng);
    } else if (c.tune.amrMinBlocks >= 8) {
      RTB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, amr_stream_kernel<false, 8, EMIT>, 128, 0));
      amr_stream_kernel<false, 8, EMIT><<<std::min(perSm * c.smCount, (int)B.nitems), 128, 0, s>>>(P, Q, nd, ng);
    } else if (c.tune.amrMinBlocks == 5) {
      RTB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, amr_stream_kernel<false, 5, EMIT>, 128, 0));
      amr_stream_kernel<false, 5, EMIT><<<std::min(perSm * c.smCount, (int)B.nitems), 128, 0, s>>>(P, Q, nd, ng);
    } else {
      RTB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&perSm, amr_stream_kernel<false, 6, EMIT>, 128, 0));
      amr_stream_kernel<false, 6, EMIT><<<std::min(perSm * c.smCount, (int)B.nitems), 128, 0, s>>>(P, Q, nd, ng);
    }
    (*launches)++;
    const int blocks = (int)std::min<int64_t>((N + 127) / 128, (int64_t)c.smCount * 16);
    amr_merge_kernel<false, true><<<blocks, 128, 0, s>>>(P, ng);
    (*launches)++;
    RTB_CUDA(cudaGetLastError());
    return RTB200_OK;
  }
  B.epochKey.clear();   // the launches below write plain (unsigned) records
  WaveParams Wp;
  for (int k = 0; k < 8; k++) Wp.sorted[k] = S.plan.dSorted[k];
  Wp.deferredCap = defCap;
  int cur = 0;  // deferred list written by the wave kernels / read by the retry kernel
  int64_t* lists[2] = {B.defA, B.defB};
  bool used[8] = {false, false, false, false, false, false, false, false};
  for (int i = 0; i < nd; i++) used[dl[i].combo] = true;
  bool prevWasWave = false;
  for (int w = 0; w < S.plan.nkeys; w++) {
    int maxCount = 0;
    for (int k = 0; k < 8; k++) {
      Wp.begin[k] = S.plan.waveStart[k][w];
      Wp.count[k] = S.plan.waveStart[k][w + 1] - S.plan.waveStart[k][w];
      if (used[k]) maxCount = std::max(maxCount, Wp.count[k]);
    }
    if (maxCount == 0) continue;
    Wp.deferred = lists[cur];
    Wp.deferredCount = B.defCount + cur;
    dim3 grid((maxCount + 15) / 16, ng);
    const bool check = !S.plan.balanced;
    // programmatic dependent launch on the previous wave (not for the first wave, nor right after a retry kernel)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = 0; cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = (c.tune.pdl && prevWasWave) ? 1 : 0;
    if (faithful) {
      if (check) RTB_CUDA(cudaLaunchKernelEx(&cfg, amr_wave_kernel<true, true, 8, EMIT>, P, Wp, ng));
      else RTB_CUDA(cudaLaunchKernelEx(&cfg, amr_wave_kernel<true, false, 8, EMIT>, P, Wp, ng));
    } else {
      if (check) RTB_CUDA(cudaLaunchKernelEx(&cfg, amr_wave_kernel<false, true, 8, EMIT>, P, Wp, ng));
      else if (c.tune.amrMinBlocks > 0 ? c.tune.amrMinBlocks <= 6 : smallWaves)
        RTB_CUDA(cudaLaunchKernelEx(&cfg, amr_wave_kernel<false, false, 6, EMIT>, P, Wp, ng));
      else RTB_CUDA(cudaLaunchKernelEx(&cfg, amr_wave_kernel<false, false, 8, EMIT>, P, Wp, ng));
    }
    prevWasWave = true;
    (*launches)++;
    if (check && (w & 15) == 15) {
      // retry what has been deferred so far (nothing on 2:1-balanced grids)
      RTB_CUDA(cudaMemsetAsync(B.defCount + (cur ^ 1), 0, sizeof(int32_t), s));
      if (faithful) amr_retry_kernel<true, EMIT><<<64, 128, 0, s>>>(P, lists[cur], B.defCount + cur, lists[cur ^ 1], B.defCount + (cur ^ 1), defCap);
      else amr_retry_kernel<false, EMIT><<<64, 128, 0, s>>>(P, lists[cur], B.defCount + cur, lists[cur ^ 1], B.defCount + (cur ^ 1), defCap);
      (*launches)++;
      cur ^= 1;
      prevWasWave = false;
    }
  }
  // drain the deferred list
  for (int iter = 0; iter < 100000 && !S.plan.balanced; iter++) {
    int32_t cnt = 0;
    RTB_CUDA(cudaMemcpyAsync(&cnt, B.defCount + cur, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    RTB_CUDA(cudaStreamSynchronize(s));
    if (cnt == 0) break;
    if (cnt > defCap) return RTB200_ERR_NOMEM;
    RTB_CUDA(cudaMemsetAsync(B.defCount + (cur ^ 1), 0, sizeof(int32_t), s));
    if (faithful) amr_retry_kernel<true, EMIT><<<256, 128, 0, s>>>(P, lists[cur], B.defCount + cur, lists[cur ^ 1], B.defCount + (cur ^ 1), defCap);
    else amr_retry_kernel<false, EMIT><<<256, 128, 0, s>>>(P, lists[cur], B.defCount + cur, lists[cur ^ 1], B.defCount + (cur ^ 1), defCap);
    (*launches)++;
    cur ^= 1;
    if (iter == 99999) return RTB200_ERR_ARG;
  }
  {
    const int blocks = (int)std::min<int64_t>((N + 127) / 128, (int64_t)c.smCount * 16);
    if (S.plan.balanced) amr_merge_kernel<false><<<blocks, 128, 0, s>>>(P, ng);
    else amr_merge_kernel<true><<<blocks, 128, 0, s>>>(P, ng);
    (*launches)++;
  }
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

int diffuse_amr(Context& c, int nAngularLevel, const double* uvb, const std::vector<Direction>& dirs, double* dJout,
                cudaStream_t s, int64_t* nsegOut) {
  const int64_t N = c.nleaf;
  AmrState& S = *state_of(c);
  if (int st = ensure_plan(c, S)) return st;
  RTB_CUDA(cudaMemsetAsync(dJout, 0, 3 * N * sizeof(double), s));
  c.lastSweepLaunches = 0;
  c.lastLaunches = 2;
  if (nsegOut) *nsegOut = 0;
  if (dirs.empty()) return RTB200_OK;
  // pattern tables: a function of the grid and of the direction list -> kept across the outer iterations
  std::string tkey = S.key;
  {
    char buf[48];
    snprintf(buf, sizeof(buf), "|%d|%a|%d|", nAngularLevel, c.boxSize, c.tune.amrSlots);
    tkey += buf;
    for (const auto& d : dirs) { snprintf(buf, sizeof(buf), "%lld,", (long long)d.iray); tkey += buf; }
  }
  if (S.tablesKey != tkey) {
    S.tables = DirTables();
    if (int st = build_dir_tables(c, nAngularLevel, dirs, S.tables)) return st;
    S.tablesKey = tkey;
  }
  DirTables& T = S.tables;
  const int ndir = (int)dirs.size();
  const int ngroups = (int)T.groups.size();
  AmrBuffers& B = S.buffers;
  // the cached buffers count as used memory: keep their batch size instead of choosing a smaller one every call
  const bool keep = B.batch > 0 && B.batchNdir == ndir && B.batchTune == c.tune.amrBatch && B.batchN == N;
  if (!keep) B.release();   // so that the new choice sees the memory they held
  const int batch = keep ? std::min(B.batch, ngroups) : choose_batch(c, ngroups);
  const int64_t defCap = std::max<int64_t>(1 << 16, std::min<int64_t>((int64_t)batch * kGroup * N, (int64_t)1 << 26));
  int st = RTB200_OK;
  {
    char buf[96];
    snprintf(buf, sizeof(buf), "%d:%lld:%d:%lld:%d", T.perDir, (long long)N, batch, (long long)defCap, (int)S.plan.balanced);   // (J per group or per item)
    if (B.sizeKey != buf) {
      B.release();
      st = alloc_batch(B, T, N, batch, defCap, false, S.plan.balanced);  // (release() also forgets the cached neighbour tables)
      if (st) B.release();
      else { B.sizeKey = buf; B.batch = batch; B.batchNdir = ndir; B.batchTune = c.tune.amrBatch; B.batchN = N; }
    }
  }
  int64_t launches = 0;
  const bool faithful = c.mathMode == RTB200_MATH_FAITHFUL;
  const double* etaSrc = c.sweepEta();   // emission or the scattering source: the sweep kernels' EMIT instantiations
  const bool emit = etaSrc != nullptr;
  const int cpyBlocks = (int)std::min<int64_t>((3 * N + 255) / 256, (int64_t)c.smCount * 16);
  if (!st) {
    if (emit) interleave_kappa_kernel<true><<<cpyBlocks, 256, 0, s>>>(c.dKappa, B.kappaA, N, etaSrc);
    else interleave_kappa_kernel<false><<<cpyBlocks, 256, 0, s>>>(c.dKappa, B.kappaA, N);
    RTB_CUDA(cudaMemsetAsync(B.JA, 0, 3 * N * sizeof(double), s));
    launches += 1;
  }
  for (int g0 = 0; g0 < ngroups && !st; g0 += batch)
    st = (emit ? run_batch<true> : run_batch<false>)(c, S, T, g0, std::min(batch, ngroups - g0), uvb, dJout, s, faithful, B,
                                                     defCap, &launches);
  if (!st) {
    deinterleave3_kernel<<<cpyBlocks, 256, 0, s>>>(B.JA, dJout, N);
    launches += 1;
  }
  if (!st && nsegOut) {
    // segment count: leaves per (level, layer) times the layer's segments -- from the host tables
    std::vector<std::vector<int64_t>> hist[3];  // per physical sweep axis: [level][layer] leaf counts
    for (int a = 0; a < 3; a++) {
      hist[a].resize(c.maxLevel + 1);
      for (int L = 0; L <= c.maxLevel; L++) hist[a][L].assign((size_t)c.nx << L, 0);
    }
    for (int64_t l = 0; l < N; l++) {
      const int L = c.hLevel[l];
      hist[0][L][c.hLeafX[l]]++; hist[1][L][c.hLeafY[l]]++; hist[2][L][c.hLeafZ[l]]++;
    }
    int64_t nseg = 0;
    for (int d = 0; d < ndir; d++) {
      const AmrDir& A = T.dirs[d];
      const int ax = A.inv[0];
      for (int L = 0; L <= c.maxLevel; L++) {
        const int nL = c.nx << L;
        for (int i = 0; i < nL; i++) {
          const int phys = A.refl[ax] ? nL - 1 - i : i;
          const int64_t cnt = hist[ax][L][phys];
          if (!cnt) continue;
          const DevPattern& p = T.pats[(size_t)A.patBase + T.levelOff[L] + i];
          nseg += cnt * (1 + p.active[1] + p.active[2]);
        }
      }
    }
    *nsegOut = nseg;
  }
  cudaStreamSynchronize(s);
  if (!B.epochKey.empty()) {   // a streamed sweep that gave up leaves records of both signs behind
    int32_t gaveUp = 0;
    if (cudaMemcpy(&gaveUp, B.defCount + 1, sizeof(int32_t), cudaMemcpyDeviceToHost) != cudaSuccess || gaveUp) B.epochKey.clear();
  }
  if (st) B.epochKey.clear();
  c.lastSweepLaunches = launches;
  c.lastLaunches = launches + 2;
  return st;
}

// debugging export: upstream leaf per ray for one direction (xy, yz, xz)
int amr_neighbours(Context& c, const Direction& d, int32_t* nbHost) {
  const int64_t N = c.nleaf;
  if (c.uniform && !c.tune.forceAmr) {
    // implicit on a uniform grid: the (i-1), (k-1), (j-1) cell of the rotated lattice when the ray is active
    std::vector<RayPattern> pat;
    layer_patterns_level0(d.phi, d.theta, c.nx, pat);
    ZoneStrides zs = zone_strides(d.izone, c.nx);
    const int n = c.nx;
    for (int i = 0; i < n; i++) {
      if (pat[i].status) return pat[i].status;
      for (int j = 0; j < n; j++)
        for (int k = 0; k < n; k++) {
          const int64_t leaf = zs.origin + i * zs.stride[0] + j * zs.stride[1] + k * zs.stride[2];
          nbHost[leaf] = i > 0 ? (int32_t)(leaf - zs.stride[0]) : -1;
          nbHost[N + leaf] = !pat[i].yzActive ? -2 : (k > 0 ? (int32_t)(leaf - zs.stride[2]) : -1);
          nbHost[2 * N + leaf] = !pat[i].xzActive ? -2 : (j > 0 ? (int32_t)(leaf - zs.stride[1]) : -1);
        }
    }
    return RTB200_OK;
  }
  std::vector<Direction> one{d};
  DirTables T;
  if (int st = build_dir_tables(c, 3, one, T)) return st;
  AmrBuffers B;
  if (int st = alloc_batch(B, T, N, 1, 16, true, true)) { B.release(); return st; }
  cudaStream_t s = c.stream;
  RTB_CUDA(cudaMemcpyAsync(B.pats, T.pats.data(), T.pats.size() * sizeof(DevPattern), cudaMemcpyHostToDevice, s));
  T.dirs[0].group = 0; T.dirs[0].lane = 0;
  RTB_CUDA(cudaMemcpyAsync(B.dirs, T.dirs.data(), sizeof(AmrDir), cudaMemcpyHostToDevice, s));
  RTB_CUDA(cudaMemcpyAsync(B.groups, T.groups.data(), sizeof(int2), cudaMemcpyHostToDevice, s));
  RTB_CUDA(cudaMemcpyAsync(B.levelOff, T.levelOff.data(), T.levelOff.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  AmrParams P;
  std::memset(&P, 0, sizeof(P));
  P.groups = B.groups;
  P.child = c.tree.child; P.lx = c.tree.leafX; P.ly = c.tree.leafY; P.lz = c.tree.leafZ; P.level = c.dLevel;
  P.pats = B.pats; P.levelOff = B.levelOff; P.dirs = B.dirs; P.nb = B.nb; P.code = B.code; P.err = c.dErr;
  P.N = N; P.n = c.nx; P.maxLevel = c.maxLevel;
  dim3 grid((unsigned)((N + 15) / 16), 1);
  amr_neighbour_kernel<<<grid, 128, 0, s>>>(P, 1);
  RTB_CUDA(cudaMemcpyAsync(nbHost, B.nb, (size_t)3 * N * sizeof(int32_t), cudaMemcpyDeviceToHost, s));
  RTB_CUDA(cudaStreamSynchronize(s));
  B.release();
  // selector / activity errors found while threading are reported by the sweep, not by this view
  cudaMemset(c.dErr, 0, 64);
  return RTB200_OK;
}

// debugging export: the wave of every leaf in the sweep order of one direction (its reflection combination)
int amr_waves(Context& c, const Direction& d, int32_t* waveOfLeaf, int32_t* nwaves) {
  AmrState& S = *state_of(c);
  if (int st = ensure_plan(c, S)) return st;
  const ZoneMap m = zone_map(d.izone);
  int combo = 0;
  for (int cc = 0; cc < 3; cc++)
    if (m.refl[cc]) combo |= 1 << cc;
  const std::vector<int32_t>& start = S.plan.waveStart[combo];
  for (int w = 0; w < S.plan.nkeys; w++)
    for (int32_t q = start[w]; q < start[w + 1]; q++) waveOfLeaf[S.plan.sorted[combo][(size_t)q]] = w;
  if (nwaves) *nwaves = S.plan.nkeys;
  return RTB200_OK;
}

}  // namespace rtb
