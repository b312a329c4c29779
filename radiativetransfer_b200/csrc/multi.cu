// Multi-GPU inside the library: one handle drives all GPUs of a node.
//
// The reference is one serial program (`program pointTransfer`, equiSources.f90:1230 `do while`): its driver calls the
// diffuse block (:1372-1808) and the source loop (:1256-1370) once per outer iteration.  To let that unchanged driver
// use 8 GPUs, the device group lives BEHIND the C-ABI: rtb200_create_multi(ngpus) gives a handle that the same
// rtb200_grid_set / rtb200_diffuse / rtb200_point / rtb200_grid_update_species calls accept (one process, N devices,
// one host thread per device while a call runs).  rtb200_create_rank(...) is the same group with one process per GPU
// (torchrun): the members are joined by an NCCL unique id and everything below is identical.
//
// Data path of a step (G = ranks, N = leaves, slab = ceil(N / G) leaves per rank):
//   species in     every rank copies ITS slab of HI / HeI / HeII from the caller's host arrays (1/G of the PCIe traffic
//                  per GPU) and the slabs are all-gathered over NVLink (NCCL, in place).
//   sweep / rays   every rank holds the whole grid and works on its shard of the directions (whole zones, longest
//                  processing time first) or of the sources (round robin); no exchange.
//   reduction      per-leaf sums over the ranks are only needed slab-wise by what follows (photo-rates, ionisation
//                  equilibrium, the copy back to the host): a REDUCE-SCATTER, half the traffic of an all-reduce.
//                  Mode 1 (default where peer access exists) is a kernel of this library: every rank publishes its
//                  full-size partial result in an exchange buffer mapped into all peers (cudaDeviceEnablePeerAccess in
//                  one process, cudaIpc handles between processes); after a flag hand-shake in peer memory ONE kernel
//                  per rank reads its slab of all G partial results over NVLink (P2P loads), adds them in rank order
//                  (fixed order: bit-reproducible) and applies the epilogue on the fly -- diffuse photo-rates
//                  (equiSources.f90:3546-3553) or the accumulation into the caller's rate fields.  Mode 0 is
//                  ncclReduceScatter followed by the epilogue kernel (the comparison baseline; also the fallback).
//   results out    every rank copies its slab of the results into the caller's arrays.
// NCCL is loaded with dlopen at group creation (libnccl.so.2 of the nvidia-nccl-cu12 wheel or the system one): a
// single-GPU user of librtb200.so needs no NCCL.
#include <dlfcn.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <thread>

#include "rtb200_internal.h"

namespace rtb {

namespace {

// ---- NCCL entry points, resolved at run time ------------------------------------------------------------------------
struct NcclId { char internal[128]; };
typedef void* NcclComm;
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(NcclId*) = nullptr;
  int (*CommInitRank)(NcclComm*, int, NcclId, int) = nullptr;
  int (*CommInitAll)(NcclComm*, int, const int*) = nullptr;
  int (*CommDestroy)(NcclComm) = nullptr;
  int (*ReduceScatter)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, NcclComm, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
constexpr int kNcclChar = 0, kNcclFloat64 = 8, kNcclSum = 0;

NcclApi& nccl() {
  static NcclApi api;
  return api;
}

int nccl_load() {
  NcclApi& a = nccl();
  if (a.lib) return RTB200_OK;
  const char* names[] = {getenv("RTB200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    if (!nm || !nm[0]) continue;
    a.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (a.lib) break;
  }
  if (!a.lib) {
    set_cuda_error("dlopen(libnccl.so.2): set RTB200_NCCL_LIB or LD_LIBRARY_PATH", cudaErrorSharedObjectInitFailed, __FILE__, __LINE__);
    return RTB200_ERR_CUDA;
  }
#define RTB_SYM(field, name)                                  \
  a.field = (decltype(a.field))dlsym(a.lib, name);            \
  if (!a.field) {                                             \
    set_cuda_error("dlsym(" name ")", cudaErrorSharedObjectSymbolNotFound, __FILE__, __LINE__); \
    a.lib = nullptr;                                          \
    return RTB200_ERR_CUDA;                                   \
  }
  RTB_SYM(GetUniqueId, "ncclGetUniqueId")
  RTB_SYM(CommInitRank, "ncclCommInitRank")
  RTB_SYM(CommInitAll, "ncclCommInitAll")
  RTB_SYM(CommDestroy, "ncclCommDestroy")
  RTB_SYM(ReduceScatter, "ncclReduceScatter")
  RTB_SYM(AllGather, "ncclAllGather")
  RTB_SYM(GroupStart, "ncclGroupStart")
  RTB_SYM(GroupEnd, "ncclGroupEnd")
  RTB_SYM(GetErrorString, "ncclGetErrorString")
#undef RTB_SYM
  return RTB200_OK;
}

#define RTB_NCCL(call)                                                                              \
  do {                                                                                              \
    int r_ = (call);                                                                                \
    if (r_ != 0) {                                                                                  \
      char msg_[256];                                                                               \
      snprintf(msg_, sizeof(msg_), "%s -> NCCL: %s", #call, nccl().GetErrorString ? nccl().GetErrorString(r_) : "?"); \
      rtb::set_cuda_error(msg_, cudaErrorUnknown, __FILE__, __LINE__);                              \
      return RTB200_ERR_CUDA;                                                                       \
    }                                                                                               \
  } while (0)

constexpr int kMaxRanks = 16;
static_assert(kMaxRanks <= kNgMaxRanks, "room for every rank's Ng sums");
constexpr double kZoneCostX = 1.0, kZoneCostY = 1.03, kZoneCostZ = 1.10;

// ---- peer-memory reduce-scatter with fused epilogue -------------------------------------------------------------------
struct PeerReduceParams {
  const double* src[kMaxRanks];   // exchange buffer of every rank, mapped into this device: [nf][gstride]
  unsigned long long* flags;      // [kMaxRanks] in THIS device's memory: flags[p] = last step rank p has published
  unsigned long long step;
  int32_t* err;
  int nranks;
  int64_t off, cnt;               // this rank's slab: leaves [off, off + cnt)
  int64_t gstride;                // field stride of the exchange buffers (padded leaf count)
  int64_t slab;                   // field stride of the slab outputs
  double* out;                    // [nf][slab] reduced fields (J or rate deposits)
  // epilogue 1: diffuse photo-rates from the reduced J (equiSources.f90:3546-3553); kout = [3][slab] k24, k25, k26
  double* kout;
  double fourPi, a0, a1, a2, b3, c2, c3;
  int kAccumulate;                // 1: kout += (krate fields keep their point-source part), 0: kout =
  // epilogue 2: out = base + sum (accumulation into the caller's rate fields), base = [nf][slab] or NULL
  const double* base;
};

__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// Publishes "my partial result of step `step` is complete" into every peer's flag array.  Runs after the kernels that
// wrote the exchange buffer, on the same stream.
struct PeerFlagPtrs {
  unsigned long long* p[kMaxRanks];
};
__global__ void peer_signal_kernel_v(const __grid_constant__ PeerFlagPtrs F, int nranks, int myRank, unsigned long long step) {
  __threadfence_system();
  if ((int)threadIdx.x < nranks)
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(F.p[threadIdx.x] + myRank), "l"(step) : "memory");
}

// One kernel: wait for all ranks' publications, then out[f][i] = sum_p src[p][f][off + i] in rank order, epilogue fused.
// NF = 3 (Jmean1..3) or 6 (rate deposits).  VEC: two leaves per thread and access (16-byte P2P loads).
template <int NF, bool VEC>
__global__ void __launch_bounds__(256) peer_reduce_kernel(const __grid_constant__ PeerReduceParams P) {
  __shared__ int sTimedOut;
  if (threadIdx.x == 0) sTimedOut = 0;
  __syncthreads();
  if ((int)threadIdx.x < P.nranks) {
    const long long t0 = clock64();
    while (ld_acquire_sys(P.flags + threadIdx.x) < P.step) {
      __nanosleep(200);
      if (clock64() - t0 > 40000000000LL) {   // ~20 s: a peer died; report instead of hanging the device
        atomicExch(P.err, RTB200_ERR_CUDA);
        sTimedOut = 1;
        break;
      }
    }
  }
  __syncthreads();
  if (sTimedOut) return;
  const int64_t n = VEC ? P.cnt / 2 : P.cnt;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (VEC) {
      double2 s[NF];
#pragma unroll
      for (int f = 0; f < NF; f++)
        s[f] = __ldcg(reinterpret_cast<const double2*>(P.src[0] + (int64_t)f * P.gstride + P.off) + i);
      for (int p = 1; p < P.nranks; p++) {
        double2 v[NF];
#pragma unroll
        for (int f = 0; f < NF; f++)
          v[f] = __ldcg(reinterpret_cast<const double2*>(P.src[p] + (int64_t)f * P.gstride + P.off) + i);
#pragma unroll
        for (int f = 0; f < NF; f++) { s[f].x = __dadd_rn(s[f].x, v[f].x); s[f].y = __dadd_rn(s[f].y, v[f].y); }
      }
      if (P.base) {
#pragma unroll
        for (int f = 0; f < NF; f++) {
          const double2 b = reinterpret_cast<const double2*>(P.base + (int64_t)f * P.slab)[i];
          s[f].x = __dadd_rn(b.x, s[f].x); s[f].y = __dadd_rn(b.y, s[f].y);
        }
      }
#pragma unroll
      for (int f = 0; f < NF; f++) reinterpret_cast<double2*>(P.out + (int64_t)f * P.slab)[i] = s[f];
      if (NF == 3 && P.kout) {
        double2* k24 = reinterpret_cast<double2*>(P.kout) + i;
        double2* k25 = reinterpret_cast<double2*>(P.kout + P.slab) + i;
        double2* k26 = reinterpret_cast<double2*>(P.kout + 2 * P.slab) + i;
        double2 o24 = P.kAccumulate ? *k24 : make_double2(0., 0.), o25 = P.kAccumulate ? *k25 : make_double2(0., 0.),
                o26 = P.kAccumulate ? *k26 : make_double2(0., 0.);
        {
          const double t1 = P.fourPi * s[0].x, t2 = P.fourPi * s[1].x, t3 = P.fourPi * s[2].x;
          o24.x = o24.x + t1 * P.a0 + t2 * P.a1 + t3 * P.a2; o25.x = o25.x + t3 * P.b3; o26.x = o26.x + t2 * P.c2 + t3 * P.c3;
        }
        {
          const double t1 = P.fourPi * s[0].y, t2 = P.fourPi * s[1].y, t3 = P.fourPi * s[2].y;
          o24.y = o24.y + t1 * P.a0 + t2 * P.a1 + t3 * P.a2; o25.y = o25.y + t3 * P.b3; o26.y = o26.y + t2 * P.c2 + t3 * P.c3;
        }
        *k24 = o24; *k25 = o25; *k26 = o26;
      }
    } else {
      double s[NF];
#pragma unroll
      for (int f = 0; f < NF; f++) s[f] = __ldcg(P.src[0] + (int64_t)f * P.gstride + P.off + i);
      for (int p = 1; p < P.nranks; p++) {
#pragma unroll
        for (int f = 0; f < NF; f++) s[f] = __dadd_rn(s[f], __ldcg(P.src[p] + (int64_t)f * P.gstride + P.off + i));
      }
      if (P.base) {
#pragma unroll
        for (int f = 0; f < NF; f++) s[f] = __dadd_rn(P.base[(int64_t)f * P.slab + i], s[f]);
      }
#pragma unroll
      for (int f = 0; f < NF; f++) P.out[(int64_t)f * P.slab + i] = s[f];
      if (NF == 3 && P.kout) {
        double* k24 = P.kout + i; double* k25 = P.kout + P.slab + i; double* k26 = P.kout + 2 * P.slab + i;
        const double t1 = P.fourPi * s[0], t2 = P.fourPi * s[1], t3 = P.fourPi * s[2];
        const double o24 = P.kAccumulate ? *k24 : 0., o25 = P.kAccumulate ? *k25 : 0., o26 = P.kAccumulate ? *k26 : 0.;
        *k24 = o24 + t1 * P.a0 + t2 * P.a1 + t3 * P.a2;
        *k25 = o25 + t3 * P.b3;
        *k26 = o26 + t2 * P.c2 + t3 * P.c3;
      }
    }
  }
}

// epilogues of the NCCL path (mode 0), on the reduced slab
__global__ void slab_rates_kernel(const double* __restrict__ J, int64_t cnt, int64_t slab, double fourPi, double a0,
                                  double a1, double a2, double b3, double c2, double c3, int accumulate, double* kout) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x) {
    const double t1 = fourPi * J[i], t2 = fourPi * J[slab + i], t3 = fourPi * J[2 * slab + i];
    const double o24 = accumulate ? kout[i] : 0., o25 = accumulate ? kout[slab + i] : 0., o26 = accumulate ? kout[2 * slab + i] : 0.;
    kout[i] = o24 + t1 * a0 + t2 * a1 + t3 * a2;
    kout[slab + i] = o25 + t3 * b3;
    kout[2 * slab + i] = o26 + t2 * c2 + t3 * c3;
  }
}
__global__ void slab_add_kernel(double* __restrict__ out, const double* __restrict__ base, int64_t total) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = __dadd_rn(base[i], out[i]);
}
// [nf][N] -> [nf][gstride] (only when the leaf count is not a multiple of the rank count)
__global__ void restride_kernel(const double* __restrict__ in, int64_t N, double* __restrict__ out, int64_t gstride, int nf) {
  const int64_t total = (int64_t)nf * gstride;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t f = i / gstride, j = i - f * gstride;
    out[i] = j < N ? in[f * N + j] : 0.;
  }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------------
struct Member {                     // one local device
  Context c;
  int rank = 0;                     // global rank
  NcclComm comm = nullptr;
  double* exch[2] = {nullptr, nullptr};     // exchange buffers [6][npad]: this rank's full-size partial results
  unsigned long long* flags = nullptr;      // [kMaxRanks]
  double* peerExch[2][kMaxRanks] = {};      // every rank's exchange buffers as seen from this device
  unsigned long long* peerFlags[kMaxRanks] = {};
  std::vector<void*> ipcOpened;             // mappings to close
  double* Jslab = nullptr;                  // [3][slab]
  double* Kslab = nullptr;                  // [3][slab] krate24, krate25, krate26 (diffuse photo-rates, + point part)
  double* Rslab = nullptr;                  // [6][slab] point-source rate fields of the slab
  double* Rbase = nullptr;                  // [6][slab] staging of the caller's rate fields (host API)
  bool haveR = false;                       // Rslab holds the point-source rates of the current outer iteration
  cudaEvent_t ev = nullptr;
  cudaStream_t copyStream = nullptr;                    // slab uploads of update_species, one event per species
  cudaEvent_t evCopy[3] = {nullptr, nullptr, nullptr};
  int64_t nsegLast = 0;
  // source iteration (scattering set): [3][npad] all-gather stage of the source | [3][slab] J of the previous
  // iteration | [kMaxRanks] slab residuals of every rank | this rank's residual word
  double* scat = nullptr;
  size_t scatBytes = 0;
};

struct Multi {
  int nranks = 1, nlocal = 1, rank0 = 0;
  bool multiProcess = false;
  int reduceMode = 1;               // 1 = peer-memory kernel, 0 = NCCL reduce-scatter
  bool peerOk = false;
  std::vector<Member*> mem;
  int64_t nleaf = 0, slab = 0, npad = 0;
  unsigned long long step = 0;
  // direction shards of the last (nAngularLevel, ray list, nx): cached
  std::string shardKey;
  std::vector<std::vector<int32_t>> shards;
  // relative time per segment of zones sweeping along x, y, z (same fit: y +3%, z +10%: the z-major copy and its
  // transposed merge); set_tuning "zone_cost_x/y/z"
  double zoneClassCost[3] = {kZoneCostX, kZoneCostY, kZoneCostZ};
};

namespace {

template <class F>
int for_each_member(Multi& m, F f) {
  if (m.nlocal == 1) return f(*m.mem[0], 0);
  std::vector<int> st((size_t)m.nlocal, 0);
  std::vector<std::thread> th;
  th.reserve((size_t)m.nlocal);
  for (int i = 0; i < m.nlocal; i++) th.emplace_back([&, i] { st[i] = f(*m.mem[i], i); });
  for (auto& t : th) t.join();
  for (int s : st)
    if (s) return s;
  return RTB200_OK;
}

inline int64_t slab_off(const Multi& m, int rank) { return std::min<int64_t>((int64_t)rank * m.slab, m.nleaf); }
inline int64_t slab_cnt(const Multi& m, int rank) { return std::min<int64_t>(m.slab, m.nleaf - slab_off(m, rank)); }

void free_exchange(Multi& m) {
  for (Member* q : m.mem) {
    cudaSetDevice(q->c.device);
    cudaDeviceSynchronize();
    for (void* p : q->ipcOpened) cudaIpcCloseMemHandle(p);
    q->ipcOpened.clear();
    cudaFree(q->exch[0]); cudaFree(q->exch[1]); cudaFree(q->flags);
    cudaFree(q->Jslab); cudaFree(q->Kslab); cudaFree(q->Rslab); cudaFree(q->Rbase);
    cudaFree(q->scat); q->scat = nullptr; q->scatBytes = 0;
    q->c.dWarmTaken = nullptr;
    q->exch[0] = q->exch[1] = nullptr; q->flags = nullptr;
    q->Jslab = q->Kslab = q->Rslab = q->Rbase = nullptr;
    q->haveR = false;
    memset(q->peerExch, 0, sizeof(q->peerExch));
    memset(q->peerFlags, 0, sizeof(q->peerFlags));
  }
}

typedef int (*PFN_cuMemGetAddressRange)(unsigned long long*, size_t*, unsigned long long);

struct IpcPacket {                  // what a rank tells the others about its exchange area
  cudaIpcMemHandle_t h[3];          // exch[0], exch[1], flags
  unsigned long long offset[3];     // pointer - allocation base (cudaIpcOpenMemHandle maps the whole allocation)
};

// allocate the exchange area of every member for the current grid and map every rank's area into every member
int setup_exchange(Multi& m) {
  free_exchange(m);
  const size_t exBytes = (size_t)6 * m.npad * sizeof(double);
  const size_t slabBytes = (size_t)m.slab * sizeof(double);
  for (Member* q : m.mem) {
    RTB_CUDA(cudaSetDevice(q->c.device));
    for (int b = 0; b < 2; b++) {
      RTB_CUDA(cudaMalloc((void**)&q->exch[b], exBytes));
      RTB_CUDA(cudaMemset(q->exch[b], 0, exBytes));
    }
    RTB_CUDA(cudaMalloc((void**)&q->flags, kMaxRanks * sizeof(unsigned long long)));
    RTB_CUDA(cudaMemset(q->flags, 0, kMaxRanks * sizeof(unsigned long long)));
    RTB_CUDA(cudaMalloc((void**)&q->Jslab, 3 * slabBytes));
    RTB_CUDA(cudaMalloc((void**)&q->Kslab, 3 * slabBytes));
    RTB_CUDA(cudaMalloc((void**)&q->Rslab, 6 * slabBytes));
    RTB_CUDA(cudaMalloc((void**)&q->Rbase, 6 * slabBytes));
    RTB_CUDA(cudaMemset(q->Jslab, 0, 3 * slabBytes));
    RTB_CUDA(cudaMemset(q->Kslab, 0, 3 * slabBytes));
    RTB_CUDA(cudaMemset(q->Rslab, 0, 6 * slabBytes));
    RTB_CUDA(cudaDeviceSynchronize());
  }
  m.step = 0;
  m.peerOk = false;
  if (m.nranks == 1) {
    Member* q = m.mem[0];
    for (int b = 0; b < 2; b++) q->peerExch[b][0] = q->exch[b];
    q->peerFlags[0] = q->flags;
    m.peerOk = true;
    return RTB200_OK;
  }
  if (!m.multiProcess) {
    // one process: unified addressing, the peers' pointers are usable once peer access is enabled
    bool ok = true;
    for (Member* q : m.mem) {
      RTB_CUDA(cudaSetDevice(q->c.device));
      for (Member* p : m.mem) {
        if (p == q) continue;
        int can = 0;
        RTB_CUDA(cudaDeviceCanAccessPeer(&can, q->c.device, p->c.device));
        if (!can) { ok = false; continue; }
        cudaError_t e = cudaDeviceEnablePeerAccess(p->c.device, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else if (e != cudaSuccess) { cudaGetLastError(); ok = false; }
      }
    }
    for (Member* q : m.mem)
      for (Member* p : m.mem) {
        for (int b = 0; b < 2; b++) q->peerExch[b][p->rank] = p->exch[b];
        q->peerFlags[p->rank] = p->flags;
      }
    m.peerOk = ok;
    return RTB200_OK;
  }
  // one process per GPU: exchange cudaIpc handles through an NCCL all-gather of a small byte buffer
  Member* q = m.mem[0];
  RTB_CUDA(cudaSetDevice(q->c.device));
  IpcPacket mine{};
  void* ptrs[3] = {q->exch[0], q->exch[1], q->flags};
  PFN_cuMemGetAddressRange getRange = nullptr;
  {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qr;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &qr) == cudaSuccess && fn)
      getRange = (PFN_cuMemGetAddressRange)fn;
    else cudaGetLastError();
  }
  bool ok = getRange != nullptr;
  for (int i = 0; i < 3 && ok; i++) {
    if (cudaIpcGetMemHandle(&mine.h[i], ptrs[i]) != cudaSuccess) { cudaGetLastError(); ok = false; break; }
    unsigned long long base = 0; size_t sz = 0;
    if (getRange(&base, &sz, (unsigned long long)(uintptr_t)ptrs[i]) != 0) { ok = false; break; }
    mine.offset[i] = (unsigned long long)(uintptr_t)ptrs[i] - base;
  }
  if (!ok) memset(&mine, 0xff, sizeof(mine));   // offset = ~0 marks "no handle"
  char* dPk = nullptr;
  RTB_CUDA(cudaMalloc((void**)&dPk, sizeof(IpcPacket) * (size_t)m.nranks));
  RTB_CUDA(cudaMemcpy(dPk + sizeof(IpcPacket) * (size_t)q->rank, &mine, sizeof(mine), cudaMemcpyHostToDevice));
  RTB_NCCL(nccl().AllGather(dPk + sizeof(IpcPacket) * (size_t)q->rank, dPk, sizeof(IpcPacket), kNcclChar, q->comm, q->c.stream));
  RTB_CUDA(cudaStreamSynchronize(q->c.stream));
  std::vector<IpcPacket> all((size_t)m.nranks);
  RTB_CUDA(cudaMemcpy(all.data(), dPk, sizeof(IpcPacket) * (size_t)m.nranks, cudaMemcpyDeviceToHost));
  cudaFree(dPk);
  for (int p = 0; p < m.nranks; p++)
    if (all[p].offset[0] == ~0ULL) ok = false;
  if (ok) {
    for (int p = 0; p < m.nranks && ok; p++) {
      if (p == q->rank) {
        for (int b = 0; b < 2; b++) q->peerExch[b][p] = q->exch[b];
        q->peerFlags[p] = q->flags;
        continue;
      }
      void* mapped[3] = {nullptr, nullptr, nullptr};
      for (int i = 0; i < 3; i++) {
        if (cudaIpcOpenMemHandle(&mapped[i], all[p].h[i], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
          cudaGetLastError();
          ok = false;
          break;
        }
        q->ipcOpened.push_back(mapped[i]);
      }
      if (!ok) break;
      q->peerExch[0][p] = (double*)((char*)mapped[0] + all[p].offset[0]);
      q->peerExch[1][p] = (double*)((char*)mapped[1] + all[p].offset[1]);
      q->peerFlags[p] = (unsigned long long*)((char*)mapped[2] + all[p].offset[2]);
    }
  }
  // all ranks must agree on the mode: a rank that failed to map makes everybody fall back to NCCL
  {
    double* dOk = nullptr;
    RTB_CUDA(cudaMalloc((void**)&dOk, sizeof(double) * (size_t)m.nranks));
    const double v = ok ? 1.0 : 0.0;
    RTB_CUDA(cudaMemcpy(dOk + q->rank, &v, sizeof(double), cudaMemcpyHostToDevice));
    RTB_NCCL(nccl().AllGather(dOk + q->rank, dOk, 1, kNcclFloat64, q->comm, q->c.stream));
    RTB_CUDA(cudaStreamSynchronize(q->c.stream));
    std::vector<double> oks((size_t)m.nranks);
    RTB_CUDA(cudaMemcpy(oks.data(), dOk, sizeof(double) * (size_t)m.nranks, cudaMemcpyDeviceToHost));
    cudaFree(dOk);
    for (double o : oks)
      if (o != 1.0) ok = false;
  }
  m.peerOk = ok;
  if (getenv("RTB200_VERBOSE")) fprintf(stderr, "[rtb200] rank %d: peer-memory exchange %s\n", q->rank, ok ? "mapped (cudaIpc)" : "unavailable -> NCCL");
  return RTB200_OK;
}

// ---- direction sharding (whole zones, longest processing time first; same rule as sharding.py) -----------------------
int shard_directions(int nranks, int nAngularLevel, const int32_t* rays, int32_t nrays, int nx, const double zoneClassCost[3],
                     std::vector<std::vector<int32_t>>& shards) {
  if (nAngularLevel < 1 || nAngularLevel > 8 || nranks < 1 || nx < 1) return RTB200_ERR_ARG;
  const int64_t total = 12LL << (2 * (nAngularLevel - 1));
  std::vector<int32_t> list;
  if (!rays && nrays == 0) { list.resize((size_t)total); std::iota(list.begin(), list.end(), 0); }
  else if (nrays < 0) return RTB200_ERR_ARG;
  else list.assign(rays, rays + nrays);
  struct Piece { std::vector<int32_t> r; double cost; int cls; };
  std::vector<Piece> pieces;
  std::vector<double> cost(list.size());
  std::vector<int> zone(list.size()), cls(list.size());
  std::vector<RayPattern> pat;
  const int np = std::min(nx, 64);   // segments per column scale with the layer count; 64 layers rank the directions
  for (size_t i = 0; i < list.size(); i++) {
    if (list[i] < 0 || list[i] >= total) return RTB200_ERR_ARG;
    Direction d = classify_direction(nAngularLevel, list[i]);
    if (d.status) return d.status;
    layer_patterns_level0(d.phi, d.theta, np, pat);
    // measured on B200 (profiles/r02_zone_times_256.log, least squares over the 24 zones): time of a zone task =
    // const + 0.056 ms per direction + 3.9e-4 ms per segment of a 256-cell column, i.e. a direction costs what 0.14
    // segments per layer cost, on top of its segments
    double cst = 0.14 * np;
    for (const auto& p : pat) cst += 1 + (p.xzActive ? 1 : 0) + (p.yzActive ? 1 : 0);
    const ZoneMap zm = zone_map(d.izone);
    int sweepAxis = 0;
    for (int a = 0; a < 3; a++)
      if (zm.src[a] == 0) sweepAxis = a;   // the physical axis the rotated i runs along
    cost[i] = cst * zoneClassCost[sweepAxis];
    zone[i] = d.izone;
    cls[i] = sweepAxis;
  }
  for (int z = 1; z <= 24; z++) {
    Piece p; p.cost = 0; p.cls = 0;
    for (size_t i = 0; i < list.size(); i++)
      if (zone[i] == z) { p.r.push_back(list[i]); p.cost += cost[i]; p.cls = cls[i]; }
    if (!p.r.empty()) pieces.push_back(std::move(p));
  }
  auto rayCost = [&](int32_t r) { for (size_t i = 0; i < list.size(); i++) if (list[i] == r) return cost[i]; return 0.0; };
  auto bySize = [](const Piece& a, const Piece& b) { return a.cost != b.cost ? a.cost > b.cost : a.r[0] < b.r[0]; };
  // split the largest zone pieces until there are at least 3 pieces per rank, so that LPT can balance
  while ((int)pieces.size() < 3 * nranks) {
    std::sort(pieces.begin(), pieces.end(), bySize);
    if (pieces.empty() || pieces[0].r.size() < 2) break;
    Piece a, b; a.cost = b.cost = 0; a.cls = b.cls = pieces[0].cls;
    const size_t half = pieces[0].r.size() / 2;
    for (size_t i = 0; i < pieces[0].r.size(); i++) {
      Piece& t = i < half ? a : b;
      t.r.push_back(pieces[0].r[i]); t.cost += rayCost(pieces[0].r[i]);
    }
    pieces.erase(pieces.begin());
    pieces.push_back(std::move(a)); pieces.push_back(std::move(b));
  }
  // Longest processing time first, ONE SWEEP AXIS AFTER THE OTHER, and no rank takes more than its share of an axis'
  // pieces: the zones of an axis differ in memory layout (lane axis contiguous or not, z-major copy), and a layer launch
  // runs all zone tasks of a rank together, so equal segment counts are only equal times when the ranks hold the same
  // mix (measured: three x-sweeping zones 6.3 ms, a z- and two y-sweeping zones 7.6 ms for the same segment count).
  std::vector<double> load((size_t)nranks, 0.);
  std::vector<std::vector<int>> owned((size_t)nranks);   // piece indices per rank
  for (int c = 2; c >= 0; c--) {
    std::vector<int> mine;
    for (int i = 0; i < (int)pieces.size(); i++)
      if (pieces[i].cls == c) mine.push_back(i);
    std::sort(mine.begin(), mine.end(), [&](int a, int b) { return bySize(pieces[a], pieces[b]); });
    const int quota = ((int)mine.size() + nranks - 1) / nranks;
    std::vector<int> taken((size_t)nranks, 0);
    for (int i : mine) {
      int best = -1;
      for (int r = 0; r < nranks; r++)
        if (taken[r] < quota && (best < 0 || load[r] < load[best])) best = r;
      owned[best].push_back(i);
      load[best] += pieces[i].cost;
      taken[best]++;
    }
  }
  // local improvement: swap two pieces of the same sweep axis between two ranks while that lowers the larger of the two
  // loads (the greedy pass pairs a large x-zone with whatever is left of y and z)
  for (int pass = 0; pass < 64; pass++) {
    bool improved = false;
    for (int a = 0; a < nranks; a++)
      for (int b = a + 1; b < nranks; b++)
        for (size_t ia = 0; ia < owned[a].size(); ia++)
          for (size_t ib = 0; ib < owned[b].size(); ib++) {
            const Piece& pa = pieces[owned[a][ia]];
            const Piece& pb = pieces[owned[b][ib]];
            if (pa.cls != pb.cls) continue;
            const double na = load[a] - pa.cost + pb.cost, nb = load[b] - pb.cost + pa.cost;
            if (std::max(na, nb) < std::max(load[a], load[b]) * (1. - 1e-12)) {
              std::swap(owned[a][ia], owned[b][ib]);
              load[a] = na; load[b] = nb;
              improved = true;
            }
          }
    if (!improved) break;
  }
  shards.assign((size_t)nranks, {});
  for (int r = 0; r < nranks; r++)
    for (int i : owned[r]) shards[r].insert(shards[r].end(), pieces[i].r.begin(), pieces[i].r.end());
  for (auto& s : shards) std::sort(s.begin(), s.end());
  return RTB200_OK;
}

int build_shards(Multi& m, int nAngularLevel, const int32_t* rays, int32_t nrays, int nx) {
  char key[96];
  snprintf(key, sizeof(key), "%d:%d:%d:%d:%a:%a:%a:", nAngularLevel, nx, m.nranks, nrays, m.zoneClassCost[0], m.zoneClassCost[1],
           m.zoneClassCost[2]);
  std::string k(key);
  if (rays)
    for (int i = 0; i < nrays; i++) { snprintf(key, sizeof(key), "%d,", rays[i]); k += key; }
  if (k == m.shardKey) return RTB200_OK;
  if (int st = shard_directions(m.nranks, nAngularLevel, rays, nrays, nx, m.zoneClassCost, m.shards)) return st;
  m.shardKey = k;
  return RTB200_OK;
}

// ---- the reduction step of one member ---------------------------------------------------------------------------------
struct Epilogue {
  const double* ksi = nullptr;   // [6] = ksi24[3], ksi25, ksi26[2]: photo-rates into Kslab
  int kAccumulate = 0;
  const double* base = nullptr;  // [nf][slab]: out = base + sum
};

// `nf` fields of exch[buf] (this rank's partial results, complete on stream s) -> out [nf][slab] = sum over the ranks
// step = the exchange step of this reduction (its parity selects buf); a source iteration takes one step per iteration
int reduce_member(Multi& m, Member& q, int buf, unsigned long long step, int nf, double* out, const Epilogue& ep, cudaStream_t s) {
  const int64_t off = slab_off(m, q.rank), cnt = slab_cnt(m, q.rank);
  const int blocks = (int)std::max<int64_t>(1, std::min<int64_t>((cnt / 2 + 255) / 256, (int64_t)q.c.smCount * 8));
  const bool usePeer = m.reduceMode == 1 && m.peerOk;
  if (usePeer) {
    PeerFlagPtrs F{};
    for (int p = 0; p < m.nranks; p++) F.p[p] = q.peerFlags[p];
    peer_signal_kernel_v<<<1, 32, 0, s>>>(F, m.nranks, q.rank, step);
    PeerReduceParams P{};
    for (int p = 0; p < m.nranks; p++) P.src[p] = q.peerExch[buf][p];
    P.flags = q.flags; P.step = step; P.err = q.c.dErr; P.nranks = m.nranks;
    P.off = off; P.cnt = cnt; P.gstride = m.npad; P.slab = m.slab; P.out = out;
    P.kout = ep.ksi ? q.Kslab : nullptr; P.kAccumulate = ep.kAccumulate; P.base = ep.base;
    P.fourPi = 4. * kPi;
    if (ep.ksi) { P.a0 = ep.ksi[0]; P.a1 = ep.ksi[1]; P.a2 = ep.ksi[2]; P.b3 = ep.ksi[3]; P.c2 = ep.ksi[4]; P.c3 = ep.ksi[5]; }
    const bool vec = (cnt % 2 == 0) && (off % 2 == 0) && (m.npad % 2 == 0) && (m.slab % 2 == 0);
    if (nf == 3) {
      if (vec) peer_reduce_kernel<3, true><<<blocks, 256, 0, s>>>(P);
      else peer_reduce_kernel<3, false><<<blocks, 256, 0, s>>>(P);
    } else {
      if (vec) peer_reduce_kernel<6, true><<<blocks, 256, 0, s>>>(P);
      else peer_reduce_kernel<6, false><<<blocks, 256, 0, s>>>(P);
    }
    RTB_CUDA(cudaGetLastError());
    return RTB200_OK;
  }
  // NCCL: one reduce-scatter per field (equal counts: the exchange buffers are padded to slab * nranks per field)
  if (m.nranks > 1) {
    RTB_NCCL(nccl().GroupStart());
    for (int f = 0; f < nf; f++)
      RTB_NCCL(nccl().ReduceScatter(q.exch[buf] + (size_t)f * m.npad, out + (size_t)f * m.slab, (size_t)m.slab, kNcclFloat64,
                                    kNcclSum, q.comm, s));
    RTB_NCCL(nccl().GroupEnd());
  } else {
    for (int f = 0; f < nf; f++)
      RTB_CUDA(cudaMemcpyAsync(out + (size_t)f * m.slab, q.exch[buf] + (size_t)f * m.npad, (size_t)cnt * sizeof(double),
                               cudaMemcpyDeviceToDevice, s));
  }
  if (ep.base) slab_add_kernel<<<blocks, 256, 0, s>>>(out, ep.base, (int64_t)nf * m.slab);
  if (ep.ksi && nf == 3)
    slab_rates_kernel<<<blocks, 256, 0, s>>>(out, cnt, m.slab, 4. * kPi, ep.ksi[0], ep.ksi[1], ep.ksi[2], ep.ksi[3], ep.ksi[4],
                                             ep.ksi[5], ep.kAccumulate, q.Kslab);
  RTB_CUDA(cudaGetLastError());
  return RTB200_OK;
}

// sweep of this member's direction shard into exch[buf][0..2] (padded layout); iter: see run_sweep
int sweep_member(Multi& m, Member& q, int buf, int nAngularLevel, const double* uvb, const double* beta, cudaStream_t s,
                 int iter = 0) {
  const std::vector<int32_t>& mine = m.shards[(size_t)q.rank];
  static const int32_t none = 0;
  double* target = m.npad == m.nleaf ? q.exch[buf] : q.c.dJ;
  int64_t ns = 0;
  int st = run_sweep(q.c, nAngularLevel, uvb, beta, mine.empty() ? &none : mine.data(), (int32_t)mine.size(), target, s, &ns, iter);
  if (st) return st;
  q.nsegLast = ns;
  if (target != q.exch[buf]) {
    const int64_t total = 3 * m.npad;
    restride_kernel<<<(int)std::min<int64_t>((total + 255) / 256, (int64_t)q.c.smCount * 16), 256, 0, s>>>(q.c.dJ, m.nleaf, q.exch[buf],
                                                                                                          m.npad, 3);
    RTB_CUDA(cudaGetLastError());
  }
  return RTB200_OK;
}

// RTB200_TIMING=1: rank 0 prints the host wall time of every phase of the host-buffer calls (each phase is closed with
// a stream synchronisation, so the numbers add up to more than an untimed call)
struct PhaseTimer {
  bool on;
  cudaStream_t s;
  std::chrono::steady_clock::time_point t0;
  std::string line;
  PhaseTimer(const char* what, int rank, cudaStream_t st) : on(rank == 0 && getenv("RTB200_TIMING") != nullptr), s(st) {
    if (on) { line = std::string("[rtb200 timing] ") + what + ":"; t0 = std::chrono::steady_clock::now(); }
  }
  void mark(const char* phase) {
    if (!on) return;
    cudaStreamSynchronize(s);
    const auto t1 = std::chrono::steady_clock::now();
    char b[64];
    snprintf(b, sizeof(b), " %s %.3f ms", phase, std::chrono::duration<double, std::milli>(t1 - t0).count());
    line += b;
    t0 = t1;
  }
  ~PhaseTimer() { if (on) fprintf(stderr, "%s\n", line.c_str()); }
};

int allgather_species(Multi& m, Member& q, bool hi, bool he1, bool he2, cudaStream_t s) {
  if (m.nranks == 1) return RTB200_OK;
  double* arr[3] = {hi ? q.c.dHI : nullptr, he1 ? q.c.dHeI : nullptr, he2 ? q.c.dHeII : nullptr};
  RTB_NCCL(nccl().GroupStart());
  for (double* a : arr)
    if (a) RTB_NCCL(nccl().AllGather(a + (size_t)q.rank * m.slab, a, (size_t)m.slab, kNcclFloat64, q.comm, s));
  RTB_NCCL(nccl().GroupEnd());
  return RTB200_OK;
}

int create_members(Multi* m, const int* devices) {
  for (int i = 0; i < m->nlocal; i++) {
    Member* q = new (std::nothrow) Member();
    if (!q) return RTB200_ERR_NOMEM;
    m->mem.push_back(q);
    q->rank = m->rank0 + i;
    if (int st = context_init(q->c, devices[i])) return st;
    RTB_CUDA(cudaEventCreateWithFlags(&q->ev, cudaEventDisableTiming));
    RTB_CUDA(cudaStreamCreateWithFlags(&q->copyStream, cudaStreamNonBlocking));
    for (int k = 0; k < 3; k++) RTB_CUDA(cudaEventCreateWithFlags(&q->evCopy[k], cudaEventDisableTiming));
  }
  return RTB200_OK;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------------
void multi_destroy(Multi* m) {
  if (!m) return;
  free_exchange(*m);
  for (Member* q : m->mem) {
    cudaSetDevice(q->c.device);
    if (q->comm && nccl().CommDestroy) nccl().CommDestroy(q->comm);
    if (q->ev) cudaEventDestroy(q->ev);
    for (int k = 0; k < 3; k++)
      if (q->evCopy[k]) cudaEventDestroy(q->evCopy[k]);
    if (q->copyStream) cudaStreamDestroy(q->copyStream);
    context_destroy(q->c);
    delete q;
  }
  delete m;
}

Context& multi_primary(Multi* m) { return m->mem[0]->c; }

int multi_set_math(Multi* m, int mode) {
  for (Member* q : m->mem) set_math(q->c, mode);
  return RTB200_OK;
}

int multi_set_tuning(Multi* m, const char* key, double value) {
  std::string k(key);
  if (k == "multi_reduce") { m->reduceMode = (int)value; return RTB200_OK; }
  if (k == "zone_cost_x" || k == "zone_cost_y" || k == "zone_cost_z") {
    if (!(value > 0.)) return RTB200_ERR_ARG;
    m->zoneClassCost[k.back() - 'x'] = value;
    return RTB200_OK;
  }
  for (Member* q : m->mem)
    if (int st = set_tuning(q->c, key, value)) return st;
  return RTB200_OK;
}

int multi_grid_set(Multi* m, int nx, int64_t nleaf, const int8_t* level, const double* HI, const double* HeI,
                   const double* HeII, const double* rho, const double* abun2, double physicalBoxSize) {
  m->nleaf = nleaf;
  m->slab = (nleaf + m->nranks - 1) / m->nranks;
  m->npad = m->slab * m->nranks;
  m->shardKey.clear();
  int st = for_each_member(*m, [&](Member& q, int) {
    q.c.padLeaves = m->npad - nleaf;
    return grid_set(q.c, nx, nleaf, level, HI, HeI, HeII, rho, abun2, physicalBoxSize);
  });
  if (st) return st;
  return setup_exchange(*m);
}

// every rank uploads its slab of the caller's arrays; NVLink all-gather completes the copies (in place)
int multi_update_species(Multi* m, const double* HI, const double* HeI, const double* HeII) {
  if (m->nleaf == 0) return RTB200_ERR_ARG;
  return for_each_member(*m, [&](Member& q, int) -> int {
    Context& c = q.c;
    RTB_CUDA(cudaSetDevice(c.device));
    PhaseTimer tm("update_species", q.rank, c.stream);
    RTB_CUDA(cudaDeviceSynchronize());   // see rtb200_grid_update_species: queued readers of the species first
    tm.mark("device-sync");
    const int64_t off = slab_off(*m, q.rank), cnt = slab_cnt(*m, q.rank);
    const size_t nb = (size_t)cnt * sizeof(double);
    // pipelined per species: the slab of species k+1 crosses PCIe (copy stream) while species k is all-gathered over
    // NVLink (the context's stream waits for the copy's event) -- measured at 4 GPUs before: 2.1 ms of copies, then
    // 1.3 ms of all-gathers, back to back
    const double* src[3] = {HI, HeI, HeII};
    double* dst[3] = {c.dHI, c.dHeI, c.dHeII};
    for (int k = 0; k < 3; k++) {
      if (!src[k]) continue;
      if (cnt > 0) RTB_CUDA(cudaMemcpyAsync(dst[k] + off, src[k] + off, nb, cudaMemcpyHostToDevice, q.copyStream));
      RTB_CUDA(cudaEventRecord(q.evCopy[k], q.copyStream));
      RTB_CUDA(cudaStreamWaitEvent(c.stream, q.evCopy[k], 0));
      if (int st = allgather_species(*m, q, k == 0, k == 1, k == 2, c.stream)) return st;
    }
    RTB_CUDA(cudaStreamSynchronize(c.stream));
    tm.mark("h2d-slab + all-gather");
    return RTB200_OK;
  });
}

// A per-leaf [3][nleaf] field of a device group (emission, scattering): every rank checks its slab of the caller's
// array, the ranks agree on the status (an all-gather of one word each in rank mode), then every rank uploads its slab
// and all-gathers the three fields on the devices, as multi_update_species does for the species.  `apply(c, packed)`
// installs the complete device copy [3][nleaf] in a member's context.
template <class Apply>
static int multi_set_field(Multi* m, const double* eta, Apply apply) {
  const int64_t N = m->nleaf;
  bool ok = true;
  for (Member* q : m->mem) {
    const int64_t off = slab_off(*m, q->rank), cnt = slab_cnt(*m, q->rank);
    for (int g = 0; g < 3 && ok; g++)
      for (int64_t i = off; i < off + cnt; i++) {
        const double v = eta[g * N + i];
        if (!(v >= 0. && v <= 1.7976931348623157e308)) { ok = false; break; }
      }
  }
  return for_each_member(*m, [&](Member& q, int) -> int {
    Context& c = q.c;
    RTB_CUDA(cudaSetDevice(c.device));
    RTB_CUDA(cudaDeviceSynchronize());   // queued sweeps read the current array
    const int64_t off = slab_off(*m, q.rank), cnt = slab_cnt(*m, q.rank);
    double* stage = nullptr;             // [3 fields][npad]: slab copies, completed in place by the all-gather
    RTB_CUDA(cudaMalloc((void**)&stage, (size_t)3 * m->npad * sizeof(double)));
    auto done = [&](int st) { cudaStreamSynchronize(c.stream); cudaFree(stage); return st; };
    if (m->nranks > 1) {                 // every rank learns every rank's verdict
      const double mine = ok ? 0. : 1.;
      RTB_CUDA(cudaMemcpyAsync(stage + q.rank, &mine, sizeof(double), cudaMemcpyHostToDevice, c.stream));
      if (int st = [&]() -> int {
            RTB_NCCL(nccl().AllGather(stage + q.rank, stage, 1, kNcclFloat64, q.comm, c.stream));
            return RTB200_OK;
          }())
        return done(st);
      std::vector<double> all((size_t)m->nranks);
      RTB_CUDA(cudaMemcpyAsync(all.data(), stage, all.size() * sizeof(double), cudaMemcpyDeviceToHost, c.stream));
      RTB_CUDA(cudaStreamSynchronize(c.stream));
      for (double v : all)
        if (v != 0.) return done(RTB200_ERR_ARG);
    } else if (!ok) {
      return done(RTB200_ERR_ARG);
    }
    for (int g = 0; g < 3; g++) {
      double* f = stage + (size_t)g * m->npad;
      if (cnt > 0) RTB_CUDA(cudaMemcpyAsync(f + off, eta + g * N + off, (size_t)cnt * sizeof(double), cudaMemcpyHostToDevice, c.stream));
      if (m->nranks > 1) {
        if (int st = [&]() -> int {
              RTB_NCCL(nccl().AllGather(f + (size_t)q.rank * m->slab, f, (size_t)m->slab, kNcclFloat64, q.comm, c.stream));
              return RTB200_OK;
            }())
          return done(st);
      }
    }
    // the fields side by side, [3][nleaf] as the sweeps read them
    double* packed = nullptr;
    RTB_CUDA(cudaMalloc((void**)&packed, (size_t)3 * N * sizeof(double)));
    int st = RTB200_OK;
    for (int g = 0; g < 3 && !st; g++)
      if (cudaMemcpyAsync(packed + (size_t)g * N, stage + (size_t)g * m->npad, (size_t)N * sizeof(double),
                          cudaMemcpyDeviceToDevice, c.stream) != cudaSuccess)
        st = RTB200_ERR_CUDA;
    if (!st) st = apply(c, packed);
    cudaStreamSynchronize(c.stream);
    cudaFree(packed);
    return done(st);
  });
}

// NULL clears the emission everywhere
int multi_set_emission(Multi* m, const double* eta) {
  if (m->nleaf == 0) return RTB200_ERR_ARG;
  if (!eta) return for_each_member(*m, [&](Member& q, int) { return set_emission(q.c, nullptr, false, q.c.stream); });
  return multi_set_field(m, eta, [](Context& c, const double* packed) { return set_emission(c, packed, true, c.stream); });
}

// NULL clears the scattering everywhere
int multi_set_scattering(Multi* m, const double* sigma, int32_t maxIterations, double tolerance) {
  if (m->nleaf == 0) return RTB200_ERR_ARG;
  if (!sigma) return for_each_member(*m, [&](Member& q, int) { return set_scattering(q.c, nullptr, false, 1, 0.); });
  if (maxIterations < 1 || !(tolerance >= 0.) || std::isinf(tolerance)) return RTB200_ERR_ARG;
  if (multi_primary(m).dDustSigma) return RTB200_ERR_ARG;   // one scattering medium at a time (dust.cu)
  return multi_set_field(m, sigma, [&](Context& c, const double* packed) {
    return set_scattering(c, packed, true, maxIterations, tolerance);
  });
}

// flags only: every member keeps its own history and its own slab of the stored J
int multi_set_scattering_acceleration(Multi* m, int32_t flags) {
  if (m->nleaf == 0) return RTB200_ERR_ARG;
  return for_each_member(*m, [&](Member& q, int) { return set_scattering_acceleration(q.c, flags); });
}

// scalars only: every member stores them and computes the dust of the whole grid from its complete species and its
// complete rho / abun2 (grid_set uploads the caller's full arrays on every member, in rank mode too)
int multi_set_dust(Multi* m, int mode, const double* betaDust, const double* albedo, int32_t maxIterations, double tolerance) {
  if (m->nleaf == 0 || !dust_args_ok(mode, betaDust, albedo, maxIterations, tolerance)) return RTB200_ERR_ARG;
  return for_each_member(*m, [&](Member& q, int) { return set_dust(q.c, mode, betaDust, albedo, maxIterations, tolerance); });
}

int multi_last_scattering(Multi* m, int32_t* iterations, double* residual) {
  Member& q = *m->mem[0];
  Context& c = q.c;
  if (c.scatResidPending) {   // tolerance 0: every rank's slab residual was all-gathered on the devices
    RTB_CUDA(cudaSetDevice(c.device));
    RTB_CUDA(cudaDeviceSynchronize());
    std::vector<double> all((size_t)m->nranks);
    RTB_CUDA(cudaMemcpy(all.data(), q.scat + 3 * m->npad + 3 * m->slab, all.size() * sizeof(double), cudaMemcpyDeviceToHost));
    c.lastScatResid = *std::max_element(all.begin(), all.end());
    c.scatResidPending = false;
  }
  if (iterations) *iterations = c.lastScatIter;
  if (residual) *residual = c.lastScatResid;
  return RTB200_OK;
}

int multi_get_species(Multi* m, double* HI, double* HeI, double* HeII) {
  if (m->nleaf == 0) return RTB200_ERR_ARG;
  return for_each_member(*m, [&](Member& q, int) -> int {
    Context& c = q.c;
    RTB_CUDA(cudaSetDevice(c.device));
    RTB_CUDA(cudaDeviceSynchronize());
    const int64_t off = slab_off(*m, q.rank), cnt = slab_cnt(*m, q.rank);
    const size_t nb = (size_t)cnt * sizeof(double);
    if (cnt == 0) return RTB200_OK;
    if (HI) RTB_CUDA(cudaMemcpy(HI + off, c.dHI + off, nb, cudaMemcpyDeviceToHost));
    if (HeI) RTB_CUDA(cudaMemcpy(HeI + off, c.dHeI + off, nb, cudaMemcpyDeviceToHost));
    if (HeII) RTB_CUDA(cudaMemcpy(HeII + off, c.dHeII + off, nb, cudaMemcpyDeviceToHost));
    return RTB200_OK;
  });
}

int multi_chemistry_tables(Multi* m, int nratec, double logtem0, double logtem9, double dlogtem, const double* const k[6]) {
  return for_each_member(*m, [&](Member& q, int) { return chemistry_set_tables(q.c, nratec, logtem0, logtem9, dlogtem, k); });
}

int multi_chemistry_temperature(Multi* m, const double* tgas) {
  return for_each_member(*m, [&](Member& q, int) { return chemistry_set_temperature(q.c, tgas); });
}

int multi_device_error(Multi* m) {
  int first = 0;
  for (Member* q : m->mem) {
    const int e = device_error(q->c);
    if (e && !first) first = e;
  }
  return first;
}

// the stored J of the warm start goes on every local member (in rank mode the other ranks learn it from the holding
// flags all-gathered at the start of their next call)
static void drop_stored_j(Multi& m) {
  for (Member* q : m.mem) q->c.scatWarm = false;
}

// Source iteration of one member (scattering set), iterations k = 1, 2, ...  Every iteration is an exchange step of its
// own, step0 + k, so that the peer reduction's double buffering (DESIGN.md 5) keeps its parity:
//   1. the sweep of the shard with the current source (opacities and sigma once, in the first),
//   2. the reduction into Jslab (with the epilogue ep: photo-rates are overwritten, so the last iteration's stay),
//   3. the slab's source pass: eta_th + sigma * J into this rank's part of the stage, the slab residual,
//   4. the all-gather of the three source fields, copied into the effective buffer [3][nleaf],
//   5. with a tolerance, an all-gather of the slab residuals: every rank takes the same max and stops after the same k.
// With the acceleration flags (ng.cu) the warm start takes x_0 from the rank's Jprev slab, and an Ng step runs between
// 5 and 4: the slab's five sums, their all-gather, the same solve on every rank and the slab's combine pass.
// Returns the number of iterations in *iters.
static int scatter_member(Multi& m, Member& q, unsigned long long step0, int nAngularLevel, const double* uvb,
                          const double* beta, const Epilogue& ep, cudaStream_t s, int* iters) {
  Context& c = q.c;
  // with the flag, every rank takes the same path below; whether x_0 is the stored J is decided on the devices from
  // every rank's holding of one, so a rank that lost its J (a failed call) turns the whole group cold
  const bool warm = (c.scatAccel & RTB200_SCATTER_WARM_START) != 0;
  const bool ng = (c.scatAccel & RTB200_SCATTER_NG) != 0;
  const double holds = c.scatWarm ? 1. : 0.;
  c.scatWarm = false;   // the Jprev slab holds a returned J again only when this call completes
  const int64_t N = m.nleaf, off = slab_off(m, q.rank), cnt = slab_cnt(m, q.rank);
  // + one word: whether the warm start was taken
  const size_t need = (size_t)(3 * m.npad + 3 * m.slab + kMaxRanks + 2) * sizeof(double);
  if (int st = ensure_buffer((void**)&q.scat, &q.scatBytes, need)) return st;
  double* stage = q.scat;
  double* Jprev = stage + 3 * m.npad;
  double* all = Jprev + 3 * m.slab;
  unsigned long long* resid = (unsigned long long*)(all + kMaxRanks);
  int32_t* warmTaken = (int32_t*)(resid + 1);
  const size_t nb = (size_t)3 * N * sizeof(double);
  NgBuffers ngb{};
  if (ng) {
    if (int st = ng_buffers(c, m.slab, &ngb)) return st;
    RTB_CUDA(cudaMemsetAsync(ngb.count, 0, sizeof(int32_t), s));
  }
  const double* sigmaSlab = nullptr;   // set after the dust (if any) is computed for this call
  const double* etaThSlab = c.dEta ? c.dEta + off : nullptr;
  double* stageSlab = stage + (size_t)q.rank * m.slab;
  auto share_eta = [&]() -> int {      // the ranks' source slabs into every rank's effective buffer
    if (m.nranks > 1) {
      RTB_NCCL(nccl().GroupStart());
      for (int g = 0; g < 3; g++) {
        double* f = stage + (size_t)g * m.npad;
        RTB_NCCL(nccl().AllGather(f + (size_t)q.rank * m.slab, f, (size_t)m.slab, kNcclFloat64, q.comm, s));
      }
      RTB_NCCL(nccl().GroupEnd());
    }
    for (int g = 0; g < 3; g++)
      RTB_CUDA(cudaMemcpyAsync(c.dEtaEff + (size_t)g * N, stage + (size_t)g * m.npad, (size_t)N * sizeof(double),
                               cudaMemcpyDeviceToDevice, s));
    return RTB200_OK;
  };
  if (warm) {
    // every rank's holding into all[0 .. nranks), then x_0 = the Jprev slab if all hold one, else 0 (eta_1 = eta_th then,
    // bit for bit); eta_1 = eta_th + sigma * x_0 by the slab's source pass (Jslab, overwritten by the first reduction,
    // takes its copy of x_0), then shared as in every iteration; dust computes its sigma from the current species first
    RTB_CUDA(cudaMemcpyAsync(all + q.rank, &holds, sizeof(double), cudaMemcpyHostToDevice, s));
    if (m.nranks > 1) RTB_NCCL(nccl().AllGather(all + q.rank, all, 1, kNcclFloat64, q.comm, s));
    if (int st = launch_warm_start_agree(c, all, m.nranks, Jprev, 3 * m.slab, warmTaken, s)) return st;
    if (c.dustMode && c.dDustSigma)
      if (int st = launch_compute_opacities_dust(c, beta, s)) return st;
    sigmaSlab = c.scatterSigma() + off;
    if (int st = launch_scatter_source(c, cnt, Jprev, q.Jslab, m.slab, sigmaSlab, etaThSlab, N, stageSlab, m.npad, resid, s))
      return st;
    if (int st = share_eta()) return st;
  } else {
    // J_0 = 0, eta_1 = eta_th
    RTB_CUDA(cudaMemsetAsync(Jprev, 0, (size_t)3 * m.slab * sizeof(double), s));
    if (c.dEta) RTB_CUDA(cudaMemcpyAsync(c.dEtaEff, c.dEta, nb, cudaMemcpyDeviceToDevice, s));
    else RTB_CUDA(cudaMemsetAsync(c.dEtaEff, 0, nb, s));
  }
  auto gather_resid = [&]() -> int {   // every rank's slab residual into all[0 .. nranks)
    RTB_CUDA(cudaMemcpyAsync(all + q.rank, resid, sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (m.nranks > 1) RTB_NCCL(nccl().AllGather(all + q.rank, all, 1, kNcclFloat64, q.comm, s));
    return RTB200_OK;
  };
  int64_t nsTotal = 0;
  int k = 1;
  int cycle = 0;   // sweeps since the call's start or the last attempted extrapolation
  double r = 0.;
  for (;; k++) {
    const unsigned long long step = step0 + (unsigned long long)k;
    const int buf = (int)(step & 1);
    if (int st = sweep_member(m, q, buf, nAngularLevel, uvb, beta, s, k)) return st;
    nsTotal += q.nsegLast;
    if (int st = reduce_member(m, q, buf, step, 3, q.Jslab, ep, s)) return st;
    sigmaSlab = c.scatterSigma() + off;
    cycle++;
    const bool extrapolate = ng && cycle == 4 && k < c.scatMaxIter;
    if (ng && cycle >= 2)   // Ng keeps y of the cycle's sweeps 1..3: the Jprev slab holds y_{k-1} until the source pass
      RTB_CUDA(cudaMemcpyAsync(ngb.hist[cycle - 2], Jprev, (size_t)3 * m.slab * sizeof(double), cudaMemcpyDeviceToDevice, s));
    RTB_CUDA(cudaMemsetAsync(resid, 0, sizeof(unsigned long long), s));
    if (int st = launch_scatter_source(c, cnt, q.Jslab, Jprev, m.slab, sigmaSlab, etaThSlab, N, stageSlab, m.npad, resid, s))
      return st;
    if (!extrapolate)
      if (int st = share_eta()) return st;
    c.lastLaunches += 1;
    if (c.scatTol > 0.) {
      if (int st = gather_resid()) return st;
      std::vector<double> v((size_t)m.nranks);
      RTB_CUDA(cudaMemcpyAsync(v.data(), all, v.size() * sizeof(double), cudaMemcpyDeviceToHost, s));
      RTB_CUDA(cudaStreamSynchronize(s));
      r = *std::max_element(v.begin(), v.end());
      if (r <= c.scatTol) break;
    }
    if (extrapolate) {   // I0..I3 = y_k (Jslab), y_{k-1}, y_{k-2}, y_{k-3} of the slab; every rank solves with all sums
      if (int st = launch_ng_partials(ngb, cnt, q.Jslab, m.slab, q.rank, s)) return st;
      if (m.nranks > 1) RTB_NCCL(nccl().AllGather(ngb.sums + 5 * q.rank, ngb.sums, 5, kNcclFloat64, q.comm, s));
      if (int st = launch_ng_apply(c, ngb, m.nranks, cnt, q.Jslab, Jprev, m.slab, sigmaSlab, etaThSlab, N, stageSlab,
                                   m.npad, s))
        return st;
      if (int st = share_eta()) return st;
      c.lastLaunches += 4;
      cycle = 0;
    }
    if (k == c.scatMaxIter) break;
  }
  if (c.scatTol == 0.)   // read by rtb200_last_scattering: no host round trip in the call
    if (int st = gather_resid()) return st;
  RTB_CUDA(cudaEventRecord(c.evStop, s));
  q.nsegLast = nsTotal;
  c.lastScatIter = k;
  c.lastScatResid = r;
  c.scatResidPending = c.scatTol == 0.;
  c.lastWarm = false;
  c.dWarmTaken = warm ? warmTaken : nullptr;   // rtb200_last_scattering_acceleration reads it once the call's work is done
  c.ngPending = ng;
  c.scatWarm = true;   // the source pass left y_k in the Jprev slab
  *iters = k;
  return RTB200_OK;
}

// resident step of one member on stream s: opacities + sweep of the shard + reduce-scatter (+ photo-rates)
// (+ ionisation equilibrium on the slab + all-gather of the new species)
static int diffuse_resident_member(Multi& m, Member& q, int nAngularLevel, const double* uvb, const double* beta,
                                   const double* ksi6, int chemistry, cudaStream_t s, int* iters) {
  Epilogue ep;
  ep.ksi = ksi6;
  ep.kAccumulate = 0;
  if (q.c.scatterSigma()) {   // source iteration, steps m.step .. m.step + iterations - 1; chemistry once, after it
    if (int st = scatter_member(m, q, m.step - 1, nAngularLevel, uvb, beta, ep, s, iters)) return st;
  } else {
    const int buf = (int)(m.step & 1);
    if (int st = sweep_member(m, q, buf, nAngularLevel, uvb, beta, s)) return st;
    if (int st = reduce_member(m, q, buf, m.step, 3, q.Jslab, ep, s)) return st;
  }
  if (chemistry) {
    if (!ksi6) return RTB200_ERR_ARG;
    const int64_t off = slab_off(m, q.rank), cnt = slab_cnt(m, q.rank);
    if (int st = chemistry_run_slab(q.c, off, cnt, q.haveR ? q.Rslab : nullptr, m.slab, q.Jslab, m.slab, ksi6, nullptr, s))
      return st;
    if (int st = allgather_species(m, q, true, true, true, s)) return st;
    q.haveR = false;   // the rates of this outer iteration are consumed (setZeroRates, equiSources.f90:1246)
  }
  return RTB200_OK;
}

int multi_diffuse_resident(Multi* m, int nAngularLevel, const double* uvb, const double* beta, const double* ksi6,
                           int chemistry, void* const* streams, int64_t* nseg) {
  if (m->nleaf == 0 || !uvb || !beta) return RTB200_ERR_ARG;
  if (int st = build_shards(*m, nAngularLevel, nullptr, 0, multi_primary(m).nx)) return st;
  m->step++;
  std::vector<int> iters((size_t)m->nlocal, 1);
  for (Member* q : m->mem) q->c.lastScatIter = 0, q->c.lastScatResid = 0., q->c.scatResidPending = false, q->c.lastNgCount = 0,
      q->c.lastWarm = false, q->c.ngPending = false, q->c.dWarmTaken = nullptr;
  int st = for_each_member(*m, [&](Member& q, int i) -> int {
    RTB_CUDA(cudaSetDevice(q.c.device));
    return diffuse_resident_member(*m, q, nAngularLevel, uvb, beta, ksi6, chemistry,
                                   streams ? (cudaStream_t)streams[i] : q.c.stream, &iters[(size_t)i]);
  });
  if (st) drop_stored_j(*m);   // a failed solve is no starting guess, on any member
  m->step += (unsigned long long)(iters[0] - 1);   // the ranks agree on the iteration count
  if (nseg) {
    *nseg = 0;
    for (Member* q : m->mem) *nseg += q->nsegLast;
  }
  return st;
}

int multi_diffuse_host(Multi* m, int nAngularLevel, const double* uvb, const double* beta, const int32_t* rays,
                       int32_t nrays, double* J1, double* J2, double* J3, int64_t* nseg) {
  if (m->nleaf == 0 || !uvb || !beta) return RTB200_ERR_ARG;
  const bool scatter = multi_primary(m).scatterSigma() != nullptr;
  if (scatter && rays) {   // the J of a direction subset is not the mean intensity the source needs
    drop_stored_j(*m);
    return RTB200_ERR_ARG;
  }
  if (int st = build_shards(*m, nAngularLevel, rays, nrays, multi_primary(m).nx)) return st;
  m->step++;
  std::vector<int> iters((size_t)m->nlocal, 1);
  for (Member* q : m->mem) q->c.lastScatIter = 0, q->c.lastScatResid = 0., q->c.scatResidPending = false, q->c.lastNgCount = 0,
      q->c.lastWarm = false, q->c.ngPending = false, q->c.dWarmTaken = nullptr;
  int st = for_each_member(*m, [&](Member& q, int i) -> int {
    Context& c = q.c;
    RTB_CUDA(cudaSetDevice(c.device));
    const int buf = (int)(m->step & 1);
    PhaseTimer tm("diffuse", q.rank, c.stream);
    if (scatter) {
      if (int e = scatter_member(*m, q, m->step - 1, nAngularLevel, uvb, beta, Epilogue(), c.stream, &iters[(size_t)i])) return e;
      tm.mark("source iteration");
    } else {
      if (int e = sweep_member(*m, q, buf, nAngularLevel, uvb, beta, c.stream)) return e;
      tm.mark("opacities+sweep+merge");
      if (int e = reduce_member(*m, q, buf, m->step, 3, q.Jslab, Epilogue(), c.stream)) return e;
      tm.mark("reduce-scatter");
    }
    const int64_t off = slab_off(*m, q.rank), cnt = slab_cnt(*m, q.rank);
    const size_t nb = (size_t)cnt * sizeof(double);
    if (cnt > 0) {
      RTB_CUDA(cudaMemcpyAsync(J1 + off, q.Jslab, nb, cudaMemcpyDeviceToHost, c.stream));
      RTB_CUDA(cudaMemcpyAsync(J2 + off, q.Jslab + m->slab, nb, cudaMemcpyDeviceToHost, c.stream));
      RTB_CUDA(cudaMemcpyAsync(J3 + off, q.Jslab + 2 * m->slab, nb, cudaMemcpyDeviceToHost, c.stream));
    }
    RTB_CUDA(cudaStreamSynchronize(c.stream));
    tm.mark("d2h-slab");
    const int de = device_error(c);
    tm.mark("status");
    return de;
  });
  if (st) drop_stored_j(*m);   // a failed solve is no starting guess, on any member
  m->step += (unsigned long long)(iters[0] - 1);   // the ranks agree on the iteration count
  if (nseg) {
    *nseg = 0;
    for (Member* q : m->mem) *nseg += q->nsegLast;
  }
  return st;
}

// point sources of one member: its share of the source list (round robin over the ranks) into exch[buf][0..5]
static int point_member(Multi& m, Member& q, int buf, const PointInputs& in, std::vector<int>& mineIdx,
                        std::vector<double>& diag, cudaStream_t s) {
  mineIdx.clear();
  for (int i = q.rank; i < in.nsrc; i += m.nranks) mineIdx.push_back(i);
  std::vector<int32_t> leaf(mineIdx.size()), wt(mineIdx.size());
  for (size_t i = 0; i < mineIdx.size(); i++) { leaf[i] = in.srcLeaf[mineIdx[i]]; wt[i] = in.srcWeight[mineIdx[i]]; }
  PointInputs mine = in;
  mine.nsrc = (int)mineIdx.size(); mine.srcLeaf = leaf.data(); mine.srcWeight = wt.data();
  // point_solve deposits into a [6][nleaf] array: with a padded exchange layout it works on the context's own rate
  // buffer and the result is re-strided afterwards
  const size_t nb = (size_t)m.nleaf * sizeof(double);
  double* target = q.exch[buf];
  if (m.npad != m.nleaf) {
    if (!q.c.dRates) RTB_CUDA(cudaMalloc((void**)&q.c.dRates, 6 * nb));
    target = q.c.dRates;
  }
  RTB_CUDA(cudaMemsetAsync(target, 0, 6 * nb, s));
  diag.assign(mineIdx.size() * 320, 0.);
  int64_t ns = 0;
  int st = point_solve(q.c, mine, target, diag.data(), &ns, nullptr, 0, nullptr, nullptr, s);
  if (st) return st;
  q.nsegLast = ns;
  if (target != q.exch[buf]) {
    const int64_t total = 6 * m.npad;
    restride_kernel<<<(int)std::min<int64_t>((total + 255) / 256, (int64_t)q.c.smCount * 16), 256, 0, s>>>(target, m.nleaf, q.exch[buf],
                                                                                                          m.npad, 6);
    RTB_CUDA(cudaGetLastError());
  }
  return RTB200_OK;
}

static void scatter_diag(const std::vector<int>& idx, const std::vector<double>& d, double* rem, double* bnd, double* dust,
                         double* spec, int32_t* hpl) {
  for (size_t i = 0; i < idx.size(); i++) {
    const double* p = d.data() + i * 320;
    const size_t s = (size_t)idx[i];
    if (rem) memcpy(rem + s * 7, p, 56);
    if (bnd) memcpy(bnd + s * 7, p + 7, 56);
    if (dust) dust[s] = p[14];
    if (hpl) hpl[s] = (int32_t)p[15];
    if (spec) memcpy(spec + s * 300, p + 16, 2400);
  }
}

int multi_point_host(Multi* m, const PointInputs& in, double* const k[6], double* rem, double* bnd, double* dust,
                     double* spec, int32_t* hpl, int64_t* nseg) {
  for (int i = 0; i < 6; i++)
    if (!k[i]) return RTB200_ERR_ARG;
  if (m->nleaf == 0 || in.nsrc < 0) return RTB200_ERR_ARG;
  m->step++;
  int st = for_each_member(*m, [&](Member& q, int) -> int {
    Context& c = q.c;
    RTB_CUDA(cudaSetDevice(c.device));
    const int buf = (int)(m->step & 1);
    const int64_t off = slab_off(*m, q.rank), cnt = slab_cnt(*m, q.rank);
    const size_t nb = (size_t)cnt * sizeof(double);
    // the caller's rate fields are ACCUMULATED (equiSources.f90:3249-3260): its slab goes up, the sum comes back
    if (cnt > 0)
      for (int f = 0; f < 6; f++)
        RTB_CUDA(cudaMemcpyAsync(q.Rbase + (size_t)f * m->slab, k[f] + off, nb, cudaMemcpyHostToDevice, c.stream));
    std::vector<int> idx;
    std::vector<double> diag;
    if (int e = point_member(*m, q, buf, in, idx, diag, c.stream)) return e;
    Epilogue ep;
    ep.base = q.Rbase;
    if (int e = reduce_member(*m, q, buf, m->step, 6, q.Rslab, ep, c.stream)) return e;
    q.haveR = true;
    if (cnt > 0)
      for (int f = 0; f < 6; f++)
        RTB_CUDA(cudaMemcpyAsync(k[f] + off, q.Rslab + (size_t)f * m->slab, nb, cudaMemcpyDeviceToHost, c.stream));
    RTB_CUDA(cudaStreamSynchronize(c.stream));
    scatter_diag(idx, diag, rem, bnd, dust, spec, hpl);
    return device_error(c);
  });
  if (nseg) {
    *nseg = 0;
    for (Member* q : m->mem) *nseg += q->nsegLast;
  }
  return st;
}

// resident point pass: Rslab = sum over the ranks of this pass's deposits (setZeroRates first, equiSources.f90:1246)
int multi_point_resident(Multi* m, const PointInputs& in, void* const* streams, double* rem, double* bnd, double* dust,
                         double* spec, int32_t* hpl, int64_t* nseg) {
  if (m->nleaf == 0 || in.nsrc < 0) return RTB200_ERR_ARG;
  m->step++;
  int st = for_each_member(*m, [&](Member& q, int i) -> int {
    RTB_CUDA(cudaSetDevice(q.c.device));
    cudaStream_t s = streams ? (cudaStream_t)streams[i] : q.c.stream;
    const int buf = (int)(m->step & 1);
    std::vector<int> idx;
    std::vector<double> diag;
    if (int e = point_member(*m, q, buf, in, idx, diag, s)) return e;
    if (int e = reduce_member(*m, q, buf, m->step, 6, q.Rslab, Epilogue(), s)) return e;
    q.haveR = true;
    scatter_diag(idx, diag, rem, bnd, dust, spec, hpl);
    return RTB200_OK;
  });
  if (nseg) {
    *nseg = 0;
    for (Member* q : m->mem) *nseg += q->nsegLast;
  }
  return st;
}

}  // namespace rtb

using namespace rtb;

extern "C" {

int rtb200_comm_unique_id(char* id128) {
  if (!id128) return RTB200_ERR_ARG;
  if (int st = nccl_load()) return st;
  NcclId id;
  RTB_NCCL(nccl().GetUniqueId(&id));
  memcpy(id128, id.internal, 128);
  return RTB200_OK;
}

int rtb200_create_multi(int ngpus, const int* devices, rtb200_ctx** out) {
  if (!out) return RTB200_ERR_ARG;
  *out = nullptr;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_cuda_error("cudaGetDeviceCount", e == cudaSuccess ? cudaErrorNoDevice : e, __FILE__, __LINE__);
    return RTB200_ERR_CUDA;
  }
  if (ngpus < 1 || ngpus > ndev || ngpus > kMaxRanks) return RTB200_ERR_ARG;
  std::vector<int> dev((size_t)ngpus);
  for (int i = 0; i < ngpus; i++) {
    dev[i] = devices ? devices[i] : i;
    if (dev[i] < 0 || dev[i] >= ndev) return RTB200_ERR_ARG;
    for (int j = 0; j < i; j++)
      if (dev[j] == dev[i]) return RTB200_ERR_ARG;
  }
  if (ngpus > 1)
    if (int st = nccl_load()) return st;
  Multi* m = new (std::nothrow) Multi();
  rtb200_ctx* h = new (std::nothrow) rtb200_ctx();
  if (!m || !h) { delete m; delete h; return RTB200_ERR_NOMEM; }
  m->nranks = ngpus; m->nlocal = ngpus; m->rank0 = 0; m->multiProcess = false;
  int st = create_members(m, dev.data());
  if (!st && ngpus > 1) {
    std::vector<NcclComm> comms((size_t)ngpus, nullptr);
    int r = nccl().CommInitAll(comms.data(), ngpus, dev.data());
    if (r != 0) {
      set_cuda_error(nccl().GetErrorString(r), cudaErrorUnknown, __FILE__, __LINE__);
      st = RTB200_ERR_CUDA;
    } else {
      for (int i = 0; i < ngpus; i++) m->mem[i]->comm = comms[i];
    }
  }
  if (st) { multi_destroy(m); delete h; return st; }
  h->m = m;
  *out = h;
  return RTB200_OK;
}

int rtb200_create_rank(int device, int nranks, int rank, const char* id128, rtb200_ctx** out) {
  if (!out) return RTB200_ERR_ARG;
  *out = nullptr;
  if (nranks < 1 || nranks > kMaxRanks || rank < 0 || rank >= nranks || (nranks > 1 && !id128)) return RTB200_ERR_ARG;
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0) {
    set_cuda_error("cudaGetDeviceCount", e == cudaSuccess ? cudaErrorNoDevice : e, __FILE__, __LINE__);
    return RTB200_ERR_CUDA;
  }
  if (device < 0 || device >= ndev) return RTB200_ERR_ARG;
  if (nranks > 1)
    if (int st = nccl_load()) return st;
  Multi* m = new (std::nothrow) Multi();
  rtb200_ctx* h = new (std::nothrow) rtb200_ctx();
  if (!m || !h) { delete m; delete h; return RTB200_ERR_NOMEM; }
  m->nranks = nranks; m->nlocal = 1; m->rank0 = rank; m->multiProcess = nranks > 1;
  int st = create_members(m, &device);
  if (!st && nranks > 1) {
    NcclId id;
    memcpy(id.internal, id128, 128);
    cudaSetDevice(device);
    int r = nccl().CommInitRank(&m->mem[0]->comm, nranks, id, rank);
    if (r != 0) {
      set_cuda_error(nccl().GetErrorString(r), cudaErrorUnknown, __FILE__, __LINE__);
      st = RTB200_ERR_CUDA;
    }
  }
  if (st) { multi_destroy(m); delete h; return st; }
  h->m = m;
  *out = h;
  return RTB200_OK;
}

int rtb200_multi_info(rtb200_ctx* h, int32_t* nranks, int32_t* nlocal, int32_t* firstRank, int64_t* slab, int32_t* reduceMode) {
  if (!h) return RTB200_ERR_ARG;
  if (!h->m) {
    if (nranks) *nranks = 1;
    if (nlocal) *nlocal = 1;
    if (firstRank) *firstRank = 0;
    if (slab) *slab = h->c.nleaf;
    if (reduceMode) *reduceMode = -1;
    return RTB200_OK;
  }
  Multi& m = *h->m;
  if (nranks) *nranks = m.nranks;
  if (nlocal) *nlocal = m.nlocal;
  if (firstRank) *firstRank = m.rank0;
  if (slab) *slab = m.slab;
  if (reduceMode) *reduceMode = (m.reduceMode == 1 && m.peerOk) ? 1 : 0;
  return RTB200_OK;
}

int rtb200_multi_slab(rtb200_ctx* h, int local, int64_t* offset, int64_t* count, double** J_device, double** K_device,
                      double** R_device) {
  if (!h || !h->m || local < 0 || local >= h->m->nlocal) return RTB200_ERR_ARG;
  Multi& m = *h->m;
  Member& q = *m.mem[local];
  if (offset) *offset = slab_off(m, q.rank);
  if (count) *count = slab_cnt(m, q.rank);
  if (J_device) *J_device = q.Jslab;
  if (K_device) *K_device = q.Kslab;
  if (R_device) *R_device = q.Rslab;
  return RTB200_OK;
}

int rtb200_multi_slab_get(rtb200_ctx* h, int local, double* J3, double* K3, double* R6) {
  if (!h || !h->m || local < 0 || local >= h->m->nlocal) return RTB200_ERR_ARG;
  Multi& m = *h->m;
  Member& q = *m.mem[local];
  RTB_CUDA(cudaSetDevice(q.c.device));
  RTB_CUDA(cudaDeviceSynchronize());
  const size_t nb = (size_t)m.slab * sizeof(double);
  if (J3) RTB_CUDA(cudaMemcpy(J3, q.Jslab, 3 * nb, cudaMemcpyDeviceToHost));
  if (K3) RTB_CUDA(cudaMemcpy(K3, q.Kslab, 3 * nb, cudaMemcpyDeviceToHost));
  if (R6) RTB_CUDA(cudaMemcpy(R6, q.Rslab, 6 * nb, cudaMemcpyDeviceToHost));
  return device_error(q.c);
}

int rtb200_shard_directions(int nranks, int nAngularLevel, int nx, const double* zoneCost3, int rank, int32_t* rays,
                            int32_t cap, int32_t* nrays) {
  if (!nrays || rank < 0 || rank >= nranks) return RTB200_ERR_ARG;
  const double dflt[3] = {kZoneCostX, kZoneCostY, kZoneCostZ};
  std::vector<std::vector<int32_t>> shards;
  if (int st = shard_directions(nranks, nAngularLevel, nullptr, 0, nx, zoneCost3 ? zoneCost3 : dflt, shards)) return st;
  const auto& s = shards[(size_t)rank];
  *nrays = (int32_t)s.size();
  if (rays)
    for (int32_t i = 0; i < std::min<int32_t>(cap, (int32_t)s.size()); i++) rays[i] = s[i];
  return RTB200_OK;
}

int rtb200_multi_shard(rtb200_ctx* h, int nAngularLevel, int rank, int32_t* rays, int32_t cap, int32_t* nrays) {
  if (!h || !h->m || !nrays || rank < 0 || rank >= h->m->nranks) return RTB200_ERR_ARG;
  Multi& m = *h->m;
  if (int st = build_shards(m, nAngularLevel, nullptr, 0, m.nleaf ? multi_primary(&m).nx : 32)) return st;
  const auto& s = m.shards[(size_t)rank];
  *nrays = (int32_t)s.size();
  if (rays)
    for (int32_t i = 0; i < std::min<int32_t>(cap, (int32_t)s.size()); i++) rays[i] = s[i];
  return RTB200_OK;
}

int rtb200_multi_diffuse_resident(rtb200_ctx* h, int nAngularLevel, const double* uvb, const double* beta, const double* ksi6,
                                  int chemistry, void* const* streams, int64_t* nseg) {
  if (!h || !h->m) return RTB200_ERR_ARG;
  return multi_diffuse_resident(h->m, nAngularLevel, uvb, beta, ksi6, chemistry, streams, nseg);
}

int rtb200_multi_point_resident(rtb200_ctx* h, int nWave, const double* wavelength, const double* lum, const double* metallicity,
                                double coefSpectrum, const double* aDust, int dustApproximation, int maxPixelLevel, int32_t nsrc,
                                const int32_t* srcLeaf, const int32_t* srcWeight, void* const* streams, double* ndotRemaining,
                                double* ndotBoundary, double* ndotDust, double* ndotSpectrum, int32_t* highestPixelLevel,
                                int64_t* nseg) {
  if (!h || !h->m) return RTB200_ERR_ARG;
  PointInputs in;
  in.nWave = nWave; in.wavelength = wavelength; in.lum = lum; in.metallicity = metallicity; in.coefSpectrum = coefSpectrum;
  in.aDust = aDust; in.dust = dustApproximation; in.maxPixelLevel = maxPixelLevel; in.nsrc = nsrc; in.srcLeaf = srcLeaf;
  in.srcWeight = srcWeight;
  return multi_point_resident(h->m, in, streams, ndotRemaining, ndotBoundary, ndotDust, ndotSpectrum, highestPixelLevel, nseg);
}

int rtb200_multi_sync(rtb200_ctx* h) {
  if (!h || !h->m) return RTB200_ERR_ARG;
  int first = 0;
  for (Member* q : h->m->mem) {
    cudaSetDevice(q->c.device);
    if (cudaDeviceSynchronize() != cudaSuccess && !first) first = RTB200_ERR_CUDA;
    const int e = device_error(q->c);
    if (e && !first) first = e;
  }
  return first;
}

}  // extern "C"
