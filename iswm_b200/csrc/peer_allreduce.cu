// peer_allreduce.cu — gradient / scalar all-reduce over NVLink 5 / NVSwitch PEER MEMORY, as plain stream-ordered kernels.
//
// The reference trains under nn.DataParallel (train.py:970): gradients are reduce-added across replicas every step. Here
// every rank owns a gradient buffer in SYMMETRIC memory (same size on every GPU, each rank's buffer mapped into every other
// rank's address space; the mapping comes from torch.distributed._symmetric_memory on the Python side, this file only sees
// raw peer pointers). A bucket is reduced by three launches on one stream:
//   1. peer_barrier_kernel   every rank has produced its bucket (flags in peer memory, release / acquire at system scope)
//   2. peer_allreduce_kernel rank r sums slice r of the bucket over all ranks' buffers - loads over NVLink in a FIXED rank
//                            order, so the sums are bit-identical on every rank and from run to run - and stores the result
//                            into every rank's buffer (two-shot all-reduce: reduce-scatter by pull, all-gather by push)
//   3. peer_barrier_kernel   every rank's stores have landed
// No host synchronisation and no library call: the whole data-parallel train step, collectives included, is captured in
// ONE CUDA graph (iswm_b200.graphs.GraphedTrainStep), which the NCCL path could not be (DESIGN 3b).
// Waits are bounded (about 4 s of SM clocks): a rank that never arrives makes its peers record an abort code and return.
#include "common.cuh"

namespace iswm {

constexpr int kMaxPeers = 8;

struct PeerPtrs {
  void* p[kMaxPeers];
};

__device__ __forceinline__ void st_release_sys(uint32_t* addr, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* addr) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(addr) : "memory");
  return v;
}

// flags: every rank owns uint32 flags[kMaxPeers] in symmetric memory (slot q = "rank q has reached barrier number v").
// epoch: this rank's private device counter of barriers executed (all ranks run the same sequence, so the counters agree).
// Thread q < world of the calling block signals rank q and waits for rank q's signal; the caller synchronises the block after.
__device__ __forceinline__ void barrier_arrive_wait(const PeerPtrs& flags, int rank, int world, uint32_t e, int* abort_flag, int& bad) {
  const int q = threadIdx.x;
  if (q < world) {
    __threadfence_system();                                   // everything this GPU wrote before the barrier is visible system-wide
    st_release_sys(reinterpret_cast<uint32_t*>(flags.p[q]) + rank, e);
    const uint32_t* mine = reinterpret_cast<const uint32_t*>(flags.p[rank]) + q;
    const long long t0 = clock64();
    int it = 0;
    // (int32) difference: correct across the counter's wrap
    while ((int32_t)(ld_acquire_sys(mine) - e) < 0) {
      if (((++it) & 255) == 0) {
        if (*((volatile int*)abort_flag) != 0 || clock64() - t0 > 8000000000ll) {
          atomicCAS(abort_flag, 0, 31);
          bad = 1;
          break;
        }
      }
    }
  }
}

__global__ void peer_barrier_kernel(PeerPtrs flags, int rank, int world, uint32_t* epoch, int* abort_flag) {
  pdl_wait();
  pdl_launch();
  const int q = threadIdx.x;
  __shared__ int bad;
  if (q == 0) bad = 0;
  __syncthreads();
  const uint32_t e = *epoch + 1;
  barrier_arrive_wait(flags, rank, world, e, abort_flag, bad);
  __syncthreads();
  if (q == 0) *epoch = e;
  (void)bad;
}

// Rank r reduces elements [lo_r, hi_r) of [off, off + n) (equal slices, multiples of 4 floats) and pushes the sums to all.
__global__ void __launch_bounds__(512)
peer_allreduce_f32_kernel(PeerPtrs bufs, int rank, int world, long long off, long long n) {
  pdl_wait();
  pdl_launch();
  const long long per = (((n + world - 1) / world) + 3) & ~3ll;
  const long long lo = min(n, (long long)rank * per), hi = min(n, lo + per);
  const long long nvec = (hi - lo) >> 2;                       // n and per are multiples of 4
  const long long base = off + lo;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 v[kMaxPeers];
#pragma unroll
    for (int p = 0; p < kMaxPeers; p++)
      if (p < world) v[p] = __ldcv(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(bufs.p[p]) + base) + i);   // volatile: peers' data, never cached stale
#pragma unroll
    for (int p = 0; p < kMaxPeers; p++)
      if (p < world) { acc.x += v[p].x; acc.y += v[p].y; acc.z += v[p].z; acc.w += v[p].w; }
#pragma unroll
    for (int p = 0; p < kMaxPeers; p++)
      if (p < world) reinterpret_cast<float4*>(reinterpret_cast<float*>(bufs.p[p]) + base)[i] = acc;
  }
}

// Small vectors (class histogram: C int64; loss numerators: a few doubles): every rank publishes its values in its own
// symmetric slot region, a barrier, every rank sums all ranks' regions in rank order. Each call SITE of a step uses its own
// region (slot_off): a region is rewritten one whole step later, with barriers of the same step in between, so a slow peer
// can never read the next step's values. 8-byte slots, slot_off + n <= the region the caller allocated.
constexpr int kSmallMax = 64;
template <typename T>
__global__ void peer_small_publish_kernel(PeerPtrs slots, int rank, const T* src, int n, int slot_off) {
  pdl_wait();
  pdl_launch();
  T* mine = reinterpret_cast<T*>(slots.p[rank]) + slot_off;
  for (int i = threadIdx.x; i < n; i += blockDim.x) mine[i] = src[i];
}
template <typename T>
__global__ void peer_small_sum_kernel(PeerPtrs slots, int world, T* dst, int n, int slot_off) {
  pdl_wait();
  pdl_launch();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    T acc = 0;
    for (int p = 0; p < world; p++) acc += __ldcv(reinterpret_cast<const T*>(slots.p[p]) + slot_off + i);
    dst[i] = acc;
  }
}

// Synchronised BatchNorm statistics. Every rank's engine carves the SAME offsets of a symmetric fp64 arena for the same
// BatchNorm (sizes depend on channel counts only), so a peer's vector is read in place at arena.p[peer] + src_off - no publish
// copy. One launch per exchange, one block:
//   1. this rank's row count goes into the word after the first job's vector (its replica copies), so counts of unequal
//      shards are exchanged rather than assumed;
//   2. barrier (signal every rank, bounded wait; skipped when flags.p[0] is null: a one-rank fold);
//   3. dst[i] = sum over ranks 0..world-1, in that order, of (sum over the vector's replica copies, in order) - the same bits
//      on every rank - and dst[n] = the global count.
// A separate kernel rather than peer reads inside every block of the BatchNorm kernels: one block reads world x n values over
// NVLink, where every apply block doing so would read ~3 x 148 x world x n (about 100 MB per BatchNorm at C = 2048).
constexpr int kSyncBnMaxJobs = 4;
constexpr int kSyncBnThreads = 512;
struct SyncBnJobs {
  long long src_off[kSyncBnMaxJobs];      // fp64 elements from the arena base
  double* dst[kSyncBnMaxJobs];            // local: n sums + 1 count
  int n[kSyncBnMaxJobs];
  int rep[kSyncBnMaxJobs];
  int njobs;
};

__global__ void __launch_bounds__(kSyncBnThreads)
syncbn_exchange_kernel(PeerPtrs arena, PeerPtrs flags, int rank, int world, uint32_t* epoch, int* abort_flag, SyncBnJobs jobs,
                       double count) {
  pdl_wait();
  pdl_launch();
  __shared__ int bad;
  const int t = threadIdx.x;
  const long long cnt_off = jobs.src_off[0] + (long long)jobs.n[0] * jobs.rep[0];
  if (t == 0) {
    bad = 0;
    reinterpret_cast<double*>(arena.p[rank])[cnt_off] = count;
    __threadfence_system();
  }
  __syncthreads();
  const bool peers = flags.p[0] != nullptr;
  uint32_t e = 0;
  if (peers) {
    e = *epoch + 1;
    barrier_arrive_wait(flags, rank, world, e, abort_flag, bad);
    __syncthreads();
  }
  for (int j = 0; j < jobs.njobs; j++) {
    const int n = jobs.n[j], rep = jobs.rep[j];
    const long long off = jobs.src_off[j];
    for (int i = t; i < n; i += kSyncBnThreads) {
      double v[kMaxPeers];
#pragma unroll
      for (int p = 0; p < kMaxPeers; p++) {
        if (p < world) {
          const double* src = reinterpret_cast<const double*>(arena.p[p]) + off + i;
          double a = __ldcv(src);                             // volatile: peers' data, never cached stale
          for (int r = 1; r < rep; r++) a += __ldcv(src + (long long)r * n);
          v[p] = a;
        }
      }
      double acc = v[0];
#pragma unroll
      for (int p = 1; p < kMaxPeers; p++)
        if (p < world) acc += v[p];
      jobs.dst[j][i] = acc;
    }
  }
  if (t == 0) {
    double acc = __ldcv(reinterpret_cast<const double*>(arena.p[0]) + cnt_off);
    for (int p = 1; p < world; p++) acc += __ldcv(reinterpret_cast<const double*>(arena.p[p]) + cnt_off);
    for (int j = 0; j < jobs.njobs; j++) jobs.dst[j][jobs.n[j]] = acc;
    if (peers) *epoch = e;
  }
  (void)bad;
}

}  // namespace iswm

using namespace iswm;

static int fill_ptrs(PeerPtrs& pp, const void* const* ptrs, int world, const char* what) {
  ISWM_REQUIRE(world >= 1 && world <= kMaxPeers, "%s: world size %d (1..%d)", what, world, kMaxPeers);
  for (int i = 0; i < kMaxPeers; i++) pp.p[i] = nullptr;
  for (int i = 0; i < world; i++) {
    ISWM_REQUIRE(ptrs[i] != nullptr, "%s: null peer pointer for rank %d", what, i);
    pp.p[i] = const_cast<void*>(ptrs[i]);
  }
  return 0;
}

static int* barrier_abort_flag() {
  static thread_local int* cached = nullptr;                 // one per device context in practice (one process per GPU)
  if (!cached && cudaMalloc(&cached, sizeof(int)) == cudaSuccess) cudaMemset(cached, 0, sizeof(int));
  return cached;
}

extern "C" int iswm_peer_barrier(const void* const* flag_ptrs, int rank, int world, uint32_t* d_epoch, void* stream) {
  ISWM_REQUIRE(flag_ptrs && d_epoch && rank >= 0 && rank < world, "peer_barrier: bad arguments");
  PeerPtrs pp;
  if (int rc = fill_ptrs(pp, flag_ptrs, world, "peer_barrier")) return rc;
  int* abort_flag = barrier_abort_flag();
  ISWM_REQUIRE(abort_flag, "peer_barrier: cannot allocate the abort flag");
  launch_k(peer_barrier_kernel, dim3(1), dim3(32), 0, static_cast<cudaStream_t>(stream), pp, rank, world, d_epoch, abort_flag);
  return check_launch("peer_barrier");
}

extern "C" int iswm_peer_allreduce_f32(const void* const* buf_ptrs, int rank, int world, int64_t offset, int64_t n, int max_blocks, void* stream) {
  ISWM_REQUIRE(buf_ptrs && rank >= 0 && rank < world && offset >= 0 && n >= 0, "peer_allreduce_f32: bad arguments");
  ISWM_REQUIRE((offset % 4) == 0 && (n % 4) == 0, "peer_allreduce_f32: offset=%lld and n=%lld must be multiples of 4 floats", (long long)offset, (long long)n);
  if (n == 0) return 0;
  PeerPtrs pp;
  if (int rc = fill_ptrs(pp, buf_ptrs, world, "peer_allreduce_f32")) return rc;
  for (int i = 0; i < world; i++) ISWM_REQUIRE((reinterpret_cast<uintptr_t>(buf_ptrs[i]) & 15) == 0, "peer_allreduce_f32: buffers must be 16-byte aligned");
  const long long per = (((n + world - 1) / world) + 3) & ~3ll;
  long long blocks = (per / 4 + 511) / 512;
  const int cap = max_blocks > 0 ? max_blocks : 2 * num_sms();
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  launch_k(peer_allreduce_f32_kernel, dim3((unsigned)blocks), dim3(512), 0, static_cast<cudaStream_t>(stream), pp, rank, world, (long long)offset, (long long)n);
  return check_launch("peer_allreduce_f32");
}

extern "C" int iswm_peer_small_publish(const void* const* slot_ptrs, int rank, int world, const void* d_src, int n, int slot_off, int is_f64, void* stream) {
  ISWM_REQUIRE(slot_ptrs && d_src && n >= 0 && n <= kSmallMax && slot_off >= 0 && rank >= 0 && rank < world, "peer_small_publish: bad arguments (n <= %d)", kSmallMax);
  PeerPtrs pp;
  if (int rc = fill_ptrs(pp, slot_ptrs, world, "peer_small_publish")) return rc;
  if (is_f64) launch_k(peer_small_publish_kernel<double>, dim3(1), dim3(64), 0, static_cast<cudaStream_t>(stream), pp, rank, static_cast<const double*>(d_src), n, slot_off);
  else launch_k(peer_small_publish_kernel<long long>, dim3(1), dim3(64), 0, static_cast<cudaStream_t>(stream), pp, rank, static_cast<const long long*>(d_src), n, slot_off);
  return check_launch("peer_small_publish");
}

extern "C" int iswm_peer_small_sum(const void* const* slot_ptrs, int world, void* d_dst, int n, int slot_off, int is_f64, void* stream) {
  ISWM_REQUIRE(slot_ptrs && d_dst && n >= 0 && n <= kSmallMax && slot_off >= 0, "peer_small_sum: bad arguments (n <= %d)", kSmallMax);
  PeerPtrs pp;
  if (int rc = fill_ptrs(pp, slot_ptrs, world, "peer_small_sum")) return rc;
  if (is_f64) launch_k(peer_small_sum_kernel<double>, dim3(1), dim3(64), 0, static_cast<cudaStream_t>(stream), pp, world, static_cast<double*>(d_dst), n, slot_off);
  else launch_k(peer_small_sum_kernel<long long>, dim3(1), dim3(64), 0, static_cast<cudaStream_t>(stream), pp, world, static_cast<long long*>(d_dst), n, slot_off);
  return check_launch("peer_small_sum");
}

extern "C" int iswm_syncbn_exchange(const iswm_syncbn_job* jobs, int n_jobs, const void* const* arena_ptrs, const void* const* flag_ptrs,
                                    int rank, int world, double count, uint32_t* d_epoch, void* stream) {
  ISWM_REQUIRE(jobs && n_jobs >= 1 && n_jobs <= kSyncBnMaxJobs, "syncbn_exchange: 1..%d jobs", kSyncBnMaxJobs);
  ISWM_REQUIRE(arena_ptrs && rank >= 0 && rank < world && count >= 1.0, "syncbn_exchange: bad arguments");
  ISWM_REQUIRE(flag_ptrs || world == 1, "syncbn_exchange: %d ranks need the barrier flags", world);
  ISWM_REQUIRE(!flag_ptrs || d_epoch, "syncbn_exchange: the barrier needs its epoch counter");
  PeerPtrs arena, flags;
  if (int rc = fill_ptrs(arena, arena_ptrs, world, "syncbn_exchange")) return rc;
  for (int i = 0; i < kMaxPeers; i++) flags.p[i] = nullptr;
  if (flag_ptrs)
    if (int rc = fill_ptrs(flags, flag_ptrs, world, "syncbn_exchange")) return rc;
  SyncBnJobs sj{};
  for (int j = 0; j < n_jobs; j++) {
    const iswm_syncbn_job& J = jobs[j];
    ISWM_REQUIRE(J.dst && J.n > 0 && J.src_off >= 0 && J.replicas >= 1, "syncbn_exchange: job %d: bad slot", j);
    sj.src_off[j] = J.src_off; sj.dst[j] = J.dst; sj.n[j] = J.n; sj.rep[j] = J.replicas;
  }
  sj.njobs = n_jobs;
  int* abort_flag = barrier_abort_flag();
  ISWM_REQUIRE(abort_flag, "syncbn_exchange: cannot allocate the abort flag");
  launch_k(syncbn_exchange_kernel, dim3(1), dim3(kSyncBnThreads), 0, static_cast<cudaStream_t>(stream), arena, flags, rank, world, d_epoch,
           abort_flag, sj, count);
  return check_launch("syncbn_exchange");
}
