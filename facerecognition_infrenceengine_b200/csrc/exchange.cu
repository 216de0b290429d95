// Multi-GPU tail over NVLink peer memory, no collective-library call on the data path (SURVEY.md section 8e).
//
// Every rank's exchange buffer (peer-mapped into all ranks, e.g. a torch symmetric-memory allocation) holds,
// per call parity and source rank, the source's local top-k block as PACKETS: 8-byte words {payload, epoch},
// stored with single 8-byte writes, so a packet is valid exactly when its epoch word matches - the data is
// its own flag (the low-latency protocol of collective libraries): no fence, no separate flag, no grid-wide
// rendezvous.  Three packet planes per block: row low word, row high word, score bits.
//
//   PUSH  every local result is pushed by a kernel of the local match itself, the moment it is final:
//           select_rescore_kernel (tc_match.cu)   each query's top-k, plus the call's hello packets
//           scan_f32_flagged_kernel (scan_f32.cu) the queries redone by the exact fallback (its last CTA)
//           exchange_push_kernel (here)           everything, for variants without a select stage
//   POLL  exchange_merge_kernel then only WAITS and merges: one warp per query polls the `world` lists of that
//         query in its OWN buffer until their packets carry the call's epoch, and folds them.  Because it is a
//         later kernel of the same stream than every local push, none of its CTAs can wait for a push that
//         sits in a CTA which is not resident yet (round 1 had both in one kernel: with another stream's
//         kernels holding SMs, resident pollers of two GPUs could wait for each other's non-resident pushers).
//
// Handshake and failure reporting.  A rank's first push of a call is a hello packet {(nq << 5) | k, epoch}
// into every rank's header.  The poll kernel checks the hellos first: a peer that is in a different call
// (call-count mismatch) or disagrees on (nq, k) is REPORTED - status record in the header, sentinel results,
// FRG_ERR_STATE from frg_exchange_status - instead of waited on.  Every wait is bounded (XPush::timeout_ns,
// default 2 s, FRG_EXCHANGE_TIMEOUT_MS): a dead or diverged peer costs one timeout, never a hung GPU and
// never a trap that would poison the CUDA context of a long-running service.
//
// Double buffering by epoch parity: a rank can be at most one call ahead of a peer (it cannot finish call
// e+1 before the peer has pushed e+1, which the peer does only after its call e completed in stream order),
// so the packets of parity e&1 are never overwritten while a slower peer still reads call e.
#include <cstdlib>

#include "merge_device.cuh"

namespace frg {

__device__ __forceinline__ uint2 ld_packet(const uint2* p) {
  uint2 v;
  asm volatile("ld.relaxed.sys.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// the first failure of a call wins the status record; everybody else sees code != 0 and stops waiting
__device__ __noinline__ void record_failure(XStatus* st, uint32_t code, uint32_t peer, uint32_t epoch,
                                            uint32_t seen_epoch, uint32_t want_hello, uint32_t seen_hello,
                                            uint32_t query) {
  if (atomicCAS(&st->code, 0u, 0xffffffffu) == 0u) {
    st->peer = peer; st->epoch = epoch; st->seen_epoch = seen_epoch;
    st->want_hello = want_hello; st->seen_hello = seen_hello; st->query = query;
    __threadfence();
    atomicExch(&st->code, code);
  }
}

// the packet planes this rank RECEIVES for the call's parity, with bounded waits
struct PacketLists {
  const unsigned char* mine;       // this rank's exchange buffer
  int world;
  int64_t block_cap, nslots;
  uint32_t epoch, hello;
  unsigned long long deadline;     // %globaltimer value after which a missing packet is a failure
  XStatus* status;

  // false: gave up (deadline passed, or another warp has already recorded a failure)
  __device__ __forceinline__ bool wait(const uint2* p, uint2* out) const {
    uint2 v = ld_packet(p);
    unsigned spins = 0;
    while (v.y != epoch) {
      __nanosleep(64);
      v = ld_packet(p);
      if ((++spins & 31u) == 0u && v.y != epoch) {
        if (ld_volatile_u32(&status->code) != 0u || global_ns() > deadline) { *out = v; return false; }
      }
    }
    *out = v;
    return true;
  }

  // lanes over the source ranks: every rank must be in THIS call with THIS (nq, k)
  __device__ __forceinline__ bool hellos_ok(int lane) const {
    bool ok = true;
    for (int p = lane; p < world; p += 32) {
      const uint2* h = reinterpret_cast<const uint2*>(mine) + (epoch & 1u) * kExchangeMaxWorld + p;
      uint2 v;
      if (!wait(h, &v)) { record_failure(status, kXHelloTimeout, p, epoch, v.y, hello, v.x, 0); ok = false; }
      else if (v.x != hello) { record_failure(status, kXHelloMismatch, p, epoch, v.y, hello, v.x, 0); ok = false; }
    }
    return __all_sync(0xffffffffu, ok);
  }

  __device__ __forceinline__ void load(int part, size_t in_part, int64_t* r, float* s) const {
    const uint2* b = reinterpret_cast<const uint2*>(
        mine + kExchangeHeader + (size_t(epoch & 1u) * world + part) * size_t(block_cap));
    uint2 lo, hi, sc;
    if (wait(b + in_part, &lo) && wait(b + nslots + in_part, &hi) && wait(b + 2 * nslots + in_part, &sc)) {
      *r = int64_t((uint64_t(hi.x) << 32) | uint64_t(lo.x));
      *s = __uint_as_float(sc.x);
      return;
    }
    record_failure(status, kXDataTimeout, uint32_t(part), epoch, lo.y, hello, 0u, uint32_t(in_part));
    *r = -1;                       // dropped by the merge; the whole result is void anyway (status != 0)
    *s = kNoScore;
  }
};

// hello + the local top-k of every query -> every rank.  One warp per query, lanes over (peer, slot).
__global__ void __launch_bounds__(128)
exchange_push_kernel(const XPush x, const int64_t* __restrict__ local_rows, const float* __restrict__ local_scores,
                     int nq, int k) {
  const int lane = threadIdx.x & 31;
  const int warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  pdl_wait();             // the local match's results
  pdl_trigger();
  if (warp == 0)
    for (int p = lane; p < x.world; p += 32) xpush_hello(x, p);
  for (int q = warp; q < nq; q += nwarps) {
    for (int c = lane; c < x.world * k; c += 32) {
      const int peer = c / k, j = c - peer * k;
      const int64_t slot = int64_t(q) * k + j;
      xpush_slot(x, (x.rank + 1 + peer) % x.world, slot, local_rows[slot], local_scores[slot]);
    }
  }
}

template <int KMAX>
__global__ void __launch_bounds__(128)
exchange_merge_kernel(const XPush x, int nq, int k, int metric, float threshold,
                      int64_t* __restrict__ out_rows, float* __restrict__ out_scores,
                      uint8_t* __restrict__ out_accept) {
  const int lane = threadIdx.x & 31;
  const int warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int nwarps = gridDim.x * (blockDim.x >> 5);
  pdl_wait();             // every local push has been issued by an earlier kernel of this stream
  unsigned char* mine = x.peer_bufs[x.rank];
  XStatus* status = reinterpret_cast<XStatus*>(mine + kExchangeStatusOff);
  const PacketLists lists{mine, x.world, x.block_cap, x.nslots, x.epoch, x.hello, global_ns() + x.timeout_ns, status};
  bool ok = warp < nq ? lists.hellos_ok(lane) : true;
  for (int q = warp; q < nq; q += nwarps) {
    if (ok) {
      merge_lists<int64_t, KMAX>(lists, x.world, k, k, metric, threshold, 0, 0, q, q, out_rows, out_scores, out_accept);
      __syncwarp();
      ok = ld_volatile_u32(&status->code) == 0u;
    }
    if (!ok) {
      // a void call returns "no match" everywhere; frg_exchange_status tells the host why
      for (int j = lane; j < k; j += 32) {
        out_rows[size_t(q) * k + j] = kNoRow;
        out_scores[size_t(q) * k + j] = metric == FRG_METRIC_EUCLIDEAN ? INFINITY : kNoScore;
      }
      if (lane == 0 && out_accept) out_accept[q] = 0;
    }
  }
}

static unsigned long long exchange_timeout_ns() {
  static const unsigned long long v = []() {
    const char* e = getenv("FRG_EXCHANGE_TIMEOUT_MS");
    const long ms = e ? atol(e) : 2000;
    return (unsigned long long)(ms < 1 ? 1 : ms) * 1000000ull;
  }();
  return v;
}

void exchange_fill_defaults(XPush* x, int nq, int k) {
  x->hello = (uint32_t(nq) << 5) | uint32_t(k);
  x->nslots = int64_t(nq) * k;
  x->timeout_ns = exchange_timeout_ns();
}

int launch_exchange_push(const XPush& x, const int64_t* local_rows, const float* local_scores, int nq, int k,
                         int sm_count, cudaStream_t st) {
  if (nq <= 0) return FRG_OK;
  int grid = (nq + 3) / 4;
  if (grid > 4 * sm_count) grid = 4 * sm_count;
  FRG_CUDA(launch_kernel(exchange_push_kernel, dim3(grid), dim3(128), 0, st, x, local_rows, local_scores, nq, k));
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

int launch_exchange_merge(const XPush& x, int nq, int k, int metric, float threshold, int sm_count,
                          int64_t* out_rows, float* out_scores, uint8_t* out_accept, cudaStream_t st) {
  if (nq <= 0) return FRG_OK;
  int grid = (nq + 3) / 4;
  if (grid > 4 * sm_count) grid = 4 * sm_count;
  if (grid < 1) grid = 1;
#define FRG_XM(K)                                                                                              \
  FRG_CUDA(launch_kernel(exchange_merge_kernel<K>, dim3(grid), dim3(128), 0, st, x, nq, k, metric, threshold, \
                         out_rows, out_scores, out_accept))
  if (k == 1) FRG_XM(1);
  else if (k <= 4) FRG_XM(4);
  else if (k <= 8) FRG_XM(8);
  else FRG_XM(16);
#undef FRG_XM
  note_launch(nullptr);
  FRG_CUDA(cudaGetLastError());
  return FRG_OK;
}

}  // namespace frg
