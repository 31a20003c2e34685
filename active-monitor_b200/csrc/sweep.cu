// sweep.cu — the am_sweep handle and the C-ABI entry points of libamsweep.
//
// Owns one shard of the HealthCheck record array in HBM (16 SoA columns,
// SURVEY.md Appendix B.1) on one CUDA device, the staging area for
// upsert / remove / post_result calls coming from the controller's goroutines
// (hcc.go:170-188 Reconcile workers, hcc.go:635/:662/:821/:836 watch loops),
// and the launch of the tick's kernels (sweep_kernels.cuh) that replace the
// per-CR schedule ladder and remedy state machine for every record at once.
//
// Shape of the host side (round 2; profiles/r02_e2e_breakdown.md has the timings):
//   * staged events are 64-bit words (slot, arg) (+ 96-B records for upserts) in pinned
//     memory, double-buffered: a tick swaps the buffers under the staging lock and
//     releases it at once — callers never wait for a copy or a kernel;
//   * posted events are copied to the device in chunks WHILE they are being posted (copy
//     stream), so at tick time only the tail is left;
//   * the list rebuild writes (u32 local index, u8 action) straight into mapped pinned
//     host memory and the statistics into a mapped struct: ONE stream synchronisation per
//     tick, no device-to-host copy call, and am_sweep_tick_view hands that memory to the
//     caller without another pass;
//   * every device operation of a handle is ordered after the previous one even when they
//     are issued on different streams (am_sweep_tick_device takes the caller's stream).
//
// There is deliberately no CPU path in this file: without a CUDA device
// am_sweep_create fails with AM_E_DEVICE.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <mutex>
#include <new>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "sweep_internal.h"
#include "sweep_kernels.cuh"
#include "tz.h"

using namespace amsweep;

namespace amsweep_host {
unsigned stage_results(uint64_t n, const uint64_t* idx, const uint8_t* phase, const uint8_t* remedy, uint64_t capacity,
                       uint32_t op_result_kind, uint64_t* ops);
void widen_list(uint64_t n, uint64_t base, const uint32_t* idx32, const uint8_t* act8, uint64_t* idx64, uint32_t* act32);
unsigned stage_slots(uint64_t n, const uint64_t* idx, uint64_t capacity, uint32_t arg0, uint32_t arg_step, uint64_t* ops);
}  // namespace amsweep_host

namespace {
// Reason of the last failed am_sweep_create, process-wide: a cgo caller may be moved to
// another OS thread between the failing call and am_last_error_detail(NULL).
std::mutex g_create_mu;
std::string g_create_error;
void set_create_error(const std::string& s) {
  std::lock_guard<std::mutex> lk(g_create_mu);
  g_create_error = s;
}

struct PinnedBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes, unsigned flags = cudaHostAllocDefault) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 2 + 4096;
    cudaError_t e = cudaHostAlloc(&p, want, flags);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 2 + 4096;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// One of the two staging areas for controller events.  The pinned arrays are appended to
// under am_sweep::mu; the device twins receive them in chunks on the copy stream.
struct Staging {
  PinnedBuf ops, recs;   // an op = one 64-bit word: slot | arg << 32
  DevBuf d_ops, d_recs;
  size_t n_ops = 0, n_recs = 0;
  size_t flushed_ops = 0, flushed_recs = 0;  // already enqueued for copy to the device twins
  uint32_t n_state = 0, n_result = 0;
  // am_sweep_post_result calls that have reserved a range of the op arrays and are filling it
  // OUTSIDE the lock (the controller's workers post concurrently, hcc.go:170-188): while there are
  // any, the arrays may not move, nothing past `flushed_ops` is known complete, and the drain waits
  int writers = 0;
  size_t done_ops = 0;  // every op below this index is staged completely (== n_ops when writers == 0)
  std::vector<std::pair<size_t, size_t>> done_ranges;  // completed ranges above the prefix (other writers still below them)
  uint64_t hwm = 0;                          // highest upserted slot + 1
  cudaEvent_t copied = nullptr;              // the last copy out of the pinned arrays
  bool copy_pending = false;
  cudaEvent_t drained = nullptr;             // the last kernel that read the device twins
  bool drain_pending = false;
};

// One of the two buffer sets a tick writes (by tick parity): a consumer of tick k — the
// list rebuild, or the NVLink exchange on another stream — overlaps the sweep of tick k+1.
struct TickSet {
  TickOut out{};
  unsigned long long* acc = nullptr;
  cudaEvent_t consumed = nullptr;
  bool consumed_pending = false;
};

constexpr size_t kFlushOps = 32768;   // staged ops per early host-to-device chunk
constexpr size_t kFlushRecs = 8192;   // staged upsert records per early chunk
}  // namespace

struct am_sweep {
  int device = 0;
  uint64_t capacity = 0, cap_padded = 0, shard_base = 0;
  uint64_t n_records = 0;  // high-water mark
  DevCols cols{};
  TickSet set[2];
  uint32_t parity = 0;
  int last_shard_parity = -1;
  uint32_t* due_idx[2] = {nullptr, nullptr};   // HBM list ring (streaming mode)
  uint8_t* due_action[2] = {nullptr, nullptr};
  // host-visible list of the last host tick: mapped pinned memory written by expand_kernel
  PinnedBuf host_out;
  uint64_t host_out_entries = 0;  // capacity in entries
  uint64_t host_n = 0;            // entries of the last host tick
  am_tick_stats_t* h_stats = nullptr;  // pinned + mapped
  am_tick_stats_t* d_stats_mapped = nullptr;
  cudaStream_t stream = nullptr;   // the handle's own stream
  cudaStream_t cstream = nullptr;  // staging copies
  cudaStream_t last_stream = nullptr;  // where the handle's last device operation was issued
  bool has_last = false;
  cudaEvent_t ev_last = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaEvent_t evp[3] = {nullptr, nullptr, nullptr};  // profiling: before sweep, after sweep, after publish
  bool profiling = false, profiled = false;
  std::mutex mu;  // guards the staging areas
  std::condition_variable cv;  // a staging area's `writers` dropped to zero
  std::atomic_flag ticking = ATOMIC_FLAG_INIT;
  Staging stage[2];
  int cur = 0;                // the staging area callers append to
  uint32_t* marks = nullptr;  // [3 * cap_padded] per-slot {latest state op, latest phase, latest remedy phase}
  PinnedBuf pin_in;
  DevBuf dev_in;
  // named time zones: one UTC offset per registered zone (tz.h) on the device, refreshed when the
  // registry grows or a tick leaves the window [tz_lo, tz_hi) in which no zone changes its offset
  uint64_t tz_version = ~0ull;
  uint32_t tz_n = 0;  // zones + 1; 0 or 1 = nothing registered
  int64_t tz_lo = 0, tz_hi = 0;
  bool tz_aligned = true;  // every offset a whole number of minutes
  DevBuf tz_off, tz_table;
  PinnedBuf tz_pin;
  cudaEvent_t tz_copied = nullptr;
  bool tz_copy_pending = false;
  std::string last_error;
  uint64_t launches = 0;
  double last_ms = -1.0;
  uint64_t seed = 0;
  bool early_results = true;  // AMSWEEP_EARLY_RESULTS=0: every posted result is applied inside the sweep
  Staging* pend_clear = nullptr;  // a host tick's drain leaves clear_marks_kernel for after the tick's kernels
  size_t pend_clear_n = 0;
  // am_sweep_run_ticks_view(AM_SWEEP_BLOCKED): one TickOut per tick of a block, allocated on first use
  TickRing ring{};
  uint32_t ring_slots = 0;
  uint32_t* ring_totals = nullptr;  // [kMaxBlockTicks] pinned + mapped: each slot's emitted count
};

namespace {

#define AM_CUDA(h, expr)                                                              \
  do {                                                                                \
    cudaError_t _e = (expr);                                                          \
    if (_e != cudaSuccess) {                                                          \
      char _b[512];                                                                   \
      snprintf(_b, sizeof _b, "%s -> %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      if (h) (h)->last_error = _b; else set_create_error(_b);                         \
      return _e == cudaErrorMemoryAllocation ? AM_E_NOMEM : AM_E_DEVICE;              \
    }                                                                                 \
  } while (0)

// Column k (0..15, AM_RECORD_COLUMNS order) of a column set, untyped; its element size is kColumns[k].elem.
template <typename Cols>  // am_record_cols_t or const am_record_cols_t
auto& column(Cols& c, int k) {
  using Ptr = typename std::conditional<std::is_const<Cols>::value, void* const, void*>::type;
  return reinterpret_cast<Ptr*>(&c)[k];
}

struct TickGuard {
  am_sweep* h;
  bool ok;
  explicit TickGuard(am_sweep* hh) : h(hh), ok(!hh->ticking.test_and_set(std::memory_order_acquire)) {}
  ~TickGuard() { if (ok) h->ticking.clear(std::memory_order_release); }
};

// Every device operation of a handle is ordered after the previous one.  They normally
// share a stream; when the stream changes (am_sweep_tick_device on a caller stream, then a
// read on the handle's own, ...) the new stream waits for an event recorded on the old one.
int order_on(am_sweep* h, cudaStream_t s) {
  if (h->has_last && h->last_stream != s) {
    AM_CUDA(h, cudaEventRecord(h->ev_last, h->last_stream));
    AM_CUDA(h, cudaStreamWaitEvent(s, h->ev_last, 0));
  }
  h->last_stream = s;
  h->has_last = true;
  return AM_OK;
}

// Grow a pinned staging array (called under h->mu); keeps the contents.  Copies out of the
// old array may still be in flight on the copy stream: wait for them before it is freed.
cudaError_t grow_pinned(am_sweep* h, PinnedBuf& b, size_t used_bytes, size_t want_bytes, bool copies_in_flight) {
  if (want_bytes <= b.cap) return cudaSuccess;
  void* np = nullptr;
  size_t ncap = want_bytes * 2 + 65536;
  cudaError_t e = cudaHostAlloc(&np, ncap, cudaHostAllocDefault);
  if (e != cudaSuccess) return e;
  if (used_bytes) memcpy(np, b.p, used_bytes);
  if (b.p) {
    if (copies_in_flight) cudaStreamSynchronize(h->cstream);
    cudaFreeHost(b.p);
  }
  b.p = np;
  b.cap = ncap;
  return cudaSuccess;
}

// Enqueue the not-yet-copied part of a staging area on the copy stream, if the device
// twins are large enough (they are grown at drain time only).  Called under h->mu by the
// posting threads (chunk threshold) and by the drain (everything).
cudaError_t flush_staging(am_sweep* h, Staging& st, bool all, size_t upto = SIZE_MAX) {
  // ops: everything below `upto` is complete.  Without an explicit bound that is all of them, or, while
  // posting calls are still filling reserved ranges, the completed prefix.
  if (upto == SIZE_MAX) upto = st.writers ? st.done_ops : st.n_ops;
  const size_t pend = upto > st.flushed_ops ? upto - st.flushed_ops : 0;
  if (pend && (all || pend >= kFlushOps) && st.d_ops.cap >= upto * 8) {
    cudaError_t e = cudaMemcpyAsync((uint64_t*)st.d_ops.p + st.flushed_ops, (const uint64_t*)st.ops.p + st.flushed_ops,
                                    pend * 8, cudaMemcpyHostToDevice, h->cstream);
    if (e != cudaSuccess) return e;
    st.flushed_ops = upto;
    st.copy_pending = true;
  }
  const size_t pr = st.n_recs - st.flushed_recs;
  if (pr && (all || pr >= kFlushRecs) && st.d_recs.cap >= st.n_recs * sizeof(am_record_t)) {
    cudaError_t e = cudaMemcpyAsync((am_record_t*)st.d_recs.p + st.flushed_recs,
                                    (const am_record_t*)st.recs.p + st.flushed_recs, pr * sizeof(am_record_t),
                                    cudaMemcpyHostToDevice, h->cstream);
    if (e != cudaSuccess) return e;
    st.flushed_recs = st.n_recs;
    st.copy_pending = true;
  }
  return cudaSuccess;
}

// A reserved range [a, b) of the op arrays is completely staged (called under h->mu): extend the
// completed prefix, absorbing ranges that finished earlier above it.
void complete_range(Staging& st, size_t a, size_t b) {
  if (a != st.done_ops) { st.done_ranges.emplace_back(a, b); return; }
  st.done_ops = b;
  for (bool again = true; again && !st.done_ranges.empty();) {
    again = false;
    for (size_t k = 0; k < st.done_ranges.size(); ++k)
      if (st.done_ranges[k].first == st.done_ops) {
        st.done_ops = st.done_ranges[k].second;
        st.done_ranges[k] = st.done_ranges.back();
        st.done_ranges.pop_back();
        again = true;
        break;
      }
  }
}

// Make room for `n` more staged ops (and `nrec` more upsert records) in the current staging area;
// called with h->mu held through `lk`.  The pinned arrays move when they grow: calls that are
// still filling a reserved range outside the lock are waited for first.
int reserve_staging(am_sweep* h, std::unique_lock<std::mutex>& lk, size_t n, size_t nrec, Staging** out) {
  for (;;) {
    Staging& st = h->stage[h->cur];
    if (st.n_ops + n > 0x3FFFFFF0ull || st.n_recs + nrec > 0x3FFFFFF0ull) return AM_E_NOSPACE;
    const size_t want = (st.n_ops + n) * 8, want_r = (st.n_recs + nrec) * sizeof(am_record_t);
    if (st.ops.cap < want || (nrec && st.recs.cap < want_r)) {
      if (st.writers) { h->cv.wait(lk); continue; }  // (the drain may have swapped the areas meanwhile)
      AM_CUDA(h, cudaSetDevice(h->device));
      const bool inflight = st.flushed_ops || st.flushed_recs || st.copy_pending;
      AM_CUDA(h, grow_pinned(h, st.ops, st.n_ops * 8, want, inflight));
      if (nrec) AM_CUDA(h, grow_pinned(h, st.recs, st.n_recs * sizeof(am_record_t), want_r, inflight));
    }
    *out = &st;
    return AM_OK;
  }
}

// Apply staged upserts / removes / results on stream `s` (called with the tick guard held).
// The staging lock is held only for the buffer swap.
// clear_marks_kernel of a drain that deferred it (host ticks: the sweep does not touch the marks, and the
// host waits for an event recorded BEFORE this launch — 15 us off the tick's latency)
int finish_deferred_clear(am_sweep* h, cudaStream_t s) {
  Staging* st = h->pend_clear;
  if (!st) return AM_OK;
  h->pend_clear = nullptr;
  const size_t n = h->pend_clear_n;
  const unsigned B = 256, G = (unsigned)((n + B - 1) / B);
  AM_LAUNCH_PDL(clear_marks_kernel, G, B, s, h->marks, (const uint2*)st->d_ops.p, (uint32_t)n);
  h->launches++;
  AM_CUDA(h, cudaGetLastError());
  AM_CUDA(h, cudaEventRecord(st->drained, s));
  st->drain_pending = true;
  return AM_OK;
}

int drain_staged(am_sweep* h, cudaStream_t s, const int64_t* tick_T = nullptr, bool defer_clear = false) {
  Staging* st;
  {
    std::unique_lock<std::mutex> lk(h->mu);
    st = &h->stage[h->cur];
    h->cv.wait(lk, [&] { return st->writers == 0; });  // posting calls still filling their ranges
    if (st->n_ops == 0) return AM_OK;
    // callers are about to append to the other area: its previous copies must have left it
    Staging& nx = h->stage[h->cur ^ 1];
    if (nx.copy_pending) {
      AM_CUDA(h, cudaEventSynchronize(nx.copied));
      nx.copy_pending = false;
    }
    // ... and the kernels of its previous drain must be done with its device twins before
    // the chunked copies of the coming events overwrite them (asynchronous ticks only)
    if (nx.drain_pending) {
      AM_CUDA(h, cudaStreamWaitEvent(h->cstream, nx.drained, 0));
      nx.drain_pending = false;
    }
    h->cur ^= 1;
  }
  // from here on `st` is private to this (single) ticking thread
  const size_t n = st->n_ops, nrec = st->n_recs;
  if (st->hwm > h->n_records) h->n_records = st->hwm;  // every upserted slot extends the swept range
  if (st->d_ops.cap < n * 8 || st->d_recs.cap < nrec * sizeof(am_record_t)) {
    // grow the device twins (frees synchronise) and copy everything again
    AM_CUDA(h, cudaStreamSynchronize(h->cstream));
    AM_CUDA(h, st->d_ops.reserve(n * 8));
    AM_CUDA(h, st->d_recs.reserve(nrec * sizeof(am_record_t)));
    st->flushed_ops = st->flushed_recs = 0;
  }
  AM_CUDA(h, flush_staging(h, *st, true));
  AM_CUDA(h, cudaEventRecord(st->copied, h->cstream));
  st->copy_pending = true;
  AM_CUDA(h, cudaStreamWaitEvent(s, st->copied, 0));
  const uint2* d_ops = (const uint2*)st->d_ops.p;
  const am_record_t* d_recs = (const am_record_t*)st->d_recs.p;
  const unsigned B = 256, G = (unsigned)((n + B - 1) / B);
  AM_LAUNCH(mark_ops_kernel, G, B, s, h->marks, d_ops, (uint32_t)n);
  h->launches++;
  if (st->n_state) {
    AM_LAUNCH_PDL(apply_state_ops_kernel, G, B, s, h->cols, h->marks, d_ops, d_recs, (uint32_t)n);
    h->launches++;
  }
  // A tick's drain applies sparse results right away (apply_results_now_kernel: no second memory round trip
  // in the sweep, and the posted bits never pass through the flags as a separate step); a read's drain, or a
  // batch touching more than an eighth of the records, leaves them pending in the flags for the sweep's own
  // streaming path (apply_result_ops_kernel).
  if (tick_T && st->n_result && h->early_results && (uint64_t)st->n_result * 8 <= h->n_records) {
    TickSet& ts = h->set[h->parity];  // the buffer set of the tick being prepared
    if (ts.consumed_pending) {        // (its statistics may still be read by an exchange on another stream)
      AM_CUDA(h, cudaStreamWaitEvent(s, ts.consumed, 0));
      ts.consumed_pending = false;
    }
    AM_LAUNCH_PDL(apply_results_now_kernel, G, B, s, h->cols, h->marks, d_ops, (uint32_t)n, *tick_T, ts.acc);
    h->launches++;
  } else if (st->n_result) {
    AM_LAUNCH_PDL(apply_result_ops_kernel, G, B, s, h->cols.flags, h->marks, d_ops, (uint32_t)n);
    h->launches++;
  }
  if (defer_clear) {  // (the caller runs finish_deferred_clear on the same stream before anything else touches the handle)
    h->pend_clear = st;
    h->pend_clear_n = n;
    AM_CUDA(h, cudaGetLastError());
  } else {
    AM_LAUNCH_PDL(clear_marks_kernel, G, B, s, h->marks, d_ops, (uint32_t)n);
    h->launches++;
    AM_CUDA(h, cudaGetLastError());
    AM_CUDA(h, cudaEventRecord(st->drained, s));
    st->drain_pending = true;
  }
  st->n_ops = st->n_recs = st->flushed_ops = st->flushed_recs = 0;
  st->done_ops = 0;
  st->done_ranges.clear();
  st->n_state = st->n_result = 0;
  st->hwm = 0;
  return AM_OK;
}

// Where the rebuilt list goes: HBM (device-resident pipelines), mapped host memory (host
// ticks) or nowhere (am_sweep_tick_shard: the exchange rebuilds the global list).
struct ListOut {
  void* idx = nullptr;      // u32 local indices
  uint8_t* act = nullptr;
  uint64_t cap = 0;
  uint32_t* count = nullptr;          // min(n_emitted, cap), device memory, may be NULL
  am_tick_stats_t* stats = nullptr;   // device or mapped host memory, may be NULL
  bool expand = true;
};

// The zones' UTC offsets at T on the device.  Per tick: one uncontended lock for the registry version
// and two compares; the offsets themselves are recomputed (tz_eval.h, host) and copied — a few hundred
// bytes — only when a zone was registered or T left the window in which no zone changes its offset.
int refresh_zones(am_sweep* h, int64_t T, cudaStream_t s) {
  if (amsweep_tz::snapshot(nullptr, nullptr, nullptr) == h->tz_version && T >= h->tz_lo && T < h->tz_hi) return AM_OK;
  std::vector<int32_t> offs;
  int64_t until = 0;
  bool aligned = true;
  const uint64_t v = amsweep_tz::offsets_at(T, &offs, &until, &aligned);
  h->tz_version = v;
  h->tz_n = (uint32_t)offs.size();
  h->tz_lo = T;
  h->tz_hi = until;
  h->tz_aligned = aligned;
  if (h->tz_n <= 1) {  // nothing registered: every T is fine until the registry grows
    h->tz_lo = INT64_MIN;
    h->tz_hi = INT64_MAX;
    return AM_OK;
  }
  const size_t bytes = (amsweep_tz::kMaxZones + 1) * sizeof(int32_t);
  AM_CUDA(h, h->tz_off.reserve(bytes));
  AM_CUDA(h, h->tz_table.reserve((amsweep_tz::kMaxZones + 1) * sizeof(TickWords)));
  AM_CUDA(h, h->tz_pin.reserve(bytes));
  if (!h->tz_copied) AM_CUDA(h, cudaEventCreateWithFlags(&h->tz_copied, cudaEventDisableTiming));
  if (h->tz_copy_pending) AM_CUDA(h, cudaEventSynchronize(h->tz_copied));  // the previous copy has left the pinned array
  memcpy(h->tz_pin.p, offs.data(), offs.size() * sizeof(int32_t));
  // (stream-ordered after every earlier tick of the handle: none of them still reads the old offsets)
  AM_CUDA(h, cudaMemcpyAsync(h->tz_off.p, h->tz_pin.p, offs.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  AM_CUDA(h, cudaEventRecord(h->tz_copied, s));
  h->tz_copy_pending = true;
  return AM_OK;
}

int launch_tick(am_sweep* h, int64_t T, uint32_t mode, const ListOut& o, cudaStream_t s) {
  if (h->n_records == 0) {
    // nothing to sweep: publish zeros without a launch
    if (o.stats) AM_CUDA(h, cudaMemsetAsync(o.stats, 0, sizeof(am_tick_stats_t), s));
    if (o.count) AM_CUDA(h, cudaMemsetAsync(o.count, 0, 4, s));
    return AM_OK;
  }
  TickSet& ts = h->set[h->parity];
  if (ts.consumed_pending) {  // an exchange on another stream may still be reading this buffer set
    AM_CUDA(h, cudaStreamWaitEvent(s, ts.consumed, 0));
    ts.consumed_pending = false;
  }
  SweepParams p{};
  p.c = h->cols;
  p.n_records = h->n_records;
  p.shard_base = h->shard_base;
  p.seed = h->seed;
  p.T = T;
  p.words = tick_words_from_unix(T);
  p.n_tiles = tiles_of(h->n_records);
  p.mode = mode;
  p.out = ts.out;
  p.acc = ts.acc;
  {  // named time zones: one UTC offset per zone, valid at T
    const int rc = refresh_zones(h, T, s);
    if (rc != AM_OK) return rc;
  }
  // off the minute no 5-field schedule can fire: the mask columns are not read.  (A zone whose UTC
  // offset is not a whole number of minutes — historical local mean times — moves the local minute
  // boundary: every tick then reads the masks.)
  int64_t sec_of_min = T % 60;
  if (sec_of_min < 0) sec_of_min += 60;
  const bool masks = sec_of_min == 0 || (mode & AM_SWEEP_FULL_SCAN) || (h->tz_n > 1 && !h->tz_aligned);
  if (masks && h->tz_n > 1) {  // the tick's wall clock per zone, from the cached offsets
    AM_LAUNCH_PDL(tz_words_kernel, (h->tz_n + 63) / 64, 64, s, (const int32_t*)h->tz_off.p, (TickWords*)h->tz_table.p, T,
                  h->tz_n);
    h->launches++;
    p.tz_table = (const TickWords*)h->tz_table.p;
  }
  if (h->profiling) AM_CUDA(h, cudaEventRecord(h->evp[0], s));
  const bool closed = (mode & AM_SWEEP_CLOSED_LOOP) != 0;
  if (o.expand) {  // single-stream tick: the sweep's launch hides behind its predecessor (the previous tick's publish, the drain)
    if (closed && masks) AM_LAUNCH_PDL(AM_SWEEP_KERNEL(true, true), p.n_tiles, kBlock, s, p);
    else if (closed) AM_LAUNCH_PDL(AM_SWEEP_KERNEL(true, false), p.n_tiles, kBlock, s, p);
    else if (masks) AM_LAUNCH_PDL(AM_SWEEP_KERNEL(false, true), p.n_tiles, kBlock, s, p);
    else AM_LAUNCH_PDL(AM_SWEEP_KERNEL(false, false), p.n_tiles, kBlock, s, p);
  } else {
    // am_sweep_tick_shard: a plain launch.  (An early-launched sweep could park its CTAs on every SM ahead of the
    // previous tick's exchange on the other stream; measured at two GPUs it made no difference — 126 us per step
    // either way — so the simpler form stays.)
    if (closed && masks) AM_LAUNCH(AM_SWEEP_KERNEL(true, true), p.n_tiles, kBlock, s, p);
    else if (closed) AM_LAUNCH(AM_SWEEP_KERNEL(true, false), p.n_tiles, kBlock, s, p);
    else if (masks) AM_LAUNCH(AM_SWEEP_KERNEL(false, true), p.n_tiles, kBlock, s, p);
    else AM_LAUNCH(AM_SWEEP_KERNEL(false, false), p.n_tiles, kBlock, s, p);
  }
  if (h->profiling) AM_CUDA(h, cudaEventRecord(h->evp[1], s));
  ScanParams sc{};
  sc.group_count = ts.out.group_count;
  sc.group_prefix = ts.out.group_prefix;
  sc.acc = ts.acc;
  sc.out_count = o.count;
  sc.n_groups = groups_of(h->n_records);
  sc.cap = (uint32_t)(o.cap > 0xFFFFFFFFull ? 0xFFFFFFFFull : o.cap);
  AM_LAUNCH_PDL(scan_groups_kernel, 1, 1024, s, sc);
  h->launches += 2;
  if (o.expand) {
    ExpandParams e{};
    e.src[0].bitmap = ts.out.bitmap;
    e.src[0].group_prefix = ts.out.group_prefix;
    e.src[0].tile_exc = ts.out.tile_exc;
    e.src[0].exc_seg = ts.out.exc_seg;
    e.src[0].base = 0;  // local indices
    e.src[0].n_groups = sc.n_groups;
    e.src[0].n_tiles = p.n_tiles;
    e.out_idx = o.idx;
    e.out_act = o.act;
    e.acc = ts.acc;
    e.stats_base = h->shard_base;
    e.cap = o.idx ? o.cap : 0;
    e.world = 1;
    e.stats_rank = 0;
    e.idx_bytes = 4;
    AM_LAUNCH_PDL(expand_kernel, dim3(sc.n_groups, 1), kExpandThreads, s, e);
    AM_LAUNCH_PDL(publish_kernel, 1, 32, s, ts.acc, o.stats, h->n_records);
    h->launches += 2;
  }
  if (h->profiling) { AM_CUDA(h, cudaEventRecord(h->evp[2], s)); h->profiled = true; }
  h->parity ^= 1;
  AM_CUDA(h, cudaGetLastError());
  return AM_OK;
}

// mapped pinned memory for the list of a host tick: u32 indices, then u8 actions
int reserve_host_out(am_sweep* h, uint64_t entries) {
  if (entries <= h->host_out_entries) return AM_OK;
  const uint64_t want = (entries + entries / 4 + 4095) / 4096 * 4096;
  AM_CUDA(h, cudaStreamSynchronize(h->stream));
  AM_CUDA(h, h->host_out.reserve(want * 5, cudaHostAllocMapped));
  h->host_out_entries = want;
  return AM_OK;
}

// Grow the mapped list buffer to hold `entries`, keeping its first `used` entries (a run of ticks
// appends list after list).  The buffer moves: nothing on the device may still write into it.
int grow_host_out(am_sweep* h, uint64_t entries, uint64_t used) {
  if (entries <= h->host_out_entries) return AM_OK;
  const uint64_t want = (entries + entries / 4 + 4095) / 4096 * 4096;
  AM_CUDA(h, cudaStreamSynchronize(h->stream));
  void* np = nullptr;
  AM_CUDA(h, cudaHostAlloc(&np, want * 5, cudaHostAllocMapped));
  if (used) {
    memcpy(np, h->host_out.p, used * 4);
    memcpy((uint8_t*)np + want * 4, (const uint8_t*)h->host_out.p + h->host_out_entries * 4, used);
  }
  h->host_out.release();
  h->host_out.p = np;
  h->host_out.cap = want * 5;
  h->host_out_entries = want;
  return AM_OK;
}

void release_ring(am_sweep* h) {
  TickOut& b = h->ring.base;
  for (uint32_t* p : {b.bitmap, b.group_count, b.group_prefix, b.tile_exc, b.exc_seg}) if (p) cudaFree(p);
  b = TickOut{};
  h->ring_slots = 0;
}

// The tick ring, `slots` ticks deep, at the strides of the handle's capacity (amsweep.h has the size).
int reserve_ring(am_sweep* h, uint32_t slots) {
  if (slots <= h->ring_slots) return AM_OK;
  AM_CUDA(h, cudaStreamSynchronize(h->stream));
  release_ring(h);
  TickRing& r = h->ring;
  r.tiles = h->cap_padded / kTile;
  r.groups = (r.tiles + kGroupTiles - 1) / kGroupTiles;
  r.bitmap_words = r.groups * kGroupWords;
  r.exc_words = r.tiles * kTile;
  const int rc = [&]() -> int {
    if (!h->ring_totals) AM_CUDA(h, cudaHostAlloc((void**)&h->ring_totals, kMaxBlockTicks * 4, cudaHostAllocMapped));
    const uint64_t words[5] = {r.bitmap_words, r.groups, r.groups + 1, r.tiles, r.exc_words};
    uint32_t** arrays[5] = {&r.base.bitmap, &r.base.group_count, &r.base.group_prefix, &r.base.tile_exc, &r.base.exc_seg};
    for (int k = 0; k < 5; ++k) {  // zero: bitmap words past the last CTA are never written; group counts start at 0
      AM_CUDA(h, cudaMalloc((void**)arrays[k], slots * words[k] * 4));
      AM_CUDA(h, cudaMemsetAsync(*arrays[k], 0, slots * words[k] * 4, h->stream));
    }
    return AM_OK;
  }();
  if (rc != AM_OK) {
    release_ring(h);
    return rc;
  }
  h->ring_slots = slots;
  return AM_OK;
}

// am_sweep_run_ticks_view without AM_SWEEP_BLOCKED: one tick after the other, each list expanded into
// the list buffer behind the previous one, one synchronisation per tick.  start[k]: tick k's first entry.
int run_lists_ticks(am_sweep* h, int64_t unix_sec0, uint64_t n_ticks, uint32_t mode, am_tick_stats_t* stats,
                    uint64_t* start) {
  uint64_t used = 0;
  for (uint64_t k = 0; k < n_ticks; ++k) {
    int rc = grow_host_out(h, used + h->n_records, used);
    if (rc != AM_OK) return rc;
    ListOut o;
    if (h->host_out_entries) {
      void* d = nullptr;
      AM_CUDA(h, cudaHostGetDevicePointer(&d, h->host_out.p, 0));
      o.idx = (uint32_t*)d + used;
      o.act = (uint8_t*)d + h->host_out_entries * 4 + used;
      o.cap = h->host_out_entries - used;
    }
    o.stats = h->d_stats_mapped;
    rc = launch_tick(h, unix_sec0 + (int64_t)k, mode, o, h->stream);
    if (rc != AM_OK) return rc;
    AM_CUDA(h, cudaStreamSynchronize(h->stream));
    stats[k] = *h->h_stats;
    stats[k].n_records = h->n_records;
    start[k] = used;
    used = (used + stats[k].n_emitted + 3) & ~3ull;  // expand_kernel writes 16-B aligned quads of indices
  }
  return AM_OK;
}

// am_sweep_run_ticks_view with AM_SWEEP_BLOCKED: per block of K ticks, sweep_block_kernel<., true> fills K
// slots of the tick ring, ring_scan_kernel turns them into offsets and totals, the host waits once and
// sizes the list buffer, and expand_kernel rebuilds the K lists, up to kMaxWorld ticks per launch.
// The block length (AMSWEEP_BLOCK_TICKS), the cut at zone-offset changes and the BlockParams are those of the
// block loop of am_sweep_run_ticks: a change to one belongs in the other.
int run_lists_blocked(am_sweep* h, int64_t unix_sec0, uint64_t n_ticks, uint32_t mode, am_tick_stats_t* stats,
                      uint64_t* start) {
  uint64_t block_ticks = kDefaultBlockTicks;
  if (const char* e = getenv("AMSWEEP_BLOCK_TICKS")) { long v = atol(e); if (v >= 1 && v <= kMaxBlockTicks) block_ticks = (uint64_t)v; }
  int rc = reserve_ring(h, (uint32_t)(block_ticks < n_ticks ? block_ticks : n_ticks));
  if (rc != AM_OK) return rc;
  am_tick_stats_t* d_stats = nullptr;
  AM_CUDA(h, cudaMalloc((void**)&d_stats, n_ticks * sizeof(am_tick_stats_t)));
  struct FreeOnExit {
    void* p;
    ~FreeOnExit() { cudaFree(p); }
  } free_on_exit{d_stats};
  AM_CUDA(h, cudaMemsetAsync(d_stats, 0, n_ticks * sizeof(am_tick_stats_t), h->stream));
  uint32_t* d_totals = nullptr;
  AM_CUDA(h, cudaHostGetDevicePointer((void**)&d_totals, h->ring_totals, 0));
  const uint32_t n_groups = groups_of(h->n_records), n_tiles = tiles_of(h->n_records);
  const unsigned grid = (unsigned)((h->n_records + kBlockRecords - 1) / kBlockRecords);
  uint64_t used = 0;
  for (uint64_t k = 0; k < n_ticks;) {
    const int64_t T = unix_sec0 + (int64_t)k;
    rc = refresh_zones(h, T, h->stream);
    if (rc != AM_OK) return rc;
    uint64_t K = n_ticks - k < block_ticks ? n_ticks - k : block_ticks;
    if (h->tz_n > 1 && h->tz_hi < T + (int64_t)K) K = (uint64_t)(h->tz_hi - T);  // (tz_hi > T after the refresh)
    BlockParams b{};
    b.c = h->cols;
    b.n_records = h->n_records;
    b.shard_base = h->shard_base;
    b.seed = h->seed;
    b.T0 = T;
    b.K = (uint32_t)K;
    b.tz_off = h->tz_n > 1 ? (const int32_t*)h->tz_off.p : nullptr;
    b.stats = reinterpret_cast<unsigned long long*>(d_stats + k);
    b.ring = h->ring;
    // exception counts and group counts of the K slots start at zero whatever an earlier call left behind
    // (ring_scan_kernel re-arms the group counts, but a call that failed in between would not have run it)
    AM_CUDA(h, cudaMemsetAsync(h->ring.base.tile_exc, 0, K * h->ring.tiles * 4, h->stream));
    AM_CUDA(h, cudaMemsetAsync(h->ring.base.group_count, 0, K * h->ring.groups * 4, h->stream));
    if (mode & AM_SWEEP_CLOSED_LOOP) AM_LAUNCH(AM_BLOCK_KERNEL(true, true), grid, kBlockThreads, h->stream, b);
    else AM_LAUNCH(AM_BLOCK_KERNEL(false, true), grid, kBlockThreads, h->stream, b);
    AM_LAUNCH(ring_scan_kernel, (unsigned)K, kRingScanThreads, h->stream, h->ring, n_groups, d_totals);
    h->launches += 2;
    AM_CUDA(h, cudaGetLastError());
    AM_CUDA(h, cudaStreamSynchronize(h->stream));
    // the K lists back to back from `used`; each expand launch starts 16-B aligned
    uint64_t end = used;
    for (uint64_t j = 0; j < K; ++j) {
      if (j % kMaxWorld == 0) end = (end + 3) & ~3ull;
      start[k + j] = end;
      end += h->ring_totals[j];
    }
    rc = grow_host_out(h, end, used);
    if (rc != AM_OK) return rc;
    void* d = nullptr;
    if (h->host_out.p) AM_CUDA(h, cudaHostGetDevicePointer(&d, h->host_out.p, 0));
    for (uint64_t j0 = 0; j0 < K; j0 += kMaxWorld) {
      const uint64_t nj = K - j0 < (uint64_t)kMaxWorld ? K - j0 : (uint64_t)kMaxWorld;
      const uint64_t s0 = start[k + j0];
      ExpandParams e{};
      for (uint64_t j = 0; j < nj; ++j) {
        const uint64_t t = j0 + j;
        ExpandSrc& src = e.src[j];
        src.bitmap = h->ring.base.bitmap + t * h->ring.bitmap_words;
        src.group_prefix = h->ring.base.group_prefix + t * (h->ring.groups + 1);
        src.tile_exc = h->ring.base.tile_exc + t * h->ring.tiles;
        src.exc_seg = h->ring.base.exc_seg + t * h->ring.exc_words;
        src.base = 0;  // local indices
        src.n_groups = n_groups;
        src.n_tiles = n_tiles;
      }
      e.out_idx = d ? (void*)((uint32_t*)d + s0) : nullptr;
      e.out_act = d ? (uint8_t*)d + h->host_out_entries * 4 + s0 : nullptr;
      e.cap = d ? h->host_out_entries - s0 : 0;
      e.acc = nullptr;  // the statistics come from the block kernel
      e.world = (int)nj;
      e.stats_rank = 0;
      e.idx_bytes = 4;
      AM_LAUNCH(expand_kernel, dim3(n_groups, (unsigned)nj), kExpandThreads, h->stream, e);
      h->launches++;
    }
    AM_CUDA(h, cudaGetLastError());
    used = end;
    k += K;
  }
  AM_CUDA(h, cudaStreamSynchronize(h->stream));
  AM_CUDA(h, cudaMemcpy(stats, d_stats, n_ticks * sizeof(am_tick_stats_t), cudaMemcpyDeviceToHost));
  for (uint64_t k = 0; k < n_ticks; ++k) stats[k].n_records = h->n_records;
  return AM_OK;
}

// One host tick: drain, four kernels, one synchronisation; the list lands in h->host_out.
int host_tick(am_sweep* h, int64_t unix_sec, uint32_t mode, am_tick_stats_t* stats) {
  AM_CUDA(h, cudaSetDevice(h->device));
  int rc = order_on(h, h->stream);
  if (rc != AM_OK) return rc;
  rc = drain_staged(h, h->stream, &unix_sec, /*defer_clear=*/true);
  struct ClearOnExit {  // whatever happens below, the marks are cleared before the handle is used again
    am_sweep* h;
    ~ClearOnExit() { (void)finish_deferred_clear(h, h->stream); }
  } clear_on_exit{h};
  if (rc != AM_OK) return rc;
  rc = reserve_host_out(h, h->n_records);
  if (rc != AM_OK) return rc;
  ListOut o;
  if (h->host_out_entries) {
    void* d = nullptr;
    AM_CUDA(h, cudaHostGetDevicePointer(&d, h->host_out.p, 0));
    o.idx = d;
    o.act = (uint8_t*)d + h->host_out_entries * 4;
    o.cap = h->host_out_entries;
  }
  o.stats = h->d_stats_mapped;
  AM_CUDA(h, cudaEventRecord(h->ev0, h->stream));
  rc = launch_tick(h, unix_sec, mode, o, h->stream);
  if (rc != AM_OK) return rc;
  AM_CUDA(h, cudaEventRecord(h->ev1, h->stream));
  rc = finish_deferred_clear(h, h->stream);  // behind the event the host waits for
  if (rc != AM_OK) return rc;
  AM_CUDA(h, cudaEventSynchronize(h->ev1));
  float ms = 0;
  AM_CUDA(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->last_ms = ms;
  am_tick_stats_t st = *h->h_stats;
  st.n_records = h->n_records;
  h->host_n = st.n_emitted;
  if (stats) *stats = st;
  return AM_OK;
}

}  // namespace

namespace amsweep {
bool shard_last_tick(am_sweep* h, ShardTick* out) {
  if (!h || h->last_shard_parity < 0) return false;
  const TickSet& ts = h->set[h->last_shard_parity];
  out->out = ts.out;
  out->acc = ts.acc;
  out->shard_base = h->shard_base;
  out->n_records = h->n_records;
  out->n_groups = groups_of(h->n_records);
  out->n_tiles = tiles_of(h->n_records);
  out->parity = h->last_shard_parity;
  out->device = h->device;
  return true;
}
int shard_order_consumer(am_sweep* h, cudaStream_t s) {
  if (h->has_last && h->last_stream != s) {
    AM_CUDA(h, cudaEventRecord(h->ev_last, h->last_stream));
    AM_CUDA(h, cudaStreamWaitEvent(s, h->ev_last, 0));
  }
  return AM_OK;
}
int shard_launch_expand(am_sweep* h, const ExpandParams& e, uint32_t groups_x, uint32_t world_y, cudaStream_t s) {
  AM_LAUNCH(expand_kernel, dim3(groups_x, world_y), kExpandThreads, s, e);
  h->launches++;
  AM_CUDA(h, cudaGetLastError());
  return AM_OK;
}
int shard_launch_publish(am_sweep* h, unsigned long long* acc, am_tick_stats_t* out_stats, uint64_t n_records,
                         cudaStream_t s) {
  AM_LAUNCH(publish_kernel, 1, 32, s, acc, out_stats, n_records);
  h->launches++;
  AM_CUDA(h, cudaGetLastError());
  return AM_OK;
}
int shard_mark_consumed(am_sweep* h, int parity, cudaStream_t s) {
  TickSet& ts = h->set[parity & 1];
  AM_CUDA(h, cudaEventRecord(ts.consumed, s));
  ts.consumed_pending = true;
  return AM_OK;
}
}  // namespace amsweep

extern "C" {

const char* am_last_error_detail(const am_sweep_t* h) {
  if (h) return h->last_error.c_str();
  static thread_local std::string copy;  // stable storage for the returned pointer
  std::lock_guard<std::mutex> lk(g_create_mu);
  copy = g_create_error;
  return copy.c_str();
}

int am_sweep_create(am_sweep_t** out, int device_id, uint64_t capacity, uint64_t shard_base) {
  if (!out || capacity == 0 || capacity > 0xFFFFF000ull) return AM_E_INVAL;
  *out = nullptr;
  am_sweep* none = nullptr;
  int ndev = 0;
  AM_CUDA(none, cudaGetDeviceCount(&ndev));
  if (device_id < 0 || device_id >= ndev) {
    set_create_error("no such CUDA device");
    return AM_E_DEVICE;
  }
  AM_CUDA(none, cudaSetDevice(device_id));
  am_sweep* h = new (std::nothrow) am_sweep();
  if (!h) return AM_E_NOMEM;
  h->device = device_id;
  h->capacity = capacity;
  h->cap_padded = (capacity + kTile - 1) / kTile * kTile;
  h->shard_base = shard_base;
  if (const char* e = getenv("AMSWEEP_EARLY_RESULTS")) h->early_results = atoi(e) != 0;  // (A/B of the two result paths)
  int rc = [&]() -> int {
    AM_CUDA(h, cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    AM_CUDA(h, cudaStreamCreateWithFlags(&h->cstream, cudaStreamNonBlocking));
    AM_CUDA(h, cudaEventCreateWithFlags(&h->ev_last, cudaEventDisableTiming));
    AM_CUDA(h, cudaEventCreate(&h->ev0));
    AM_CUDA(h, cudaEventCreate(&h->ev1));
    for (int k = 0; k < 3; ++k) AM_CUDA(h, cudaEventCreate(&h->evp[k]));
    for (int b = 0; b < 2; ++b) {
      AM_CUDA(h, cudaEventCreateWithFlags(&h->stage[b].copied, cudaEventDisableTiming));
      AM_CUDA(h, cudaEventCreateWithFlags(&h->stage[b].drained, cudaEventDisableTiming));
      AM_CUDA(h, cudaEventCreateWithFlags(&h->set[b].consumed, cudaEventDisableTiming));
    }
    for (int k = 0; k < kNumCols; ++k) {
      void*& p = column(h->cols, k);
      AM_CUDA(h, cudaMalloc(&p, h->cap_padded * kColumns[k].elem));
      AM_CUDA(h, cudaMemsetAsync(p, 0, h->cap_padded * kColumns[k].elem, h->stream));
    }
    AM_LAUNCH(fill_u32_kernel, 1184, 256, h->stream, h->cols.flags, AM_F_TOMBSTONE, h->cap_padded);
    h->launches++;
    const size_t ntiles = h->cap_padded / kTile;
    const size_t ngroups = (ntiles + kGroupTiles - 1) / kGroupTiles;
    for (int b = 0; b < 2; ++b) {
      TickOut& t = h->set[b].out;
      // bitmap words past the last tile of the last group are never written: they stay zero
      AM_CUDA(h, cudaMalloc((void**)&t.bitmap, ngroups * kGroupWords * 4));
      AM_CUDA(h, cudaMemsetAsync(t.bitmap, 0, ngroups * kGroupWords * 4, h->stream));
      AM_CUDA(h, cudaMalloc((void**)&t.group_count, ngroups * 4));
      AM_CUDA(h, cudaMemsetAsync(t.group_count, 0, ngroups * 4, h->stream));
      AM_CUDA(h, cudaMalloc((void**)&t.group_prefix, (ngroups + 1) * 4));
      AM_CUDA(h, cudaMemsetAsync(t.group_prefix, 0, (ngroups + 1) * 4, h->stream));
      AM_CUDA(h, cudaMalloc((void**)&t.tile_exc, ntiles * 4));
      AM_CUDA(h, cudaMemsetAsync(t.tile_exc, 0, ntiles * 4, h->stream));
      AM_CUDA(h, cudaMalloc((void**)&t.exc_seg, h->cap_padded * 4));
      AM_CUDA(h, cudaMemsetAsync(t.exc_seg, 0, h->cap_padded * 4, h->stream));  // expand_kernel prefetches past the counts
      AM_CUDA(h, cudaMalloc((void**)&h->set[b].acc, kNumAcc * 8));
      AM_CUDA(h, cudaMemsetAsync(h->set[b].acc, 0, kNumAcc * 8, h->stream));
    }
    AM_CUDA(h, cudaMalloc((void**)&h->marks, h->cap_padded * 12));
    AM_CUDA(h, cudaMemsetAsync(h->marks, 0, h->cap_padded * 12, h->stream));
    for (int b = 0; b < 2; ++b) {
      AM_CUDA(h, cudaMalloc((void**)&h->due_idx[b], h->cap_padded * 4));
      AM_CUDA(h, cudaMalloc((void**)&h->due_action[b], h->cap_padded));
    }
    AM_CUDA(h, cudaHostAlloc((void**)&h->h_stats, sizeof(am_tick_stats_t), cudaHostAllocMapped));
    memset(h->h_stats, 0, sizeof(am_tick_stats_t));
    AM_CUDA(h, cudaHostGetDevicePointer((void**)&h->d_stats_mapped, h->h_stats, 0));
    AM_CUDA(h, cudaGetLastError());
    AM_CUDA(h, cudaStreamSynchronize(h->stream));
    return AM_OK;
  }();
  if (rc != AM_OK) {
    set_create_error(h->last_error);
    am_sweep_destroy(h);
    return rc;
  }
  *out = h;
  return AM_OK;
}

void am_sweep_destroy(am_sweep_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();  // ticks may have been issued on caller streams
  for (int k = 0; k < kNumCols; ++k) if (column(h->cols, k)) cudaFree(column(h->cols, k));
  for (int b = 0; b < 2; ++b) {
    TickOut& t = h->set[b].out;
    if (t.bitmap) cudaFree(t.bitmap);
    if (t.group_count) cudaFree(t.group_count);
    if (t.group_prefix) cudaFree(t.group_prefix);
    if (t.tile_exc) cudaFree(t.tile_exc);
    if (t.exc_seg) cudaFree(t.exc_seg);
    if (h->set[b].acc) cudaFree(h->set[b].acc);
    if (h->set[b].consumed) cudaEventDestroy(h->set[b].consumed);
    if (h->due_idx[b]) cudaFree(h->due_idx[b]);
    if (h->due_action[b]) cudaFree(h->due_action[b]);
    Staging& st = h->stage[b];
    st.ops.release(); st.recs.release();
    st.d_ops.release(); st.d_recs.release();
    if (st.copied) cudaEventDestroy(st.copied);
    if (st.drained) cudaEventDestroy(st.drained);
  }
  if (h->marks) cudaFree(h->marks);
  release_ring(h);
  if (h->ring_totals) cudaFreeHost(h->ring_totals);
  if (h->h_stats) cudaFreeHost(h->h_stats);
  h->host_out.release();
  h->pin_in.release(); h->dev_in.release();
  h->tz_off.release(); h->tz_table.release(); h->tz_pin.release();
  if (h->tz_copied) cudaEventDestroy(h->tz_copied);
  if (h->ev_last) cudaEventDestroy(h->ev_last);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  for (int k = 0; k < 3; ++k) if (h->evp[k]) cudaEventDestroy(h->evp[k]);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->cstream) cudaStreamDestroy(h->cstream);
  delete h;
}

uint64_t am_sweep_size(const am_sweep_t* h) { return h ? h->n_records : 0; }
uint64_t am_sweep_capacity(const am_sweep_t* h) { return h ? h->capacity : 0; }
int am_sweep_device(const am_sweep_t* h) { return h ? h->device : -1; }
double am_sweep_last_kernel_ms(const am_sweep_t* h) { return h ? h->last_ms : -1.0; }
uint64_t am_sweep_launch_count(const am_sweep_t* h) { return h ? h->launches : 0; }
void* am_sweep_column_ptr(am_sweep_t* h, int id) {
  return (h && id >= 0 && id < kNumCols) ? column(h->cols, id) : nullptr;
}
int am_sweep_set_profiling(am_sweep_t* h, int on) {
  if (!h) return AM_E_INVAL;
  h->profiling = on != 0;
  h->profiled = false;
  return AM_OK;
}
int am_sweep_last_profile(am_sweep_t* h, double* sweep_ms, double* rest_ms) {
  if (!h || !h->profiled) return AM_E_INVAL;
  AM_CUDA(h, cudaSetDevice(h->device));
  AM_CUDA(h, cudaEventSynchronize(h->evp[2]));
  float a = 0, b = 0;
  AM_CUDA(h, cudaEventElapsedTime(&a, h->evp[0], h->evp[1]));
  AM_CUDA(h, cudaEventElapsedTime(&b, h->evp[1], h->evp[2]));
  if (sweep_ms) *sweep_ms = a;
  if (rest_ms) *rest_ms = b;
  return AM_OK;
}
void* am_sweep_stream(am_sweep_t* h) { return h ? (void*)h->stream : nullptr; }
int am_sweep_set_seed(am_sweep_t* h, uint64_t seed) {
  if (!h) return AM_E_INVAL;
  h->seed = seed;
  return AM_OK;
}

int am_sweep_load_range(am_sweep_t* h, uint64_t first, uint64_t n, const am_record_cols_t* cols) {
  if (!h || !cols || first + n > h->capacity || first + n < first) return AM_E_INVAL;
  if (n == 0) return AM_OK;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  AM_CUDA(h, cudaSetDevice(h->device));
  int rc = order_on(h, h->stream);
  if (rc != AM_OK) return rc;
  for (int k = 0; k < kNumCols; ++k) {
    const size_t elem = kColumns[k].elem;
    char* dst = (char*)column(h->cols, k) + first * elem;
    const void* src = column(*cols, k);
    if (src) AM_CUDA(h, cudaMemcpyAsync(dst, src, n * elem, cudaMemcpyHostToDevice, h->stream));
    else AM_CUDA(h, cudaMemsetAsync(dst, 0, n * elem, h->stream));
  }
  AM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (first + n > h->n_records) h->n_records = first + n;
  return AM_OK;
}

int am_sweep_upsert(am_sweep_t* h, uint64_t n, const uint64_t* idx, const am_record_t* recs) {
  if (!h || (n && (!idx || !recs))) return AM_E_INVAL;
  if (n == 0) return AM_OK;
  std::unique_lock<std::mutex> lk(h->mu);
  Staging* stp = nullptr;
  if (int rc = reserve_staging(h, lk, n, n, &stp)) return rc;
  Staging& st = *stp;
  AM_CUDA(h, cudaSetDevice(h->device));
  // nothing is committed (counters unchanged) when a slot is out of range
  if (amsweep_host::stage_slots(n, idx, h->capacity, kOpUpsert | (uint32_t)st.n_recs, 1u, (uint64_t*)st.ops.p + st.n_ops))
    return AM_E_RANGE;
  am_record_t* dst = (am_record_t*)st.recs.p + st.n_recs;
  uint64_t hwm = st.hwm;
  for (uint64_t k = 0; k < n; ++k) {
    dst[k] = recs[k];
    dst[k].flags &= ~AM_F_TOMBSTONE;
    dst[k].reserved = 0;
    if (idx[k] + 1 > hwm) hwm = idx[k] + 1;
  }
  st.hwm = hwm;
  complete_range(st, st.n_ops, st.n_ops + n);
  st.n_ops += n; st.n_recs += n;
  st.n_state += (uint32_t)n;
  AM_CUDA(h, flush_staging(h, st, false));
  return AM_OK;
}

int am_sweep_remove(am_sweep_t* h, uint64_t n, const uint64_t* idx) {
  if (!h || (n && !idx)) return AM_E_INVAL;
  if (n == 0) return AM_OK;
  std::unique_lock<std::mutex> lk(h->mu);
  Staging* stp = nullptr;
  if (int rc = reserve_staging(h, lk, n, 0, &stp)) return rc;
  Staging& st = *stp;
  AM_CUDA(h, cudaSetDevice(h->device));
  if (amsweep_host::stage_slots(n, idx, h->capacity, kOpRemove, 0u, (uint64_t*)st.ops.p + st.n_ops)) return AM_E_RANGE;
  complete_range(st, st.n_ops, st.n_ops + n);
  st.n_ops += n;
  st.n_state += (uint32_t)n;
  AM_CUDA(h, flush_staging(h, st, false));
  return AM_OK;
}

int am_sweep_post_result(am_sweep_t* h, uint64_t n, const uint64_t* idx, const uint8_t* phase,
                         const uint8_t* remedy_phase) {
  if (!h || (n && (!idx || !phase))) return AM_E_INVAL;
  if (n == 0) return AM_OK;
  // Reserve a range of the op arrays under the lock, fill it outside: the controller's workers
  // (hcc.go:170-188) post concurrently and the per-entry pass is the cost of a post.  Per slot the
  // call order is the reservation order.
  std::unique_lock<std::mutex> lk(h->mu);
  Staging* stp = nullptr;
  if (int rc = reserve_staging(h, lk, n, 0, &stp)) return rc;
  Staging& st = *stp;
  const size_t a = st.n_ops;
  st.n_ops += n;
  st.n_result += (uint32_t)n;
  ++st.writers;  // the drain and any growth of the arrays now wait for this call
  uint64_t* const oo = (uint64_t*)st.ops.p + a;
  lk.unlock();
  // validate and stage in vectorised passes of one copy chunk each; a single large post hands every
  // finished chunk to the copy stream before staging the next (when no other call is staging).
  // phase -> flag bits: {none, Succeeded, Failed} -> {0, PENDING_OK, PENDING_FAIL}
  unsigned bad = 0;
  cudaError_t ce = cudaSuccess;
  for (uint64_t off = 0; off < n && !bad; off += kFlushOps) {
    const uint64_t m = n - off < kFlushOps ? n - off : kFlushOps;
    bad = amsweep_host::stage_results(m, idx + off, phase + off, remedy_phase ? remedy_phase + off : nullptr, h->capacity,
                                      kOpResult, oo + off);
    if (!bad && off + m < n) {
      lk.lock();
      if (st.writers == 1 && ce == cudaSuccess && cudaSetDevice(h->device) == cudaSuccess)
        ce = flush_staging(h, st, false, a + off + m);  // everything below is complete: this call is the only one staging
      lk.unlock();
    }
  }
  // nothing of a call with a bad entry takes effect: its range is already part of the sequence (later
  // calls may have reserved behind it), so it becomes ops that mark and set nothing
  if (bad)
    for (uint64_t k = 0; k < n; ++k) oo[k] = (uint64_t)kOpResult << 32;
  lk.lock();
  complete_range(st, a, a + n);
  // Hand the completed prefix to the copy stream, a chunk at a time, even while other calls are staging.
  // The range is claimed under the lock; the copy is issued outside it (a copy call under the lock
  // serialised every worker behind the CUDA API: 0.38 ms per post with ten workers), while this call still
  // counts as a writer — the drain, which records the "copied" event, waits for it.
  size_t c_lo = 0, c_hi = 0;
  if (ce == cudaSuccess && st.done_ops > st.flushed_ops && st.done_ops - st.flushed_ops >= kFlushOps && st.d_ops.cap >= st.done_ops * 8) {
    c_lo = st.flushed_ops;
    c_hi = st.done_ops;
    st.flushed_ops = c_hi;
    st.copy_pending = true;
  }
  const uint64_t* src = (const uint64_t*)st.ops.p;  // (the array cannot move while this call is a writer)
  lk.unlock();
  if (c_hi > c_lo && (ce = cudaSetDevice(h->device)) == cudaSuccess)
    ce = cudaMemcpyAsync((uint64_t*)st.d_ops.p + c_lo, src + c_lo, (c_hi - c_lo) * 8, cudaMemcpyHostToDevice, h->cstream);
  lk.lock();
  if (--st.writers == 0) h->cv.notify_all();
  if (bad) return (bad & 1u) ? AM_E_RANGE : AM_E_INVAL;
  AM_CUDA(h, ce);
  return AM_OK;
}

int am_sweep_tick(am_sweep_t* h, int64_t unix_sec, uint32_t mode, uint64_t* due_idx,
                  uint32_t* due_action, uint64_t cap, uint64_t* n_out, am_tick_stats_t* stats) {
  if (!h || (cap && (!due_idx || !due_action))) return AM_E_INVAL;
  if (unix_sec >= (1ll << 55) || unix_sec <= -(1ll << 55)) return AM_E_RANGE;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  int rc = host_tick(h, unix_sec, mode, stats);
  if (rc != AM_OK) return rc;
  const uint64_t n = h->host_n;
  if (n_out) *n_out = n;
  const uint64_t ncopy = n < cap ? n : cap;
  if (ncopy)  // widen into the caller's (Go) memory
    amsweep_host::widen_list(ncopy, h->shard_base, (const uint32_t*)h->host_out.p,
                             (const uint8_t*)h->host_out.p + h->host_out_entries * 4, due_idx, due_action);
  return n > cap ? AM_E_NOSPACE : AM_OK;
}

int am_sweep_tick_view(am_sweep_t* h, int64_t unix_sec, uint32_t mode, am_tick_view_t* view,
                       am_tick_stats_t* stats) {
  if (!h || !view) return AM_E_INVAL;
  if (unix_sec >= (1ll << 55) || unix_sec <= -(1ll << 55)) return AM_E_RANGE;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  int rc = host_tick(h, unix_sec, mode, stats);
  if (rc != AM_OK) return rc;
  view->idx_local = (const uint32_t*)h->host_out.p;
  view->action = h->host_out.p ? (const uint8_t*)h->host_out.p + h->host_out_entries * 4 : nullptr;
  view->n = h->host_n;
  view->shard_base = h->shard_base;
  return AM_OK;
}

int am_sweep_last_list(am_sweep_t* h, uint64_t offset, uint64_t* due_idx, uint32_t* due_action,
                       uint64_t cap, uint64_t* n_out) {
  if (!h || (cap && (!due_idx || !due_action))) return AM_E_INVAL;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  const uint64_t n = h->host_n;
  if (offset > n) return AM_E_RANGE;
  const uint64_t left = n - offset, ncopy = left < cap ? left : cap;
  if (n_out) *n_out = left;
  if (ncopy)
    amsweep_host::widen_list(ncopy, h->shard_base, (const uint32_t*)h->host_out.p + offset,
                             (const uint8_t*)h->host_out.p + h->host_out_entries * 4 + offset, due_idx, due_action);
  return left > cap ? AM_E_NOSPACE : AM_OK;
}

int am_sweep_tick_device(am_sweep_t* h, int64_t unix_sec, uint32_t mode, void* d_due_idx,
                         void* d_due_action, uint64_t cap, void* d_count, void* d_stats,
                         void* cuda_stream) {
  if (!h || (cap && (!d_due_idx || !d_due_action))) return AM_E_INVAL;
  if (unix_sec >= (1ll << 55) || unix_sec <= -(1ll << 55)) return AM_E_RANGE;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  AM_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;  // NULL == CUDA default stream
  int rc = order_on(h, s);
  if (rc != AM_OK) return rc;
  rc = drain_staged(h, s, &unix_sec);
  if (rc != AM_OK) return rc;
  ListOut o;
  o.idx = d_due_idx;
  o.act = (uint8_t*)d_due_action;
  o.cap = cap;
  o.count = (uint32_t*)d_count;
  o.stats = (am_tick_stats_t*)d_stats;
  return launch_tick(h, unix_sec, mode, o, s);
}

int am_sweep_tick_shard(am_sweep_t* h, int64_t unix_sec, uint32_t mode, void* cuda_stream) {
  if (!h) return AM_E_INVAL;
  if (unix_sec >= (1ll << 55) || unix_sec <= -(1ll << 55)) return AM_E_RANGE;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  AM_CUDA(h, cudaSetDevice(h->device));
  cudaStream_t s = (cudaStream_t)cuda_stream;
  int rc = order_on(h, s);
  if (rc != AM_OK) return rc;
  rc = drain_staged(h, s, &unix_sec);
  if (rc != AM_OK) return rc;
  if (h->n_records == 0) return AM_E_INVAL;  // an empty shard has nothing to exchange
  ListOut o;
  o.expand = false;
  const int parity = (int)h->parity;
  rc = launch_tick(h, unix_sec, mode, o, s);
  if (rc == AM_OK) h->last_shard_parity = parity;
  return rc;
}

int am_sweep_run_ticks(am_sweep_t* h, int64_t unix_sec0, uint64_t n_ticks, uint32_t mode,
                       uint64_t seed, am_tick_stats_t* stats_out) {
  if (!h || !stats_out) return AM_E_INVAL;
  if (n_ticks == 0) return AM_OK;
  if (n_ticks > (1ull << 24)) return AM_E_INVAL;
  if (unix_sec0 >= (1ll << 55) - (int64_t)n_ticks || unix_sec0 <= -(1ll << 55)) return AM_E_RANGE;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  AM_CUDA(h, cudaSetDevice(h->device));
  int rc = order_on(h, h->stream);
  if (rc != AM_OK) return rc;
  rc = drain_staged(h, h->stream, &unix_sec0);
  if (rc != AM_OK) return rc;
  h->seed = seed;
  am_tick_stats_t* d_stats = nullptr;
  AM_CUDA(h, cudaMalloc((void**)&d_stats, n_ticks * sizeof(am_tick_stats_t)));
  const bool blocked = (mode & AM_SWEEP_BLOCKED) != 0 && h->n_records != 0;
  if (blocked) {  // the block kernel accumulates into the rows
    if (cudaError_t e = cudaMemsetAsync(d_stats, 0, n_ticks * sizeof(am_tick_stats_t), h->stream); e != cudaSuccess) {
      h->last_error = cudaGetErrorString(e);
      cudaFree(d_stats);
      return AM_E_DEVICE;
    }
  }
  if (cudaError_t e = cudaEventRecord(h->ev0, h->stream); e != cudaSuccess) {
    h->last_error = cudaGetErrorString(e);
    rc = AM_E_DEVICE;
  }
  // (run_lists_blocked repeats this block loop for am_sweep_run_ticks_view: a change here belongs there too.)
  // Temporal blocking (sweep_block.cuh): up to kMaxBlockTicks ticks per pass over the columns.  A block
  // never spans an instant at which a registered zone changes its UTC offset (the kernel holds one
  // offset per zone for the whole block).
  uint64_t block_ticks = kDefaultBlockTicks;
  if (const char* e = getenv("AMSWEEP_BLOCK_TICKS")) { long v = atol(e); if (v >= 1 && v <= kMaxBlockTicks) block_ticks = (uint64_t)v; }
  for (uint64_t k = 0; blocked && k < n_ticks && rc == AM_OK;) {
    const int64_t T = unix_sec0 + (int64_t)k;
    rc = refresh_zones(h, T, h->stream);
    if (rc != AM_OK) break;
    uint64_t K = n_ticks - k < block_ticks ? n_ticks - k : block_ticks;
    if (h->tz_n > 1 && h->tz_hi < T + (int64_t)K) K = (uint64_t)(h->tz_hi - T);  // (tz_hi > T after the refresh)
    BlockParams b{};
    b.c = h->cols;
    b.n_records = h->n_records;
    b.shard_base = h->shard_base;
    b.seed = h->seed;
    b.T0 = T;
    b.K = (uint32_t)K;
    b.tz_off = h->tz_n > 1 ? (const int32_t*)h->tz_off.p : nullptr;
    b.stats = reinterpret_cast<unsigned long long*>(d_stats + k);
    const unsigned grid = (unsigned)((h->n_records + kBlockRecords - 1) / kBlockRecords);
    if (mode & AM_SWEEP_CLOSED_LOOP) AM_LAUNCH(sweep_block_kernel<true>, grid, kBlockThreads, h->stream, b);
    else AM_LAUNCH(sweep_block_kernel<false>, grid, kBlockThreads, h->stream, b);
    h->launches++;
    if (cudaError_t e = cudaGetLastError(); e != cudaSuccess) { h->last_error = cudaGetErrorString(e); rc = AM_E_DEVICE; }
    k += K;
  }
  for (uint64_t k = 0; !blocked && k < n_ticks && rc == AM_OK; ++k) {
    ListOut o;
    o.idx = h->due_idx[k & 1];
    o.act = h->due_action[k & 1];
    o.cap = h->cap_padded;
    o.stats = d_stats + k;
    rc = launch_tick(h, unix_sec0 + (int64_t)k, mode, o, h->stream);
  }
  if (rc == AM_OK) {
    cudaError_t e = cudaEventRecord(h->ev1, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e == cudaSuccess) e = cudaMemcpy(stats_out, d_stats, n_ticks * sizeof(am_tick_stats_t), cudaMemcpyDeviceToHost);
    float ms = 0;
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    if (e != cudaSuccess) { h->last_error = cudaGetErrorString(e); rc = AM_E_DEVICE; }
    else h->last_ms = ms;
    if (blocked && rc == AM_OK)
      for (uint64_t k = 0; k < n_ticks; ++k) stats_out[k].n_records = h->n_records;
  }
  cudaFree(d_stats);
  return rc;
}

int am_sweep_run_ticks_view(am_sweep_t* h, int64_t unix_sec0, uint64_t n_ticks, uint32_t mode, uint64_t seed,
                            am_tick_stats_t* stats_out, am_tick_view_t* views) {
  if (!h || !stats_out || !views) return AM_E_INVAL;
  if (n_ticks == 0) return AM_OK;
  if (n_ticks > (1ull << 24)) return AM_E_INVAL;
  if (unix_sec0 >= (1ll << 55) - (int64_t)n_ticks || unix_sec0 <= -(1ll << 55)) return AM_E_RANGE;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  AM_CUDA(h, cudaSetDevice(h->device));
  int rc = order_on(h, h->stream);
  if (rc != AM_OK) return rc;
  // No tick time: posted results stay pending in the flags, and the first tick's sweep or block kernel
  // applies and counts them (a block kernel publishes only what it counts itself).
  rc = drain_staged(h, h->stream);
  if (rc != AM_OK) return rc;
  h->seed = seed;
  h->host_n = 0;  // the list buffer is about to hold a run of lists, no longer the last tick's
  std::vector<uint64_t> start(n_ticks);
  AM_CUDA(h, cudaEventRecord(h->ev0, h->stream));
  if ((mode & AM_SWEEP_BLOCKED) && h->n_records != 0)
    rc = run_lists_blocked(h, unix_sec0, n_ticks, mode, stats_out, start.data());
  else
    rc = run_lists_ticks(h, unix_sec0, n_ticks, mode & ~AM_SWEEP_BLOCKED, stats_out, start.data());
  if (rc != AM_OK) return rc;
  AM_CUDA(h, cudaEventRecord(h->ev1, h->stream));
  AM_CUDA(h, cudaEventSynchronize(h->ev1));
  float ms = 0;
  AM_CUDA(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
  h->last_ms = ms;
  const uint8_t* act = h->host_out.p ? (const uint8_t*)h->host_out.p + h->host_out_entries * 4 : nullptr;
  for (uint64_t k = 0; k < n_ticks; ++k) {
    views[k].idx_local = h->host_out.p ? (const uint32_t*)h->host_out.p + start[k] : nullptr;
    views[k].action = act ? act + start[k] : nullptr;
    views[k].n = stats_out[k].n_emitted;
    views[k].shard_base = h->shard_base;
  }
  return AM_OK;
}

static int read_impl(am_sweep_t* h, uint64_t first, uint64_t n, const uint64_t* idx, am_record_cols_t* out);

int am_sweep_repeat_after_sec(am_sweep_t* h, int64_t unix_sec, uint64_t first, uint64_t n, int64_t* out) {
  if (!h || (n && !out)) return AM_E_INVAL;
  if (first + n > h->capacity || first + n < first || n > 0xFFFFFFFFull) return AM_E_INVAL;
  if (unix_sec >= (1ll << 55) || unix_sec <= -(1ll << 55)) return AM_E_RANGE;
  if (n == 0) return AM_OK;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  AM_CUDA(h, cudaSetDevice(h->device));
  int rc = order_on(h, h->stream);
  if (rc != AM_OK) return rc;
  rc = drain_staged(h, h->stream);
  if (rc != AM_OK) return rc;
  AM_CUDA(h, h->dev_in.reserve(n * 8));
  AM_CUDA(h, h->pin_in.reserve(n * 8));
  AM_LAUNCH(next_fire_kernel, (unsigned)((n + 127) / 128), 128, h->stream, h->cols, (uint32_t)first, (uint32_t)n,
            unix_sec, (int64_t*)h->dev_in.p);
  h->launches++;
  AM_CUDA(h, cudaGetLastError());
  AM_CUDA(h, cudaMemcpyAsync(h->pin_in.p, h->dev_in.p, n * 8, cudaMemcpyDeviceToHost, h->stream));
  AM_CUDA(h, cudaStreamSynchronize(h->stream));
  memcpy(out, h->pin_in.p, n * 8);
  {  // schedules bound to a named time zone (marked -1, never a real value): Next() on the host
    std::vector<uint64_t> zi;
    for (uint64_t k = 0; k < n; ++k) if (out[k] == -1) zi.push_back(first + k);
    if (!zi.empty()) {
      std::vector<uint64_t> mi(zi.size()), hr(zi.size()), dm(zi.size()), mo(zi.size()), dw(zi.size());
      std::vector<uint32_t> fl(zi.size());
      am_record_cols_t c{};
      c.minute = mi.data(); c.hour = hr.data(); c.dom = dm.data(); c.month = mo.data(); c.dow = dw.data(); c.flags = fl.data();
      const int rrc = read_impl(h, 0, zi.size(), zi.data(), &c);
      if (rrc != AM_OK) return rrc;
      for (size_t k = 0; k < zi.size(); ++k) {
        am_cron_t cr{mi[k], hr[k], dm[k], mo[k], dw[k], 0, AM_CRON_SPEC, (int32_t)(fl[k] >> AM_F_TZ_SHIFT)};
        out[zi[k] - first] = am_cron_repeat_after_sec(&cr, unix_sec);
      }
    }
  }
  return AM_OK;
}

int am_sweep_next_due(am_sweep_t* h, int64_t unix_sec, int64_t* next_out) {
  if (!h || !next_out) return AM_E_INVAL;
  if (unix_sec >= (1ll << 55) || unix_sec <= -(1ll << 55)) return AM_E_RANGE;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  AM_CUDA(h, cudaSetDevice(h->device));
  int rc = order_on(h, h->stream);
  if (rc != AM_OK) return rc;
  rc = drain_staged(h, h->stream);
  if (rc != AM_OK) return rc;
  *next_out = INT64_MAX;  // nothing will ever be due (empty shard, only tombstones / exhausted schedules)
  if (h->n_records == 0) return AM_OK;
  AM_CUDA(h, h->dev_in.reserve(8));
  AM_CUDA(h, h->pin_in.reserve(8));
  AM_CUDA(h, cudaMemsetAsync(h->dev_in.p, 0xFF, 8, h->stream));
  AM_LAUNCH(next_due_kernel, 148 * 8, 256, h->stream, h->cols, h->n_records, unix_sec, (unsigned long long*)h->dev_in.p);
  h->launches++;
  AM_CUDA(h, cudaGetLastError());
  AM_CUDA(h, cudaMemcpyAsync(h->pin_in.p, h->dev_in.p, 8, cudaMemcpyDeviceToHost, h->stream));
  AM_CUDA(h, cudaStreamSynchronize(h->stream));
  const unsigned long long key = *(const unsigned long long*)h->pin_in.p;
  if (key != ~0ull) *next_out = (int64_t)(key ^ (1ull << 63));
  return AM_OK;
}

static int read_impl(am_sweep_t* h, uint64_t first, uint64_t n, const uint64_t* idx, am_record_cols_t* out);

int am_sweep_read(am_sweep_t* h, uint64_t first, uint64_t n, const uint64_t* idx,
                  am_record_cols_t* out) {
  if (!h || !out) return AM_E_INVAL;
  if (n == 0) return AM_OK;
  TickGuard g(h);
  if (!g.ok) return AM_E_BUSY;
  AM_CUDA(h, cudaSetDevice(h->device));
  {  // a read observes every upsert / remove / result staged before it
    int rc = order_on(h, h->stream);
    if (rc != AM_OK) return rc;
    rc = drain_staged(h, h->stream);
    if (rc != AM_OK) return rc;
  }
  return read_impl(h, first, n, idx, out);
}

// (tick guard held, staged events drained, h->stream ordered)
static int read_impl(am_sweep_t* h, uint64_t first, uint64_t n, const uint64_t* idx, am_record_cols_t* out) {
  if (!idx) {
    if (first + n > h->capacity || first + n < first) return AM_E_INVAL;
    for (int k = 0; k < kNumCols; ++k) {
      void* dst = column(*out, k);
      if (!dst) continue;
      const size_t elem = kColumns[k].elem;
      AM_CUDA(h, cudaMemcpyAsync(dst, (char*)column(h->cols, k) + first * elem, n * elem, cudaMemcpyDeviceToHost, h->stream));
    }
    AM_CUDA(h, cudaStreamSynchronize(h->stream));
    return AM_OK;
  }
  if (n > 0xFFFFFFFFull) return AM_E_INVAL;
  for (uint64_t k = 0; k < n; ++k)
    if (idx[k] >= h->capacity) return AM_E_RANGE;
  const size_t o_idx = n * sizeof(am_record_t), total = o_idx + n * 4;
  AM_CUDA(h, h->pin_in.reserve(total));
  AM_CUDA(h, h->dev_in.reserve(total));
  uint32_t* hidx = (uint32_t*)((char*)h->pin_in.p + o_idx);
  for (uint64_t k = 0; k < n; ++k) hidx[k] = (uint32_t)idx[k];
  char* dp = (char*)h->dev_in.p;
  AM_CUDA(h, cudaMemcpyAsync(dp + o_idx, hidx, n * 4, cudaMemcpyHostToDevice, h->stream));
  AM_LAUNCH(gather_records_kernel, (unsigned)((n + 255) / 256), 256, h->stream, h->cols,
            (const uint32_t*)(dp + o_idx), (am_record_t*)dp, (uint32_t)n);
  h->launches++;
  AM_CUDA(h, cudaGetLastError());
  AM_CUDA(h, cudaMemcpyAsync(h->pin_in.p, dp, n * sizeof(am_record_t), cudaMemcpyDeviceToHost, h->stream));
  AM_CUDA(h, cudaStreamSynchronize(h->stream));
  const am_record_t* r = (const am_record_t*)h->pin_in.p;
#define AM_SCATTER(name) \
  if (out->name)         \
    for (uint64_t k = 0; k < n; ++k) out->name[k] = r[k].name;
  AM_RECORD_COLUMNS(AM_SCATTER)
#undef AM_SCATTER
  return AM_OK;
}

}  // extern "C"
