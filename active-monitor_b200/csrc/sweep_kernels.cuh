// sweep_kernels.cuh — the per-tick schedule-evaluation sweep for sm_100a.
//
// One launch evaluates every HealthCheck record of a shard at one wall-clock
// second T (SURVEY.md Appendix B.3).  It replaces, for N records at once, the
// per-CR decisions of the reference controller (hcc.go = internal/controllers/
// healthcheck_controller.go):
//     hcc.go:227        Workflow.Resource == nil      -> record skipped
//     hcc.go:238-250    pause rule                    -> AM_ACT_STOPPED
//     hcc.go:251-263    cron arm (robfig bitmasks)    -> matches(T), A.7
//     hcc.go:264, :751  interval / timer              -> T - finishedAt >= ras
//     hcc.go:635-661    Succeeded transition          -> apply_result()
//     hcc.go:662-722    Failed transition + remedy gate
//     hcc.go:821-851    remedy result counters
//
// Shape of the kernel (pure integer work, HBM-bandwidth bound, no tensor cores):
//   * records live as SoA columns in HBM; a CTA of 256 threads owns one tile of
//     1024 consecutive records, a warp owns 128 of them;
//   * every warp-level load instruction is fully coalesced: lane L reads the
//     16 B (two u64 records) or 8 B (two i32 records) at column + (w + 2L),
//     twice per tile ("halves"), so 16 independent loads are in flight per
//     lane before the first use (a __syncwarp() after them keeps ptxas from
//     delaying half of them).  Staging the tile in shared memory instead —
//     per-lane cp.async, TMA bulk copies one-shot, and a persistent two-stage
//     TMA pipeline — was built, verified and measured 6-15 % slower for this
//     streaming, near-issue-bound kernel (DESIGN.md section 3);
//   * the tick's broken-down time is computed once per tick as one-hot words
//     and reaches every CTA through the kernel parameters (constant bank); a
//     5-field schedule fires iff minute&M && hour&H && month&Mo && dayMatches
//     (five ANDs, no loop);
//   * remedy/counter columns are touched only by lanes whose record has a
//     posted result (or is due, in closed-loop mode): 56 B/record otherwise;
//   * the emitted set leaves the kernel as a BITMAP (one bit per record: the four
//     warp ballots the kernel takes anyway, interleaved into four 32-record words
//     per warp, one 128-B line per tile) plus a per-tile list of EXCEPTIONS — the
//     few records whose action is anything but the bare AM_ACT_SUBMIT_HC; no
//     dependency between CTAs.  scan_groups_kernel (one CTA) turns the per-group
//     popcounts into exclusive offsets and expand_kernel rebuilds the contiguous
//     ascending (index, action) list from bitmap + exceptions — for the local shard
//     or, on several GPUs, for every rank's bitmap after the NVLink exchange
//     (gather_kernels.cuh): 1 bit per record crosses the wire instead of 5 bytes per
//     entry.  Round 1 wrote (u32, u8) segments and compacted them (16.7 MB written +
//     33 MB moved per tick at the bench density); a single-pass decoupled look-back was
//     measured before that and rejected (profiles/r01a_lookback_sweep_ncu.csv);
//   * per-tick statistics are reduced lane -> warp (redux) -> CTA -> global (fire-and-
//     forget RED); kernel boundaries (programmatic dependent launches) are the only
//     global synchronisation, so the sweep kernel has one __syncthreads, no fences and
//     no completion tickets.
#pragma once
#ifndef AMSWEEP_EMULATE  // tests/emu compiles this file for the CPU (cuda_emu.h supplies the model)
#include <cuda_runtime.h>
#endif
#include <stdint.h>

#include "../../include/amsweep.h"
#include "civil.h"

#include "sweep_types.h"

namespace amsweep {

// ---- streaming loads / stores: every byte is touched once per tick --------
template <typename T>
__device__ __forceinline__ T ld_stream(const T* p) { return __ldcs(p); }
template <typename T>
__device__ __forceinline__ void st_stream(T* p, T v) { __stcs(p, v); }

// Segment entries are written once by the sweep and read once, a few tens of
// microseconds later, by expand_kernel: keep them L2-resident (evict_last)
// while 560 MB of evict_first column data streams past them.
#ifndef AMSWEEP_EMULATE
__device__ __forceinline__ uint64_t l2_evict_last_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void st_keep_u32(uint32_t* p, uint32_t v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.u32 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_keep_u8(uint8_t* p, uint32_t v, uint64_t pol) {
  asm volatile("st.global.L2::cache_hint.u8 [%0], %1, %2;" ::"l"(p), "r"(v), "l"(pol) : "memory");
}
// programmatic dependent launch (sm_90+): see AM_LAUNCH_PDL
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#else  // CPU emulation: plain stores, the cache policy has no meaning
inline void pdl_wait() {}
inline void pdl_trigger() {}
inline uint64_t l2_evict_last_policy() { return 0; }
inline void st_keep_u32(uint32_t* p, uint32_t v, uint64_t) { *p = v; }
inline void st_keep_u8(uint8_t* p, uint32_t v, uint64_t) { *p = (uint8_t)v; }
#endif

__device__ __forceinline__ uint64_t sm64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
__device__ __forceinline__ uint64_t outcome_key(uint64_t seed, uint64_t gidx, uint64_t t) {
  return sm64(sm64(seed ^ sm64(gidx)) + t);
}

// the low 16 bits of x -> the even bit positions of a 32-bit word
__device__ __forceinline__ uint32_t spread16(uint32_t x) {
  x &= 0xFFFFu;
  x = (x | (x << 8)) & 0x00FF00FFu;
  x = (x | (x << 4)) & 0x0F0F0F0Fu;
  x = (x | (x << 2)) & 0x33333333u;
  x = (x | (x << 1)) & 0x55555555u;
  return x;
}

// bit i of a 4-bit value -> byte i of a word (0/1 each)
__device__ __forceinline__ uint32_t spread4(uint32_t v) { return ((v & 0xFu) * 0x00204081u) & 0x01010101u; }

// Mutable per-record state carried through the result state machine.
struct RecState {
  uint32_t flags;
  int64_t fa;       // finishedAt
  int32_t s, f;     // SuccessCount, FailedCount
  int32_t rs, rf, rt;  // RemedySuccessCount, RemedyFailedCount, RemedyTotalRuns
  int64_t rfa;      // RemedyFinishedAt, 0 == nil
  int32_t limit, reset;
};

// watchRemedyWorkflow result, hcc.go:821-851
__device__ __forceinline__ void remedy_result(RecState& r, int64_t T, bool ok, uint32_t& res) {
  if (ok) { r.rs = (int32_t)((uint32_t)r.rs + 1u); res += 1u << 16; }
  else    { r.rf = (int32_t)((uint32_t)r.rf + 1u); res += 1u << 24; }
  r.rt = (int32_t)((uint32_t)r.rs + (uint32_t)r.rf);
  r.rfa = T;
}

// Step 1 of B.3: apply a posted workflow result.  Returns action bits; `res`
// counts {ok, fail, remedy_ok, remedy_fail} in its four bytes (a record can
// take two results in one closed-loop tick) for the metrics counters.
__device__ __forceinline__ uint32_t apply_result(RecState& r, int64_t T, uint32_t& res) {
  uint32_t act = 0;
  const uint32_t f = r.flags;
  // watchWorkflowReschedule re-arms the repeat timer after either outcome (hcc.go:745-752)
  const uint32_t armed = (f & (AM_F_PENDING_OK | AM_F_PENDING_FAIL)) ? AM_F_TIMER_ARMED : 0u;
  if (f & AM_F_PENDING_OK) {  // hcc.go:635-661
    r.s = (int32_t)((uint32_t)r.s + 1u);
    r.fa = T;
    res += 1u;
    if ((f & AM_F_HAS_REMEDY) && r.rt >= 1) {  // :649
      r.rt = r.rs = r.rf = 0;
      r.rfa = 0;
      act |= AM_ACT_RESET_ON_PASS;
    }
  } else if (f & AM_F_PENDING_FAIL) {  // hcc.go:662-722
    r.f = (int32_t)((uint32_t)r.f + 1u);
    r.fa = T;
    res += 1u << 8;
    if (f & AM_F_HAS_REMEDY) {  // :677
      bool run = false;
      if (r.limit != 0 && r.reset != 0) {  // :679
        if (r.limit > r.rt) {               // :681
          run = true;
        } else if (r.rfa == 0) {
          act |= AM_ACT_ANOMALY;  // nil RemedyFinishedAt at :690 (N3)
        } else {
          // int(now.Sub(RemedyFinishedAt).Seconds()): Sub saturates at
          // +-9223372036 s, far outside the i32 resetInterval domain
          int64_t d = (int64_t)((uint64_t)T - (uint64_t)r.rfa);
          d = d > 9223372036ll ? 9223372036ll : (d < -9223372036ll ? -9223372036ll : d);
          if ((int64_t)r.reset >= d) {  // :692
            act |= AM_ACT_REMEDY_SKIP;
          } else {  // :695-704
            r.rt = r.rs = r.rf = 0;
            r.rfa = 0;
            act |= AM_ACT_RESET_ON_INTERVAL;
            run = true;
          }
        }
      } else {  // :712-719
        run = true;
      }
      if (run) {
        act |= AM_ACT_RUN_REMEDY;
        if (f & AM_F_REMEDY_PENDING) remedy_result(r, T, (f & AM_F_REMEDY_OUTCOME_OK) != 0, res);
      }
    }
  } else if (f & AM_F_REMEDY_PENDING) {  // remedy finished on its own
    remedy_result(r, T, (f & AM_F_REMEDY_OUTCOME_OK) != 0, res);
  }
  r.flags = (f & ~(AM_F_PENDING_OK | AM_F_PENDING_FAIL | AM_F_REMEDY_PENDING | AM_F_REMEDY_OUTCOME_OK)) | armed;
  return act;
}

// Action bits of apply_result <-> the carry bits of the flags word (AM_F_CARRY_MASK): RUN_REMEDY (0x02)
// in bit 11, REMEDY_SKIP .. ANOMALY (0x10 .. 0x80) in bits 12 .. 15.
__device__ __forceinline__ uint32_t carried_actions(uint32_t f) { return ((f >> 10) & AM_ACT_RUN_REMEDY) | ((f >> 8) & 0xF0u); }
__device__ __forceinline__ uint32_t carry_of_actions(uint32_t a) { return ((a & AM_ACT_RUN_REMEDY) << 10) | ((a & 0xF0u) << 8); }
static_assert(AM_F_CARRY_SHIFT == 11 && AM_ACT_RUN_REMEDY == 0x02u && AM_ACT_REMEDY_SKIP == 0x10u && AM_ACT_ANOMALY == 0x80u,
              "carry bit layout");

// Is the record evaluated at all: kinds 1..5 are; tombstones, NO_RESOURCE (hcc.go:227) and host-fallback are not.
// (The sweep expands the macro in place, on the kind it has already extracted: only then does the compiler fold it
// into the kind tests of the ladder — through the function, sweep_tick_kernel<1,0> issues 8 more instructions.)
#define AM_EVALUATED(f, kind) (((0x3Eu >> (kind)) & 1u) && !((f) & AM_F_TOMBSTONE))
__device__ __forceinline__ bool evaluated(uint32_t f) { return AM_EVALUATED(f, f & AM_KIND_MASK); }

// Closed-loop harness (config 5, DESIGN §6.7): a due record completes in the same tick with its preset
// outcome — failed iff key byte 0 < the record's failp8, remedy succeeded iff key byte 1 < kRemedyOkBelow
// — taken like a posted result (hcc.go:635-724).  Returns the action bits of that result.
constexpr uint32_t kRemedyOkBelow = 179;  // of 256: a remedy succeeds 70 % of the time
__device__ __forceinline__ uint32_t complete_closed_loop(RecState& s, uint64_t seed, uint64_t gidx, int64_t T, uint32_t& res) {
  const uint64_t k = outcome_key(seed, gidx, (uint64_t)T);
  const uint32_t failp = (s.flags >> AM_F_FAILP_SHIFT) & 0xFFu;
  const bool fail = (uint32_t)(k & 0xFF) < failp;
  const bool rem_ok = (uint32_t)((k >> 8) & 0xFF) < kRemedyOkBelow;
  s.flags |= (fail ? AM_F_PENDING_FAIL : AM_F_PENDING_OK) | AM_F_REMEDY_PENDING | (rem_ok ? AM_F_REMEDY_OUTCOME_OK : 0u);
  return apply_result(s, T, res);
}

// Results applied (metrics.MonitorSuccess / Error; hcc.go:635-722, :821-851): the four byte counters of
// apply_result's `res` {ok, fail, remedy ok, remedy fail} summed over the warp (two redux over 16-bit halves).
// Lane q < 4 receives counter q, the other lanes 0.
__device__ __forceinline__ uint32_t warp_result_counts(uint32_t res, int lane) {
  uint32_t lo = 0, hi = 0;
  if (__any_sync(kFull, res != 0)) {
    lo = __reduce_add_sync(kFull, (res & 0xFFu) | ((res & 0xFF00u) << 8));           // ok | fail<<16
    hi = __reduce_add_sync(kFull, ((res >> 16) & 0xFFu) | ((res >> 8) & 0xFF0000u));  // remedy ok | fail<<16
  }
  return lane < 4 ? ((lane < 2 ? lo : hi) >> ((lane & 1) * 16)) & 0xFFFFu : 0u;
}

// robfig SpecSchedule matching against the tick's one-hot wall-clock words (Appendix A: five ANDs and
// the dom/dow star rule).  Branch-free: every term is evaluated (no short-circuit control flow).
__device__ __forceinline__ bool cron_matches(const TickWords& t, uint64_t mi, uint64_t hr, uint64_t dm, uint64_t mo, uint64_t dw) {
  const bool fld = ((mi & t.minute) != 0) & ((hr & t.hour) != 0) & ((mo & t.month) != 0);
  const bool dmm = (dm & t.dom) != 0, dwm = (dw & t.dow) != 0;
  const bool star = ((dm | dw) >> 63) != 0;  // robfig dayMatches
  return (t.sec0 != 0) & fld & (star ? (dmm & dwm) : (dmm | dwm));
}
// A schedule bound to a named time zone ("CRON_TZ=Zone ...", robfig parser.go / hcc.go:253,
// SpecSchedule.Location): the same match against the zone's wall clock.  `z` points at the zone's entry
// of the tick's word table (tz_words_kernel).  Rare records: kept out of line.  (Deriving the words from
// T + offset inside this call instead of loading them cost the 10 M-record sweep 8 us — half of all warps
// hold a zone-bound record at 0.6 % of the records and ran ~100 more instructions each.)
__device__ __noinline__ bool cron_matches_in_zone(const TickWords* z, uint64_t mi, uint64_t hr, uint64_t dm, uint64_t mo,
                                                  uint64_t dw) {
  const TickWords t = *z;
  return cron_matches(t, mi, hr, dm, mo, dw);
}

// The tick's wall clock in every registered zone as one-hot words: T + the zone's UTC offset, broken
// down.  The offsets are kept by the launcher (valid until a zone changes its offset); this is one
// thread per zone and no memory traffic to speak of, launched with programmatic serialisation ahead of
// the sweep — only when zones are registered.
__global__ void tz_words_kernel(const int32_t* __restrict__ tz_off, TickWords* __restrict__ table, int64_t T, uint32_t n) {
  pdl_wait();
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) table[k] = tick_words_from_unix(T + (int64_t)tz_off[k]);
}

// ---------------------------------------------------------------------------
// The sweep.  CLOSED = closed-loop harness (SURVEY §8d config 5): a due record
// completes in the same tick with its preset outcome.
// ---------------------------------------------------------------------------
constexpr int kMinBlocks = 3;  // CTAs per SM with the mask columns; one more without them
// MASKS = the five cron-field columns are read and matched.  Off the minute a
// 5-field schedule cannot fire (ParseStandard pins Second to 1<<0), so the
// launcher picks MASKS=false unless AM_SWEEP_FULL_SCAN is set: 40 of the 56
// bytes per record and all of the mask arithmetic disappear at compile time.
template <bool CLOSED, bool MASKS>
__global__ void __launch_bounds__(kBlock, MASKS ? kMinBlocks : kMinBlocks + 1) sweep_tick_kernel(const SweepParams p) {
  // one row per warp, written unconditionally: no zero-initialisation, no shared
  // atomics, and therefore a single __syncthreads in the whole kernel
  __shared__ uint32_t s_warp_tot[kWarps], s_warp_exc[kWarps];
  __shared__ uint32_t s_ballot[kWarps][4];  // each warp's four emitted-record ballots
  __shared__ uint32_t s_wres[kWarps][4];    // posted results applied: ok, fail, remedy ok, remedy fail

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const uint32_t tile = blockIdx.x;
  const uint32_t tile_base = tile * (uint32_t)kTile;
  const int64_t T = p.T;
  pdl_wait();  // the sweep is launched while its predecessor (the previous tick's publish, or the drain) still runs

  // ---- phase A: issue every schedule-column load of this lane up front ----
  // half h covers records r0(h) .. r0(h)+1, r0 = tile_base + warp*128 + h*64 + lane*2
  uint32_t r0[2];
  ulonglong2 mi[2], hr[2], dm[2], mo[2], dw[2];
  longlong2 fa[2];
  int2 ras[2];
  uint2 fl[2];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    r0[h] = tile_base + (uint32_t)(warp * kRecPerWarp + h * 64 + lane * 2);
    fl[h] = ld_stream(reinterpret_cast<const uint2*>(p.c.flags + r0[h]));
    ras[h] = ld_stream(reinterpret_cast<const int2*>(p.c.ras + r0[h]));
    fa[h] = ld_stream(reinterpret_cast<const longlong2*>(p.c.finished_at + r0[h]));
  }
  if (MASKS) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      mi[h] = ld_stream(reinterpret_cast<const ulonglong2*>(p.c.minute + r0[h]));
      hr[h] = ld_stream(reinterpret_cast<const ulonglong2*>(p.c.hour + r0[h]));
      dm[h] = ld_stream(reinterpret_cast<const ulonglong2*>(p.c.dom + r0[h]));
      mo[h] = ld_stream(reinterpret_cast<const ulonglong2*>(p.c.month + r0[h]));
      dw[h] = ld_stream(reinterpret_cast<const ulonglong2*>(p.c.dow + r0[h]));
    }
  }

  // Scheduling fence: a warp-level memory-ordering point.  ptxas may not sink the loads
  // above across it, so all 16 are issued before any of the arithmetic below (without it
  // the second half's loads were delayed behind the first half's compute: -30 % bandwidth).
  __syncwarp();

  // The tick's broken-down time: one-hot words computed once per tick (civil.h) and
  // delivered through the kernel parameters, i.e. the constant bank / uniform
  // registers — cheaper than staging them in shared memory, which cost every CTA a
  // serial thread-0 section and a barrier (profiles/r01_summary.md).
  const TickWords w = p.words;
  // named time zones are rare: one vote per warp decides whether the per-record zone lookup exists at all
  const uint32_t fl_or = fl[0].x | fl[0].y | fl[1].x | fl[1].y;
  const bool warp_tz = MASKS && p.tz_table != nullptr && __any_sync(kFull, (fl_or >> AM_F_TZ_SHIFT) != 0);

  uint32_t act[2][2];
  uint32_t res_lane = 0;  // 4 x 8-bit counts of results applied by this lane
  uint32_t nfl[2][2];     // flags / finishedAt after this tick
  int64_t nfa[2][2];
  bool dirty[2] = {false, false};
  uint32_t needy = 0, due_bits = 0;  // bit (2h+j): record needs the remedy/counter columns / is due

  // ---- schedule decision for the lane's four records ------------------------
#pragma unroll
  for (int h = 0; h < 2; ++h) {
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const uint32_t f = j ? fl[h].y : fl[h].x;
      const int32_t rasv = j ? ras[h].y : ras[h].x;
      const int64_t fav = j ? fa[h].y : fa[h].x;
      const uint32_t kind = f & AM_KIND_MASK;
      const bool live = AM_EVALUATED(f, kind);
      const bool has_result = (f & (AM_F_PENDING_OK | AM_F_PENDING_FAIL)) != 0;
      const bool pending = (f & (AM_F_PENDING_OK | AM_F_PENDING_FAIL | AM_F_REMEDY_PENDING)) != 0;
      // step 1 sets finishedAt = T before the due decision is taken
      const int64_t fa_eff = has_result ? T : fav;
      const int64_t elapsed = (int64_t)((uint64_t)T - (uint64_t)fa_eff);
      // not(hcc.go:264): "elapsed < RepeatAfterSec && timer != nil" skips; a posted result re-arms
      // the timer in this very tick (step 1 runs first), and without a timer (controller restart,
      // hcc.go:161) the reference submits whatever finishedAt says
      const bool armed = has_result || (f & AM_F_TIMER_ARMED) != 0;
      const bool due_iv = !((elapsed < (int64_t)rasv) & armed);
      bool due_cron = false;
      if (MASKS) {
        const uint64_t miv = j ? mi[h].y : mi[h].x, hrv = j ? hr[h].y : hr[h].x;
        const uint64_t dmv = j ? dm[h].y : dm[h].x, mov = j ? mo[h].y : mo[h].x;
        const uint64_t dwv = j ? dw[h].y : dw[h].x;
        due_cron = cron_matches(w, miv, hrv, dmv, mov, dwv);
        if (warp_tz) {  // warp-uniform: some record of this warp is bound to a named time zone
          const uint32_t tz = f >> AM_F_TZ_SHIFT;
          // the zone's wall clock instead of UTC's — behind a real call: inlined, ptxas turned the zone
          // lookup of all four records into predicated instructions that EVERY warp issues (+24 LDG,
          // +40 address IMADs per warp: 84 -> 96 us per 10 M-record tick, profiles/r02_summary.md)
          if (tz) due_cron = cron_matches_in_zone(p.tz_table + tz, miv, hrv, dmv, mov, dwv);
        }
      }
      const bool is_iv = ((0x14u >> kind) & 1u) != 0;  // INTERVAL or CRON_EVERY
      const bool due = live && (is_iv ? due_iv : (kind == AM_KIND_CRON_SPEC && due_cron));
      const bool stopped_now = live && kind == AM_KIND_STOPPED && !(f & AM_F_STOPPED_REPORTED);
      act[h][j] = (due ? AM_ACT_SUBMIT_HC : 0u) | (stopped_now ? AM_ACT_STOPPED : 0u) |
                  ((live && kind == AM_KIND_PARSE_ERROR) ? AM_ACT_PARSE_ERROR : 0u);
      nfl[h][j] = f;
      nfa[h][j] = fav;
      if (stopped_now) {  // hcc.go:238-250: Status "Stopped", FinishedAt = now
        nfl[h][j] = f | AM_F_STOPPED_REPORTED;
        nfa[h][j] = T;
        dirty[h] = true;
      }
      if (live && (pending || (CLOSED && due))) needy |= 1u << (2 * h + j);
      if (due) due_bits |= 1u << (2 * h + j);
    }
  }

  // ---- results applied at this tick's drain (apply_results_now_kernel) left their action bits in the
  //      flags' carry bits: emit and clear them.  Rare (a posted "Succeeded" carries nothing): one vote
  //      per warp keeps the per-record form out of the common path.
  if (__any_sync(kFull, (fl_or & AM_F_CARRY_MASK) != 0)) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const uint32_t f = j ? fl[h].y : fl[h].x;
        if (f & AM_F_CARRY_MASK) {
          act[h][j] |= carried_actions(f);
          nfl[h][j] &= ~AM_F_CARRY_MASK;
          dirty[h] = true;
        }
      }
    }
  }

  // ---- results + remedy state machine (hcc.go:633-724, 819-852) -------------------
  // Two shapes, chosen per warp by how many lanes have work:
  //  dense  (>= 16 lanes, e.g. half of all checks reporting a result this tick): per
  //         pair of records, vector loads of the eight remedy/counter columns and the
  //         state machine predicated per record — the bytes are needed anyway and 16-B
  //         transactions keep the LSU count low;
  //  sparse (a few due/posted records per warp): a warp loop in which every lane takes
  //         its next needy record with scalar accesses — the loop runs once or twice
  //         instead of four predicated copies of the state machine.
  if (__popc(__ballot_sync(kFull, needy != 0)) >= 16) {
    // both halves' loads first (sixteen more in flight per lane: the mask registers are dead by now),
    // then the state machines, then the stores — a half's stores would otherwise fence the other
    // half's loads behind them (the compiler cannot tell the columns apart)
    int2 lim[2], rst[2], sc[2], fc[2], rsc[2], rfc[2], rtc[2];
    longlong2 rfa[2];
    auto load_half = [&](int h) {
      if ((needy >> (2 * h)) & 3u) {
        const uint32_t r = r0[h];
        lim[h] = ld_stream(reinterpret_cast<const int2*>(p.c.runs_limit + r));
        rst[h] = ld_stream(reinterpret_cast<const int2*>(p.c.reset_interval + r));
        sc[h] = ld_stream(reinterpret_cast<const int2*>(p.c.success + r));
        fc[h] = ld_stream(reinterpret_cast<const int2*>(p.c.failed + r));
        rsc[h] = ld_stream(reinterpret_cast<const int2*>(p.c.remedy_success + r));
        rfc[h] = ld_stream(reinterpret_cast<const int2*>(p.c.remedy_failed + r));
        rtc[h] = ld_stream(reinterpret_cast<const int2*>(p.c.remedy_total + r));
        rfa[h] = ld_stream(reinterpret_cast<const longlong2*>(p.c.remedy_finished_at + r));
      }
    };
    if (MASKS) {  // (the variants without the mask columns run at 64 registers: one half at a time there)
      load_half(0);
      load_half(1);
      __syncwarp();
    }
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const uint32_t nb = (needy >> (2 * h)) & 3u;
      if (!MASKS) load_half(h);
      if (nb) {
        const uint32_t r = r0[h];
        int32_t ns[2] = {sc[h].x, sc[h].y}, nf[2] = {fc[h].x, fc[h].y};
        int32_t nrs[2] = {rsc[h].x, rsc[h].y}, nrf[2] = {rfc[h].x, rfc[h].y}, nrt[2] = {rtc[h].x, rtc[h].y};
        int64_t nrfa[2] = {rfa[h].x, rfa[h].y};
        const int32_t limv[2] = {lim[h].x, lim[h].y}, rstv[2] = {rst[h].x, rst[h].y};
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if ((nb >> j) & 1u) {
            RecState s{nfl[h][j], nfa[h][j], ns[j], nf[j], nrs[j], nrf[j], nrt[j], nrfa[j], limv[j], rstv[j]};
            uint32_t res = 0;
            uint32_t a = apply_result(s, T, res);
            if (CLOSED && ((due_bits >> (2 * h + j)) & 1u)) a |= complete_closed_loop(s, p.seed, p.shard_base + r + (uint32_t)j, T, res);
            act[h][j] |= a;
            res_lane += res;
            nfl[h][j] = s.flags; nfa[h][j] = s.fa;
            ns[j] = s.s; nf[j] = s.f; nrs[j] = s.rs; nrf[j] = s.rf; nrt[j] = s.rt; nrfa[j] = s.rfa;
          }
        }
        dirty[h] = true;  // a result always clears its PENDING flags
        if (ns[0] != sc[h].x || ns[1] != sc[h].y) st_stream(reinterpret_cast<int2*>(p.c.success + r), make_int2(ns[0], ns[1]));
        if (nf[0] != fc[h].x || nf[1] != fc[h].y) st_stream(reinterpret_cast<int2*>(p.c.failed + r), make_int2(nf[0], nf[1]));
        if (nrs[0] != rsc[h].x || nrs[1] != rsc[h].y)
          st_stream(reinterpret_cast<int2*>(p.c.remedy_success + r), make_int2(nrs[0], nrs[1]));
        if (nrf[0] != rfc[h].x || nrf[1] != rfc[h].y)
          st_stream(reinterpret_cast<int2*>(p.c.remedy_failed + r), make_int2(nrf[0], nrf[1]));
        if (nrt[0] != rtc[h].x || nrt[1] != rtc[h].y)
          st_stream(reinterpret_cast<int2*>(p.c.remedy_total + r), make_int2(nrt[0], nrt[1]));
        if (nrfa[0] != rfa[h].x || nrfa[1] != rfa[h].y)
          st_stream(reinterpret_cast<longlong2*>(p.c.remedy_finished_at + r), make_longlong2(nrfa[0], nrfa[1]));
      }
    }
    needy = 0;
  }
  while (__any_sync(kFull, needy != 0)) {
    if (needy) {
      const int b = __ffs(needy) - 1;
      needy &= needy - 1;
      const uint32_t i = r0[0] + (uint32_t)(64 * (b >> 1) + (b & 1));
      const int32_t lim = ld_stream(p.c.runs_limit + i), rst = ld_stream(p.c.reset_interval + i);
      const int32_t sc = ld_stream(p.c.success + i), fc = ld_stream(p.c.failed + i);
      const int32_t rsc = ld_stream(p.c.remedy_success + i), rfc = ld_stream(p.c.remedy_failed + i);
      const int32_t rtc = ld_stream(p.c.remedy_total + i);
      const int64_t rfa = ld_stream(p.c.remedy_finished_at + i);
      const uint32_t f0 = b == 0 ? nfl[0][0] : b == 1 ? nfl[0][1] : b == 2 ? nfl[1][0] : nfl[1][1];
      const int64_t fa0 = b == 0 ? nfa[0][0] : b == 1 ? nfa[0][1] : b == 2 ? nfa[1][0] : nfa[1][1];
      RecState s{f0, fa0, sc, fc, rsc, rfc, rtc, rfa, lim, rst};
      uint32_t res = 0;
      uint32_t a = apply_result(s, T, res);
      if (CLOSED && ((due_bits >> b) & 1u)) a |= complete_closed_loop(s, p.seed, p.shard_base + i, T, res);
      res_lane += res;  // per lane at most 4 records x 2 results per byte
      if (s.s != sc) st_stream(p.c.success + i, s.s);
      if (s.f != fc) st_stream(p.c.failed + i, s.f);
      if (s.rs != rsc) st_stream(p.c.remedy_success + i, s.rs);
      if (s.rf != rfc) st_stream(p.c.remedy_failed + i, s.rf);
      if (s.rt != rtc) st_stream(p.c.remedy_total + i, s.rt);
      if (s.rfa != rfa) st_stream(p.c.remedy_finished_at + i, s.rfa);
      // (a record "Stopped" in this very tick already carries STOPPED_REPORTED and
      // finishedAt = T in nfl/nfa, and apply_result preserves both: the pause rule of
      // hcc.go:238-250 and a posted result commute)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (q == b) {
          act[q >> 1][q & 1] |= a;
          nfl[q >> 1][q & 1] = s.flags;
          nfa[q >> 1][q & 1] = s.fa;
        }
      }
      if (b < 2) dirty[0] = true; else dirty[1] = true;  // a result always clears its PENDING flags
    }
  }
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    if (dirty[h]) {
      st_stream(reinterpret_cast<uint2*>(p.c.flags + r0[h]), make_uint2(nfl[h][0], nfl[h][1]));
      st_stream(reinterpret_cast<longlong2*>(p.c.finished_at + r0[h]), make_longlong2(nfa[h][0], nfa[h][1]));
    }
  }

  // ---- the emitted set as a bitmap, non-default actions as exceptions -------------
  // e..: records with any action; x..: records whose action is not the bare SUBMIT_HC (rare
  // unless results are being applied: their ballots are only taken when the warp has any)
  const unsigned e00 = __ballot_sync(kFull, act[0][0] != 0), e01 = __ballot_sync(kFull, act[0][1] != 0);
  const unsigned e10 = __ballot_sync(kFull, act[1][0] != 0), e11 = __ballot_sync(kFull, act[1][1] != 0);
  const uint32_t warp_total = __popc(e00) + __popc(e01) + __popc(e10) + __popc(e11);
  unsigned x00 = 0, x01 = 0, x10 = 0, x11 = 0;
  if (__any_sync(kFull, (act[0][0] | act[0][1] | act[1][0] | act[1][1]) > 1u)) {
    x00 = __ballot_sync(kFull, act[0][0] > 1u); x01 = __ballot_sync(kFull, act[0][1] > 1u);
    x10 = __ballot_sync(kFull, act[1][0] > 1u); x11 = __ballot_sync(kFull, act[1][1] > 1u);
  }
  const uint32_t xtot0 = __popc(x00) + __popc(x01);
  const uint32_t warp_exc = xtot0 + __popc(x10) + __popc(x11);
  // the four ballots go to shared memory as they are; warp 0 interleaves them into the tile's 32
  // bitmap words after the barrier (once per tile instead of once per warp)
  if (lane < 4) s_ballot[warp][lane] = lane == 0 ? e00 : (lane == 1 ? e01 : (lane == 2 ? e10 : e11));
  if (lane == 0) { s_warp_tot[warp] = warp_total; s_warp_exc[warp] = warp_exc; }

  // ---- results applied this tick (feeds metrics.MonitorSuccess/Error): lane ->
  //      warp (two redux over 16-bit halves) -> per-warp shared row.  The action
  //      statistics and index checksums are derived from the emitted entries
  //      by expand_kernel, so records that emit nothing cost nothing here.
  {
    const uint32_t v = warp_result_counts(res_lane, lane);
    if (lane < 4) s_wres[warp][lane] = v;
  }
  __syncthreads();

  // ---- tile write-out: one 128-B line of bitmap words, the counts, the exceptions ---
  // Everything written here is read once, a few tens of microseconds later, by
  // expand_kernel (and by the NVLink push): keep it L2-resident (evict_last) while the
  // evict_first column data streams past.
  const uint64_t keep = l2_evict_last_policy();
  if (warp == 0) {
    // Word `lane` of the tile = word k = lane & 3 of warp lane >> 2: its records 32k .. 32k+31 are
    // half k>>1, lanes 16(k&1) .. +15, two records per lane — the two ballots of that half, 16
    // bits each, interleaved.
    const int ww = lane >> 2, hh = (lane >> 1) & 1;
    const unsigned sh16 = (unsigned)(lane & 1) * 16u;
    const uint32_t word = spread16(s_ballot[ww][2 * hh] >> sh16) | (spread16(s_ballot[ww][2 * hh + 1] >> sh16) << 1);
    st_keep_u32(p.out.bitmap + (size_t)tile * kTileWords + lane, word, keep);
    if (lane < 4) {  // result counters (RED, no return value)
      uint32_t sv = 0;
#pragma unroll
      for (int k = 0; k < kWarps; ++k) sv += s_wres[k][lane];
      if (sv) atomicAdd(&p.acc[10 + lane], (unsigned long long)sv);
    }
    if (lane == 4 || lane == 5) {
      uint32_t tot = 0;
#pragma unroll
      for (int k = 0; k < kWarps; ++k) tot += lane == 4 ? s_warp_tot[k] : s_warp_exc[k];
      if (lane == 4) { if (tot) atomicAdd(&p.out.group_count[tile / kGroupTiles], tot); }
      else st_keep_u32(p.out.tile_exc + tile, tot, keep);
    }
  }
  if (warp_exc) {  // warp-uniform; rare unless results are being applied
    uint32_t base = tile_base;
#pragma unroll
    for (int k = 0; k < kWarps; ++k) base += (k < warp) ? s_warp_exc[k] : 0u;
    const unsigned lt = (1u << lane) - 1u;
    uint32_t rank[2];
    rank[0] = __popc(x00 & lt) + __popc(x01 & lt);
    rank[1] = xtot0 + __popc(x10 & lt) + __popc(x11 & lt);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t pos = base + rank[h];
#pragma unroll
      for (int j = 0; j < 2; ++j)
        if (act[h][j] > 1u) {
          const uint32_t off = (uint32_t)(warp * kRecPerWarp + h * 64 + lane * 2 + j);  // record within the tile
          st_keep_u32(p.out.exc_seg + pos, (off << 8) | act[h][j], keep);
          ++pos;
        }
    }
  }
}

// ---------------------------------------------------------------------------
// Per-group emitted counts -> exclusive offsets.  One CTA: the array is a few KB (one u32
// per 8192 records; 1221 for 10 M records) and the work is O(groups) whatever the shard size
// — round 1 had every compaction CTA re-sum all earlier groups, O(groups^2) loads per tick.
// Also publishes n_emitted early (acc[1], and min(n_emitted, cap) for device-side consumers
// of the list) and zeroes the group counters again for the next tick.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) scan_groups_kernel(const ScanParams p) {
  __shared__ uint32_t s_warp[32];
  __shared__ uint32_t s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_carry = 0;
  pdl_wait();  // the sweep's REDs into group_count are complete and visible
  pdl_trigger();
  __syncthreads();
  for (uint32_t g0 = 0; g0 < p.n_groups; g0 += blockDim.x) {
    const uint32_t g = g0 + (uint32_t)tid;
    const uint32_t c = g < p.n_groups ? p.group_count[g] : 0u;
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t up = __shfl_up_sync(kFull, incl, d);
      if (lane >= d) incl += up;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {  // exclusive scan of the 32 warp totals
      const uint32_t t = s_warp[lane];
      uint32_t wi = t;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t up = __shfl_up_sync(kFull, wi, d);
        if (lane >= d) wi += up;
      }
      s_warp[lane] = wi - t;
    }
    __syncthreads();
    const uint32_t carry = s_carry;
    const uint32_t excl = carry + s_warp[warp] + incl - c;
    if (g < p.n_groups) {
      p.group_prefix[g] = excl;
      p.group_count[g] = 0;  // re-armed for the next tick that uses this buffer set
    }
    __syncthreads();  // every thread has read s_carry / s_warp of this round
    if (tid == (int)blockDim.x - 1) s_carry = excl + c;
    __syncthreads();
  }
  if (tid == 0) {
    const uint32_t total = s_carry;
    p.group_prefix[p.n_groups] = total;
    p.acc[1] = (unsigned long long)total;  // n_emitted
    if (p.out_count) *p.out_count = total < p.cap ? total : p.cap;
  }
}

// ---------------------------------------------------------------------------
// Bitmap + exceptions -> the contiguous ascending (index, action) list.  One CTA per
// (group, rank): thread t owns bitmap words 2t, 2t+1 of the group (64 records).  The CTA's position
// in the output is rank offset + group_prefix[g]; the in-group rank of a set bit is the
// exclusive popcount prefix of its word (warp shuffles + 4 warp totals) plus the bits below
// it.  Offsets and action bytes are staged in shared memory — defaults first, then the
// tile's exceptions patched in by rank lookup — and written out as destination-aligned
// quads (16 B of indices + 4 B of actions per store), so the same kernel can write into
// HBM, into a peer-visible exchange buffer or straight into mapped host memory.  While
// writing, every thread counts action bits and checksums global indices for the shard
// whose statistics this GPU owns.
// ---------------------------------------------------------------------------
constexpr int kExpandThreads = 128;  // one thread per PAIR of bitmap words (64 records): the kernel is
                                     // instruction-bound, and the per-thread fixed cost halves per entry
__global__ void __launch_bounds__(kExpandThreads, 8) expand_kernel(const ExpandParams p) {
  // staged so that shared index j <-> output position (start & ~3) + j: a destination-aligned
  // quad of the output is one aligned 8-B (offsets) + one 4-B (actions) shared load
  __shared__ __align__(16) uint16_t s_off[kGroupRecords + 8];
  __shared__ __align__(16) uint8_t s_act[kGroupRecords + 8];
  __shared__ uint32_t s_w[kGroupWords];
  __shared__ uint16_t s_wpre[kGroupWords];
  __shared__ uint32_t s_warp[4];
  __shared__ uint32_t s_nx[8];
  __shared__ uint32_t s_cnt[4][8];            // per-warp counts of the 8 action bits among the exceptions
  __shared__ unsigned long long s_chk[4][2];  // per-warp xor / sum of emitted global indices
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = blockIdx.y;
  const uint32_t g = blockIdx.x;
  const ExpandSrc& src = p.src[r];
  if (g >= src.n_groups) return;  // uniform per CTA
  pdl_wait();
  pdl_trigger();
  // ---- every global load of the CTA is issued here, before the first use: the kernel is a chain
  //      of L2 latencies otherwise (one CTA moves 1 KB in and ~14 KB out)
  const uint2 w2 = __ldcs(reinterpret_cast<const uint2*>(src.bitmap + (size_t)g * kGroupWords) + tid);
  uint64_t start = src.group_prefix[g];
  const uint32_t cnt = src.group_prefix[g + 1] - (uint32_t)start;
  // Exceptions: half-warp (tile & 1) of warp (tile >> 1) patches tile `tile` of the group; its first
  // 16 entries are fetched speculatively (the segment is always mapped; entries past the count are
  // never used)
  const uint32_t tsub = (uint32_t)tid >> 4, l16 = (uint32_t)tid & 15u;  // tile within the group, lane within the half-warp
  const uint32_t tile = g * kGroupTiles + tsub;
  const bool tile_ok = tile < src.n_tiles;
  const uint32_t nx = tile_ok ? src.tile_exc[tile] : 0u;
  const uint32_t e_first = tile_ok ? __ldcs(src.exc_seg + (size_t)tile * kTile + l16) : 0u;
  for (int q = 0; q < r; ++q) start += p.src[q].group_prefix[p.src[q].n_groups];
  if (cnt == 0) return;  // uniform per CTA: nothing emitted by these 8192 records
  const uint32_t sh = (uint32_t)start & 3u;

  // ---- ranks: exclusive popcount prefix over the group's 256 words (two per thread)
  const uint32_t c_lo = (uint32_t)__popc(w2.x), c = c_lo + (uint32_t)__popc(w2.y);
  uint32_t incl = c;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t up = __shfl_up_sync(kFull, incl, d);
    if (lane >= d) incl += up;
  }
  if (lane == 31) s_warp[warp] = incl;
  if (l16 == 0) s_nx[tsub] = nx;
  *reinterpret_cast<uint2*>(&s_w[2 * tid]) = w2;
  // default action for every staged entry (and the padding around them), 4 bytes per store
  for (uint32_t j = (uint32_t)tid * 4u; j < sh + cnt + 4u; j += 4u * kExpandThreads)
    *reinterpret_cast<uint32_t*>(&s_act[j]) = 0x01010101u * AM_ACT_SUBMIT_HC;
  __syncthreads();
  uint32_t before = 0;
#pragma unroll
  for (int k = 0; k < 4; ++k) before += k < warp ? s_warp[k] : 0u;
  const uint32_t excl = before + incl - c;
  *reinterpret_cast<uint32_t*>(&s_wpre[2 * tid]) = excl | ((excl + c_lo) << 16);
  {  // two 32-bit loops (a 64-bit find-first-set / clear-lowest pair costs twice the instructions)
    uint32_t pos = sh + excl;
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      uint32_t ww = hf ? w2.y : w2.x;
      const uint32_t rec0 = (uint32_t)tid * 64u + (uint32_t)hf * 32u - 1u;  // __ffs is 1-based
      while (ww) {
        s_off[pos++] = (uint16_t)(rec0 + (uint32_t)__ffs((int)ww));
        ww &= ww - 1u;
      }
    }
  }
  __syncthreads();
  // ---- exceptions of this half-warp's tile: action bytes other than the default.  Their action
  //      bits are counted here (the default entries all carry SUBMIT_HC and nothing else).
  const bool stats = p.acc != nullptr && r == p.stats_rank;
  uint32_t c0 = 0, c1 = 0;
  for (uint32_t i = l16; i < nx; i += 16u) {
    const uint32_t e = i < 16u ? e_first : __ldcs(src.exc_seg + (size_t)tile * kTile + i);
    const uint32_t off = tsub * (uint32_t)kTile + (e >> 8);
    const uint32_t wd = off >> 5;
    const uint32_t rk = (uint32_t)s_wpre[wd] + (uint32_t)__popc(s_w[wd] & ((1u << (off & 31u)) - 1u));
    s_act[sh + rk] = (uint8_t)e;
    c0 += spread4(e);
    c1 += spread4(e >> 4);
  }
  if (stats) {
    // statistics of this warp's slice of the group: action bits from the exceptions (a lane holds
    // at most 64 of them: byte counters), index checksums from the bitmap words themselves — the
    // sum over the set bits b of word t of (32 t + b) = popc(w) 32 t + sum_j 2^j popc(w & M_j)
    uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    if (__any_sync(kFull, nx != 0)) {
      a0 = __reduce_add_sync(kFull, (c0 & 0xFFu) | ((c0 & 0xFF00u) << 8));
      a1 = __reduce_add_sync(kFull, ((c0 >> 16) & 0xFFu) | ((c0 >> 8) & 0xFF0000u));
      a2 = __reduce_add_sync(kFull, (c1 & 0xFFu) | ((c1 & 0xFF00u) << 8));
      a3 = __reduce_add_sync(kFull, ((c1 >> 16) & 0xFFu) | ((c1 >> 8) & 0xFF0000u));
    }
    if (lane < 8) {
      const uint32_t qv = lane < 2 ? a0 : (lane < 4 ? a1 : (lane < 6 ? a2 : a3));
      s_cnt[warp][lane] = (qv >> ((lane & 1) * 16)) & 0xFFFFu;
    }
    uint32_t osum = 0;
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const uint32_t w = hf ? w2.y : w2.x;
      osum += (uint32_t)__popc(w) * ((uint32_t)(2 * tid + hf) * 32u) + (uint32_t)__popc(w & 0xAAAAAAAAu) +
              2u * (uint32_t)__popc(w & 0xCCCCCCCCu) + 4u * (uint32_t)__popc(w & 0xF0F0F0F0u) +
              8u * (uint32_t)__popc(w & 0xFF00FF00u) + 16u * (uint32_t)__popc(w & 0xFFFF0000u);
    }
    const uint32_t wsum = __reduce_add_sync(kFull, osum);  // < 2^25 per warp
    if (lane == 0) s_chk[warp][1] = wsum;
  }
  __syncthreads();

  // ---- write-out: destination-aligned quads
  const uint64_t obase = src.base + (uint64_t)g * kGroupRecords;
  const uint64_t sbase = p.stats_base + (uint64_t)g * kGroupRecords;
  const uint64_t pos_base = start - sh;  // multiple of 4
  const uint32_t n_stage = sh + cnt;
  unsigned long long cx = 0;
  // any quad, entry by entry: the ragged first / last quad of the group, the end of a short buffer
  auto write_ragged = [&](uint32_t j) {
    const uint2 o2 = *reinterpret_cast<const uint2*>(&s_off[4u * j]);
    const uint32_t a4 = *reinterpret_cast<const uint32_t*>(&s_act[4u * j]);
    const uint32_t off[4] = {o2.x & 0xFFFFu, o2.x >> 16, o2.y & 0xFFFFu, o2.y >> 16};
    const uint64_t pos0 = pos_base + 4ull * j;
    const uint32_t k_lo = j == 0 ? sh : 0u;
    const uint32_t k_hi = n_stage - 4u * j < 4u ? n_stage - 4u * j : 4u;
#pragma unroll
    for (uint32_t k = 0; k < 4; ++k) {
      if (k < k_lo || k >= k_hi) continue;
      if (stats) cx ^= sbase + off[k];
      const uint64_t pos = pos0 + k;
      if (pos >= p.cap) continue;
      if (p.idx_bytes == 4) reinterpret_cast<uint32_t*>(p.out_idx)[pos] = (uint32_t)(obase + off[k]);
      else reinterpret_cast<uint64_t*>(p.out_idx)[pos] = obase + off[k];
      p.out_act[pos] = (uint8_t)(a4 >> (8 * k));
    }
  };
  // Interior quads [q_lo, q_hi): all four slots belong to this group and fit the caller's buffer — no
  // per-entry predicates (they were two thirds of this loop's 71 instructions per quad).  The index
  // checksum runs on the low words: a group's indices share their high word unless the group straddles
  // a multiple of 2^32 (then every quad takes the entry-by-entry form), and four equal high words cancel.
  const uint32_t q_lo = sh ? 1u : 0u;
  uint32_t q_hi = n_stage >> 2;
  {
    const uint64_t cap_q = p.cap >> 2, base_q = pos_base >> 2;
    const uint64_t room = cap_q > base_q ? cap_q - base_q : 0;
    if (room < q_hi) q_hi = (uint32_t)room;
    if ((uint32_t)sbase > 0xFFFFFFFFu - kGroupRecords) q_hi = q_lo;  // (uniform per CTA)
    if (q_hi < q_lo) q_hi = q_lo;
  }
  const uint32_t n_quads = (n_stage + 3u) >> 2;
  if (q_lo && (uint32_t)tid == 0u) write_ragged(0);
  for (uint32_t j = q_hi + (uint32_t)tid; j < n_quads; j += blockDim.x) write_ragged(j);
  {
    const uint32_t b32 = (uint32_t)obase, s32 = (uint32_t)sbase;
    uint32_t cx32 = 0;
    for (uint32_t j = q_lo + (uint32_t)tid; j < q_hi; j += blockDim.x) {
      const uint2 o2 = *reinterpret_cast<const uint2*>(&s_off[4u * j]);
      const uint32_t a4 = *reinterpret_cast<const uint32_t*>(&s_act[4u * j]);
      const uint32_t o0 = o2.x & 0xFFFFu, o1 = o2.x >> 16, o2_ = o2.y & 0xFFFFu, o3 = o2.y >> 16;
      const uint64_t q = (pos_base >> 2) + j;
      if (p.idx_bytes == 4) {
        reinterpret_cast<uint4*>(p.out_idx)[q] = make_uint4(b32 + o0, b32 + o1, b32 + o2_, b32 + o3);
      } else {
        ulonglong2* d = reinterpret_cast<ulonglong2*>(p.out_idx) + 2 * q;
        d[0] = make_ulonglong2(obase + o0, obase + o1);
        d[1] = make_ulonglong2(obase + o2_, obase + o3);
      }
      reinterpret_cast<uint32_t*>(p.out_act)[q] = a4;
      cx32 ^= (s32 + o0) ^ (s32 + o1) ^ (s32 + o2_) ^ (s32 + o3);
    }
    if (stats) cx ^= (unsigned long long)cx32;
  }
  // statistics: warp -> CTA -> global RED
  if (stats) {
    const uint32_t xl = __reduce_xor_sync(kFull, (uint32_t)cx), xh = __reduce_xor_sync(kFull, (uint32_t)(cx >> 32));
    if (lane == 0) s_chk[warp][0] = ((unsigned long long)xh << 32) | xl;
    __syncthreads();
    if (tid < 8) {
      uint32_t v = 0, n_exc = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) v += s_cnt[k][tid];
#pragma unroll
      for (int k = 0; k < 8; ++k) n_exc += s_nx[k];
      if (tid == 0) v += cnt - n_exc;  // every default entry is a bare SUBMIT_HC
      if (v) atomicAdd(&p.acc[2 + tid], (unsigned long long)v);
    }
    if (tid == 8) {
      unsigned long long x = 0, t = 0;
#pragma unroll
      for (int k = 0; k < 4; ++k) { x ^= s_chk[k][0]; t += s_chk[k][1]; }
      atomicXor(&p.acc[14], x);
      atomicAdd(&p.acc[15], t + (unsigned long long)cnt * sbase);
    }
  }
}

// One warp, after the kernel boundary that completes every expand CTA's REDs: publish the
// tick's am_tick_stats_t (device or mapped-host memory) and re-arm the accumulators.
__global__ void publish_kernel(unsigned long long* acc, am_tick_stats_t* out_stats, uint64_t n_records) {
  const int k = threadIdx.x;
  if (k >= kNumAcc) return;
  pdl_wait();
  unsigned long long v = acc[k];
  acc[k] = 0;
  if (k == 0) v = n_records;
  if (out_stats) reinterpret_cast<unsigned long long*>(out_stats)[k] = v;
}

// ---- small maintenance kernels (create / read) -----------------------------
__global__ void fill_u32_kernel(uint32_t* p, uint32_t v, uint64_t n) {
  uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

// RepeatAfterSec as the reference derives it at reconcile time (hcc.go:259-262):
// for a 5-field schedule Next(T) - T (robfig SpecSchedule.Next, cron_next_utc), for
// "@every d" and interval checks the stored interval, 0 for everything else.  One
// thread per record; the day scan diverges, which is fine for an on-demand query
// (status display, timer-wheel bucketing) that is not part of the per-tick path.
__global__ void next_fire_kernel(DevCols c, uint32_t first, uint32_t n, int64_t T, int64_t* out) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t i = first + k;
  const uint32_t f = c.flags[i];
  const uint32_t kind = f & AM_KIND_MASK;
  int64_t v = 0;
  if (!(f & AM_F_TOMBSTONE)) {
    if (kind == AM_KIND_CRON_SPEC && (f >> AM_F_TZ_SHIFT) != 0)
      v = -1;  // bound to a named time zone: the host evaluates Next() (am_cron_next), marked here
    else if (kind == AM_KIND_CRON_SPEC)
      v = repeat_after_from_next(cron_next_utc(c.minute[i], c.hour[i], c.dom[i], c.month[i], c.dow[i], T), T);
    else if (kind == AM_KIND_INTERVAL || kind == AM_KIND_CRON_EVERY)
      v = c.ras[i];
  }
  out[k] = v;
}

// The earliest second after T at which a tick of this shard would emit anything, given the state
// as it is (no further upserts / results): the wake-up time of the reference's earliest timer
// (time.AfterFunc, hcc.go:751) or cron activation (hcc.go:262) — the 1 Hz ticker may sleep until
// then.  Pending results, an unreported "Stopped" and parse errors (requeued after 1 s, hcc.go:204)
// are due at once.  Grid-stride, one record per thread and step; lane -> warp (shuffles) -> global
// atomicMin on a biased unsigned key.
__global__ void next_due_kernel(DevCols c, uint64_t n, int64_t T, unsigned long long* out_biased) {
  unsigned long long best = ~0ull;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
    const uint32_t f = c.flags[i];
    const uint32_t kind = f & AM_KIND_MASK;
    if (!evaluated(f)) continue;
    int64_t due = INT64_MAX;
    if ((f & (AM_F_PENDING_OK | AM_F_PENDING_FAIL | AM_F_REMEDY_PENDING)) || kind == AM_KIND_PARSE_ERROR ||
        (kind == AM_KIND_STOPPED && !(f & AM_F_STOPPED_REPORTED))) {
      due = T + 1;
    } else if (kind == AM_KIND_INTERVAL || kind == AM_KIND_CRON_EVERY) {
      const int64_t at = (int64_t)((uint64_t)c.finished_at[i] + (uint64_t)(int64_t)c.ras[i]);
      due = ((f & AM_F_TIMER_ARMED) && at > T + 1) ? at : T + 1;
    } else if (kind == AM_KIND_CRON_SPEC && (f >> AM_F_TZ_SHIFT) != 0) {
      due = T + 60 - ((T % 60) + 60) % 60;  // zone-bound: not before the next whole minute (a safe lower bound)
    } else if (kind == AM_KIND_CRON_SPEC) {
      const int64_t nx = cron_next_utc(c.minute[i], c.hour[i], c.dom[i], c.month[i], c.dow[i], T);
      if (nx != kNoNextFire) due = nx;
    }
    const unsigned long long key = (unsigned long long)due ^ (1ull << 63);  // order-preserving bias
    best = key < best ? key : best;
  }
#pragma unroll
  for (int d = 16; d; d >>= 1) {
    const unsigned long long o = __shfl_xor_sync(kFull, best, d);
    best = o < best ? o : best;
  }
  if ((threadIdx.x & 31) == 0 && best != ~0ull) atomicMin(out_biased, best);
}

// ---- staged controller events (upsert / remove / post_result) ---------------
// Events reach the library from many goroutines between two ticks; per slot
// they must take effect in call order.  An event's tick-local sequence number
// is its position in the staged arrays (1-based).  mark: atomicMax of the sequence into
// the slot's mark triple {latest upsert/remove, latest workflow phase, latest remedy
// phase}; apply: only the marked winners write — the latest upsert/remove, then the latest
// workflow phase and the latest remedy phase if they were posted after it (an older
// result belongs to the replaced CR).  The two phases are tracked independently: the
// reference observes them in separate watch loops (hcc.go:607-756 and :788-852), so a
// "Failed" and a remedy "Succeeded" posted by two calls before one tick must both
// survive.  clear: marks back to zero.  No host-side hashing or sorting.
// A staged op is a uint2 (slot, arg): arg = kind in the top 2 bits; low 30 bits: record index
// (upsert) or flag bits (result).
constexpr uint32_t kOpUpsert = 0u << 30, kOpRemove = 1u << 30, kOpResult = 2u << 30, kOpKindMask = 3u << 30;
constexpr uint32_t kHcBits = AM_F_PENDING_OK | AM_F_PENDING_FAIL;
constexpr uint32_t kRemedyBits = AM_F_REMEDY_PENDING | AM_F_REMEDY_OUTCOME_OK;

__global__ void mark_ops_kernel(uint32_t* marks, const uint2* __restrict__ ops, uint32_t n) {
  pdl_wait();  // (launched with programmatic stream serialisation: nothing of the predecessor is touched before this)
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint2 op = ops[k];
  const uint32_t i = op.x, arg = op.y;
  if ((arg & kOpKindMask) != kOpResult) { atomicMax(&marks[3u * i], k + 1u); return; }
  if (arg & kHcBits) atomicMax(&marks[3u * i + 1u], k + 1u);
  if (arg & AM_F_REMEDY_PENDING) atomicMax(&marks[3u * i + 2u], k + 1u);
}

// upserts (hcc.go:170-188 Reconcile) and removes (hcc.go:175-186)
__global__ void apply_state_ops_kernel(DevCols c, const uint32_t* __restrict__ marks, const uint2* __restrict__ ops,
                                       const am_record_t* __restrict__ recs, uint32_t n) {
  pdl_wait();  // (launched with programmatic stream serialisation: nothing of the predecessor is touched before this)
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint2 op = ops[k];
  const uint32_t i = op.x, arg = op.y;
  const uint32_t kind = arg & kOpKindMask;
  if (kind == kOpResult || marks[3u * i] != k + 1u) return;
  if (kind == kOpRemove) { c.flags[i] = AM_F_TOMBSTONE; return; }
  const am_record_t r = recs[arg & ~kOpKindMask];
#define AM_STORE(name) c.name[i] = r.name;
  AM_RECORD_COLUMNS(AM_STORE)
#undef AM_STORE
}

// terminal phases observed by the watch loops (hcc.go:635/:662/:821/:836).  The winner of
// the workflow phase and the winner of the remedy phase may be two different ops of the
// same slot: each rewrites only its own bit group, atomically.
__global__ void apply_result_ops_kernel(uint32_t* flags, const uint32_t* __restrict__ marks, const uint2* __restrict__ ops,
                                        uint32_t n) {
  pdl_wait();  // (launched with programmatic stream serialisation: nothing of the predecessor is touched before this)
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint2 op = ops[k];
  const uint32_t i = op.x, arg = op.y;
  if ((arg & kOpKindMask) != kOpResult) return;
  const uint32_t s = marks[3u * i];
  if (k + 1u < s) return;  // posted before the slot's latest upsert / remove
  uint32_t clr = 0, set = 0;
  if ((arg & kHcBits) && marks[3u * i + 1u] == k + 1u) { clr |= kHcBits; set |= arg & kHcBits; }
  if ((arg & AM_F_REMEDY_PENDING) && marks[3u * i + 2u] == k + 1u) { clr |= kRemedyBits; set |= arg & kRemedyBits; }
  if (clr) {
    atomicAnd(&flags[i], ~clr);
    atomicOr(&flags[i], set);
  }
}

// Results posted between two ticks, applied while the tick drains them instead of inside its sweep.
// In the sweep a record with a posted result costs its warp a second, dependent memory round trip
// (the remedy / counter columns) behind the streaming loads; with a result on ~2 % of the records
// nine warps in ten pay it and the tick's sweep slows from 84 to 143 us at 10 M records
// (profiles/r02_e2e_breakdown.json).  Here every result is its own thread: the slot's owner (see below)
// merges the posted bits into the flags, gathers the state columns its case needs, runs the same
// apply_result and scatters what changed — this kernel REPLACES apply_result_ops_kernel for such a drain.  The action bits go
// into the flags' carry bits for the sweep of the SAME tick to emit (it clears them); the finishedAt /
// timer-armed state it leaves is exactly what the sweep's own step 1 would have decided on.  Only the
// tick's drain does this (T is the tick's second) and only when results are sparse; a read drains
// without it, and a dense batch is cheaper as the sweep's streaming path.
__global__ void apply_results_now_kernel(DevCols c, const uint32_t* __restrict__ marks, const uint2* __restrict__ ops, uint32_t n,
                                         int64_t T, unsigned long long* acc) {
  pdl_wait();  // (launched with programmatic stream serialisation: nothing of the predecessor is touched before this)
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  constexpr uint32_t kPend = AM_F_PENDING_OK | AM_F_PENDING_FAIL | AM_F_REMEDY_PENDING;
  uint32_t res = 0;
  uint2 op = make_uint2(0u, 0u);
  if (k < n) op = ops[k];
  if (k < n && (op.y & kOpKindMask) == kOpResult) {
    const uint32_t i = op.x, arg = op.y;
    const uint32_t s_state = marks[3u * i], hcw = marks[3u * i + 1u], rmw = marks[3u * i + 2u];
    // The winners of the slot's two phase groups (apply_result_ops_kernel's rule: the latest op of a group, if
    // it was posted after the slot's latest upsert / remove) may be two different ops; ONE thread owns the
    // slot here — the workflow-phase winner, else the remedy-phase winner — and takes the other group's
    // bits from that op, so the flags are read and written once, without atomics.
    const bool hc_valid = hcw != 0u && hcw >= s_state, rm_valid = rmw != 0u && rmw >= s_state;
    const bool mine_hc = hc_valid && hcw == k + 1u, mine_rm = rm_valid && rmw == k + 1u;
    if (mine_hc || (mine_rm && !hc_valid)) {
      uint32_t f = c.flags[i];
      if (mine_hc) f = (f & ~kHcBits) | (arg & kHcBits);
      if (rm_valid) f = (f & ~kRemedyBits) | ((mine_rm ? arg : ops[rmw - 1u].y) & kRemedyBits);
      if (!evaluated(f) || !(f & kPend)) {
        c.flags[i] = f;  // (a record the sweep does not evaluate keeps its posted result)
      } else {
        // Gather only what this result can touch (every column is its own 32-B sector of a random record):
        // a "Succeeded" on a check without remedy reads its success counter and nothing else — two gathers
        // instead of ten; with all ten the kernel took as long (56 us for 0.18 M results) as the sweep's own
        // sparse path it replaces.  What apply_result reads, by case (hcc.go:635-724, :821-851):
        //   Succeeded: SuccessCount;            with a remedy workflow: RemedyTotalRuns (reset on pass)
        //   Failed:    FailedCount;             with a remedy workflow: the gate (limit, reset interval, total, finishedAt)
        //   a remedy outcome (applied only behind a Failed that runs the remedy, or on its own): the remedy counters
        const bool r_ok = (f & AM_F_PENDING_OK) != 0, r_fail = !r_ok && (f & AM_F_PENDING_FAIL) != 0;
        const bool remedy_state = ((r_ok || r_fail) && (f & AM_F_HAS_REMEDY)) || (!r_ok && !r_fail);
        RecState s{};
        s.flags = f;  // (finishedAt is only ever overwritten with T by a workflow result: not read)
        if (r_ok) s.s = c.success[i];
        if (r_fail) s.f = c.failed[i];
        if (remedy_state) {
          s.rs = c.remedy_success[i]; s.rf = c.remedy_failed[i]; s.rt = c.remedy_total[i];
          s.rfa = c.remedy_finished_at[i]; s.limit = c.runs_limit[i]; s.reset = c.reset_interval[i];
        }
        const RecState b = s;
        const uint32_t a = apply_result(s, T, res);
        if (r_ok || r_fail) c.finished_at[i] = s.fa;
        if (s.s != b.s) c.success[i] = s.s;
        if (s.f != b.f) c.failed[i] = s.f;
        if (s.rs != b.rs) c.remedy_success[i] = s.rs;
        if (s.rf != b.rf) c.remedy_failed[i] = s.rf;
        if (s.rt != b.rt) c.remedy_total[i] = s.rt;
        if (s.rfa != b.rfa) c.remedy_finished_at[i] = s.rfa;
        c.flags[i] = s.flags | carry_of_actions(a);  // pending bits cleared, timer armed, action bits for this tick's sweep
      }
    }
  }
  // results applied: warp -> global RED, as the sweep does per tile
  const int lane = threadIdx.x & 31;
  const uint32_t v = warp_result_counts(res, lane);
  if (v) atomicAdd(&acc[10 + lane], (unsigned long long)v);
}

__global__ void clear_marks_kernel(uint32_t* marks, const uint2* __restrict__ ops, uint32_t n) {
  pdl_wait();  // (launched with programmatic stream serialisation: nothing of the predecessor is touched before this)
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t i = ops[k].x;
  marks[3u * i] = 0;
  marks[3u * i + 1u] = 0;
  marks[3u * i + 2u] = 0;
}

__global__ void gather_records_kernel(DevCols c, const uint32_t* __restrict__ idx, am_record_t* out,
                                      uint32_t n) {
  uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t i = idx[k];
  am_record_t r;
#define AM_LOAD(name) r.name = c.name[i];
  AM_RECORD_COLUMNS(AM_LOAD)
#undef AM_LOAD
  r.reserved = 0;
  out[k] = r;
}

}  // namespace amsweep

#include "sweep_block.cuh"
