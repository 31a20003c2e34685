// sweep_block.cuh — K consecutive one-second ticks per pass over the columns ("temporal blocking",
// SURVEY §7 step 9; the timer-wheel reading of §8f-1 / hcc.go:751).
//
// am_sweep_run_ticks streams seconds back to back (BASELINE config 5: one simulated day = 86 400 ticks).
// With one sweep per tick every tick re-reads 16..56 B per record to find the ~4 % that are due.  But
// nothing reaches a record from outside between the ticks of such a run, so its whole future inside a
// block of K ticks (96 by default) follows from its own columns: this kernel loads a record ONCE, then steps it from
// event to event in registers — the reference's own shape, a timer per HealthCheck (time.AfterFunc,
// hcc.go:751) instead of a scan per second:
//
//   interval / "@every" check   next event = finishedAt + repeatAfterSec (hcc.go:264), every tick while no
//                               timer is armed (controller restart, hcc.go:161)
//   5-field cron                next event = the next tick whose LOCAL second is 0 (robfig activates on
//                               the minute; the zone's offset decides which UTC second that is)
//   parse error                 every tick (hcc.go:254-257: warning + requeue)
//   stopped                     once (hcc.go:238-250)
//   posted result / carry bits  the first tick of the block
//
// and at an event tick evaluates EXACTLY what sweep_tick_kernel evaluates for that (record, tick) —
// the same ladder, and the same helpers of sweep_kernels.cuh for the rest: evaluated, apply_result,
// complete_closed_loop — so the per-tick statistics and the
// columns after the block are bit-identical to K single ticks (tests: run_ticks blocked == unblocked ==
// oracle).  Work is O(events), not O(records x ticks); the columns are read and written once per K
// ticks.  Reported separately from the K = 1 roofline number.
//
// am_sweep_run_ticks wants per-tick statistics only (am_tick_stats_t): sweep_block_kernel<CLOSED, false>.
// am_sweep_run_ticks_view also wants every tick's (index, action) list: sweep_block_kernel<CLOSED, true>
// additionally leaves, per tick of the block, exactly what sweep_tick_kernel leaves for one tick — an
// emitted bitmap, per-group counts and per-tile exception segments (TickOut) — in slot t of a TickRing.
// ring_scan_kernel turns the counts into offsets for all K slots at once, and the unchanged expand_kernel
// rebuilds up to 16 ticks' lists per launch (its "ranks" are the ticks; its output, their concatenation).
#pragma once

#include <type_traits>

namespace amsweep {

constexpr int kMaxBlockTicks = 128;
constexpr int kDefaultBlockTicks = 96;  // 16.0 us per tick; 64: 18.1, 128: 17.3 (tools/r02_run17.sh, 10 M records, config 5)
constexpr int kBlockThreads = 128;
// Occupancy is what this kernel wants: its warps wait on each other (per-class lists of different lengths, one
// barrier before the flush) and on shared atomics.  256 threads at 94 registers = 2 CTAs per SM: 27.3 us per tick,
// 52 % of the stall samples at the final barrier.  128 threads: 23.2.  128 threads capped at 64 registers (8 CTAs per
// SM, 4 bytes of spills): 18.0; the same at 256 threads / 4 CTAs: 16.8.  (tools/r02_run15.sh .. r02_run17.sh)
constexpr int kBlockMinCtas = 8;
constexpr int kBlockRecords = 4 * kBlockThreads;  // four consecutive records per thread in the classification pass
constexpr int kBlockClasses = 4;                  // by expected number of events in the block: <= 2, <= 8, <= 24, more
constexpr int kBlockWords = kBlockRecords / 32;   // emitted-bitmap words of one CTA per tick
static_assert(kTile == 2 * kBlockRecords && kGroupRecords % kBlockRecords == 0, "a tile is two block CTAs");

// K TickOut slots back to back, one per tick of a block (am_sweep_run_ticks_view with AM_SWEEP_BLOCKED).
// Slot t of each array starts at t * (its per-slot stride); the strides are those of the handle's
// capacity, so every slot has the layout expand_kernel reads.
struct TickRing {
  TickOut base;           // slot 0
  uint64_t bitmap_words;  // per-slot strides, in u32 elements: n_groups * 256
  uint64_t groups;        // group_count; group_prefix has groups + 1 per slot
  uint64_t tiles;         // tile_exc
  uint64_t exc_words;     // exc_seg: tiles * 1024
};

struct BlockParams {
  DevCols c;
  uint64_t n_records, shard_base, seed;
  int64_t T0;                  // first tick of the block
  uint32_t K;                  // ticks in the block, <= kMaxBlockTicks
  const int32_t* tz_off;       // per-zone UTC offsets valid for the whole block (NULL: no zone registered)
  unsigned long long* stats;   // K rows of 16 accumulators (am_tick_stats_t layout), zero on entry
  TickRing ring;               // sweep_block_kernel<., true> only: tile_exc and group_count zero on entry
};

// first tick index u > t at which the LOCAL second (UTC + off) is 0
__device__ __forceinline__ int64_t next_local_minute(int64_t T0, int64_t t, int32_t off) {
  int64_t m = (T0 + t + 1 + (int64_t)off) % 60;
  if (m < 0) m += 60;
  return t + 1 + (m ? 60 - m : 0);
}

// Per-CTA statistics of a block of ticks, in shared memory.
struct BlockStats {
  uint32_t cnt[kMaxBlockTicks][13];   // [0] emitted, [1..8] action bits, [9..12] results applied
  uint32_t sum[kMaxBlockTicks];       // sum of CTA-local offsets of the emitted records
  uint32_t x[kMaxBlockTicks][2];      // xor of the emitted global indices
  // records that emit the same bare action on EVERY tick from some tick on (a parse error: hcc.go:254-257
  // warns on every pass; an open-loop check that stays due): registered once, as a delta at their first
  // such tick, and integrated over the ticks when the CTA flushes.  [.][0] = SUBMIT_HC, [.][1] = PARSE_ERROR
  uint32_t c_cnt[kMaxBlockTicks][2], c_sum[kMaxBlockTicks][2], c_x[kMaxBlockTicks][2][2];
  uint16_t list[kBlockClasses][kBlockRecords];  // records with events, by class
  uint32_t n_list[kBlockClasses];
};

// What the lists add: 8 768 B (static shared memory 25 168 B instead of 16 400; with the 1 KB reserved per CTA,
// 26 192 B instead of 17 424: still 8 CTAs per SM).  Still 64 registers; the spills grow to 16 B (closed loop)
// and 28 B stored / 60 B loaded (open loop), from 4 and 12 B without the lists (ptxas, CUDA 12.9).
struct BlockLists {
  uint32_t emit[kMaxBlockTicks][kBlockWords];  // records of the CTA with an event action at tick t
  uint32_t c_parse[kBlockWords];               // constant emitter of PARSE_ERROR (else of SUBMIT_HC)
  uint8_t c_from[kBlockRecords];               // first tick of the record's constant action; 0xFF: none
};
struct BlockStatsLists : BlockStats {
  BlockLists lists;
};

// (record loc of the CTA at cta_base, tick t) emits `act`, which is not a bare SUBMIT_HC: an entry of
// the tile's exception segment in slot t.  Two CTAs share a tile; expand_kernel finds an entry's place
// from its offset, so their order within the segment does not matter.
__device__ __forceinline__ void ring_exception(const TickRing& r, int64_t t, uint64_t cta_base, uint32_t loc, uint32_t act) {
  const uint64_t tile = cta_base / kTile;
  const uint32_t off = (uint32_t)(cta_base % kTile) + loc;
  const uint32_t pos = atomicAdd(r.base.tile_exc + (uint64_t)t * r.tiles + tile, 1u);
  r.base.exc_seg[(uint64_t)t * r.exc_words + tile * kTile + pos] = (off << 8) | act;
}

template <bool LISTS = false>
__device__ __forceinline__ void block_constant(BlockStats& S, int which, int64_t t_from, int64_t K, uint64_t g, uint32_t loc,
                                               BlockLists* L = nullptr) {
  if (t_from >= K) return;
  atomicAdd(&S.c_cnt[t_from][which], 1u);
  atomicAdd(&S.c_sum[t_from][which], loc);
  atomicXor(&S.c_x[t_from][which][0], (uint32_t)g);
  atomicXor(&S.c_x[t_from][which][1], (uint32_t)(g >> 32));
  if constexpr (LISTS) {  // (a record becomes a constant emitter at most once)
    L->c_from[loc] = (uint8_t)t_from;
    if (which) atomicOr(&L->c_parse[loc >> 5], 1u << (loc & 31u));
  }
}

// One record through the block, event by event (see the header of this file).
template <bool CLOSED, bool LISTS = false>
__device__ __forceinline__ void block_record(const BlockParams& p, BlockStats& S, uint64_t cta_base, uint32_t loc,
                                             BlockLists* L = nullptr) {
  constexpr uint32_t kPend = AM_F_PENDING_OK | AM_F_PENDING_FAIL | AM_F_REMEDY_PENDING;
  const int64_t K = (int64_t)p.K;
  const uint64_t i = cta_base + loc;
  const uint64_t g = p.shard_base + i;
  uint32_t f = ld_stream(p.c.flags + i);
  const int32_t rasv = ld_stream(p.c.ras + i);
  int64_t fa = ld_stream(p.c.finished_at + i);
  const uint32_t kind = f & AM_KIND_MASK;
  const bool is_iv = ((0x14u >> kind) & 1u) != 0;  // INTERVAL or CRON_EVERY
  const bool is_cron = kind == AM_KIND_CRON_SPEC;
  int32_t zoff = 0;
  uint64_t mi = 0, hr = 0, dm = 0, mo = 0, dw = 0;
  if (is_cron) {
    const uint32_t tz = f >> AM_F_TZ_SHIFT;
    if (tz && p.tz_off) zoff = p.tz_off[tz];
    mi = ld_stream(p.c.minute + i); hr = ld_stream(p.c.hour + i); dm = ld_stream(p.c.dom + i);
    mo = ld_stream(p.c.month + i); dw = ld_stream(p.c.dow + i);
  }
  // remedy / counter state: every due record needs it in closed loop, a posted result in open loop
  RecState s{};
  const bool with_state = CLOSED || (f & kPend) != 0;
  if (with_state) {
    s.limit = ld_stream(p.c.runs_limit + i); s.reset = ld_stream(p.c.reset_interval + i);
    s.s = ld_stream(p.c.success + i); s.f = ld_stream(p.c.failed + i);
    s.rs = ld_stream(p.c.remedy_success + i); s.rf = ld_stream(p.c.remedy_failed + i);
    s.rt = ld_stream(p.c.remedy_total + i); s.rfa = ld_stream(p.c.remedy_finished_at + i);
  }
  const RecState s0 = s;
  const uint32_t f0 = f;
  const int64_t fa0 = fa;

  auto next_event = [&](int64_t t) -> int64_t {  // the first tick index > t at which this record can act
    if (kind == AM_KIND_PARSE_ERROR) return t + 1;
    if (kind == AM_KIND_STOPPED) return (f & AM_F_STOPPED_REPORTED) ? K : t + 1;
    if (is_iv) {
      if (!(f & AM_F_TIMER_ARMED)) return t + 1;  // no timer: the reference submits on every pass
      const int64_t d = fa + (int64_t)rasv - p.T0;  // elapsed >= ras  <=>  tick index >= d
      return d > t + 1 ? d : t + 1;
    }
    return next_local_minute(p.T0, t, zoff);  // 5-field schedule
  };

  int64_t t = (f & (kPend | AM_F_CARRY_MASK)) ? 0 : next_event(-1);
  while (t < K) {
    const int64_t T = p.T0 + t;
    // ---- exactly sweep_tick_kernel's decision for (record, T) ----
    const bool has_result = (f & (AM_F_PENDING_OK | AM_F_PENDING_FAIL)) != 0;
    const bool pending = (f & kPend) != 0;
    const int64_t fa_eff = has_result ? T : fa;
    const int64_t elapsed = (int64_t)((uint64_t)T - (uint64_t)fa_eff);
    const bool armed = has_result || (f & AM_F_TIMER_ARMED) != 0;
    const bool due_iv = !((elapsed < (int64_t)rasv) & armed);
    bool due_cron = false;
    if (is_cron) {
      const TickWords w = tick_words_from_unix(T + (int64_t)zoff);
      due_cron = cron_matches(w, mi, hr, dm, mo, dw);
    }
    const bool due = is_iv ? due_iv : (is_cron && due_cron);
    const bool stopped_now = kind == AM_KIND_STOPPED && !(f & AM_F_STOPPED_REPORTED);
    uint32_t act = (due ? AM_ACT_SUBMIT_HC : 0u) | (stopped_now ? AM_ACT_STOPPED : 0u) |
                   (kind == AM_KIND_PARSE_ERROR ? AM_ACT_PARSE_ERROR : 0u);
    if (f & AM_F_CARRY_MASK) {
      act |= carried_actions(f);
      f &= ~AM_F_CARRY_MASK;
    }
    if (stopped_now) {  // hcc.go:238-250
      f |= AM_F_STOPPED_REPORTED;
      fa = T;
    }
    uint32_t res = 0;
    if (pending || (CLOSED && due)) {
      s.flags = f;
      s.fa = fa;
      uint32_t a = apply_result(s, T, res);
      if (CLOSED && due) a |= complete_closed_loop(s, p.seed, g, T, res);
      act |= a;
      f = s.flags;
      fa = s.fa;
    }
    // ---- this tick's statistics (what expand_kernel derives from the emitted list) ----
    if (act) {
      atomicAdd(&S.cnt[t][0], 1u);
      uint32_t bits = act;
      while (bits) {
        const int b = __ffs((int)bits) - 1;
        bits &= bits - 1u;
        atomicAdd(&S.cnt[t][1 + b], 1u);
      }
      atomicXor(&S.x[t][0], (uint32_t)g);
      atomicXor(&S.x[t][1], (uint32_t)(g >> 32));
      atomicAdd(&S.sum[t], loc);
      if constexpr (LISTS) {
        atomicOr(&L->emit[t][loc >> 5], 1u << (loc & 31u));
        if (act != AM_ACT_SUBMIT_HC) ring_exception(p.ring, t, cta_base, loc, act);
      }
    }
    if (res) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if ((res >> (8 * q)) & 0xFFu) atomicAdd(&S.cnt[t][9 + q], (res >> (8 * q)) & 0xFFu);
    }
    // from here on the same bare action on every tick, and nothing changes any more?
    if (kind == AM_KIND_PARSE_ERROR) { block_constant<LISTS>(S, 1, t + 1, K, g, loc, L); break; }
    if (!CLOSED && is_iv && due) { block_constant<LISTS>(S, 0, t + 1, K, g, loc, L); break; }  // stays due: nothing completes it in open loop
    t = next_event(t);
  }

  // ---- write back what changed ----
  if (f != f0) st_stream(p.c.flags + i, f);
  if (fa != fa0) st_stream(p.c.finished_at + i, fa);
  if (with_state) {
    if (s.s != s0.s) st_stream(p.c.success + i, s.s);
    if (s.f != s0.f) st_stream(p.c.failed + i, s.f);
    if (s.rs != s0.rs) st_stream(p.c.remedy_success + i, s.rs);
    if (s.rf != s0.rf) st_stream(p.c.remedy_failed + i, s.rf);
    if (s.rt != s0.rt) st_stream(p.c.remedy_total + i, s.rt);
    if (s.rfa != s0.rfa) st_stream(p.c.remedy_finished_at + i, s.rfa);
  }
}

template <bool CLOSED, bool LISTS = false>
__global__ void __launch_bounds__(kBlockThreads, kBlockMinCtas) sweep_block_kernel(const BlockParams p) {
  __shared__ typename std::conditional<LISTS, BlockStatsLists, BlockStats>::type S;
  BlockLists* L = nullptr;
  const int tid = threadIdx.x;
  {
    uint32_t* z = reinterpret_cast<uint32_t*>(&S);
    constexpr int kZero = (int)(offsetof(BlockStats, list) / 4);  // everything before the lists
    for (int k = tid; k < kZero; k += kBlockThreads) z[k] = 0;
    if (tid < kBlockClasses) S.n_list[tid] = 0;
  }
  if constexpr (LISTS) {
    L = &S.lists;
    for (uint32_t k = (uint32_t)tid; k < p.K * kBlockWords; k += kBlockThreads) (&L->emit[0][0])[k] = 0;
    if (tid < kBlockWords) L->c_parse[tid] = 0;
    reinterpret_cast<uint32_t*>(L->c_from)[tid] = 0xFFFFFFFFu;  // (kBlockRecords = 4 x kBlockThreads)
  }
  __syncthreads();

  const uint64_t cta_base = (uint64_t)blockIdx.x * kBlockRecords;
  const int64_t K = (int64_t)p.K;
  constexpr uint32_t kPend = AM_F_PENDING_OK | AM_F_PENDING_FAIL | AM_F_REMEDY_PENDING;

  // ---- pass 1: classify.  16 B per record (flags, repeatAfterSec, finishedAt), four records per thread.
  //      Records that cannot act inside the block — the majority: an armed timer that fires later — cost
  //      nothing more; records that emit the same action on every tick are registered as constants;
  //      the others go onto a list by their expected number of events, so that the lanes of a warp of
  //      pass 2 run loops of similar length (per-lane ownership ran at 4 of 32 lanes active: one
  //      "@every 500ms" check keeps its lane busy for 64 events while its neighbours have none).
  {
    const uint32_t loc0 = 4u * (uint32_t)tid;
    const uint64_t i0 = cta_base + loc0;  // columns are padded to whole tiles; slots past n_records are tombstones
    const uint4 f4 = ld_stream(reinterpret_cast<const uint4*>(p.c.flags + i0));
    const int4 r4 = ld_stream(reinterpret_cast<const int4*>(p.c.ras + i0));
    const longlong2 a01 = ld_stream(reinterpret_cast<const longlong2*>(p.c.finished_at + i0));
    const longlong2 a23 = ld_stream(reinterpret_cast<const longlong2*>(p.c.finished_at + i0 + 2));
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint32_t f = q == 0 ? f4.x : q == 1 ? f4.y : q == 2 ? f4.z : f4.w;
      const int32_t rasv = q == 0 ? r4.x : q == 1 ? r4.y : q == 2 ? r4.z : r4.w;
      const int64_t fa = q == 0 ? a01.x : q == 1 ? a01.y : q == 2 ? a23.x : a23.y;
      const uint32_t loc = loc0 + (uint32_t)q;
      const uint32_t kind = f & AM_KIND_MASK;
      if (!evaluated(f)) continue;
      const bool first_tick = (f & (kPend | AM_F_CARRY_MASK)) != 0;  // a posted result / carried action: an event at tick 0
      const uint64_t g = p.shard_base + cta_base + loc;
      int64_t n_ev = 0;  // expected events in the block (an upper bound is fine: it only picks the list)
      if (kind == AM_KIND_PARSE_ERROR) {
        if (!first_tick) { block_constant<LISTS>(S, 1, 0, K, g, loc, L); continue; }
        n_ev = 1;
      } else if (kind == AM_KIND_STOPPED) {
        n_ev = (first_tick || !(f & AM_F_STOPPED_REPORTED)) ? 1 : 0;
      } else if (kind == AM_KIND_CRON_SPEC) {
        int32_t zoff = 0;
        const uint32_t tz = f >> AM_F_TZ_SHIFT;
        if (tz && p.tz_off) zoff = p.tz_off[tz];
        const int64_t m0 = next_local_minute(p.T0, -1, zoff);
        n_ev = (first_tick ? 1 : 0) + (m0 < K ? 1 + (K - 1 - m0) / 60 : 0);
      } else {  // INTERVAL / CRON_EVERY
        const int64_t step = rasv > 0 ? (int64_t)rasv : 1;
        if (!(f & AM_F_TIMER_ARMED) || first_tick) {
          if (!CLOSED && !first_tick) { block_constant<LISTS>(S, 0, 0, K, g, loc, L); continue; }  // due on every tick, nothing changes
          n_ev = 1 + (K - 1) / step;
        } else {
          int64_t d = fa + (int64_t)rasv - p.T0;
          if (d < 0) d = 0;
          if (d >= K) continue;  // its timer fires after the block
          if (!CLOSED) { block_constant<LISTS>(S, 0, d, K, g, loc, L); continue; }  // due from tick d on
          n_ev = 1 + (K - 1 - d) / step;
        }
      }
      if (n_ev <= 0) continue;
      const int c = n_ev <= 2 ? 0 : (n_ev <= 8 ? 1 : (n_ev <= 24 ? 2 : 3));
      S.list[c][atomicAdd(&S.n_list[c], 1u)] = (uint16_t)loc;
    }
  }
  __syncthreads();
  // (Measured and dropped: a second kernel for the longest loops, run in full warps — slower, its lanes
  //  all sit on the same tick and collide on every shared atomic; grouping the lanes of a warp by tick
  //  with match.any + redux before the atomics, and 128-thread CTAs — slower still, 40 vs 27 us per tick:
  //  the collectives cost more than the conflicts they remove.  profiles/r02_summary.md.)

  // ---- pass 2: the listed records, longest loops first; the warps start at different places so that the
  //      (short) head of every list does not always land on warp 0
#pragma unroll 1
  for (int c = kBlockClasses - 1; c >= 0; --c) {
    const uint32_t n = S.n_list[c];
    for (uint32_t k = ((uint32_t)tid + (uint32_t)(kBlockThreads / 4) * (uint32_t)c) & (kBlockThreads - 1); k < n; k += kBlockThreads)
      block_record<CLOSED, LISTS>(p, S, cta_base, S.list[c][k], L);
  }
  __syncthreads();

  // ---- integrate the constant emitters over the ticks (thread t: everything registered at ticks <= t)
  for (int t = tid; t < (int)p.K; t += kBlockThreads) {
    uint32_t c0 = 0, c1 = 0, s0 = 0, s1 = 0, x0 = 0, x1 = 0;
    for (int u = 0; u <= t; ++u) {
      c0 += S.c_cnt[u][0]; c1 += S.c_cnt[u][1];
      s0 += S.c_sum[u][0]; s1 += S.c_sum[u][1];
      x0 ^= S.c_x[u][0][0] ^ S.c_x[u][1][0];
      x1 ^= S.c_x[u][0][1] ^ S.c_x[u][1][1];
    }
    S.cnt[t][0] += c0 + c1;
    S.cnt[t][1] += c0;      // AM_ACT_SUBMIT_HC   (bit 0)
    S.cnt[t][4] += c1;      // AM_ACT_PARSE_ERROR (bit 3)
    S.sum[t] += s0 + s1;
    S.x[t][0] ^= x0;
    S.x[t][1] ^= x1;
  }
  __syncthreads();

  // ---- CTA -> global: one RED per non-zero (tick, field) ----
  const unsigned long long gbase = (unsigned long long)(p.shard_base + cta_base);
  for (uint32_t k = (uint32_t)tid; k < p.K * 16u; k += kBlockThreads) {
    const uint32_t t = k >> 4, fld = k & 15u;
    unsigned long long* dst = p.stats + (size_t)t * kNumAcc + fld;
    if (fld >= 1 && fld <= 13) {
      const uint32_t v = S.cnt[t][fld - 1];
      if (v) atomicAdd(dst, (unsigned long long)v);
    } else if (fld == 14) {
      const unsigned long long x = ((unsigned long long)S.x[t][1] << 32) | S.x[t][0];
      if (x) atomicXor(dst, x);
    } else if (fld == 15) {
      const uint32_t cnt = S.cnt[t][0];
      if (cnt) atomicAdd(dst, (unsigned long long)cnt * gbase + S.sum[t]);
    }
  }

  if constexpr (LISTS) {
    // ---- the constant emitters join the bitmap of every tick from their first one on: warp w owns words
    //      w, w + 4, ... (one ballot per word and tick); a parse error is an exception on each of them
    const uint32_t lane = (uint32_t)tid & 31u;
    for (int w = tid >> 5; w < kBlockWords; w += kBlockThreads / 32) {
      const uint32_t loc = 32u * (uint32_t)w + lane;
      const uint32_t from = L->c_from[loc];
      const bool parse = ((L->c_parse[w] >> lane) & 1u) != 0;
      if (!__any_sync(kFull, from != 0xFFu)) continue;  // (warp-uniform)
      for (uint32_t t = 0; t < p.K; ++t) {
        const bool on = from <= t;
        const uint32_t m = __ballot_sync(kFull, on);
        if (lane == 0) L->emit[t][w] |= m;
        if (on && parse) ring_exception(p.ring, t, cta_base, loc, AM_ACT_PARSE_ERROR);
      }
    }
    __syncthreads();
    // ---- slot t: this CTA's 16 bitmap words (64 B), and its emitted count into the group's counter
    const uint64_t word0 = cta_base / 32, group = cta_base / kGroupRecords;
    for (uint32_t k = (uint32_t)tid; k < p.K * kBlockWords; k += kBlockThreads) {
      const uint32_t t = k / kBlockWords, w = k % kBlockWords;
      p.ring.base.bitmap[(uint64_t)t * p.ring.bitmap_words + word0 + w] = L->emit[t][w];
    }
    for (uint32_t t = (uint32_t)tid; t < p.K; t += kBlockThreads)
      if (S.cnt[t][0]) atomicAdd(p.ring.base.group_count + (uint64_t)t * p.ring.groups + group, S.cnt[t][0]);
  }
}

// Per-slot group offsets of a tick ring: one CTA per tick, the scan of scan_groups_kernel over that
// slot's group counts.  Re-arms the counts and writes each tick's total to totals[t] (mapped host
// memory: the host sizes its list buffer from them before expand_kernel runs).
constexpr int kRingScanThreads = 256;
__global__ void __launch_bounds__(kRingScanThreads) ring_scan_kernel(const TickRing r, uint32_t n_groups, uint32_t* totals) {
  __shared__ uint32_t s_warp[kRingScanThreads / 32];
  __shared__ uint32_t s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint64_t t = blockIdx.x;
  uint32_t* count = r.base.group_count + t * r.groups;
  uint32_t* prefix = r.base.group_prefix + t * (r.groups + 1);
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (uint32_t g0 = 0; g0 < n_groups; g0 += kRingScanThreads) {
    const uint32_t g = g0 + (uint32_t)tid;
    const uint32_t c = g < n_groups ? count[g] : 0u;
    uint32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t up = __shfl_up_sync(kFull, incl, d);
      if (lane >= d) incl += up;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    uint32_t before = s_carry;
    for (int k = 0; k < warp; ++k) before += s_warp[k];
    const uint32_t excl = before + incl - c;
    if (g < n_groups) {
      prefix[g] = excl;
      count[g] = 0;
    }
    __syncthreads();  // every thread has read s_carry / s_warp of this round
    if (tid == kRingScanThreads - 1) s_carry = excl + c;
    __syncthreads();
  }
  if (tid == 0) {
    prefix[n_groups] = s_carry;
    totals[t] = s_carry;
  }
}

}  // namespace amsweep
