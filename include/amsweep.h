/*
 * amsweep.h — C-ABI of libamsweep: the B200-native per-tick HealthCheck
 * schedule-evaluation sweep for keikoproj/active-monitor.
 *
 * This header is the drop-in boundary (SURVEY.md §8b).  Every entry point
 * names the reference decision it replaces; `hcc.go` abbreviates
 * internal/controllers/healthcheck_controller.go of the reference.
 *
 * Conventions (cgo-friendly):
 *   - plain C, fixed-width integers, flat arrays; no callbacks, no torch types;
 *   - every input is COPIED during the call, the library never retains caller
 *     memory; outputs go to caller-provided buffers (capacity passed in);
 *   - return value: 0 on success, negative AM_E_* on failure; never aborts,
 *     never throws across the boundary;
 *   - per-record anomalies are DATA (action bit AM_ACT_ANOMALY), not failures;
 *   - there is NO CPU fallback: without a CUDA device am_sweep_create fails
 *     with AM_E_DEVICE;
 *   - every am_sweep_* / am_gather_* call makes the handle's device the
 *     calling thread's current CUDA device (cudaSetDevice) and leaves it so.
 */
#ifndef AMSWEEP_H_
#define AMSWEEP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AMSWEEP_ABI_VERSION 2

/* ---- error codes ------------------------------------------------------- */
#define AM_OK 0
#define AM_E_INVAL (-1)       /* NULL pointer, bad argument                   */
#define AM_E_RANGE (-2)       /* value outside the HBM column's domain (N1)   */
#define AM_E_NOSPACE (-3)     /* caller buffer too small; needed size returned */
#define AM_E_DEVICE (-4)      /* CUDA failure; see am_last_error_detail       */
#define AM_E_NOMEM (-5)       /* host or device allocation failed             */
#define AM_E_PARSE (-6)       /* cron spec rejected (robfig error text in err) */
#define AM_E_UNSUPPORTED (-7) /* valid spec the device path does not evaluate
                                 (a 256th distinct CRON_TZ zone): keep it on
                                 the Go path                                  */
#define AM_E_BUSY (-8)        /* second concurrent am_sweep_tick on a handle  */

/* ---- cron (replaces cron.ParseStandard, hcc.go:253; robfig/cron v3.0.1) - */
#define AM_CRON_ERROR 0
#define AM_CRON_SPEC 1  /* SpecSchedule: five uint64 masks, bit 63 = starBit  */
#define AM_CRON_EVERY 2 /* ConstantDelaySchedule: delay_sec > 0               */

#define AM_STAR_BIT (1ull << 63)

typedef struct am_cron {
  uint64_t minute, hour, dom, month, dow; /* robfig SpecSchedule fields      */
  int64_t delay_sec;                      /* ConstantDelaySchedule.Delay / s  */
  int32_t kind;                           /* AM_CRON_*                        */
  int32_t tz_id;                          /* SpecSchedule.Location: 0 = time.Local ==
                                             UTC (distroless image, Dockerfile:25),
                                             else an am_tz_lookup id           */
} am_cron_t;

/* Parse `spec[0..len)` exactly as cron.ParseStandard does.  On a rejected
 * spec returns AM_E_PARSE, sets out->kind = AM_CRON_ERROR and writes the
 * robfig-style message (NUL-terminated, truncated to errcap) into err. */
int am_cron_parse(const char* spec, size_t len, am_cron_t* out, char* err, size_t errcap);

/* Named time zones.  robfig resolves a "TZ=" / "CRON_TZ=" prefix with time.LoadLocation and
 * evaluates the schedule in that zone (parser.go; call site hcc.go:253).  Here a zone is registered
 * once per process under a small id (1..255; "", "UTC" and "Local" are 0: the shipped image runs in
 * UTC) read from the system's TZif files ($ZONEINFO, /usr/share/zoneinfo, ...: Go's search path);
 * am_cron_parse does this by itself and returns the id in am_cron_t.tz_id; classify carries it in
 * the record's flags (AM_F_TZ_SHIFT); each tick evaluates such records against their zone's wall
 * clock on the device.  AM_E_PARSE: unknown zone (robfig: "provided bad location");
 * AM_E_UNSUPPORTED: more than 255 distinct zones in one process. */
int am_tz_lookup(const char* name, size_t len, int32_t* tz_id);
/* UTC offset, seconds east, of a registered zone at a UTC instant (0 for id 0). */
int am_tz_offset(int32_t tz_id, int64_t unix_sec, int32_t* utoff_out);

/* matches(T) of SURVEY Appendix A.7 for one schedule and one UTC second:
 * 1 if a SpecSchedule fires exactly at unix_sec, else 0 (host helper; the
 * device evaluates the same predicate inside the sweep kernel). */
int am_cron_matches(const am_cron_t* c, int64_t unix_sec);

/* Schedule.Next(t) for whole-second t (hcc.go:262): first activation strictly
 * after unix_sec, or INT64_MIN when none within five years (robfig returns the
 * zero time).  UTC only. */
int64_t am_cron_next(const am_cron_t* c, int64_t unix_sec);

/* RepeatAfterSec as hcc.go:262 derives it for a clock reading with a non-zero
 * nanosecond part (SURVEY B.4 N2): whole seconds from floor(now) to Next(now).
 * When Next() finds nothing (Go zero time) Sub saturates and the Go value is
 * int(minDuration/Second)+1 = -9223372035, returned as is. */
int64_t am_cron_repeat_after_sec(const am_cron_t* c, int64_t unix_sec);

/* ---- record schema (SURVEY Appendix B.1) -------------------------------- */
/* flags word */
#define AM_KIND_MASK 0x7u
#define AM_KIND_NO_RESOURCE 0u   /* Workflow.Resource == nil, hcc.go:227       */
#define AM_KIND_STOPPED 1u       /* ras<=0 && cron=="", hcc.go:238             */
#define AM_KIND_INTERVAL 2u      /* ras>0 (cron ignored), hcc.go:264           */
#define AM_KIND_CRON_SPEC 3u     /* ras<=0 && 5-field/descriptor, hcc.go:251   */
#define AM_KIND_CRON_EVERY 4u    /* ras<=0 && "@every d", hcc.go:251           */
#define AM_KIND_PARSE_ERROR 5u   /* ParseStandard error, hcc.go:254-257        */
#define AM_KIND_HOST_FALLBACK 6u /* AM_E_UNSUPPORTED specs (a 256th distinct time
                                    zone): not evaluated on the device          */
#define AM_F_HAS_REMEDY (1u << 3)        /* !RemedyWorkflow.IsEmpty()          */
#define AM_F_PENDING_OK (1u << 4)        /* workflow phase Succeeded posted    */
#define AM_F_PENDING_FAIL (1u << 5)      /* workflow phase Failed posted       */
#define AM_F_REMEDY_PENDING (1u << 6)    /* a remedy outcome is attached       */
#define AM_F_REMEDY_OUTCOME_OK (1u << 7) /* ... and it is Succeeded            */
#define AM_F_TOMBSTONE (1u << 8)         /* removed / never upserted           */
#define AM_F_STOPPED_REPORTED (1u << 9)  /* "Stopped" status already written   */
#define AM_F_TIMER_ARMED (1u << 10)      /* RepeatTimersByName holds a timer for the
                                            check (hcc.go:264 "&& timer != nil";
                                            armed by hcc.go:745-752 after a result) */
#define AM_F_CARRY_SHIFT 11              /* bits 11..15: library-internal.  Action bits of a posted result the
                                          * library applied while draining the staged calls of a tick (before
                                          * that tick's sweep, which emits and clears them): never set in a
                                          * record a caller sees or supplies                                */
#define AM_F_CARRY_MASK (0x1Fu << AM_F_CARRY_SHIFT)
#define AM_F_TZ_SHIFT 24                 /* bits 24..31: time zone of a 5-field schedule
                                            ("CRON_TZ=Zone ..."), 0 = UTC; am_tz_lookup   */
#define AM_F_TZ_MASK (0xFFu << AM_F_TZ_SHIFT)
#define AM_F_FAILP_SHIFT 16              /* closed-loop harness: P(fail)*256   */
#define AM_F_FAILP_MASK (0xFFu << AM_F_FAILP_SHIFT)

/* action byte emitted per record per tick (0 = nothing to do) */
#define AM_ACT_SUBMIT_HC 0x01u         /* hcc.go:269-288 submit the workflow   */
#define AM_ACT_RUN_REMEDY 0x02u        /* hcc.go:683/705/714 processRemedy     */
#define AM_ACT_STOPPED 0x04u           /* hcc.go:238-250 write status Stopped  */
#define AM_ACT_PARSE_ERROR 0x08u       /* hcc.go:254-257 warning event+requeue */
#define AM_ACT_REMEDY_SKIP 0x10u       /* hcc.go:692-693                       */
#define AM_ACT_RESET_ON_PASS 0x20u     /* hcc.go:649-660                       */
#define AM_ACT_RESET_ON_INTERVAL 0x40u /* hcc.go:695-704                       */
#define AM_ACT_ANOMALY 0x80u           /* nil RemedyFinishedAt at hcc.go:690   */

/* One HealthCheck as the controller sees it (api/v1alpha1/healthcheck_types.go
 * :32-44 spec, :47-66 status); Go `int` is int64. */
typedef struct am_healthcheck {
  int64_t repeat_after_sec;      /* Spec.RepeatAfterSec                        */
  const char* cron;              /* Spec.Schedule.Cron (not NUL-terminated)    */
  size_t cron_len;               /* 0 == ""                                    */
  int32_t has_resource;          /* Spec.Workflow.Resource != nil              */
  int32_t has_remedy;            /* !Spec.RemedyWorkflow.IsEmpty()             */
  int64_t remedy_runs_limit;     /* Spec.RemedyRunsLimit                       */
  int64_t remedy_reset_interval; /* Spec.RemedyResetInterval                   */
  int64_t finished_at;           /* Status.FinishedAt.Unix()                   */
  int64_t remedy_finished_at;    /* Status.RemedyFinishedAt.Unix()             */
  int32_t finished_at_set;       /* Status.FinishedAt != nil                   */
  int32_t remedy_finished_at_set;
  int64_t success_count, failed_count;
  int64_t remedy_success_count, remedy_failed_count, remedy_total_runs;
  uint32_t fail_p8;              /* closed-loop harness only, 0..255           */
  uint32_t timer_armed;          /* r.GetTimerByName(name) != nil (hcc.go:264):
                                    0 after a controller restart (hcc.go:161 starts
                                    with an empty RepeatTimersByName), so the first
                                    evaluation submits whatever finishedAt says   */
} am_healthcheck_t;

/* One packed record = one element of each SoA column. */
typedef struct am_record {
  uint64_t minute, hour, dom, month, dow;
  int64_t finished_at;        /* nil => 0 (hcc.go:231-235)                     */
  int64_t remedy_finished_at; /* nil => 0 (nil-ness matters: N3)               */
  int32_t ras;                /* RepeatAfterSec | @every delay                 */
  uint32_t flags;
  int32_t runs_limit, reset_interval;
  int32_t success, failed, remedy_success, remedy_failed, remedy_total;
  int32_t reserved;
} am_record_t;

/* Ladder classification at upsert, in the order hcc.go:227 -> 238 -> 251 ->
 * 264 (SURVEY B.2).  Returns AM_OK, AM_E_RANGE (value does not fit the column,
 * N1) or AM_E_UNSUPPORTED (record gets AM_KIND_HOST_FALLBACK).  A cron parse
 * error is NOT a call failure: kind = AM_KIND_PARSE_ERROR, like the reference's
 * per-reconcile error. */
int am_healthcheck_classify(const am_healthcheck_t* hc, am_record_t* out);

/* The same ladder for n HealthChecks at once (SURVEY.md 8f-2, bulk ingest at
 * controller start: the informer's initial list replays every CR through
 * Reconcile, hcc.go:170).  Records are independent, so the batch is split
 * over n_threads host threads (<= 0: one per hardware thread).  rc_out[i]
 * (may be NULL) receives what am_healthcheck_classify returns for record i;
 * the call itself returns AM_OK, or AM_E_INVAL / AM_E_NOMEM.  *n_not_ok (may
 * be NULL) counts records whose rc is not AM_OK. */
int am_healthcheck_classify_batch(const am_healthcheck_t* hcs, uint64_t n, am_record_t* out,
                                  int32_t* rc_out, int n_threads, uint64_t* n_not_ok);

/* HealthCheck manifests as the API server serves them (JSON: one object, an array of objects, or a
 * List with "items") -> packed records, natively: one structural pass, then field extraction by the
 * JSON tags of api/v1alpha1/healthcheck_types.go:32-66 / :88-102 and the ladder, split over n_threads
 * host threads (<= 0: all).  For the informer's initial list at controller start (hcc.go:170) and for
 * restores from a dump.  `timer_armed` is applied to every record (0 after a restart, hcc.go:161).
 * out / rc_out (may be NULL) hold `cap` entries; *n_out = HealthChecks found; AM_E_NOSPACE when
 * cap is too small (nothing written), AM_E_PARSE when the document is not JSON of that shape.
 * rc_out[i]: what am_healthcheck_classify returned, or AM_E_PARSE for a malformed object / time. */
int am_healthcheck_ingest_json(const char* json, size_t len, uint32_t timer_armed, am_record_t* out,
                               int32_t* rc_out, uint64_t cap, uint64_t* n_out, int n_threads);

/* RemedyWorkflow.IsEmpty (api/v1alpha1/healthcheck_types.go:104-106):
 * reflect.DeepEqual against the zero value — note a non-nil empty rbacRules
 * slice is NOT empty. */
int am_remedy_is_empty(size_t generate_name_len, int resource_is_nil, int64_t timeout,
                       int rbac_rules_is_nil);

/* SoA view used by bulk load / upsert / read.  Any pointer may be NULL:
 * on input a NULL column means "all zero", on output "do not read". */
typedef struct am_record_cols {
  uint64_t *minute, *hour, *dom, *month, *dow;
  int32_t* ras;
  uint32_t* flags;
  int64_t* finished_at;
  int32_t *runs_limit, *reset_interval;
  int32_t *success, *failed, *remedy_success, *remedy_failed, *remedy_total;
  int64_t* remedy_finished_at;
} am_record_cols_t;

/* ---- the sweep ---------------------------------------------------------- */
typedef struct am_sweep am_sweep_t;

typedef struct am_tick_stats {
  uint64_t n_records;  /* slots swept (high-water mark of this shard)        */
  uint64_t n_emitted;  /* records with a non-zero action                      */
  uint64_t n_submit_hc, n_run_remedy, n_stopped, n_parse_error;
  uint64_t n_remedy_skip, n_reset_on_pass, n_reset_on_interval, n_anomaly;
  uint64_t n_result_ok, n_result_fail; /* feed metrics.MonitorSuccess/Error,
                                          collector.go:19-31 (workflow=healthCheck) */
  uint64_t n_remedy_ok, n_remedy_fail; /* same vectors, workflow=remedy        */
  uint64_t idx_xor, idx_sum;           /* checksum of emitted global indices   */
} am_tick_stats_t;

#define AM_SWEEP_CLOSED_LOOP 0x1u /* harness: a due record completes instantly
                                     with its preset outcome (SURVEY B.3)     */
#define AM_SWEEP_FULL_SCAN 0x2u   /* read every schedule column even on ticks
                                     where no 5-field cron can fire (sec!=0)  */
#define AM_SWEEP_BLOCKED 0x4u     /* am_sweep_run_ticks(_view) only: temporal blocking.  Blocks of consecutive
                                     ticks (96; AMSWEEP_BLOCK_TICKS, at most 128) are evaluated in one pass over the columns,
                                     every record stepped from event to event (its next repeat timer,
                                     hcc.go:751; its next cron minute) — per-tick statistics and the
                                     columns afterwards are identical to tick-by-tick evaluation.
                                     am_sweep_run_ticks returns statistics only; the per-tick lists
                                     of a blocked run come from am_sweep_run_ticks_view            */

/* One shard of the record array on one CUDA device.  `capacity` slots are
 * allocated up front; `shard_base` is added to local indices wherever a
 * global index is reported (multi-GPU index-range sharding, SURVEY §8e). */
int am_sweep_create(am_sweep_t** out, int device_id, uint64_t capacity, uint64_t shard_base);
void am_sweep_destroy(am_sweep_t*);

/* Bulk load of a contiguous index range [first, first+n) — informer re-list
 * after (re)start (SURVEY §5 "failure detection / recovery").  The columns are
 * taken as they are: they must be values this library produced
 * (am_healthcheck_classify / am_sweep_read).  In particular
 * AM_F_REMEDY_OUTCOME_OK only has a meaning together with AM_F_REMEDY_PENDING. */
int am_sweep_load_range(am_sweep_t*, uint64_t first, uint64_t n, const am_record_cols_t* cols);

/* Reconcile of created/updated CRs (hcc.go:170-188): scatter n records to
 * local slots idx[i].  Thread-safe; staged and applied by the next tick. */
int am_sweep_upsert(am_sweep_t*, uint64_t n, const uint64_t* idx, const am_record_t* recs);

/* CR deleted (hcc.go:175-186: Stop() its timer): tombstone the slots.  A removed
 * slot reads back as flags == AM_F_TOMBSTONE; its other columns are unspecified
 * until the next upsert.  Staged calls (upsert / remove / post_result) take effect
 * per slot in call order at the next tick or read. */
int am_sweep_remove(am_sweep_t*, uint64_t n, const uint64_t* idx);

/* Terminal workflow phases observed by the watch loops (hcc.go:635, :662,
 * :821, :836).  phase / remedy_phase: 0 none, 1 Succeeded, 2 Failed.
 * Thread-safe; staged and applied at the start of the next tick.  Calls from several
 * threads (the reconcile workers, hcc.go:170-188) stage concurrently: a call holds the
 * handle's lock only to reserve its range of the staging arrays, so posting scales with
 * the caller's threads; per slot, calls take effect in the order they entered the library.
 * A call with an out-of-range slot (AM_E_RANGE) or a phase outside 0..2 (AM_E_INVAL) has
 * no effect at all. */
#define AM_PHASE_NONE 0
#define AM_PHASE_SUCCEEDED 1
#define AM_PHASE_FAILED 2
int am_sweep_post_result(am_sweep_t*, uint64_t n, const uint64_t* idx, const uint8_t* phase,
                         const uint8_t* remedy_phase);

/* One tick at wall-clock second unix_sec: drain staged ops, run the sweep
 * kernel, return the ascending list of (global index, action) for every record
 * whose action is non-zero.  Replaces, for every record at once, the decisions
 * at hcc.go:238-267, :649-660, :677-721, :821-851 and the timer at :751.
 * If n_emitted > cap: AM_E_NOSPACE, *n_out = needed, first cap entries valid.
 * Single caller at a time per handle (AM_E_BUSY otherwise). */
int am_sweep_tick(am_sweep_t*, int64_t unix_sec, uint32_t mode, uint64_t* due_idx,
                  uint32_t* due_action, uint64_t cap, uint64_t* n_out, am_tick_stats_t* stats);

/* The same tick without the per-entry pass into caller memory: `view` points at the
 * library's own pinned host buffer, which the GPU wrote directly — u32 LOCAL indices
 * (global = shard_base + idx_local[k]) and u8 actions, ascending.  A cgo caller reads
 * C memory in place (unsafe.Slice).  Valid until the next am_sweep_tick* call on the
 * handle.  Never returns AM_E_NOSPACE. */
typedef struct am_tick_view {
  const uint32_t* idx_local;
  const uint8_t* action;
  uint64_t n;
  uint64_t shard_base;
} am_tick_view_t;
int am_sweep_tick_view(am_sweep_t*, int64_t unix_sec, uint32_t mode, am_tick_view_t* view,
                       am_tick_stats_t* stats);

/* Re-read the list of the last am_sweep_tick / am_sweep_tick_view from entry `offset`
 * on (an AM_E_NOSPACE tick has consumed its one-shot actions — RUN_REMEDY, STOPPED,
 * RESET_* — on the device: fetch the rest here instead of losing them).  *n_out = entries
 * from `offset` to the end; AM_E_NOSPACE again if they exceed cap. */
int am_sweep_last_list(am_sweep_t*, uint64_t offset, uint64_t* due_idx, uint32_t* due_action,
                       uint64_t cap, uint64_t* n_out);

/* Same tick, results left in HBM: launches on `cuda_stream` (a cudaStream_t /
 * CUstream as void*; NULL = CUDA's default stream, as in every CUDA API; use
 * am_sweep_stream() for the handle's own stream) and does not synchronise.
 * d_due_idx (u32 LOCAL indices), d_due_action (u8) hold `cap` entries;
 * d_count receives min(n_emitted, cap) (u32) — the number of valid list entries;
 * d_stats (may be NULL) receives an am_tick_stats_t whose n_emitted is the full count.
 * Used for device-resident pipelines.  Stream rule: every device operation of a handle
 * is ordered after the previous one, whatever streams they were issued on (the library
 * inserts the event waits); a stream passed here must stay alive until the next call on
 * the handle has returned. */
int am_sweep_tick_device(am_sweep_t*, int64_t unix_sec, uint32_t mode, void* d_due_idx,
                         void* d_due_action, uint64_t cap, void* d_count, void* d_stats,
                         void* cuda_stream);

/* Multi-GPU tick, first half: drain + sweep + group scan only.  The emitted set stays
 * inside the handle as a bitmap (1 bit per record) plus the non-default actions;
 * am_gather_exchange ships exactly that over NVLink and rebuilds the GLOBAL list on
 * every GPU.  Two buffer sets alternate, so the exchange of tick k (on another stream)
 * may overlap am_sweep_tick_shard of tick k+1; tick k+2 waits for exchange k by itself. */
int am_sweep_tick_shard(am_sweep_t*, int64_t unix_sec, uint32_t mode, void* cuda_stream);

/* Streaming: n_ticks consecutive one-second ticks starting at unix_sec0,
 * back-to-back on the device (BASELINE config 5).  Per-tick stats are written
 * to stats_out[0..n_ticks) (host).  Emitted lists go to an HBM ring and are
 * not copied to the host (with AM_SWEEP_BLOCKED there are none); am_sweep_run_ticks_view
 * returns them.
 * `seed` keys the closed-loop outcome sequence. */
int am_sweep_run_ticks(am_sweep_t*, int64_t unix_sec0, uint64_t n_ticks, uint32_t mode,
                       uint64_t seed, am_tick_stats_t* stats_out);

/* am_sweep_run_ticks, and in addition the ascending (local index, action) list of every tick.
 * views[k] (k < n_ticks) describes tick unix_sec0 + k, in the form am_sweep_tick_view returns.
 * All lists live back to back in the library's pinned host buffer (each one or each group of up to
 * 16 starts on a multiple of 4 entries). That buffer grows to hold the whole run at 5 B per entry,
 * so choose n_ticks to match. The views stay valid until the next am_sweep_tick* /
 * am_sweep_run_ticks* call on the handle; am_sweep_last_list finds no list after this call.
 * Works with and without AM_SWEEP_BLOCKED / AM_SWEEP_CLOSED_LOOP. Both forms return identical lists,
 * statistics and columns, and these are identical to n_ticks calls of am_sweep_tick. Staged results
 * are applied, and counted, at the first tick.
 * Without AM_SWEEP_BLOCKED the ticks run one after the other, one synchronisation each. With it, a
 * block of K ticks (AMSWEEP_BLOCK_TICKS, 96 by default) costs one synchronisation: the block kernel
 * leaves each tick's emitted set in a device "tick ring" of K slots, allocated on the first blocked
 * call and kept until am_sweep_destroy: K x (4.13 B x capacity) of device memory, about 3.9 GB for
 * 10 M records at K = 96 (5.3 GB at K = 128). */
int am_sweep_run_ticks_view(am_sweep_t*, int64_t unix_sec0, uint64_t n_ticks, uint32_t mode,
                            uint64_t seed, am_tick_stats_t* stats_out, am_tick_view_t* views);

/* RepeatAfterSec of records [first, first+n) as the reference derives it at
 * reconcile time (hcc.go:259-262): Next(unix_sec) - unix_sec for a 5-field
 * schedule (robfig SpecSchedule.Next evaluated on the device; -9223372035 when
 * nothing fires within five years), the stored interval for "@every"/interval
 * checks, 0 otherwise.  On-demand query, not part of the per-tick path. */
int am_sweep_repeat_after_sec(am_sweep_t*, int64_t unix_sec, uint64_t first, uint64_t n, int64_t* out);

/* The earliest second after unix_sec at which a tick of this shard would emit anything, given
 * the state as it stands (staged events included, no further ones assumed): the wake-up time of
 * the reference's earliest repeat timer (hcc.go:751) or cron activation (hcc.go:262), evaluated on
 * the device over every record (robfig SpecSchedule.Next for 5-field schedules).  The 1 Hz ticker
 * may sleep until then — or until the next upsert / post_result, whichever comes first: ticks in
 * between return an empty list.  INT64_MAX when nothing will ever be due. */
int am_sweep_next_due(am_sweep_t*, int64_t unix_sec, int64_t* next_out);

/* Device -> host read-back of record state (status write-back, hcc.go:1445;
 * checkpoint, SURVEY §5). idx == NULL reads the range [first, first+n). */
int am_sweep_read(am_sweep_t*, uint64_t first, uint64_t n, const uint64_t* idx,
                  am_record_cols_t* out);

/* Introspection */
uint64_t am_sweep_size(const am_sweep_t*);     /* high-water mark (slots swept) */
uint64_t am_sweep_capacity(const am_sweep_t*);
int am_sweep_device(const am_sweep_t*);
/* Device time of the last am_sweep_tick / am_sweep_run_ticks sweep kernels
 * (CUDA events on the launching stream), milliseconds; <0 if none. */
double am_sweep_last_kernel_ms(const am_sweep_t*);
/* Per-kernel device timing: when on, every tick records CUDA events on the
 * launching stream before and after sweep_tick_kernel and after the rest of the
 * tick (scan + expand + publish).  am_sweep_last_profile waits for the last tick and
 * returns the two durations in milliseconds.  Off by default (the extra events
 * break the programmatic launch chain: do not time a step with it on). */
int am_sweep_set_profiling(am_sweep_t*, int on);
int am_sweep_last_profile(am_sweep_t*, double* sweep_ms, double* rest_ms);
/* Number of kernels this library has launched on the handle so far. */
uint64_t am_sweep_launch_count(const am_sweep_t*);
/* Raw device pointer of a column (for zero-copy wrapping by torch / NCCL
 * plumbing); column ids follow am_record_cols_t member order, 0..15. */
void* am_sweep_column_ptr(am_sweep_t*, int column);
int am_sweep_set_seed(am_sweep_t*, uint64_t seed);
/* The handle's own non-blocking stream (cudaStream_t as void*). */
void* am_sweep_stream(am_sweep_t*);

/* ---- multi-GPU: the global due list on every GPU, over NVLink peer memory (SURVEY §8e) --
 * One am_gather per rank (one process per GPU).  Every rank creates its exchange block,
 * exports a CUDA-IPC handle, the handles are exchanged by the caller's plumbing
 * (torch.distributed / any side channel) and connected, and the shard layout is set.
 * Then, per tick, every rank calls
 *     am_sweep_tick_shard(sweep, T, mode, stream_a);      // sweep + group scan
 *     am_gather_exchange(gather, sweep, d_stats, stream_b);
 * The exchange ships the sweep's own output — one bit per record for the emitted set,
 * group offsets, the non-default actions — into every peer's block (one kernel, 16-B peer
 * stores, no NCCL, no host round-trip) and rebuilds the GLOBAL ascending (index, action)
 * list locally from the world's bitmaps.  When its last kernel retires, out_idx / out_act
 * on EVERY rank hold that list, out_counts[0..world) the per-rank counts and
 * out_counts[world] the total; d_stats (may be NULL) receives this shard's am_tick_stats_t.
 * stream_b may differ from stream_a (the library orders them): the exchange of tick k then
 * overlaps the sweep of tick k+1.
 * Like any collective, the exchange is a rendezvous: every rank must call it the same
 * number of times.  Its device-side wait for the peers is bounded (AMSWEEP_PUSH_TIMEOUT_MS,
 * default 5000, 0 = unbounded): a peer that never arrives leaves out_counts[world] ==
 * 0xFFFFFFFF and the handle out of step (recreate it).  Argument errors are reported before
 * anything that the peers could observe happens.
 * The reference has no counterpart (single process; consumer is hcc.go:502). */
#define AM_IPC_HANDLE_BYTES 64
typedef struct am_gather am_gather_t;
/* cap_total: records of all shards together (bounds the global list).
 * idx_bytes: 8 = u64 global indices in the output; 4 = u32 (the caller guarantees every
 * global index < 2^32). */
int am_gather_create(am_gather_t** out, int device, int rank, int world, uint64_t cap_total,
                     int idx_bytes);
int am_gather_export(am_gather_t*, void* handle_out /* AM_IPC_HANDLE_BYTES */);
int am_gather_connect(am_gather_t*, const void* handles /* world x AM_IPC_HANDLE_BYTES, rank order */);
/* bases[r] / sizes[r] = first global index / number of records of rank r's shard (the same
 * arrays on every rank).  Required before am_gather_exchange. */
int am_gather_set_layout(am_gather_t*, const uint64_t* bases, const uint64_t* sizes);
int am_gather_exchange(am_gather_t*, am_sweep_t* shard, void* d_stats, void* cuda_stream);
/* One whole step of a sharded controller in one call — the multi-GPU counterpart of am_sweep_tick_view:
 * am_sweep_tick_shard of the bound shard on `sweep_stream` (draining what was posted to it), the
 * exchange on `exchange_stream`, then THIS rank's own part of the global list — its checks, as local
 * slots — extracted into the library's pinned host buffer; one synchronisation.  am_gather_bind names
 * the shard and the two streams once; the view is valid until the next call.  AM_E_DEVICE when a peer
 * did not arrive within AMSWEEP_PUSH_TIMEOUT_MS.  (The global list itself stays on the device:
 * am_gather_out_idx / _act / _counts.) */
int am_gather_bind(am_gather_t*, am_sweep_t* shard, void* sweep_stream, void* exchange_stream);
int am_gather_tick_view(am_gather_t*, int64_t unix_sec, uint32_t mode, am_tick_view_t* view, am_tick_stats_t* stats);
/* Round-1 "plain" format, kept as the measured baseline: every rank writes its FINISHED
 * list (the output of am_sweep_tick_device: u32 local indices, u8 actions, device count)
 * straight into every peer's output buffer at its global offset, 5 or 9 bytes per entry
 * on the wire.  Unbounded device-side waits. */
int am_gather_push(am_gather_t*, const void* d_idx_local /* u32 */, const void* d_act_local /* u8 */,
                   const void* d_count_local /* u32 */, uint64_t shard_base, void* cuda_stream);
void* am_gather_out_idx(am_gather_t*);    /* u64|u32[cap_total], valid after the last exchange / push retires */
void* am_gather_out_act(am_gather_t*);    /* u8[cap_total]                                    */
void* am_gather_out_counts(am_gather_t*); /* u32[world+1]                                     */
/* Device timing of one exchange (CUDA events on its stream): the NVLink push (including the
 * wait for the peers), the list rebuild (counts + expand), the statistics publication. */
int am_gather_set_profiling(am_gather_t*, int on);
int am_gather_last_profile(am_gather_t*, double* push_ms, double* rebuild_ms, double* publish_ms);
const char* am_gather_last_error(const am_gather_t*);
void am_gather_destroy(am_gather_t*);

/* ---- hand-off to the workflow side (SURVEY.md 8f-3; host only, no GPU) ---- */
/* The step AFTER the path: the 1 Hz ticker goroutine publishes the list one
 * am_sweep_tick returned; up to MaxParallel workers (hcc.go:138, the
 * MaxConcurrentReconciles of hcc.go:298) pop chunks and run
 * createSubmitWorkflow / processRemedy (hcc.go:502, :759) for them.  It
 * replaces the goroutine-per-timer fan-out of hcc.go:751 by a bounded FIFO:
 * back-pressure instead of unbounded goroutines when the cluster is slow.
 * Thread-safe for any number of publishers and poppers; never blocks. */
typedef struct am_handoff am_handoff_t;
typedef struct am_work_item {
  uint64_t idx;     /* global record index                                    */
  int64_t unix_sec; /* the tick that emitted it                               */
  uint32_t action;  /* AM_ACT_* bits (already filtered by the publish mask)   */
  uint32_t reserved;
} am_work_item_t;

int am_handoff_create(am_handoff_t** out, uint64_t capacity /* work items */);
void am_handoff_destroy(am_handoff_t*);
/* Enqueue, in order, the entries of one tick whose action has a bit of
 * action_mask set (e.g. AM_ACT_SUBMIT_HC | AM_ACT_RUN_REMEDY).  All or
 * nothing: AM_E_NOSPACE when they do not fit, nothing enqueued, *n_out = the
 * number that would have been; AM_OK: *n_out = number enqueued. */
int am_handoff_publish(am_handoff_t*, int64_t unix_sec, uint64_t n, const uint64_t* idx,
                       const uint32_t* action, uint32_t action_mask, uint64_t* n_out);
/* Dequeue up to `max` items in FIFO order (0 items is not an error). */
int am_handoff_pop(am_handoff_t*, uint64_t max, am_work_item_t* out, uint64_t* n_out);
/* Queue depth and lifetime totals (any pointer may be NULL). */
int am_handoff_stats(am_handoff_t*, uint64_t* pending, uint64_t* published, uint64_t* popped,
                     uint64_t* rejected_batches);

/* UTC broken-down time exactly as the kernel computes it (test hook):
 * out[0..6) = sec, min, hour, dom(1-31), month(1-12), dow(0=Sunday). */
void am_civil_from_unix(int64_t unix_sec, int32_t out[6]);

const char* am_strerror(int code);
const char* am_last_error_detail(const am_sweep_t*); /* NULL handle: create-time error */
int am_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* AMSWEEP_H_ */
