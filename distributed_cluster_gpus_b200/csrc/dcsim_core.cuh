/*
 * dcsim_core.cuh — the device code of the B200 batched simulator (all kernels' bodies).
 *
 * The reference's multi-DC event loop (simcore/simulator_paper_multi.py:412-480 and the leaves it calls; citations
 * are relative to the reference tree) is split where its data dependencies split it:
 *
 *   arrival pre-pass  (dcsim_generate_arrivals, one THREAD per replica)
 *       Only arrival handlers draw random numbers and routing never looks at DC state, so a replica's whole arrival
 *       sequence — instants, routed DCs, which pushes were schedulable, and the uniform / normal deviate its job size
 *       is a function of — is drawn ahead, in the reference's draw order, with all 32 lanes of a warp running the
 *       samplers.  Only what the NEXT draw depends on stays in this sequential chain (stream position, stream clocks).
 *
 *   list merge        (dcsim_merge_arrivals, one WARP per replica, lane-parallel over arrivals)
 *       Everything that hangs off an arrival without feeding back into the draws: the job size (pow / exp), the
 *       xfer_done instant t + transfer_s[ingress][dc][jtype] (SIM:580-588), and the position both events take in the
 *       replica's time-ordered list of {arrival, xfer_done} events — ties broken exactly as the heap would, by push
 *       order (SIM:163).
 *
 *   event loop        (dcsim_replica_run, one WARP per replica)
 *       The replica's working set — pending-event candidates, per-DC accumulators, a window of its event list, (small
 *       blocks:) its running-job records — is a "state block" staged in shared memory for the launch; the unbounded
 *       FIFO queues, the event lists and (large blocks) the running-job records live in HBM/L2.  How the 32 lanes are
 *       used:
 *         - pop-min: the pending events are kept as *candidates* (one per DC = earliest job_finish of that DC, the next
 *           list entry, the log tick, ...); every lane loads one candidate and three REDUX.MIN (hi word, lo word, seq)
 *           find the winner;
 *         - the per-event sweep over all DCs (SIM:429-437) runs one DC per lane;
 *         - a job_finish is one lane-parallel pass over the DC's records (compaction, next finish, power re-sum);
 *         - staging of the list window and the state block run strided across the warp;
 *         - the handlers themselves are strictly sequential per replica and run on lane 0 out of shared memory.
 *
 * All arithmetic that defines results is FP64 and is written so that, compiled with -fmad=false, every + - * /
 * happens in the reference's order with one rounding each.  log/exp/pow/sin come from CUDA's libdevice (<= 2 ulp
 * from glibc's), which is why parity with the reference is asserted at 1e-9 relative and exact event/job/RNG-word
 * counts rather than bit-for-bit.
 *
 * The file compiles two ways:
 *   - nvcc, sm_100a: DCSIM_LANES = 32, warp collectives are real (csrc/dcsim_b200.cu);
 *   - g++ with -DDCSIM_HOST_EMU (tests/hostemu/, TEST-ONLY): DCSIM_LANES = 1, collectives are identities.
 *     It exists so the handler logic can be checked against the oracle where there is no GPU; it is not
 *     linked into, or reachable from, the product library.
 */
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>
#if !defined(DCSIM_HOST_EMU)
#include <cuda_pipeline.h>
#endif

#include "../../include/dcsim_b200.h"

#ifdef DCSIM_HOST_EMU
#define DCSIM_DEV static inline
#define DCSIM_LANES 1
static inline int dcsim_lane() { return 0; }
static inline void dcsim_warp_sync() {}
static inline uint32_t dcsim_warp_min_u32(uint32_t x) { return x; }
static inline uint32_t dcsim_warp_ballot(bool p) { return p ? 1u : 0u; }
static inline uint32_t dcsim_bcast_u32(uint32_t x, int) { return x; }
static inline int dcsim_ffs(uint32_t x) { return __builtin_ffs((int)x); }
static inline uint32_t dcsim_hi(double x) { uint64_t u; memcpy(&u, &x, 8); return (uint32_t)(u >> 32); }
static inline uint32_t dcsim_lo(double x) { uint64_t u; memcpy(&u, &x, 8); return (uint32_t)u; }
static inline uint32_t dcsim_mulhi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
static inline int dcsim_bit_length(uint32_t n) { return 32 - __builtin_clz(n); }
static inline uint32_t dcsim_popc(uint32_t x) { return (uint32_t)__builtin_popcount(x); }
static inline uint32_t dcsim_lanemask_lt(int) { return 0u; }
static inline uint32_t dcsim_warp_add_u32(uint32_t x) { return x; }
static inline uint32_t dcsim_warp_max_u32(uint32_t x) { return x; }
static inline uint32_t dcsim_pick_u32(bool, uint32_t v) { return v; }
static inline void dcsim_event_sync() {}
static inline bool dcsim_event_any(bool p) { return p; }
static inline uint32_t dcsim_event_min_u32(uint32_t x) { return x; }
static inline bool dcsim_event_any_full(bool p) { return p; }
static inline void dcsim_sync_full() {}
static inline uint32_t dcsim_event_bcast_u32(uint32_t x, int) { return x; }
static inline uint32_t dcsim_event_pick_u32(bool, uint32_t v) { return v; }
#define DCSIM_INF (__builtin_inf())
#else
#define DCSIM_DEV __device__ __forceinline__
/* Lanes per replica.  32: one warp owns one replica.  8 / 16: a warp carries 4 / 2 replicas, each on an aligned group of
 * lanes; every collective below is then relative to the caller's group (the groups of a warp run different handlers
 * and only ever synchronise among themselves).  The merge kernel always uses 32. */
#ifndef DCSIM_LANES
#define DCSIM_LANES 32
#endif
#if DCSIM_LANES == 32
#define DCSIM_GROUP_SHIFT 0u
#define DCSIM_GROUP_MASK 0xffffffffu
#else
#define DCSIM_GROUP_SHIFT ((threadIdx.x & 31u) & ~(unsigned)(DCSIM_LANES - 1))
#define DCSIM_GROUP_MASK ((((1u << DCSIM_LANES) - 1u)) << DCSIM_GROUP_SHIFT)
#endif
DCSIM_DEV int dcsim_lane() { return (int)(threadIdx.x & (unsigned)(DCSIM_LANES - 1)); }
DCSIM_DEV void dcsim_warp_sync() { __syncwarp(DCSIM_GROUP_MASK); }
DCSIM_DEV uint32_t dcsim_warp_min_u32(uint32_t x) {
#if DCSIM_LANES == 32
  return __reduce_min_sync(0xffffffffu, x);
#else
  const unsigned gm = DCSIM_GROUP_MASK;
#pragma unroll
  for (int o = DCSIM_LANES / 2; o > 0; o >>= 1) { const uint32_t y = __shfl_xor_sync(gm, x, o); x = y < x ? y : x; }
  return x;
#endif
}
DCSIM_DEV uint32_t dcsim_warp_ballot(bool p) {
#if DCSIM_LANES == 32
  return __ballot_sync(0xffffffffu, p);
#else
  return (__ballot_sync(DCSIM_GROUP_MASK, p) >> DCSIM_GROUP_SHIFT) & ((1u << DCSIM_LANES) - 1u);
#endif
}
DCSIM_DEV uint32_t dcsim_bcast_u32(uint32_t x, int src) { return __shfl_sync(DCSIM_GROUP_MASK, x, src, DCSIM_LANES); }
DCSIM_DEV int dcsim_ffs(uint32_t x) { return __ffs((int)x); }
DCSIM_DEV uint32_t dcsim_hi(double x) { return (uint32_t)__double2hiint(x); }
DCSIM_DEV uint32_t dcsim_lo(double x) { return (uint32_t)__double2loint(x); }
DCSIM_DEV uint32_t dcsim_mulhi(uint32_t a, uint32_t b) { return __umulhi(a, b); }
DCSIM_DEV int dcsim_bit_length(uint32_t n) { return 32 - __clz((int)n); }
DCSIM_DEV uint32_t dcsim_popc(uint32_t x) { return (uint32_t)__popc(x); }
DCSIM_DEV uint32_t dcsim_lanemask_lt(int lane) { return (1u << lane) - 1u; }
#if DCSIM_LANES == 32
DCSIM_DEV uint32_t dcsim_warp_add_u32(uint32_t x) { return __reduce_add_sync(0xffffffffu, x); }
DCSIM_DEV uint32_t dcsim_warp_max_u32(uint32_t x) { return __reduce_max_sync(0xffffffffu, x); }
#else
DCSIM_DEV uint32_t dcsim_warp_add_u32(uint32_t x) {
#pragma unroll
  for (int o = DCSIM_LANES / 2; o > 0; o >>= 1) x += __shfl_xor_sync(DCSIM_GROUP_MASK, x, o);
  return x;
}
DCSIM_DEV uint32_t dcsim_warp_max_u32(uint32_t x) {
#pragma unroll
  for (int o = DCSIM_LANES / 2; o > 0; o >>= 1) { const uint32_t y = __shfl_xor_sync(DCSIM_GROUP_MASK, x, o); x = y > x ? y : x; }
  return x;
}
#endif
/* The value `v` of the ONE lane of the group whose `mine` is set, to every lane of the group.  A ballot with a member
 * mask that differs between the groups of a warp is executed once per distinct mask (4 serial VOTEs + the bookkeeping
 * around them: the largest single stall of the 8-lane event loop in the round-2 ncu capture); a min-butterfly is three
 * converged shuffles. */
DCSIM_DEV uint32_t dcsim_pick_u32(bool mine, uint32_t v) {
#if DCSIM_LANES == 32
  return __shfl_sync(0xffffffffu, v, __ffs((int)__ballot_sync(0xffffffffu, mine)) - 1);
#else
  return dcsim_warp_min_u32(mine ? v : 0xffffffffu);
#endif
}
/* EVENT-LEVEL collectives: called at points of the event loop that every lane of the WARP reaches together, whatever
 * its replica is doing (dcsim_replica_run keeps the loop itself warp-uniform: a replica that is done stays in it,
 * switched off, until all replicas of the warp are).  The member mask is then the constant full mask even when the
 * warp carries several replicas — a group-relative mask is a run-time value the hardware cannot know to be uniform,
 * and every collective under it pays a MATCH.ANY + REDUX.OR + branch to find out.  Shuffles still stay inside the
 * group: xor distances below DCSIM_LANES never leave an aligned group of DCSIM_LANES lanes. */
DCSIM_DEV void dcsim_event_sync() { __syncwarp(); }
DCSIM_DEV bool dcsim_event_any(bool p) {
#if DCSIM_LANES == 32
  return p; /* one replica per warp: its own flag */
#else
  return __any_sync(0xffffffffu, p) != 0;
#endif
}
DCSIM_DEV uint32_t dcsim_event_min_u32(uint32_t x) {
#if DCSIM_LANES == 32
  return __reduce_min_sync(0xffffffffu, x);
#else
#pragma unroll
  for (int o = DCSIM_LANES / 2; o > 0; o >>= 1) { const uint32_t y = __shfl_xor_sync(0xffffffffu, x, o); x = y < x ? y : x; }
  return x;
#endif
}
/* Thread-per-replica kernels (the arrival pre-pass): all 32 lanes of the warp, each with its own replica. */
DCSIM_DEV bool dcsim_event_any_full(bool p) { return __any_sync(0xffffffffu, p) != 0; }
DCSIM_DEV void dcsim_sync_full() { __syncwarp(); }
DCSIM_DEV uint32_t dcsim_event_bcast_u32(uint32_t x, int src) { return __shfl_sync(0xffffffffu, x, src, DCSIM_LANES); }
DCSIM_DEV uint32_t dcsim_event_pick_u32(bool mine, uint32_t v) { /* dcsim_pick_u32 at an event-level point */
#if DCSIM_LANES == 32
  return dcsim_pick_u32(mine, v);
#else
  return dcsim_event_min_u32(mine ? v : 0xffffffffu);
#endif
}
#define DCSIM_INF (__longlong_as_double(0x7ff0000000000000LL))
#endif

DCSIM_DEV double dcsim_hilo_f64(uint32_t hi, uint32_t lo) {
#ifdef DCSIM_HOST_EMU
  const uint64_t u = ((uint64_t)hi << 32) | (uint64_t)lo; double x; memcpy(&x, &u, 8); return x;
#else
  return __hiloint2double((int)hi, (int)lo);
#endif
}

DCSIM_DEV double dcsim_bcast_f64(double x, int src) {
#ifdef DCSIM_HOST_EMU
  (void)src; return x;
#else
  return __hiloint2double((int)dcsim_bcast_u32(dcsim_hi(x), src), (int)dcsim_bcast_u32(dcsim_lo(x), src));
#endif
}
DCSIM_DEV double dcsim_event_bcast_f64(double x, int src) {
#ifdef DCSIM_HOST_EMU
  (void)src; return x;
#else
  return __hiloint2double((int)dcsim_event_bcast_u32(dcsim_hi(x), src), (int)dcsim_event_bcast_u32(dcsim_lo(x), src));
#endif
}

/* Histogram bin of a positive latency: 4 bins per octave from 2^-20 s, from the IEEE exponent and the top two
 * mantissa bits — pure integer work, identical on host and device. */
DCSIM_DEV int dcsim_lat_bin(double lat) {
  const uint32_t hi = dcsim_hi(lat);
  const int e = (int)((hi >> 20) & 0x7ffu) - (1023 - 20);
  int idx = e * 4 + (int)((hi >> 18) & 3u);
  idx = idx < 0 ? 0 : idx;
  return idx > DCSIM_LAT_BINS - 1 ? DCSIM_LAT_BINS - 1 : idx;
}

/* Cold helpers are kept OUT OF LINE in the one-replica-per-warp build (by-value arguments only, so the context stays in
 * registers): inlining them costs the event loop registers and instruction-cache footprint on paths most launches never
 * take.  When a warp carries several replicas they are INLINED instead: a call made by one lane group while its
 * siblings are elsewhere in the loop is ruinous (the job-latency histogram's one-instruction helper measured +130 % on
 * the whole event loop as a call, < 1 % inlined: tools/hist_probe.py), and that build has registers to spare. */
#if defined(DCSIM_HOST_EMU)
#define DCSIM_COLD static
#elif DCSIM_LANES == 32
#define DCSIM_COLD static __device__ __noinline__ /* static: the core is compiled into several translation units */
#else
#define DCSIM_COLD static __device__ __forceinline__
#endif

/* One count into replica r's [2][DCSIM_LAT_BINS] histogram in HBM — fire-and-forget, nothing waits for it. */
DCSIM_COLD void dcsim_hist_add(uint32_t* hist, uint64_t r, int jt, double lat) {
  uint32_t* cell = hist + r * (uint64_t)(2 * DCSIM_LAT_BINS) + (uint32_t)(jt * DCSIM_LAT_BINS + dcsim_lat_bin(lat));
#ifdef DCSIM_HOST_EMU
  *cell += 1u;
#else
  atomicAdd(cell, 1u);
#endif
}

/* ---- candidate slots (the event set, one slot per lane) -------------------------------------- */
enum {
  CAND_DC0 = 0,      /* + d   : earliest job_finish among DC d's running jobs */
  /* behind the n_dc finish slots, densely (so that 4 DCs + 3 fit the 8 lanes of a lane group in one round):
     n_dc     the next entry of the replica's {arrival, xfer_done} list  (CAND_LIST(c))
     n_dc + 1 the log tick                                               (CAND_LOG(c))
     n_dc + 2 earliest superseded job_finish (cap_greedy re-scheduling leaves the old event in the heap, SIM:330-338) */
  CAND_N = 16        /* slots allocated (DCSIM_MAX_DC + 3 used at most); unused ones stay +inf */
};
#define DCSIM_CAND_N 16 /* == CAND_N, for the preprocessor (an enumerator reads as 0 in #if) */
#define DCSIM_SEQ_LIMIT ((1u << 28) - (1u << 20)) /* lane-group builds: see dcsim_argmin_cand */
static_assert(DCSIM_CAND_N == CAND_N, "DCSIM_CAND_N");
#define CAND_LIST(c) ((c).P->spec.n_dc)
#define CAND_LOG(c) ((c).P->spec.n_dc + 1)
#define CAND_STALE(c) ((c).P->spec.n_dc + 2)
enum { KIND_ARR_INF = 0, KIND_ARR_TRN = 1, KIND_XFER = 2, KIND_FINISH = 3, KIND_LOG = 4, KIND_STALE = 5 };

/* ---- one entry of a replica's event list (SoA: t f64, aux f64, meta u32) ----------------------
 * arrival : t = arrival instant; aux (low 32 bits) = list position of its xfer_done entry (ML_A_XIN);
 *           meta = 0 | stream << 1 | ML_A_NEXT | ML_A_XSCHED | ML_A_XIN
 * xfer    : t = xfer_done instant; aux = job size; meta = 1 | dc << 1 | jtype << 4 | ingress << 5 | arrival index << 8 */
enum : uint32_t {
  ML_XFER = 1u,
  ML_A_NEXT = 1u << 5,   /* the stream's next arrival was schedulable: its push takes a seq (SIM:591-592) */
  ML_A_XSCHED = 1u << 6, /* the xfer_done push was schedulable: it takes a seq (SIM:580-588) */
  ML_A_XIN = 1u << 7     /* ... and falls at or before end_time, i.e. it is in the list (aux holds its position) */
};
#define DCSIM_MAX_ARRIVALS (1u << 24) /* arrival index field of an xfer entry */

enum { /* per-DC f64 arrays inside the state block, each DCSIM_MAX_DC long */
  DF_ENERGY = 0,
  DF_LAST_T,     /* (kept in a register during a launch: dcsim_ctx_t::now; this slot holds it between launches)
                    util_last_ts (SIM:430-436) AND last_energy_time (models.py:100-106): both are 0.0 until the
                    first event and are set to t on every event, so one slot carries both */
  DF_UTIL_TIME, DF_UTIL_BEGIN, DF_ACC_UNIT, DF_CUR_FREQ, DF_POWER,
  DF_PSUM,       /* sum of the running jobs' n*P_gpu(f) in dict (= start) order from 0.0 (SIM:168-179): extended by one
                    addition when a job starts (the same additions a re-sum would do), re-summed when one leaves */
  DF_N
};
enum { /* per-DC i32 arrays; FIFO rings are (head index, length) so no modulo is needed */
  DI_BUSY = 0, DI_NRUN, DI_QH_INF, DI_QN_INF, DI_QH_TRN, DI_QN_TRN, DI_FMIN_SLOT, DI_N
};

/* One DC per lane on the GPU (32 lanes >= DCSIM_MAX_DC); a plain loop in the single-lane host build. */
#if DCSIM_LANES >= DCSIM_MAX_DC
#define DCSIM_FOR_EACH_DC(d, c, n) for (int d = (c).lane, once_ = 1; once_ && d < (n); once_ = 0)
#else
#define DCSIM_FOR_EACH_DC(d, c, n) for (int d = 0; d < (n); ++d)
#endif

#define DCSIM_LIST_WINDOW 32u   /* slots of the event-list ring in shared memory (list position p lives in slot p & 31) */
#define DCSIM_LIST_HALF 16u     /* refill granularity: while one half is consumed the other is (asynchronously) loaded */
/* A rejection loop that has not accepted after this many draws stops the replica with DCSIM_ST_RNG_RUNAWAY
 * instead of spinning (the reference would spin: e.g. arrivals.py:41-45 under a clipped lambda). */
#define DCSIM_REJECTION_LIMIT (1 << 24)

/* Persistent scalars of a replica (first bytes of its state block). */
struct dcsim_hdr_t {
  double now, lat_sum, lat_sum_inf, lat_sum_trn, last_t;
  double omin_t;        /* the earliest of the candidates OTHER than the list entry: (omin_t, omin_seq) in slot omin_slot, */
  uint32_t n_events, seq, jid, rng_pos;
  uint32_t cand_dirty, status, done, initialized; /* ... valid while cand_dirty == 0 (dcsim_argmin_cand) */
  uint32_t n_fin_inf, n_fin_trn, ev_arr, ev_xfer;
  uint32_t ev_fin, ev_log, omin_seq, max_run;
  uint32_t max_q, omin_slot, bandit_t, n_stale;
  uint32_t smin_slot, ml_cursor, ml_count, _r3; /* event-list cursor / length */
};

/* Byte offsets of the arrays inside a state block; computed once per handle on the host. */
struct dcsim_layout_t {
  int32_t cand_t, cand_seq;
  int32_t dc_f64, dc_i32;
  int32_t lw_t, lw_aux, lw_meta, pend_seq, xring; /* list window, pending seq per stream, seq ring of in-flight transfers */
  int32_t xring_mask;                              /* ring entries - 1 (a power of two) */
  int32_t rn_t, rn_pw, rn_tpt, rn_start, rn_size, rn_f, rn_seq, rn_meta, rn_jid;
  int32_t memo_f64, memo_n; /* per (DC, jtype): the last (n, f) a job started with and its T(n,f), n*P_gpu(f), 1/T */
  int32_t bandit_n, bandit_s;
  /* power-cap controller (algo = cap_greedy with power_cap > 0 only) */
  int32_t rn_done, rn_upd;           /* per running record: units_done, last_update (models.py:20-21) */
  int32_t st_t, st_seq;              /* stale job_finish pool */
  int32_t at_rho, at_fto, at_ref, at_idx; /* DVFS atoms scratch (freq_load_agg.py) */
  int32_t cap_stale, cap_atoms;
  int32_t total_bytes;
  int32_t rec_off;         /* the running-job records occupy [rec_off, total_bytes): the part of the block that may stay
                              in HBM/L2 while [0, rec_off) is staged in shared memory ("head staged" launch mode) */
  int32_t cap_run;
  int32_t cap_q[2];        /* FIFO entries per DC: [0]=inference [1]=training */
  int32_t lean;            /* 1: running records carry no size / f / jid (nobody reads them: no job log, bandit or cap) */
  uint64_t queue_bytes;    /* HBM bytes of one replica's FIFOs */
};

static inline int32_t dcsim_align16(int32_t x) { return (x + 15) & ~15; }

/* The head of a state block has a FIXED layout — header, event set, per-DC arrays, list window, pending seqs, the
 * base of the transfer-seq ring — so the event loop addresses it with immediate offsets (LDS [blk + imm]) instead of
 * adding a layout field from the constant bank in front of every access; only the capacity-dependent arrays behind it
 * go through dcsim_layout_t. */
enum : int32_t {
  DCSIM_OFF_CAND_T = ((int32_t)sizeof(dcsim_hdr_t) + 15) & ~15,
  DCSIM_OFF_CAND_SEQ = DCSIM_OFF_CAND_T + CAND_N * 8,
  DCSIM_OFF_DC_F64 = DCSIM_OFF_CAND_SEQ + CAND_N * 4,
  DCSIM_OFF_DC_I32 = DCSIM_OFF_DC_F64 + DF_N * DCSIM_MAX_DC * 8,
  DCSIM_OFF_LW_T = (DCSIM_OFF_DC_I32 + DI_N * DCSIM_MAX_DC * 4 + 15) & ~15,
  DCSIM_OFF_LW_AUX = DCSIM_OFF_LW_T + (int32_t)DCSIM_LIST_WINDOW * 8,
  DCSIM_OFF_LW_META = DCSIM_OFF_LW_AUX + (int32_t)DCSIM_LIST_WINDOW * 8,
  DCSIM_OFF_PEND_SEQ = DCSIM_OFF_LW_META + (int32_t)DCSIM_LIST_WINDOW * 4,
  DCSIM_OFF_XRING = (DCSIM_OFF_PEND_SEQ + 2 * DCSIM_MAX_ING * 4 + 15) & ~15
};

/* Host-side: sizes the state block from the spec's capacities. */
static inline void dcsim_make_layout(const dcsim_spec_t* sp, dcsim_layout_t* L, int job_log) {
  memset(L, 0, sizeof(*L));
  const bool bandit = sp->xfer_rule == DCSIM_START_BANDIT || sp->deq_rule == DCSIM_START_BANDIT;
  const bool cap = sp->algo == DCSIM_ALGO_CAP_GREEDY && sp->power_cap > 0.0;
  /* size (job_log.csv, cap re-timing), f (job_log.csv, bandit reward, cap) and jid (job_log.csv) of a running job
     are dead weight in the state block unless one of those readers exists: 60 -> 40 bytes per record. */
  L->lean = (job_log || bandit || cap) ? 0 : 1;
  int32_t cx = sp->cap_xfer > 0 ? sp->cap_xfer : 64;
  int32_t cr = sp->cap_run > 0 ? sp->cap_run : 16;
  cr = (cr + 3) & ~3;
  L->cap_run = cr;
  L->cap_q[0] = sp->cap_q_inf > 0 ? sp->cap_q_inf : 4096;
  L->cap_q[1] = sp->cap_q_trn > 0 ? sp->cap_q_trn : 512;
  L->cand_t = DCSIM_OFF_CAND_T; L->cand_seq = DCSIM_OFF_CAND_SEQ;
  L->dc_f64 = DCSIM_OFF_DC_F64; L->dc_i32 = DCSIM_OFF_DC_I32;
  L->lw_t = DCSIM_OFF_LW_T; L->lw_aux = DCSIM_OFF_LW_AUX; L->lw_meta = DCSIM_OFF_LW_META; L->pend_seq = DCSIM_OFF_PEND_SEQ;
  /* seq of an in-flight xfer_done, indexed by its list position: an arrival writes it, the entry reads it when the
   * cursor gets there.  cap_xfer bounds the transfers in flight; an xfer entry lies at most (arrivals + transfers in
   * between) ahead of its arrival — the merge kernel measures that distance and flags DCSIM_ST_XFER_OVERFLOW when the
   * ring is too small for it, so the bound is checked, not assumed. */
  int32_t ring = 8;
  while (ring < 2 * cx) ring <<= 1;
  L->xring = DCSIM_OFF_XRING;
  L->xring_mask = ring - 1;
  int32_t o = dcsim_align16(DCSIM_OFF_XRING + ring * 4);
  const int32_t nr = sp->n_dc * cr;
  L->memo_f64 = o; o += sp->n_dc * 2 * 4 * 8;
  L->memo_n = o; o = dcsim_align16(o + sp->n_dc * 2 * 4);
  if (bandit) {
    L->bandit_s = o; o += sp->n_dc * 2 * DCSIM_MAX_FREQ * 8;
    L->bandit_n = o; o += sp->n_dc * 2 * DCSIM_MAX_FREQ * 4;
  }
  if (cap) {
    L->cap_stale = sp->cap_stale > 0 ? ((sp->cap_stale + 3) & ~3) : 64;
    int max_levels = 1;
    for (int d = 0; d < sp->n_dc; ++d) max_levels = sp->dc[d].n_freq > max_levels ? sp->dc[d].n_freq : max_levels;
    L->cap_atoms = (nr * (max_levels - 1) + 3) & ~3;
    if (L->cap_atoms < 4) L->cap_atoms = 4;
    L->st_t = o; o += L->cap_stale * 8;
    L->at_rho = o; o += L->cap_atoms * 8;
    L->at_fto = o; o += L->cap_atoms * 8;
    L->st_seq = o; o += L->cap_stale * 4;
    L->at_ref = o; o += L->cap_atoms * 4;
    L->at_idx = o; o = dcsim_align16(o + L->cap_atoms * 4);
  }
  /* the running-job records come last: everything in front of rec_off is the "head" (always staged) */
  o = dcsim_align16(o);
  L->rec_off = o;
  L->rn_t = o; o += nr * 8;
  L->rn_pw = o; o += nr * 8;
  L->rn_tpt = o; o += nr * 8;
  L->rn_start = o; o += nr * 8;
  if (!L->lean) { L->rn_size = o; o += nr * 8; L->rn_f = o; o += nr * 8; }
  if (cap) { L->rn_done = o; o += nr * 8; L->rn_upd = o; o += nr * 8; }
  L->rn_seq = o; o += nr * 4;
  L->rn_meta = o; o += nr * 4;
  if (!L->lean) { L->rn_jid = o; o += nr * 4; }
  L->total_bytes = dcsim_align16(o);
  L->queue_bytes = (uint64_t)sp->n_dc * ((uint64_t)L->cap_q[0] + (uint64_t)L->cap_q[1]) * 16ull;
}

/* One FIFO entry in HBM: the part of a Job that survives queueing (models.py:5-27). */
struct alignas(16) dcsim_qent_t {
  double size;
  uint32_t jid;
  uint32_t ing;
};

/* Optional recorders for ONE replica of the batch (the CSV wire formats; debug trace). */
struct dcsim_recorders_t {
  dcsim_trace_rec_t* trace;
  dcsim_job_rec_t* jobs;
  dcsim_cluster_rec_t* cluster;
  uint32_t* counts; /* [0]=trace rows, [1]=job rows, [2]=cluster rows (device memory) */
  uint32_t trace_cap, jobs_cap, cluster_cap, _pad;
  int64_t trace_replica; /* local replica index, -1 = none */
  int64_t log_replica;
};

/* Per-replica result of the two pre-pass kernels. */
struct dcsim_arrhdr_t {
  uint32_t count;      /* arrivals with t <= end_time, i.e. arrival events the loop will process */
  uint32_t first_mask; /* bit s: stream s's first arrival was schedulable (took a seq at construction, SIM:154-156) */
  uint32_t rng_words;  /* words the whole run consumes */
  uint32_t status;     /* DCSIM_ST_* raised while generating / merging */
  uint32_t ml_count;   /* entries of the merged {arrival, xfer_done} list */
  uint32_t max_ahead;  /* largest distance (in list entries) between an arrival and its xfer_done entry */
  uint32_t _pad[2];
};

/* Everything a launch needs.  Passed as ONE __grid_constant__ kernel parameter, so the scenario is read
 * through the constant cache and never competes with the state blocks for shared memory / L1. */
struct dcsim_kparams_t {
  dcsim_spec_t spec;
  dcsim_layout_t L;
  dcsim_recorders_t rec;
  uint64_t n_replicas;
  uint64_t seed0;       /* Philox key of local replica 0 (base_seed + first_replica_id) */
  uint64_t max_events;  /* per replica per launch; 0 = run to the end */
  uint32_t budget32;    /* the same as one 32-bit compare: 0 (unlimited) and anything >= 2^32 become 0xffffffff (host-computed) */
  uint32_t _pad32;
  char* state;          /* [n_replicas][L.total_bytes] */
  char* queues;         /* [n_replicas][L.queue_bytes] */
  double* summary;      /* [n_replicas][DCSIM_SUMMARY_K] */
  /* arrival pre-pass output, replica-major SoA: arrival k of replica r at [r * cap_arr + k] */
  double* arr_t;        /* arrival instant */
  double* arr_raw;      /* what the job size is a function of: the clamped uniform (inference, arrivals.py:8), the normal
                           deviate z (training, arrivals.py:10-11) — or the size itself under eco_route, which routes by it */
  uint32_t* arr_meta;   /* stream (bits 0-3) | routed DC (4-6) | next arrival of the stream was schedulable (7) | raw is the size (8) */
  uint32_t* arr_pred;   /* index of the stream's previous arrival (whose processing pushed this one), 0xffffffff = the constructor */
  /* merge scratch, same indexing */
  double* arr_tx;       /* xfer_done instant of arrival k (+inf: not schedulable / unreachable) */
  uint32_t* arr_fin;    /* number of arrivals j < k whose xfer_done instant is finite */
  /* merged event list, replica-major SoA: entry p of replica r at [r * 2 * cap_arr + p] (see ML_*) */
  double* ml_t;
  double* ml_aux;
  uint32_t* ml_meta;
  struct dcsim_arrhdr_t* arr_hdr;
  uint32_t* lat_hist;   /* [n_replicas][2][DCSIM_LAT_BINS] job-latency histograms, or NULL */
  uint32_t* mt_state;   /* [624][n_replicas] Mersenne Twister states (rng = MT19937 only), else NULL */
  uint32_t cap_arr;
  uint32_t _pad33;
  double end_eps;       /* end_time + 1e-9, the _schedule cut-off (SIM:161) */
  double max_transfer;  /* largest finite transfer_s[ingress][dc][jtype] of the scenario */
#ifdef DCSIM_DEVICE_TEST_HOOKS
  double test_time_quantum; /* TEST-ONLY device builds: see dcsim_test_quantize */
#endif
};

/* ---- small typed views ------------------------------------------------------------------------ */
template <typename T>
DCSIM_DEV T* dcsim_at(char* blk, int32_t off) { return reinterpret_cast<T*>(blk + off); }

struct dcsim_ctx_t {
  const dcsim_kparams_t* P;
  char* blk;             /* this replica's state block (shared memory on the GPU) */
  char* rec;             /* base the running-job record offsets (L.rn_*) apply to: blk when the records are staged with
                            the rest of the block, the block's home in HBM/L2 when only the head is staged */
  uint32_t r;            /* local replica index (its FIFOs, list and histogram row are addressed from it on demand) */
  dcsim_hdr_t* H;
  int lane;
  bool is_traced, is_logged;
  bool is_ghost;          /* a lane group without a replica (dcsim_replica_step): reads, never writes */
  /* Hot scalars kept in registers and written back to the header when the launch ends.  seq: lane 0's copy is
   * authoritative (only lane 0 runs handlers); the others are warp-uniform. */
  uint32_t seq;          /* successful pushes (SIM:163) */
  uint32_t cursor;       /* next entry of the event list */
  double now;            /* instant of the latest processed event, 0.0 before the first.  Until the next event is popped
                            it is also util_last_ts / last_energy_time of EVERY data centre: SIM:429-437 touches them all
                            on every event, so they never differ (DF_LAST_T holds it between launches) */
};

#define DCF(c, which) (dcsim_at<double>((c).blk, DCSIM_OFF_DC_F64 + (which) * DCSIM_MAX_DC * 8))
#define DCI(c, which) (dcsim_at<int32_t>((c).blk, DCSIM_OFF_DC_I32 + (which) * DCSIM_MAX_DC * 4))
#define CAND_T(c) (dcsim_at<double>((c).blk, DCSIM_OFF_CAND_T))
#define CAND_SEQ(c) (dcsim_at<uint32_t>((c).blk, DCSIM_OFF_CAND_SEQ))
#define LW_T(c) (dcsim_at<double>((c).blk, DCSIM_OFF_LW_T))
#define LW_AUX(c) (dcsim_at<double>((c).blk, DCSIM_OFF_LW_AUX))
#define LW_META(c) (dcsim_at<uint32_t>((c).blk, DCSIM_OFF_LW_META))
#define PEND_SEQ(c) (dcsim_at<uint32_t>((c).blk, DCSIM_OFF_PEND_SEQ))
#define XRING(c) (dcsim_at<uint32_t>((c).blk, DCSIM_OFF_XRING))

/* ================================================================================================
 * Philox4x32-10 stream; definition shared with oracle/philox_random.py
 * ============================================================================================== */
DCSIM_DEV void dcsim_philox_block(uint32_t k0, uint32_t k1, uint32_t b, uint32_t out[4]) {
  uint32_t c0 = b, c1 = 0u, c2 = 0u, c3 = 0u; /* block index < 2^30 here: rng_pos is 32-bit */
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = dcsim_mulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = dcsim_mulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

DCSIM_DEV double dcsim_u53(uint32_t w0, uint32_t w1) { /* genrand_res53 on two given words */
  /* ((w0 >> 5) * 2^26 + (w1 >> 6)) / 2^53 as CPython computes it in doubles; every step there is exact (the sum is an
   * integer below 2^53), so building the integer first and converting once gives the same bits */
  return (double)(((uint64_t)(w0 >> 5) << 26) | (uint64_t)(w1 >> 6)) * (1.0 / 9007199254740992.0);
}

/* ================================================================================================
 * Model leaves, evaluated in registers at job start
 * ============================================================================================== */
/* f**3 as CPython computes it (libm pow(f, 3.0), correctly rounded for every f this path sees):
 * error-free products via fma, one final rounding. */
DCSIM_DEV double dcsim_cube(double f) {
  const double p = f * f, pe = fma(f, f, -p);
  const double q = p * f, qe = fma(p, f, -q);
  return q + (qe + pe * f);
}

/* energy_paper.py:4-12   n * (alpha_p f^3 + beta_p f + gamma_p) */
DCSIM_DEV double dcsim_task_power(int n, double f_ghz, const dcsim_coeffs_t& k) {
  const double f = f_ghz > 0.0 ? f_ghz : 0.0;
  const double per_gpu = k.alpha_p * dcsim_cube(f) + k.beta_p * f + k.gamma_p;
  return (double)(n > 0 ? n : 0) * per_gpu;
}

/* latency_paper.py:4-9 */
DCSIM_DEV double dcsim_step_time(int n_gpus, double f_ghz, const dcsim_coeffs_t& k) {
  const int n = n_gpus > 1 ? n_gpus : 1;
  const double f = f_ghz > 1e-9 ? f_ghz : 1e-9;
  const double base = k.alpha_t + k.beta_t / f;
  if (n == 1) return base;
  return (base + k.gamma_t * (double)n) / (double)n;
}

/* x % y for x >= 0, y > 0 (what CPython computes with fmod).  q = floor(fl(x/y)) is the true quotient or one
 * more (rounding is monotone and integers are representable); x - q*y is then the true remainder or a tiny
 * negative number, both exact in one fma, and the fix-up addition is exact because the true remainder is
 * representable.  Checked against fmod() on the host build (tests/test_device_core_hostemu.py). */
DCSIM_DEV double dcsim_mod_pos(double x, double y) {
  const double q = floor(x / y);
  double r = fma(-q, y, x);
  if (r < 0.0) r += y;
  return r;
}

/* ================================================================================================
 * Arrival pre-pass (one THREAD per replica)
 *
 * In every algo on this path the arrival process does not depend on data-centre state: only arrival handlers
 * draw random numbers (arrivals.py:8,11,15,44; SIM:576) and routing is random.choice or eco_route's static
 * E_unit * size score (SIM:544-553, 575-577).  So the replica's whole arrival sequence — instants, routed DCs, which
 * pushes were schedulable — can be generated ahead of the event loop, in the reference's draw order (arrival events in
 * time order; inside one: size -> route -> next gap), by one thread per replica with all 32 lanes of a warp busy,
 * instead of on one lane of the replica's warp.
 *
 * The chain is kept as short as the draw order allows: what decides the NEXT draw is only the stream position (how
 * many words each sampler consumed) and the stream clocks.  A job size never feeds back (except under eco_route), so
 * the pre-pass stores the deviate it is a function of and the merge kernel evaluates pow / exp lane-parallel; the
 * rejection samplers decide through squeeze tests, and every lane of the warp ends an arrival with ONE converged
 * log() for its next gap.
 * ============================================================================================== */
/* Thread-level Philox stream with a 32-word ring (element i at ring[i * stride]: [word][thread] in shared memory on
 * the GPU; the pointer is passed alongside the stream, not inside it, so that the accesses compile to LDS/STS).  The
 * ring is topped up ONCE per arrival, by all lanes of the warp at the same program point; refilling inside the
 * samplers instead makes 32 out-of-phase lanes drag the warp through the block function at almost every draw
 * (measured: 43 % of the pre-pass). */
#define DCSIM_TRNG_RING 32u
/* Word source = CPython's own Mersenne Twister instead of Philox (dcsim_set_rng(h, DCSIM_RNG_MT19937)): the replica
 * then IS the stock reference at random.seed(seed0 + r) (SIM:71).  State: 624 words in HBM, element i at
 * mt[i * mt_stride] ([word][replica], coalesced across the warp's replicas). */
struct dcsim_mt_t { uint32_t* mt; uint64_t mt_stride; uint32_t mti; };
/* The stream is a template over the word source so that the Philox instantiation carries no trace of the other one
 * (a run-time switch cost the pre-pass 3 %: different register allocation, more local-memory traffic). */
template <bool MT> struct dcsim_trng_t { uint32_t k0, k1, pos, filled; };
template <> struct dcsim_trng_t<true> { uint32_t k0, k1, pos, filled; dcsim_mt_t mt; };

/* MT19937 (Matsumoto & Nishimura) as CPython drives it: Modules/_randommodule.c init_by_array / genrand_uint32. */
#define DCSIM_MT_N 624u
#define DCSIM_MT_M 397u
#define DCSIM_MT_AT(g, i) ((g).mt[(uint64_t)(i) * (g).mt_stride])
DCSIM_DEV void dcsim_mt_seed(dcsim_mt_t& g, uint64_t seed) { /* random.seed(int): key = 32-bit digits of |seed| */
  const uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  const uint32_t len = key[1] ? 2u : 1u;
  uint32_t prev = 19650218u;
  DCSIM_MT_AT(g, 0) = prev;
  for (uint32_t i = 1; i < DCSIM_MT_N; ++i) { prev = 1812433253u * (prev ^ (prev >> 30)) + i; DCSIM_MT_AT(g, i) = prev; }
  uint32_t i = 1, j = 0;
  prev = DCSIM_MT_AT(g, 0);
  for (uint32_t k = DCSIM_MT_N; k; --k) {
    prev = (DCSIM_MT_AT(g, i) ^ ((prev ^ (prev >> 30)) * 1664525u)) + key[j] + j;
    DCSIM_MT_AT(g, i) = prev;
    if (++i >= DCSIM_MT_N) { DCSIM_MT_AT(g, 0) = prev; i = 1; }
    if (++j >= len) j = 0;
  }
  for (uint32_t k = DCSIM_MT_N - 1u; k; --k) {
    prev = (DCSIM_MT_AT(g, i) ^ ((prev ^ (prev >> 30)) * 1566083941u)) - i;
    DCSIM_MT_AT(g, i) = prev;
    if (++i >= DCSIM_MT_N) { DCSIM_MT_AT(g, 0) = prev; i = 1; }
  }
  DCSIM_MT_AT(g, 0) = 0x80000000u;
  g.mti = DCSIM_MT_N;
}
DCSIM_DEV uint32_t dcsim_mt_next(dcsim_mt_t& g) {
  if (g.mti >= DCSIM_MT_N) { /* regenerate the 624 words in place */
    /* word kk needs the OLD words kk, kk+1 and word kk+M (old while kk+M < N, already NEW once it wraps); the last
     * word pairs with the NEW word 0 — reading the array in place gives exactly that */
    for (uint32_t kk = 0; kk < DCSIM_MT_N; ++kk) {
      const uint32_t a = DCSIM_MT_AT(g, kk);
      const uint32_t b = DCSIM_MT_AT(g, kk + 1u < DCSIM_MT_N ? kk + 1u : 0u);
      const uint32_t m = DCSIM_MT_AT(g, kk + DCSIM_MT_M < DCSIM_MT_N ? kk + DCSIM_MT_M : kk + DCSIM_MT_M - DCSIM_MT_N);
      const uint32_t y = (a & 0x80000000u) | (b & 0x7fffffffu);
      DCSIM_MT_AT(g, kk) = m ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    g.mti = 0u;
  }
  uint32_t y = DCSIM_MT_AT(g, g.mti++);
  y ^= y >> 11;
  y ^= (y << 7) & 0x9d2c5680u;
  y ^= (y << 15) & 0xefc60000u;
  y ^= y >> 18;
  return y;
}

template <bool MT>
DCSIM_DEV void dcsim_trng_block(dcsim_trng_t<MT>& g, uint32_t* ring, int stride) { /* appends block filled/4 */
  uint32_t w[4];
  if constexpr (MT) { w[0] = dcsim_mt_next(g.mt); w[1] = dcsim_mt_next(g.mt); w[2] = dcsim_mt_next(g.mt); w[3] = dcsim_mt_next(g.mt); }
  else dcsim_philox_block(g.k0, g.k1, g.filled >> 2, w);
  const uint32_t i = g.filled & (DCSIM_TRNG_RING - 1u);
  ring[(i + 0u) * stride] = w[0]; ring[(i + 1u) * stride] = w[1];
  ring[(i + 2u) * stride] = w[2]; ring[(i + 3u) * stride] = w[3];
  g.filled += 4u;
}
template <bool MT>
DCSIM_DEV void dcsim_trng_topup(dcsim_trng_t<MT>& g, uint32_t* ring, int stride) {
  /* one block at a time: generating two with interleaved rounds (more ILP for a latency-bound kernel) measured 4 %
     SLOWER — the longer live ranges cost more than the overlap gains (profiles/r02_variants_ab.md) */
  while (g.filled - g.pos <= DCSIM_TRNG_RING - 4u) dcsim_trng_block(g, ring, stride);
}
/* A sampler out-ran the ring (a long rejection run): one more block, out of line.  The Philox flavour takes the
 * generator's fields BY VALUE — handing out &g would pin the whole generator (pos, filled) in local memory for the
 * entire kernel, a load and a store around every word drawn. */
#ifndef DCSIM_HOST_EMU
static __device__ __noinline__
#else
static
#endif
void dcsim_trng_dry_philox(uint32_t k0, uint32_t k1, uint32_t filled, uint32_t* ring, int stride) {
  uint32_t w[4];
  dcsim_philox_block(k0, k1, filled >> 2, w);
  const uint32_t i = filled & (DCSIM_TRNG_RING - 1u);
  ring[(i + 0u) * stride] = w[0]; ring[(i + 1u) * stride] = w[1];
  ring[(i + 2u) * stride] = w[2]; ring[(i + 3u) * stride] = w[3];
}
/* The samplers call dcsim_trng_need(n) once where they are about to draw n words (n <= 4: one block refills the ring
 * by that much) and then take the words without a check each.  After the per-arrival top-up the ring holds >= 29 words,
 * so only long rejection runs ever refill here. */
template <bool MT>
DCSIM_DEV void dcsim_trng_need(dcsim_trng_t<MT>& g, uint32_t* ring, int stride, uint32_t n) {
  if (g.filled - g.pos < n) {
    if constexpr (MT) dcsim_trng_block(g, ring, stride);
    else { dcsim_trng_dry_philox(g.k0, g.k1, g.filled, ring, stride); g.filled += 4u; }
  }
}
template <bool MT>
DCSIM_DEV uint32_t dcsim_trng_word(dcsim_trng_t<MT>& g, uint32_t* ring, int stride) { /* after dcsim_trng_need */
  return ring[(g.pos++ & (DCSIM_TRNG_RING - 1u)) * stride];
}
template <bool MT>
DCSIM_DEV double dcsim_trng_random(dcsim_trng_t<MT>& g, uint32_t* ring, int stride) { /* after dcsim_trng_need(2) */
  const uint32_t a = dcsim_trng_word(g, ring, stride), b = dcsim_trng_word(g, ring, stride);
  return dcsim_u53(a, b);
}

/* Constants of the thinning squeeze for one arrival stream (computed once per replica). */
struct dcsim_squeeze_t {
  double max_rate;   /* rate * (1 + |amp|), arrivals.py:40 */
  double x1_min;     /* 1-U1 >= x1_min guarantees the candidate gap w = -log(1-U1)/max_rate <= w_max */
  double eps;        /* |lambda(t+w) - lambda(t)| / max_rate <= eps for 0 <= w <= w_max (+ the slop of the cheap lambda(t)) */
  double inv_period; /* 1 / period, for the cheap phase of lambda(t) */
};
DCSIM_DEV dcsim_squeeze_t dcsim_squeeze_setup(const dcsim_arrival_t& a, double two_pi) {
  dcsim_squeeze_t q;
  const double abs_amp = a.amp < 0.0 ? -a.amp : a.amp;
  q.max_rate = a.rate * (1.0 + abs_amp);
  double w_max = 8.0 / q.max_rate;                 /* covers all but e^-8 of the candidate gaps ... */
  if (w_max > 0.002 * a.period) w_max = 0.002 * a.period; /* ... unless the rate varies too fast for that */
  q.x1_min = exp(-q.max_rate * w_max * 0.999);     /* 0.999: errs towards the exact path */
  /* lambda is rate*(1+amp*sin(2 pi t/period)) clipped at 0: Lipschitz constant rate*|amp|*2 pi/period.  The band's
   * centre lambda(t) itself is evaluated in single precision (absolute error of the sine < 1e-6, i.e. < 1e-6 of
   * max_rate in lambda/max_rate): 4e-6 of extra half-width covers it with room to spare. */
  q.eps = a.rate * abs_amp * two_pi * w_max / a.period / q.max_rate + 4e-6 + 1e-9;
  q.inv_period = a.period > 0.0 ? 1.0 / a.period : 0.0;
  return q;
}

/* sin(2 pi * frac(t / period)) good to ~1e-6 absolute: only ever used to CENTRE the squeeze band, never to decide. */
DCSIM_DEV double dcsim_sin_phase_approx(double t, double inv_period, double two_pi) {
  const double tp = t * inv_period;
  const double ph = (tp - floor(tp)) * two_pi; /* [0, 2 pi) */
#ifdef DCSIM_HOST_EMU
  return sin(ph);
#else
  float x = (float)ph;
  x = x > 3.14159274f ? x - 6.28318548f : x;   /* MUFU.SIN is accurate to 2^-21.4 on [-pi, pi] */
  return (double)__sinf(x);
#endif
}

/* arrivals.py:35-48 with random.py:617; returns the gap (+inf for a dead stream).
 *
 * Sinusoid "thinning" (arrivals.py:41-45) redraws (w, U2) until U2 <= lambda(t+w)/max_rate, keeping only the last w.
 * The decision of a candidate is taken WITHOUT log and sin whenever it is not close: w <= w_max is implied by
 * 1-U1 >= x1_min, and then lambda(t+w)/max_rate lies within eps of p0 ~ lambda(t)/max_rate, so U2 <= p0 - eps
 * accepts and U2 > p0 + eps rejects exactly as the full formula would; only candidates inside the +-eps band (or with
 * a very long gap) evaluate the reference's expression.  Same words consumed, same decisions, same w — but a thread
 * spends ~20 instructions instead of ~500 on a rejected candidate, which matters because a warp's lanes all wait
 * for the lane with the longest rejection run.  The accepted candidate's gap -log(1-U1)/max_rate is left to
 * dcsim_t_gap_finish(), which the arrival loop calls behind a warp-wide reconvergence point: written after the loop
 * in the same function, the compiler duplicated the log() into every loop exit and the lanes ran it one exit at a
 * time (ncu: 18 % of the kernel's instructions at a third of the lanes). */
/* What the draws of one inter-arrival gap leave to be done: gap = is_w ? v : -log(v) / rate. */
struct dcsim_gap_draw_t { double v, rate; bool is_w; };
template <bool MT>
DCSIM_DEV dcsim_gap_draw_t dcsim_t_gap_draw(dcsim_trng_t<MT>& g, uint32_t* ring, int stride, const dcsim_spec_t& sp, const dcsim_squeeze_t& q,
                                            int jt, double t, uint32_t* status) {
  const dcsim_arrival_t& a = sp.arr[jt];
  dcsim_gap_draw_t out;
  out.v = DCSIM_INF; out.rate = 1.0; out.is_w = true; /* a dead stream */
  if (a.mode == DCSIM_ARR_POISSON) {
    if (a.rate <= 0.0) return out;
    dcsim_trng_need(g, ring, stride, 2u);
    out.v = 1.0 - dcsim_trng_random(g, ring, stride); out.rate = a.rate; out.is_w = false;
  } else if (a.mode == DCSIM_ARR_SINUSOID) {
    const double max_rate = q.max_rate;
    double lam0 = a.rate * (1.0 + a.amp * dcsim_sin_phase_approx(t, q.inv_period, sp.two_pi));
    lam0 = lam0 > 0.0 ? lam0 : 0.0;
    const double p0 = lam0 / max_rate, p_lo = p0 - q.eps, p_hi = p0 + q.eps;
    for (int it = 0;; ++it) {
      if (it >= DCSIM_REJECTION_LIMIT) { *status |= DCSIM_ST_RNG_RUNAWAY; return out; }
      dcsim_trng_need(g, ring, stride, 4u);
      const double x1 = 1.0 - dcsim_trng_random(g, ring, stride);
      const double u2 = dcsim_trng_random(g, ring, stride);
      if (x1 >= q.x1_min) {
        if (u2 > p_hi) continue;                                                        /* certainly rejected */
        if (u2 <= p_lo) { out.v = x1; out.rate = max_rate; out.is_w = false; break; }   /* certainly accepted */
      }
      const double w = -log(x1) / max_rate;               /* in the band: the reference's expression */
      const double tc = t + w;
      double lam = a.rate * (1.0 + a.amp * sin(sp.two_pi * dcsim_mod_pos(tc, a.period) / a.period));
      lam = lam > 0.0 ? lam : 0.0;
      if (u2 <= lam / max_rate) { out.v = w; break; }
    }
  }
  return out;
}
DCSIM_DEV double dcsim_t_gap_finish(const dcsim_gap_draw_t& d) { return d.is_w ? d.v : -log(d.v) / d.rate; }
template <bool MT>
DCSIM_DEV double dcsim_t_gap(dcsim_trng_t<MT>& g, uint32_t* ring, int stride, const dcsim_spec_t& sp, const dcsim_squeeze_t& q, int jt,
                             double t, uint32_t* status) {
  return dcsim_t_gap_finish(dcsim_t_gap_draw(g, ring, stride, sp, q, jt, t, status));
}

/* arrivals.py:5-11 with random.py:541-549, 597: draws what the job size is a function of — the clamped uniform of the
 * Pareto branch, the Kinderman-Monahan normal deviate of the log-normal branch — consuming exactly the reference's words.
 * The K-M acceptance zz <= -log(u2) is decided by the bounds 1-u <= -log(u) <= (1-u)/u (1-u2 is exact: u2 is a
 * multiple of 2^-53) whenever they settle it with a 1e-6 relative margin — far more than any libm's log is off — and
 * by the reference's expression otherwise.  dcsim_size_from_raw() finishes the job. */
template <bool MT>
DCSIM_DEV double dcsim_t_size_raw(dcsim_trng_t<MT>& g, uint32_t* ring, int stride, const dcsim_spec_t& sp, int jt, uint32_t* status) {
  if (jt == DCSIM_JT_INFERENCE) {
    dcsim_trng_need(g, ring, stride, 2u);
    const double x = 1.0 - dcsim_trng_random(g, ring, stride);
    return x > sp.uniform_floor ? x : sp.uniform_floor;
  }
  double z = 0.0;
  for (int it = 0;; ++it) {
    if (it >= DCSIM_REJECTION_LIMIT) { *status |= DCSIM_ST_RNG_RUNAWAY; break; }
    dcsim_trng_need(g, ring, stride, 4u);
    const double u1 = dcsim_trng_random(g, ring, stride);
    const double u2 = 1.0 - dcsim_trng_random(g, ring, stride);
    z = sp.nv_magicconst * (u1 - 0.5) / u2;
    const double zz = z * z / 4.0;
    const double om = 1.0 - u2;
    if (zz <= om * 0.999999) break;        /* zz < 1-u2 <= -log(u2) */
    if (zz * u2 > om * 1.000001) continue; /* zz > (1-u2)/u2 >= -log(u2) */
    if (zz <= -log(u2)) break;
  }
  return z;
}

/* x % y as above when a guess of the quotient is at hand (finish_time % log_interval with the number of log ticks so
 * far: exact whenever the clock is between the q-th and the (q+1)-th multiple of y, which is where it is unless a tick
 * instant has drifted by an ulp).  With the right q the remainder x - q*y is exact in one fma (it is representable: it
 * is what fmod returns); a wrong q puts the true value outside [0, y), and no rounding can move it back inside, so
 * "the result lies in [0, y)" certifies both q and the result.  Otherwise: the division. */
DCSIM_DEV double dcsim_mod_pos_hint(double x, double y, uint32_t q_guess) {
  const double r = fma(-(double)q_guess, y, x);
  if (r >= 0.0 && r < y) return r;
  return dcsim_mod_pos(x, y);
}

/* arrivals.py:7-8 / 10-11 from the stored deviate. */
DCSIM_DEV double dcsim_size_from_raw(const dcsim_spec_t& sp, double raw, int jt) {
  if (jt == DCSIM_JT_INFERENCE) return sp.pareto_xm / pow(raw, sp.pareto_inv_alpha);
  const double v = exp(sp.lognorm_mu + raw * sp.lognorm_sigma);
  return v > sp.lognorm_floor ? v : sp.lognorm_floor;
}

/* TEST HOOK (see oracle/dcsim_oracle.c g_test_time_quantum): rounds arrival and xfer_done instants up to a multiple of a
 * quantum so that same-instant events become common and the tie-breaking below is exercised.  Compiled into the host
 * build and into the test-only device builds made with -DDCSIM_DEVICE_TEST_HOOKS (tests/test_gpu_ties.py), where the
 * quantum travels in the launch parameters (every caller has them as `P`); the product library has neither. */
#if defined(DCSIM_HOST_EMU) || defined(DCSIM_DEVICE_TEST_HOOKS)
DCSIM_DEV double dcsim_test_quantize_by(double q, double t) {
  return (q > 0.0 && !(t == DCSIM_INF)) ? ceil(t / q) * q : t;
}
#endif
#if defined(DCSIM_HOST_EMU)
static double dcsim_test_time_quantum = 0.0;
#define dcsim_test_quantize(t) dcsim_test_quantize_by(dcsim_test_time_quantum, (t))
#elif defined(DCSIM_DEVICE_TEST_HOOKS)
#define dcsim_test_quantize(t) dcsim_test_quantize_by(P->test_time_quantum, (t))
#else
#define dcsim_test_quantize(t) (t)
#endif

#define DCSIM_NO_PRED 0xffffffffu
/* Push rank of stream q's pending arrival: the constructor pushed the first arrivals in stream order (SIM:154-156),
 * every later one was pushed while its predecessor — list entry `last` — was being processed (SIM:591-592). */
DCSIM_DEV uint32_t dcsim_stream_rank(uint32_t last, int q) { return last == DCSIM_NO_PRED ? (uint32_t)q : 16u + last; }

/* One replica's arrival list.  Per-thread scratch, element s of each array at [s * stride] ([slot][thread] in shared
 * memory): `next_t` the 2*n_ing stream clocks, `last_idx` the list index of each stream's latest arrival, `ring` the
 * DCSIM_TRNG_RING staged words of the stream. */
template <bool MT>
DCSIM_DEV void dcsim_generate_arrivals(const dcsim_kparams_t* P, uint64_t r, double* next_t, uint32_t* last_idx, uint32_t* ring, int stride) {
  const dcsim_spec_t& sp = P->spec;
  const int n_streams = 2 * sp.n_ing;
  dcsim_trng_t<MT> g;
  const uint64_t key = P->seed0 + r;
  g.k0 = (uint32_t)key; g.k1 = (uint32_t)(key >> 32); g.pos = 0u; g.filled = 0u;
  if constexpr (MT) { g.mt.mt = P->mt_state + r; g.mt.mt_stride = P->n_replicas; dcsim_mt_seed(g.mt, key); }
  uint32_t status = 0u, first_mask = 0u, count = 0u;
  const double end_eps = P->end_eps;
  dcsim_squeeze_t sq[2];
  sq[0] = dcsim_squeeze_setup(sp.arr[0], sp.two_pi);
  sq[1] = dcsim_squeeze_setup(sp.arr[1], sp.two_pi);
  for (int s = 0; s < n_streams; ++s) { /* SIM:154-156 */
    dcsim_trng_topup(g, ring, stride);
    const double t = dcsim_test_quantize(0.0 + dcsim_t_gap(g, ring, stride, sp, (s & 1) ? sq[1] : sq[0], s & 1, 0.0, &status));
    const bool ok = !(t == DCSIM_INF) && !(t > end_eps);
    next_t[s * stride] = ok ? t : DCSIM_INF;
    last_idx[s * stride] = DCSIM_NO_PRED;
    if (ok) first_mask |= 1u << s;
  }
  double* out_t = P->arr_t + r * (uint64_t)P->cap_arr;
  double* out_raw = P->arr_raw + r * (uint64_t)P->cap_arr;
  uint32_t* out_meta = P->arr_meta + r * (uint64_t)P->cap_arr;
  uint32_t* out_pred = P->arr_pred + r * (uint64_t)P->cap_arr;
  const int k_bits = dcsim_bit_length((uint32_t)sp.n_dc);
  /* The loop is WARP-uniform: a replica that has ended (end_time, an overflow) stays in it, switched off, until the
   * warp's last one has — so that the lanes can be made to reconverge (a full-mask __syncwarp) between the divergent
   * part of an arrival (rejection loops of different lengths) and the part all of them share (the log of the gap). */
  bool alive = true;
  for (;;) {
    int s = -1;
    double t = DCSIM_INF;
    bool tie = false;
    if (alive) {
      for (int q = 0; q < n_streams; ++q) {
        const double tq = next_t[q * stride];
        if (tq < t) { t = tq; s = q; tie = false; } else if (tq == t) tie = true;
      }
      if (s < 0 || t > sp.end_time) alive = false; /* heap empty / SIM:427 */
      else if (tie) { /* heap order is (t, seq): pending arrivals at the same instant pop in push order (rare: ~rate * ulp(t)) */
        for (int q = s + 1; q < n_streams; ++q)
          if (next_t[q * stride] == t && dcsim_stream_rank(last_idx[q * stride], q) < dcsim_stream_rank(last_idx[s * stride], s)) s = q;
      }
      if (status) alive = false;
    }
    if (!dcsim_event_any_full(alive)) break;
    const int jt = s & 1;
    double raw = 0.0;
    int dc_sel = 0;
    uint32_t raw_is_size = 0u;
    dcsim_gap_draw_t gd;
    gd.v = DCSIM_INF; gd.rate = 1.0; gd.is_w = true;
    if (alive) {
      dcsim_trng_topup(g, ring, stride);
      raw = dcsim_t_size_raw(g, ring, stride, sp, jt, &status); /* draw order: size -> route -> next gap (SIM:540,576,591) */
      if (sp.route_rule == DCSIM_ROUTE_ECO) { /* SIM:544-553: routes by E_unit * size, so the size is needed here */
        const double size = dcsim_size_from_raw(sp, raw, jt);
        double best = sp.dc[0].eco_e_unit[jt] * size;
        for (int d = 1; d < sp.n_dc; ++d) {
          const double score = sp.dc[d].eco_e_unit[jt] * size;
          if (score < best) { best = score; dc_sel = d; }
        }
        raw = size; raw_is_size = 0x100u;
      } else { /* random.choice: random.py:242-250 */
        dcsim_trng_need(g, ring, stride, 1u);
        uint32_t v = dcsim_trng_word(g, ring, stride) >> (32 - k_bits);
        for (int it = 0; v >= (uint32_t)sp.n_dc; ++it) {
          if (it >= DCSIM_REJECTION_LIMIT) { status |= DCSIM_ST_RNG_RUNAWAY; v = 0u; break; }
          dcsim_trng_need(g, ring, stride, 1u);
          v = dcsim_trng_word(g, ring, stride) >> (32 - k_bits);
        }
        dc_sel = (int)v;
      }
      dcsim_squeeze_t q; /* selected field by field: indexing sq[] with jt would put the array in local memory */
      q.max_rate = jt ? sq[1].max_rate : sq[0].max_rate; q.x1_min = jt ? sq[1].x1_min : sq[0].x1_min;
      q.eps = jt ? sq[1].eps : sq[0].eps; q.inv_period = jt ? sq[1].inv_period : sq[0].inv_period;
      gd = dcsim_t_gap_draw(g, ring, stride, sp, q, jt, t, &status);
    }
    dcsim_sync_full(); /* every lane is back from its rejection loops */
    if (alive) {
      const double tn = dcsim_test_quantize(t + dcsim_t_gap_finish(gd));
      const bool has_next = !(tn == DCSIM_INF) && !(tn > end_eps);
      next_t[s * stride] = has_next ? tn : DCSIM_INF;
      if (count >= P->cap_arr) { status |= DCSIM_ST_ARRIVALS_OVERFLOW; alive = false; }
      else {
        out_t[count] = t;
        out_raw[count] = raw;
        out_meta[count] = (uint32_t)s | ((uint32_t)dc_sel << 4) | (has_next ? 0x80u : 0u) | raw_is_size;
        out_pred[count] = last_idx[s * stride];
        last_idx[s * stride] = count;
        ++count;
      }
    }
  }
  dcsim_arrhdr_t h;
  h.count = count; h.first_mask = first_mask; h.rng_words = g.pos; h.status = status;
  h.ml_count = 0u; h.max_ahead = 0u; h._pad[0] = h._pad[1] = 0u;
  P->arr_hdr[r] = h;
}

/* ================================================================================================
 * List merge (one WARP per replica, lane-parallel over its arrivals)
 *
 * An arrival at t is followed by its xfer_done at t + transfer_s[ingress][dc][jtype] (SIM:580-588) — a constant per
 * (ingress, DC, job type), known as soon as the arrival is.  So both kinds of event go into ONE time-ordered list and
 * the event loop needs no pool of in-flight transfers (no push, no removal, no min-rescan per transfer).  Order is the
 * heap's (t, seq): between two list events seq order is push order, and every push in the list happens while an
 * arrival is processed (the xfer_done first, then the stream's next arrival, SIM:580-592; the constructor's pushes
 * before all, in stream order) — so ties are resolved exactly from list indices alone:
 *     arrival k   pushed while arrival pred(k) was processed, after pred(k)'s own xfer_done;
 *     xfer_done j pushed while arrival j was processed.
 * The position of an event is the number of events before it; with the arrivals already in order only the transfers
 * within max_transfer of it need to be looked at.  The same pass evaluates the job sizes (pow / exp), all 32 lanes
 * on different arrivals.
 * ============================================================================================== */
DCSIM_DEV bool dcsim_finite(double x) { return !(x == DCSIM_INF); }

/* The merge works on a sliding window of the replica's arrivals kept in shared memory (a ring indexed by the arrival
 * number): what the position scans read — arrival instant, xfer_done instant, running count of finite transfers,
 * predecessor — plus what the emission needs (size, meta).  Everything is also in HBM (the pre-pass output and the
 * merge's own scratch), which is where a scan falls back to when it reaches behind the ring (very long transfers). */
#ifndef DCSIM_MERGE_RING
#define DCSIM_MERGE_RING 128u /* a power of two >= DCSIM_LANES */
#endif
struct dcsim_merge_ring_t {
  double at[DCSIM_MERGE_RING], tx[DCSIM_MERGE_RING], sz[DCSIM_MERGE_RING];
  uint32_t fin[DCSIM_MERGE_RING], pred[DCSIM_MERGE_RING], meta[DCSIM_MERGE_RING];
};

/* List positions of arrival k (pos_a) and of its xfer_done (pos_x, when `xin`): the number of list events before each.
 * CHECKED = false: every index the scans touch is known to be in the ring (the common case, decided once per chunk);
 * CHECKED = true: indices below `lo` are read from HBM.  `thr_gap` = max_transfer plus a margin far above any rounding:
 * an arrival earlier than (t - thr_gap) has its xfer_done — if it has one — before t, and so have all before it. */
template <bool CHECKED>
DCSIM_DEV void dcsim_merge_positions(const dcsim_merge_ring_t* ring, const double* at, const double* tx, const uint32_t* fin,
                                     const uint32_t* pred, uint32_t lo, uint32_t n, uint32_t k, double tk, double txk, uint32_t pk,
                                     double thr_gap, bool xin, uint32_t* pos_a, uint32_t* pos_x) {
  const uint32_t RM = DCSIM_MERGE_RING - 1u;
#define MR_AT(j) ((!CHECKED || (j) >= lo) ? ring->at[(j) & RM] : at[(j)])
#define MR_TX(j) ((!CHECKED || (j) >= lo) ? ring->tx[(j) & RM] : tx[(j)])
#define MR_FIN(j) ((!CHECKED || (j) >= lo) ? ring->fin[(j) & RM] : fin[(j)])
#define MR_PRED(j) ((!CHECKED || (j) >= lo) ? ring->pred[(j) & RM] : pred[(j)])
  /* One walk back over the earlier arrivals j serves both positions: transfer j precedes arrival k if tx_j < t_k (or
   * ties and was pushed first), and precedes transfer k if tx_j <= tx_k.  tx_k >= t_k, so the second question is
   * settled ("everything further back is earlier") no later than the first. */
  uint32_t cnt = 0u, cx = 0u;
  const double far_a = tk - thr_gap, far_x = xin ? txk - thr_gap : DCSIM_INF;
  bool x_open = xin;
  for (uint32_t j = k; j > 0u;) {
    --j;
    const double tj = MR_AT(j), txj = MR_TX(j);
    if (x_open) {
      if (tj < far_x) { cx += MR_FIN(j) + (dcsim_finite(txj) ? 1u : 0u); x_open = false; }
      else if (txj <= txk) ++cx; /* tie: pushed earlier */
    }
    if (tj < far_a) { cnt += MR_FIN(j) + (dcsim_finite(txj) ? 1u : 0u); break; } /* every finite one up to j is earlier */
    if (txj < tk || (txj == tk && pk != DCSIM_NO_PRED && j <= pk)) ++cnt;
  }
  *pos_a = k + cnt;
  *pos_x = 0xffffffffu;
  if (xin) {
    uint32_t ca = k + 1u; /* arrivals 0..k come first (their pushes precede arrival k's processing) */
    for (uint32_t i = k + 1u; i < n; ++i) { /* i < frontier: stage 1 ran until an arrival later than txk */
      const double ti = MR_AT(i);
      if (ti > txk) break;
      if (ti < txk) ++ca;
      else { const uint32_t pi = MR_PRED(i); if (pi == DCSIM_NO_PRED || pi < k) ++ca; } /* tie: arrival i was pushed before arrival k ran */
      if (MR_TX(i) < txk) ++cx;                                                         /* tie: pushed later */
    }
    *pos_x = ca + cx;
  }
#undef MR_AT
#undef MR_TX
#undef MR_FIN
#undef MR_PRED
}

DCSIM_DEV void dcsim_merge_arrivals(const dcsim_kparams_t* P, uint64_t r, int lane, dcsim_merge_ring_t* ring) {
  const dcsim_spec_t& sp = P->spec;
  dcsim_arrhdr_t* hdr = P->arr_hdr + r;
  const uint32_t n = hdr->count;
  const uint64_t ab = r * (uint64_t)P->cap_arr;
  const double* at = P->arr_t + ab;
  double* raw = P->arr_raw + ab;
  const uint32_t* am = P->arr_meta + ab;
  const uint32_t* pred = P->arr_pred + ab;
  double* tx = P->arr_tx + ab;
  uint32_t* fin = P->arr_fin + ab;
  double* mt = P->ml_t + 2ull * ab;
  double* ma = P->ml_aux + 2ull * ab;
  uint32_t* mm = P->ml_meta + 2ull * ab;
  const double end = sp.end_time, end_eps = P->end_eps, tmax = P->max_transfer;
  const double thr_gap = tmax + (end + 1.0) * 1e-12 + 1e-300; /* > max_transfer by far more than any rounding at t <= end */
  const uint32_t RM = DCSIM_MERGE_RING - 1u;

  uint32_t frontier = 0u;  /* arrivals [0, frontier) have their size / xfer_done instant / finite count (ring + HBM) */
  uint32_t fin_base = 0u;  /* finite xfer_done instants among them */
  uint32_t n_x = 0u, ahead = 0u;
  for (uint32_t k0 = 0u; k0 < n; k0 += DCSIM_LANES) {
    /* ---- stage 1, as far ahead as this chunk's scans can reach: past the chunk itself and on until an arrival later
     * than every xfer_done instant of the chunk (<= its last arrival + max_transfer) */
    const uint32_t k_last = k0 + DCSIM_LANES - 1u < n - 1u ? k0 + DCSIM_LANES - 1u : n - 1u;
    for (;;) {
      if (frontier > k_last) {
        if (frontier >= n) break;
        const double t_hi = (frontier - k_last <= DCSIM_MERGE_RING ? ring->at[k_last & RM] : at[k_last]) + thr_gap;
        if (ring->at[(frontier - 1u) & RM] > t_hi) break;
      }
      const uint32_t k = frontier + (uint32_t)lane;
      bool f = false;
      double v = DCSIM_INF, size = 0.0, tk = 0.0;
      uint32_t meta = 0u;
      if (k < n) {
        meta = am[k];
        const int stream = (int)(meta & 15u), jt = stream & 1, ing = stream >> 1, dc = (int)((meta >> 4) & 7u);
        size = raw[k];
        if (!(meta & 0x100u)) size = dcsim_size_from_raw(sp, size, jt);
        tk = at[k];
        v = dcsim_test_quantize(tk + sp.transfer_s[ing][dc][jt]); /* SIM:580: now + transfer_s, now == the arrival instant */
        f = dcsim_finite(v);
      }
      const uint32_t votes = dcsim_warp_ballot(f);
      if (k < n) {
        const uint32_t fk = fin_base + dcsim_popc(votes & dcsim_lanemask_lt(lane));
        ring->at[k & RM] = tk; ring->tx[k & RM] = v; ring->sz[k & RM] = size;
        ring->fin[k & RM] = fk; ring->pred[k & RM] = pred[k]; ring->meta[k & RM] = meta;
        tx[k] = v; fin[k] = fk; raw[k] = size; /* the HBM copies back the ring up */
      }
      fin_base += dcsim_popc(votes);
      frontier += DCSIM_LANES;
      dcsim_warp_sync(); /* ring / HBM entries written by other lanes are read below */
    }
    const uint32_t lo = frontier > DCSIM_MERGE_RING ? frontier - DCSIM_MERGE_RING : 0u; /* ring holds [lo, frontier) */
    /* every backward scan of this chunk stops at or before `lo` when the oldest ring entry is already "far" from the
       chunk's first arrival (forward scans end below the frontier by construction of stage 1) */
    const bool covered = lo == 0u || (k0 >= lo && ring->at[lo & RM] < ring->at[k0 & RM] - thr_gap);

    /* ---- stage 2: list positions of this chunk's arrivals and their xfer_done events, emission */
    const uint32_t k = k0 + (uint32_t)lane;
    if (k < n) {
      const bool kin = k >= lo;
      const double tk = kin ? ring->at[k & RM] : at[k], txk = kin ? ring->tx[k & RM] : tx[k];
      const uint32_t meta = kin ? ring->meta[k & RM] : am[k], pk = kin ? ring->pred[k & RM] : pred[k];
      const bool xs = dcsim_finite(txk) && !(txk > end_eps); /* SIM:160-163 */
      const bool xin = xs && !(txk > end);                    /* SIM:427: later events are never processed */
      uint32_t pos_a, pos_x;
      if (covered) dcsim_merge_positions<false>(ring, at, tx, fin, pred, lo, n, k, tk, txk, pk, thr_gap, xin, &pos_a, &pos_x);
      else dcsim_merge_positions<true>(ring, at, tx, fin, pred, lo, n, k, tk, txk, pk, thr_gap, xin, &pos_a, &pos_x);
      if (xin) { ++n_x; ahead = pos_x - pos_a > ahead ? pos_x - pos_a : ahead; }
      const uint32_t stream = meta & 15u;
      mt[pos_a] = tk;
      ma[pos_a] = dcsim_hilo_f64(0u, pos_x);
      mm[pos_a] = (stream << 1) | ((meta & 0x80u) ? ML_A_NEXT : 0u) | (xs ? ML_A_XSCHED : 0u) | (xin ? ML_A_XIN : 0u);
      if (xin) {
        mt[pos_x] = txk;
        ma[pos_x] = kin ? ring->sz[k & RM] : raw[k];
        mm[pos_x] = ML_XFER | (((meta >> 4) & 7u) << 1) | ((stream & 1u) << 4) | ((stream >> 1) << 5) | (k << 8);
      }
    }
    dcsim_warp_sync(); /* this chunk's ring reads are done before the next chunk's stage 1 overwrites old entries */
  }
  n_x = dcsim_warp_add_u32(n_x);
  ahead = dcsim_warp_max_u32(ahead);
  if (lane == 0) {
    hdr->ml_count = n + n_x;
    hdr->max_ahead = ahead;
    if (ahead > (uint32_t)P->L.xring_mask) hdr->status |= DCSIM_ST_XFER_OVERFLOW; /* the seq ring would wrap onto a pending entry */
  }
}

/* ================================================================================================
 * Event-set primitives
 * ============================================================================================== */
/* Strided arg-min over (t[i], seq[i]), i < n, in (t, seq) lexicographic order (SIM:163: heap key).
 * Times are >= 0, so their IEEE bit patterns order like unsigned integers and the reduction is three
 * REDUX.MIN.U32.  Returns the winning index to every lane, -1 if every entry is +inf / n == 0. */
DCSIM_DEV int dcsim_argmin_ts(const double* t, const uint32_t* seq, int n, int lane, double* t_out, uint32_t* seq_out) {
#if DCSIM_LANES == 32
  if (n <= 32) { /* the common case (pools rarely hold more than a warp's worth): one entry per lane, no loop */
    const bool in = lane < n;
    const double ti = in ? t[lane] : DCSIM_INF;
    const uint32_t s = in ? seq[lane] : 0xffffffffu;
    const uint32_t h = dcsim_hi(ti), l = dcsim_lo(ti);
    const uint32_t mh = dcsim_warp_min_u32(h);
    if (mh >= 0x7ff00000u) return -1;
    const uint32_t ml = dcsim_warp_min_u32(h == mh ? l : 0xffffffffu);
    const bool m = (h == mh) && (l == ml);
    const uint32_t ms = dcsim_warp_min_u32(m ? s : 0xffffffffu);
    const uint32_t votes = dcsim_warp_ballot(m && s == ms);
    *t_out = __hiloint2double((int)mh, (int)ml);
    *seq_out = ms;
    return dcsim_ffs(votes) - 1;
  }
#endif
  uint32_t bh = 0x7ff00000u, bl = 0u, bs = 0xffffffffu;
  int bi = -1;
  for (int i = lane; i < n; i += DCSIM_LANES) {
    const double ti = t[i];
    const uint32_t h = dcsim_hi(ti), l = dcsim_lo(ti), s = seq[i];
    if (h < bh || (h == bh && (l < bl || (l == bl && s < bs)))) { bh = h; bl = l; bs = s; bi = i; }
  }
  const uint32_t mh = dcsim_warp_min_u32(bh);
  if (mh >= 0x7ff00000u) return -1;
  const uint32_t ml = dcsim_warp_min_u32(bh == mh ? bl : 0xffffffffu);
  const bool m = (bh == mh) && (bl == ml);
  const uint32_t ms = dcsim_warp_min_u32(m ? bs : 0xffffffffu);
  const uint32_t votes = dcsim_warp_ballot(m && bs == ms && bi >= 0);
  const int src = dcsim_ffs(votes) - 1;
  const int win = (int)dcsim_bcast_u32((uint32_t)bi, src);
#ifdef DCSIM_HOST_EMU
  *t_out = t[win];
#else
  *t_out = __hiloint2double((int)mh, (int)ml);
#endif
  *seq_out = ms;
  return win;
}

/* Seq of the list entry at the cursor.  It was handed out when the push happened: an arrival's when its stream's
 * previous arrival (or the constructor) pushed it, an xfer_done's when its own arrival did. */
DCSIM_DEV uint32_t* dcsim_list_seq_slot(dcsim_ctx_t& c, uint32_t m) {
  return (m & ML_XFER) ? XRING(c) + (c.cursor & (uint32_t)c.P->L.xring_mask) : PEND_SEQ(c) + ((m >> 1) & 15u);
}

/* Pop-min over the event set.  Two halves:
 *
 *  (1) the earliest of the candidates OTHER than the list entry — per DC the earliest job_finish, the log tick, (power-cap
 *      controller) the earliest superseded job_finish: one slot per lane (two with 8 lanes and more than 5 DCs) and
 *      three min-reductions.  A warp per replica: REDUX.MIN over hi, lo, seq and a ballot.  Several replicas per warp:
 *      shuffle butterflies inside the lane group over hi, lo and (seq << 4 | slot) under the constant full mask — this is
 *      an EVENT-LEVEL point, every lane of the warp is here (dcsim_event_sync);
 *  (2) that minimum against the next list entry, read straight from the list window (entry c.cursor; the slot behind
 *      the window reads +inf), so nothing has to "publish" the next list entry: a compare on every lane.
 *
 * With several replicas per warp (1) is CACHED in the header: it changes only when one of those slots is written (a
 * job_finish, a start that becomes its DC's earliest finish, a log tick, the cap controller), whoever writes one raises
 * cand_dirty, and the reduction only runs when some replica of the warp is dirty (a clean one next to it recomputes what
 * it had).  In a saturated cluster most events are arrivals and transfers that queue: the 4 DC x 64 bench batch
 * re-reduces on a few percent of its events (event loop 126.8 -> 119.3 ms); a lightly loaded single DC is dirty on most
 * and pays for the bookkeeping (268 -> 279 ms) — profiles/r02_ab_s21_*.  What else was tried for (1), all slower: one
 * butterfly over the whole tuple (fewer dependent round trips, more instructions), every lane scanning the slots itself
 * (no shuffles at all: +20 %), probing chunks that switch the cache off when it misses (the switch costs what it saves).
 * With a warp per replica three REDUX.MIN are cheaper than the bookkeeping: no cache.
 *
 * The list's slot of the event set is never written: it stays +inf and takes part in (1) harmlessly.
 * Returns the winning candidate slot, -1 if all are +inf. */
struct dcsim_omin_t { uint32_t hi, lo, seq; int slot; bool fresh; }; /* (1); fresh: just reduced, not yet in the header */
/* Lane 0, after the event's first sync (every lane has read the header's copy by then): publishes a fresh (1).  Never
 * from a ghost lane group: with nothing staged its `blk` IS replica n-1's block in HBM, and nothing orders its store
 * against that replica's handler — landing after the handler had dirtied the event set again, it cleared cand_dirty over
 * a stale minimum and replica n-1 popped events out of order (8 lanes, DCSIM_MODE_INPLACE: tests/test_gpu_launch_modes.py).
 * A switched-off replica still publishes: its event set no longer changes, and a cache left dirty would make the whole
 * warp re-reduce on every event until its last replica ends. */
DCSIM_DEV void dcsim_omin_publish(dcsim_ctx_t& c, const dcsim_omin_t& o) {
  if (o.fresh && c.lane == 0 && !c.is_ghost) {
    c.H->omin_t = dcsim_hilo_f64(o.hi, o.lo); c.H->omin_seq = o.seq; c.H->omin_slot = (uint32_t)o.slot; c.H->cand_dirty = 0u;
  }
}
DCSIM_DEV int dcsim_argmin_cand(dcsim_ctx_t& c, dcsim_omin_t& om, double* t_out, uint32_t* seq_out) {
  const uint32_t li = c.cursor & (DCSIM_LIST_WINDOW - 1u); /* entries at and past the end of the list read (+inf, 0) */
  const uint32_t lm = LW_META(c)[li];
  uint32_t oh, ol, os;
  int oslot;
  om.fresh = false;
#if !defined(DCSIM_HOST_EMU) && DCSIM_LANES == 32
  {
    /* slot == lane, no loop; surplus lanes all look at the last slot, which is never used (+inf) */
    const int i = c.lane < DCSIM_CAND_N ? c.lane : DCSIM_CAND_N - 1;
    const double t = CAND_T(c)[i];
    const uint32_t s = CAND_SEQ(c)[i];
    const uint32_t h = dcsim_hi(t), l = dcsim_lo(t);
    oh = dcsim_event_min_u32(h);
    ol = dcsim_event_min_u32(h == oh ? l : 0xffffffffu);
    const bool m = (h == oh) && (l == ol);
    os = dcsim_event_min_u32(m ? s : 0xffffffffu);
    oslot = dcsim_ffs(__ballot_sync(0xffffffffu, m && s == os)) - 1;
  }
#else
  if (dcsim_event_any(c.H->cand_dirty != 0u)) {
#if !defined(DCSIM_HOST_EMU)
    const int i = c.lane < DCSIM_CAND_N ? c.lane : DCSIM_CAND_N - 1; /* slot == lane */
    double t = CAND_T(c)[i];
    uint32_t s = CAND_SEQ(c)[i];
    uint32_t h = dcsim_hi(t), l = dcsim_lo(t);
    uint32_t slot = (uint32_t)i;
#if DCSIM_LANES < DCSIM_CAND_N
    /* fewer lanes than slots (8 lanes): the event set of up to 5 DCs (n_dc + 3 slots) still fits one round; beyond,
     * each lane also looks at slot lane + DCSIM_LANES and keeps the earlier of its two (a scenario constant) */
    if (c.P->spec.n_dc + 3 > DCSIM_LANES) {
      const int i2 = c.lane + DCSIM_LANES;
      const double t2 = CAND_T(c)[i2];
      const uint32_t s2 = CAND_SEQ(c)[i2];
      const uint32_t h2 = dcsim_hi(t2), l2 = dcsim_lo(t2);
      if (h2 < h || (h2 == h && (l2 < l || (l2 == l && s2 < s)))) { h = h2; l = l2; s = s2; slot = (uint32_t)i2; }
    }
#endif
    oh = dcsim_event_min_u32(h);
    ol = dcsim_event_min_u32(h == oh ? l : 0xffffffffu);
    const bool m = (h == oh) && (l == ol);
    /* seq and slot in ONE reduction, as (seq << 4) | slot: the slot is 4 bits (CAND_N == 16), and a replica that ever
     * hands out seq 2^28 stops with DCSIM_ST_SEQ_OVERFLOW (dcsim_replica_run) — 2^28 pushes are ~10^8 events, a thousand
     * times the longest configuration of BASELINE.json.  (t, seq) is unique, so this only spares the pick a butterfly. */
    const uint32_t mk = dcsim_event_min_u32(m ? ((s << 4) | slot) : 0xffffffffu);
    os = oh >= 0x7ff00000u ? 0xffffffffu : mk >> 4;
    oslot = (int)(mk & 15u);
#else
    double ot = DCSIM_INF;
    os = 0xffffffffu;
    oslot = dcsim_argmin_ts(CAND_T(c), CAND_SEQ(c), CAND_N, c.lane, &ot, &os);
    if (oslot < 0) { ot = DCSIM_INF; os = 0xffffffffu; oslot = 0; }
    oh = dcsim_hi(ot); ol = dcsim_lo(ot);
#endif
    om.hi = oh; om.lo = ol; om.seq = os; om.slot = oslot; om.fresh = true;
  } else {
    const double ot = c.H->omin_t;
    oh = dcsim_hi(ot); ol = dcsim_lo(ot); os = c.H->omin_seq; oslot = (int)c.H->omin_slot;
  }
#endif
  const double lt = LW_T(c)[li];
  const uint32_t lh = dcsim_hi(lt), ll = dcsim_lo(lt);
  const uint32_t ls = *dcsim_list_seq_slot(c, lm);
  const bool list_first = lh < oh || (lh == oh && (ll < ol || (ll == ol && ls < os)));
  const uint32_t wh = list_first ? lh : oh;
  if (wh >= 0x7ff00000u) return -1;
  *t_out = dcsim_hilo_f64(wh, list_first ? ll : ol);
  *seq_out = list_first ? ls : os;
  return list_first ? CAND_LIST(c) : oslot;
}

/* SIM:160-163: an event later than end_time + 1e-9 (or at +inf) is never scheduled and takes no seq. */
DCSIM_DEV bool dcsim_schedulable(const dcsim_ctx_t& c, double t) { return !(t == DCSIM_INF) && !(t > c.P->end_eps); }

/* Lane 0.  DC d's estimated power as SIM:168-179 computes it on every event: the running jobs' powers summed in
 * dict (= start) order from 0.0 — kept in DF_PSUM, see there — then the idle term. */
DCSIM_DEV void dcsim_refresh_power(dcsim_ctx_t& c, int d) {
  const dcsim_dc_t& cfg = c.P->spec.dc[d];
  const int idle = cfg.total_gpus - DCI(c, DI_BUSY)[d];
  const double p_idle = (double)idle * (cfg.power_gating ? cfg.p_sleep : cfg.p_idle);
  DCF(c, DF_POWER)[d] = DCF(c, DF_PSUM)[d] + p_idle;
}

/* Lane 0, cold (power-cap controller only: it changes a record's power in place).  DF_PSUM of DC d from scratch. */
DCSIM_DEV void dcsim_resum_power(dcsim_ctx_t& c, int d) {
  const int n = DCI(c, DI_NRUN)[d];
  const double* pw = dcsim_at<double>(c.rec, c.P->L.rn_pw) + d * c.P->L.cap_run;
  double p_active = 0.0;
  for (int i = 0; i < n; ++i) p_active += pw[i];
  DCF(c, DF_PSUM)[d] = p_active;
}

/* Warp.  Earliest job_finish among DC d's running records -> candidate slot d. */
DCSIM_DEV void dcsim_rescan_dc(dcsim_ctx_t& c, int d) {
  const int n = DCI(c, DI_NRUN)[d];
  const int off = d * c.P->L.cap_run;
  double t; uint32_t s;
  const int k = dcsim_argmin_ts(dcsim_at<double>(c.rec, c.P->L.rn_t) + off, dcsim_at<uint32_t>(c.rec, c.P->L.rn_seq) + off,
                                n, c.lane, &t, &s);
  if (c.lane == 0) {
    CAND_T(c)[CAND_DC0 + d] = k >= 0 ? t : DCSIM_INF;
    CAND_SEQ(c)[CAND_DC0 + d] = k >= 0 ? s : 0xffffffffu;
    c.H->cand_dirty = 1u;
    DCI(c, DI_FMIN_SLOT)[d] = k;
  }
  dcsim_warp_sync();
}

/* ---- HBM FIFOs (dc.q_inf / dc.q_train, models.py:61-62) --------------------------------------- */
/* Entry `idx` of DC d's FIFO of job type jt.  One replica's FIFOs are below 4 GB (dcsim_create checks), so everything
 * but the replica's own offset is 32-bit arithmetic: one widening multiply-add instead of a chain of 64-bit ones. */
DCSIM_DEV dcsim_qent_t* dcsim_queue_at(const dcsim_ctx_t& c, int d, int jt, int idx) {
  const dcsim_layout_t& L = c.P->L;
  const uint32_t per_dc = (uint32_t)L.cap_q[0] + (uint32_t)L.cap_q[1];
  const uint32_t inner = ((uint32_t)d * per_dc + (jt ? (uint32_t)L.cap_q[0] : 0u) + (uint32_t)idx) * (uint32_t)sizeof(dcsim_qent_t);
  return reinterpret_cast<dcsim_qent_t*>(c.P->queues + ((uint64_t)c.r * (uint64_t)(uint32_t)L.queue_bytes + (uint64_t)inner));
}
DCSIM_DEV int dcsim_queue_len(dcsim_ctx_t& c, int d, int jt) { return DCI(c, jt ? DI_QN_TRN : DI_QN_INF)[d]; }
DCSIM_DEV void dcsim_enqueue(dcsim_ctx_t& c, int d, int jt, double size, uint32_t jid, uint32_t ing) {
  const int cap = c.P->L.cap_q[jt];
  int32_t* len = DCI(c, jt ? DI_QN_TRN : DI_QN_INF) + d;
  const int n = *len;
  if (n >= cap) { c.H->status |= DCSIM_ST_QUEUE_OVERFLOW; return; }
  int tail = DCI(c, jt ? DI_QH_TRN : DI_QH_INF)[d] + n;
  if (tail >= cap) tail -= cap;
  dcsim_qent_t e; e.size = size; e.jid = jid; e.ing = ing;
  *dcsim_queue_at(c, d, jt, tail) = e;
  *len = n + 1;
  if ((uint32_t)(n + 1) > c.H->max_q) c.H->max_q = (uint32_t)(n + 1);
}
DCSIM_DEV dcsim_qent_t dcsim_dequeue(dcsim_ctx_t& c, int d, int jt) {
  int32_t* head = DCI(c, jt ? DI_QH_TRN : DI_QH_INF) + d;
  const int h = *head;
  const dcsim_qent_t e = *dcsim_queue_at(c, d, jt, h);
  *head = h + 1 >= c.P->L.cap_q[jt] ? 0 : h + 1;
  DCI(c, jt ? DI_QN_TRN : DI_QN_INF)[d] -= 1;
  return e;
}

/* ================================================================================================
 * Handlers (lane 0)
 * ============================================================================================== */
/* policy.py:16-41: returns the GPU count and rewrites dc.current_freq */
DCSIM_DEV int dcsim_policy_select(dcsim_ctx_t& c, int d, int jt) {
  const dcsim_spec_t& sp = c.P->spec;
  double* cur = DCF(c, DF_CUR_FREQ) + d;
  const int free_g = sp.dc[d].total_gpus - DCI(c, DI_BUSY)[d];
  int g = free_g > 0 ? (free_g < sp.max_gpus_per_job ? free_g : sp.max_gpus_per_job) : 0;
  if (jt == DCSIM_JT_INFERENCE) {
    *cur = sp.dvfs_high;
  } else if (sp.policy_name == DCSIM_POLICY_PERF_FIRST) {
    const double cand = dcsim_queue_len(c, d, 0) > 0 ? sp.dvfs_high : sp.dc[d].default_freq;
    *cur = cand > *cur ? cand : *cur;
  } else if (sp.train_scale_out_low_freq && free_g >= 2) {
    *cur = sp.dvfs_low;
  } else {
    *cur = sp.dvfs_low > *cur ? sp.dvfs_low : *cur;
  }
  return g > 1 ? g : 1;
}

/* learners.py:20-36 */
DCSIM_COLD double dcsim_bandit_select(const dcsim_kparams_t* P, char* blk, int d, int jt) {
  const dcsim_dc_t& cfg = P->spec.dc[d];
  dcsim_hdr_t* H = reinterpret_cast<dcsim_hdr_t*>(blk);
  const uint32_t* N = dcsim_at<uint32_t>(blk, P->L.bandit_n) + (d * 2 + jt) * DCSIM_MAX_FREQ;
  const double* S = dcsim_at<double>(blk, P->L.bandit_s) + (d * 2 + jt) * DCSIM_MAX_FREQ;
  H->bandit_t += 1u;
#pragma unroll 1
  for (int i = 0; i < cfg.n_freq; ++i)
    if (N[i] < 1u) return cfg.freq_levels[i];
  double best_ucb = -1e9, best_f = cfg.freq_levels[0];
  const double two_log_t = 2.0 * log((double)H->bandit_t);
#pragma unroll 1
  for (int i = 0; i < cfg.n_freq; ++i) {
    const double n = (double)N[i];
    const double ucb = S[i] / n + sqrt(two_log_t / n);
    if (ucb > best_ucb) { best_ucb = ucb; best_f = cfg.freq_levels[i]; }
  }
  return best_f;
}

/* learners.py:38-42 with cost = E_pred = P_job * T(n, f) (SIM:716, 826-827) */
DCSIM_COLD void dcsim_bandit_update(const dcsim_kparams_t* P, char* blk, int d, int jt, int g, double f_used, double p_job) {
  const dcsim_dc_t& cfg = P->spec.dc[d];
  const double E_pred = p_job * dcsim_step_time(g, f_used, cfg.coeffs[jt]);
#pragma unroll 1
  for (int q = 0; q < cfg.n_freq; ++q) {
    if (cfg.freq_levels[q] == f_used) {
      dcsim_at<uint32_t>(blk, P->L.bandit_n)[(d * 2 + jt) * DCSIM_MAX_FREQ + q] += 1u;
      dcsim_at<double>(blk, P->L.bandit_s)[(d * 2 + jt) * DCSIM_MAX_FREQ + q] += -E_pred;
      break;
    }
  }
}

/* job_log.csv row, SIM:815-823 (unrounded) */
DCSIM_COLD void dcsim_joblog_write(const dcsim_kparams_t* P, uint32_t jid, uint32_t meta, int d, double size, double f_used,
                                   double start_s, double finish_s) {
  const uint32_t r = P->rec.counts[1];
  if (r < P->rec.jobs_cap) {
    dcsim_job_rec_t* o = P->rec.jobs + r;
    o->jid = jid; o->ingress = (uint8_t)(meta >> 17); o->jtype = (uint8_t)((meta >> 16) & 1u);
    o->dc = (uint8_t)d; o->_pad0 = 0; o->_pad1 = 0u; o->n_gpus = meta & 0xffffu; o->size = size;
    o->f_used = f_used; o->start_s = start_s; o->finish_s = finish_s;
  }
  P->rec.counts[1] = r + 1u;
}

/* SIM:680-699 (_start_job, use_dc_freq) and SIM:960-980 (_start_job_with_nf): allocate, stamp, push job_finish. */
template <bool CAP>
DCSIM_DEV void dcsim_start_job(dcsim_ctx_t& c, int d, int jt, double size, uint32_t jid, uint32_t ing, int n, double f) {
  const dcsim_layout_t& L = c.P->L;
  const dcsim_coeffs_t& k = c.P->spec.dc[d].coeffs[jt];
  int32_t* nrun = DCI(c, DI_NRUN) + d;
  const int slot = *nrun;
  if (slot >= L.cap_run) { c.H->status |= DCSIM_ST_RUN_OVERFLOW; return; }
  DCI(c, DI_BUSY)[d] += n;
  /* T(n,f), n*P_gpu(f) and 1/T cost three FP64 divisions and a cube per start (~85 instructions); jobs of one type at
   * one DC mostly start with the (n, f) of the previous one, so the last result is kept per (DC, jtype).  Same
   * operations on the same inputs: the cached values are bit-identical to recomputing. */
  double T_unit, pw_job, tpt_job;
  {
    double* mf = dcsim_at<double>(c.blk, L.memo_f64) + (d * 2 + jt) * 4; /* f, T, n*P, 1/T */
    int32_t* mn = dcsim_at<int32_t>(c.blk, L.memo_n) + (d * 2 + jt);
    if (*mn == n && mf[0] == f) {
      T_unit = mf[1]; pw_job = mf[2]; tpt_job = mf[3];
    } else {
      T_unit = dcsim_step_time(n, f, k);
      pw_job = dcsim_task_power(n, f, k);
      tpt_job = 1.0 / T_unit; /* SIM:956 */
      *mn = n; mf[0] = f; mf[1] = T_unit; mf[2] = pw_job; mf[3] = tpt_job;
    }
  }
  const double t_fin = c.now + size * T_unit;
  const int i = d * L.cap_run + slot;
  const bool ok = dcsim_schedulable(c, t_fin);
  const uint32_t seq = ok ? c.seq++ : 0xffffffffu;
  dcsim_at<double>(c.rec, L.rn_t)[i] = ok ? t_fin : DCSIM_INF; /* a dropped finish holds its GPUs for ever */
  dcsim_at<uint32_t>(c.rec, L.rn_seq)[i] = seq;
  dcsim_at<double>(c.rec, L.rn_pw)[i] = pw_job;
  dcsim_at<double>(c.rec, L.rn_tpt)[i] = tpt_job;
  dcsim_at<double>(c.rec, L.rn_start)[i] = c.now;
  dcsim_at<uint32_t>(c.rec, L.rn_meta)[i] = (uint32_t)n | ((uint32_t)jt << 16) | (ing << 17);
  if (CAP || L.lean == 0) {
    dcsim_at<double>(c.rec, L.rn_size)[i] = size;
    dcsim_at<double>(c.rec, L.rn_f)[i] = f;
    dcsim_at<uint32_t>(c.rec, L.rn_jid)[i] = jid;
  }
  if constexpr (CAP) { /* SIM:690-692: units_done = 0, last_update = now */
    dcsim_at<double>(c.rec, L.rn_done)[i] = 0.0;
    dcsim_at<double>(c.rec, L.rn_upd)[i] = c.now;
  }
  *nrun = slot + 1;
  DCF(c, DF_PSUM)[d] += pw_job; /* the addition a re-sum in dict order would end with */
  if ((uint32_t)(slot + 1) > c.H->max_run) c.H->max_run = (uint32_t)(slot + 1);
  if (ok) { /* incremental update of DC d's earliest finish */
    const double ct = CAND_T(c)[CAND_DC0 + d];
    if (t_fin < ct || (t_fin == ct && seq < CAND_SEQ(c)[CAND_DC0 + d])) {
      CAND_T(c)[CAND_DC0 + d] = t_fin; CAND_SEQ(c)[CAND_DC0 + d] = seq; DCI(c, DI_FMIN_SLOT)[d] = slot;
      c.H->cand_dirty = 1u; /* (a start that is not its DC's earliest finish leaves the event set's minimum alone) */
    }
  }
}

/* SIM:982-984  int((now % 86400) // 3600), CPython float_rem / float_floor_div for positive operands */
DCSIM_COLD int dcsim_current_hour(double now) {
  const double x = fmod(now, 86400.0);
  const double mod = fmod(x, 3600.0);
  const double div = (x - mod) / 3600.0;
  double fl = floor(div);
  if (div - fl > 0.5) fl += 1.0;
  return (int)fl;
}

/* The start rules of SIM:603-676 (at xfer_done) and SIM:892-927 (dequeue loop). */
template <bool CAP>
DCSIM_DEV void dcsim_start_by_rule(dcsim_ctx_t& c, int rule, bool at_xfer, int d, int jt, double size, uint32_t jid, uint32_t ing) {
  const dcsim_spec_t& sp = c.P->spec;
  const int free_g = sp.dc[d].total_gpus - DCI(c, DI_BUSY)[d];
  if (rule == DCSIM_START_NF_LUT) {
    const dcsim_nf_t nf = at_xfer ? sp.dc[d].nf_xfer[jt][dcsim_current_hour(c.now)] : sp.dc[d].nf_deq[jt];
    int n = nf.n < free_g ? nf.n : free_g; /* SIM:962 */
    n = n > 1 ? n : 1;
    dcsim_start_job<CAP>(c, d, jt, size, jid, ing, n, nf.f);
  } else if (rule == DCSIM_START_BANDIT) {
    int n = free_g < sp.max_gpus_per_job ? free_g : sp.max_gpus_per_job;
    const double f = dcsim_bandit_select(c.P, c.blk, d, jt);
    n = n < free_g ? n : free_g;
    n = n > 1 ? n : 1;
    dcsim_start_job<CAP>(c, d, jt, size, jid, ing, n, f);
  } else {
    const int g = dcsim_policy_select(c, d, jt);
    dcsim_start_job<CAP>(c, d, jt, size, jid, ing, g, DCF(c, DF_CUR_FREQ)[d]); /* SIM:689,696: f = dc.current_freq */
  }
}

/* The event list is streamed through a 32-slot ring in the state block, half a ring (16 entries) at a time: when the
 * cursor enters one half, the other half — just consumed — is refilled with the 16 entries after the current half.  On
 * the GPU the refill is ASYNCHRONOUS (cp.async: HBM -> shared memory without registers), so its latency, which a whole
 * warp (all of its lane groups) would otherwise sit out every 16 list events, hides behind the events of the current
 * half; dcsim_list_wait() is called before the first entry of a freshly filled half is looked at.  Slots of list
 * positions at or past the end of the list get (+inf, 0): "no event". */
DCSIM_DEV void dcsim_list_fill(dcsim_ctx_t& c, uint32_t first, uint32_t n_entries) {
  const uint64_t off = (uint64_t)c.r * 2ull * (uint64_t)c.P->cap_arr;
  const uint32_t count = c.H->ml_count;
  for (uint32_t i = (uint32_t)c.lane; i < n_entries; i += DCSIM_LANES) {
    const uint32_t p = first + i, slot = p & (DCSIM_LIST_WINDOW - 1u);
    if (p < count) {
#if !defined(DCSIM_HOST_EMU)
      if (__isShared(c.blk)) {
        __pipeline_memcpy_async(LW_T(c) + slot, c.P->ml_t + off + p, 8);
        __pipeline_memcpy_async(LW_AUX(c) + slot, c.P->ml_aux + off + p, 8);
        __pipeline_memcpy_async(LW_META(c) + slot, c.P->ml_meta + off + p, 4);
        continue;
      }
#endif
      LW_T(c)[slot] = c.P->ml_t[off + p]; LW_AUX(c)[slot] = c.P->ml_aux[off + p]; LW_META(c)[slot] = c.P->ml_meta[off + p];
    } else {
      LW_T(c)[slot] = DCSIM_INF; LW_AUX(c)[slot] = 0.0; LW_META(c)[slot] = 0u;
    }
  }
#if !defined(DCSIM_HOST_EMU)
  __pipeline_commit();
#endif
}
/* Whole lane group: every refill issued so far has landed and is visible to all lanes. */
DCSIM_DEV void dcsim_list_wait() {
#if !defined(DCSIM_HOST_EMU)
  __pipeline_wait_prior(0);
#endif
  dcsim_warp_sync();
}

/* SIM:595-678 (lane 0): the transferred job starts if its DC has a free GPU, else it queues. */
template <bool CAP>
DCSIM_DEV void dcsim_handle_xfer(dcsim_ctx_t& c, double size, uint32_t meta) {
  const dcsim_spec_t& sp = c.P->spec;
  const int d = (int)((meta >> 1) & 7u), jt = (int)((meta >> 4) & 1u);
  const uint32_t ing = (meta >> 5) & 7u, jid = (meta >> 8) + 1u; /* SIM:539: jids count arrivals */
  if (sp.dc[d].total_gpus - DCI(c, DI_BUSY)[d] > 0) {
    dcsim_start_by_rule<CAP>(c, sp.xfer_rule, true, d, jt, size, jid, ing);
    dcsim_refresh_power(c, d);
  } else {
    dcsim_enqueue(c, d, jt, size, jid, ing); /* SIM:678 */
  }
}

/* The next entry of the event list fires (whole warp: the window may need re-staging).
 * Arrival, SIM:537-592: everything random about it was drawn by the pre-pass; what remains is handing out the seqs
 * of its two pushes — the xfer_done's goes into the ring slot of that entry's list position, the stream's next
 * arrival's into the stream's pending slot.  xfer_done: dcsim_handle_xfer. */
template <bool CAP>
DCSIM_DEV void dcsim_handle_list(dcsim_ctx_t& c) {
  const uint32_t i = c.cursor & (DCSIM_LIST_WINDOW - 1u);
  if (c.lane == 0) {
    const uint32_t meta = LW_META(c)[i];
    if (meta & ML_XFER) {
      dcsim_handle_xfer<CAP>(c, LW_AUX(c)[i], meta);
    } else {
      c.H->ev_arr++;
      if (meta & ML_A_XSCHED) { /* SIM:580-588 */
        const uint32_t s = c.seq++;
        if (meta & ML_A_XIN) XRING(c)[dcsim_lo(LW_AUX(c)[i]) & (uint32_t)c.P->L.xring_mask] = s;
      }
      if (meta & ML_A_NEXT) PEND_SEQ(c)[(meta >> 1) & 15u] = c.seq++; /* SIM:591-592 */
    }
  }
  c.cursor += 1u;
  if ((c.cursor & (DCSIM_LIST_HALF - 1u)) == 0u) { /* entering the other half: it was refilled half a ring ago */
    dcsim_list_wait();                              /* (also: lane 0 is done with the half just left) */
    dcsim_list_fill(c, c.cursor + DCSIM_LIST_HALF, DCSIM_LIST_HALF);
  }
} /* (the event's closing sync follows in dcsim_event_body) */

/* SIM:701-927 minus RL/elastic branches (lane 0 part, after the record was read and before it is erased). */
DCSIM_DEV void dcsim_finish_account(dcsim_ctx_t& c, int d, int slot) {
  const dcsim_spec_t& sp = c.P->spec;
  const dcsim_layout_t& L = c.P->L;
  dcsim_hdr_t* H = c.H;
  const int i = d * L.cap_run + slot;
  const uint32_t meta = dcsim_at<uint32_t>(c.rec, L.rn_meta)[i];
  const int g = (int)(meta & 0xffffu), jt = (int)((meta >> 16) & 1u);
  int32_t* busy = DCI(c, DI_BUSY) + d;
  *busy = *busy - g > 0 ? *busy - g : 0; /* SIM:707 */
  const double now = c.now;
  DCF(c, DF_ACC_UNIT)[d] += dcsim_at<double>(c.rec, L.rn_tpt)[i] * dcsim_mod_pos_hint(now, sp.log_interval, H->ev_log); /* SIM:711 */
  const double lat = now - dcsim_at<double>(c.rec, L.rn_start)[i]; /* SIM:820 */
  H->lat_sum += lat;
  if (jt == DCSIM_JT_INFERENCE) { H->lat_sum_inf += lat; H->n_fin_inf++; } else { H->lat_sum_trn += lat; H->n_fin_trn++; }
  if (c.P->lat_hist) dcsim_hist_add(c.P->lat_hist, (uint64_t)c.r, jt, lat);
  if (L.lean == 0) { /* the readers of a finished job's size / f / jid: job_log.csv and the bandit's reward */
    const double f_used = dcsim_at<double>(c.rec, L.rn_f)[i];
    if (c.is_logged && c.P->rec.jobs)
      dcsim_joblog_write(c.P, dcsim_at<uint32_t>(c.rec, L.rn_jid)[i], meta, d, dcsim_at<double>(c.rec, L.rn_size)[i], f_used,
                         dcsim_at<double>(c.rec, L.rn_start)[i], now);
    if (sp.deq_rule == DCSIM_START_BANDIT)
      dcsim_bandit_update(c.P, c.blk, d, jt, g, f_used, dcsim_at<double>(c.rec, L.rn_pw)[i]);
  }
}

/* SIM:840-927: start queued jobs while GPUs are free, inference first when inf_priority.  `pre` is the head entry of
 * queue `pre_jt` of this DC loaded ahead of time by the caller (-1: none): the queues live in HBM and the first
 * dequeue's latency is otherwise exposed on every job_finish of a saturated DC. */
#ifndef DCSIM_PREFETCH_DEQ
#define DCSIM_PREFETCH_DEQ 1
#endif
DCSIM_DEV int dcsim_dequeue_pick(dcsim_ctx_t& c, int d) {
  if (c.P->spec.inf_priority && dcsim_queue_len(c, d, 0) > 0) return 0;
  if (dcsim_queue_len(c, d, 1) > 0) return 1;
  return -1;
}
template <bool CAP>
DCSIM_DEV void dcsim_dequeue_loop(dcsim_ctx_t& c, int d, const dcsim_qent_t& pre, int pre_jt) {
  const dcsim_spec_t& sp = c.P->spec;
  bool first = true;
  while (sp.dc[d].total_gpus - DCI(c, DI_BUSY)[d] > 0 && c.H->status == 0u) {
    const int jt = dcsim_dequeue_pick(c, d);
    if (jt < 0) break;
    dcsim_qent_t e;
    if (DCSIM_PREFETCH_DEQ && first && jt == pre_jt) { /* the head entry is already here: just advance the ring */
      int32_t* head = DCI(c, jt ? DI_QH_TRN : DI_QH_INF) + d;
      const int h = *head;
      *head = h + 1 >= c.P->L.cap_q[jt] ? 0 : h + 1;
      DCI(c, jt ? DI_QN_TRN : DI_QN_INF)[d] -= 1;
      e = pre;
    } else {
      e = dcsim_dequeue(c, d, jt);
    }
    first = false;
    dcsim_start_by_rule<CAP>(c, sp.deq_rule, false, d, jt, e.size, e.jid, e.ing);
  }
}

/* SIM:701-927, whole warp: the job_finish of DC d's earliest-finishing record (slot DI_FMIN_SLOT).
 *
 * One pass over the DC's records does everything the reference's `del dc.running_jobs[jid]` + next `_estimate_dc_power`
 * + next heap pop imply: lane j loads record j of the set WITHOUT the finished one (slot j, or j + 1 behind the hole),
 * lanes behind the hole store it one slot down (dict order is start order, models.py:60), the earliest remaining
 * finish is an arg-min over the registers, and the active power is re-summed in dict order (SIM:168-179) from the
 * registers by shuffles (a lane-0 loop over shared memory measured slower: its loads serialise behind the additions).
 * The records are touched once per job_finish — one load round trip, stores fire-and-forget — which is what lets them
 * live in HBM/L2 (RECG) when the block is large. */
template <bool CAP, bool RECG>
DCSIM_DEV void dcsim_handle_finish(dcsim_ctx_t& c, int d) {
  const dcsim_layout_t& L = c.P->L;
  const int off = d * L.cap_run;
  const int n = DCI(c, DI_NRUN)[d];
  const int k = DCI(c, DI_FMIN_SLOT)[d];
  dcsim_qent_t pre; pre.size = 0.0; pre.jid = 0u; pre.ing = 0u;
  int pre_jt = -1;
  if (c.lane == 0) {
    c.H->ev_fin++;
    if (DCSIM_PREFETCH_DEQ) { /* the dequeue loop below will want this entry: have the load in flight meanwhile */
      pre_jt = dcsim_dequeue_pick(c, d);
      if (pre_jt >= 0) pre = *dcsim_queue_at(c, d, pre_jt, DCI(c, pre_jt ? DI_QH_TRN : DI_QH_INF)[d]);
    }
    dcsim_finish_account(c, d, k); /* reads record k; writes no record */
  }
  double* rt = dcsim_at<double>(c.rec, L.rn_t) + off; double* rp = dcsim_at<double>(c.rec, L.rn_pw) + off;
  double* rv = dcsim_at<double>(c.rec, L.rn_tpt) + off; double* ra = dcsim_at<double>(c.rec, L.rn_start) + off;
  uint32_t* rq = dcsim_at<uint32_t>(c.rec, L.rn_seq) + off; uint32_t* rm = dcsim_at<uint32_t>(c.rec, L.rn_meta) + off;
  const bool full = L.lean == 0;
  const int n1 = n - 1;
  uint32_t bh = 0x7ff00000u, bl = 0u, bs = 0xffffffffu;
  int bi = -1;
  double psum = 0.0;
  dcsim_warp_sync(); /* lane 0's reads of record k are done before anybody overwrites slot k */
  /* (issuing the pass's loads BEFORE lane 0's accounting, so that the two L2 round trips overlap, measured slower:
     the loop then carries lane 0's code with every record field live — profiles/r02_variants_ab.md) */
  for (int base = 0; base < n1; base += DCSIM_LANES) {
    const int j = base + c.lane;
    const bool act = j < n1, moved = act && j >= k;
    const int src = moved ? j + 1 : j;
    double a_t = DCSIM_INF, a_pw = 0.0, a_tpt = 0.0, a_start = 0.0, a_size = 0.0, a_f = 0.0, a_done = 0.0, a_upd = 0.0;
    uint32_t a_seq = 0xffffffffu, a_meta = 0u, a_jid = 0u;
    if (act) { a_t = rt[src]; a_seq = rq[src]; a_pw = rp[src]; }
    if (moved) {
      a_tpt = rv[src]; a_start = ra[src]; a_meta = rm[src];
      if (full) { a_size = dcsim_at<double>(c.rec, L.rn_size)[off + src]; a_f = dcsim_at<double>(c.rec, L.rn_f)[off + src];
                  a_jid = dcsim_at<uint32_t>(c.rec, L.rn_jid)[off + src]; }
      if constexpr (CAP) { a_done = dcsim_at<double>(c.rec, L.rn_done)[off + src]; a_upd = dcsim_at<double>(c.rec, L.rn_upd)[off + src]; }
    }
    {
      const int cnt = n1 - base < DCSIM_LANES ? n1 - base : DCSIM_LANES;
#if DCSIM_LANES >= 4
      /* SIM:168-179: dict order, from 0.0.  Four at a time: lanes at and past cnt hold 0.0, and x + 0.0 == x exactly */
      for (int i = 0; i < cnt; i += 4) {
        psum += dcsim_bcast_f64(a_pw, i); psum += dcsim_bcast_f64(a_pw, i + 1);
        psum += dcsim_bcast_f64(a_pw, i + 2); psum += dcsim_bcast_f64(a_pw, i + 3);
      }
#else
      for (int i = 0; i < cnt; ++i) psum += dcsim_bcast_f64(a_pw, i); /* SIM:168-179: dict order, from 0.0 */
#endif
    }
    {
      const uint32_t h = dcsim_hi(a_t), l = dcsim_lo(a_t);
      if (act && (h < bh || (h == bh && (l < bl || (l == bl && a_seq < bs))))) { bh = h; bl = l; bs = a_seq; bi = j; }
    }
    dcsim_warp_sync(); /* every lane holds its record before the slot it came from is overwritten */
    if (moved) {
      rt[j] = a_t; rq[j] = a_seq; rp[j] = a_pw; rv[j] = a_tpt; ra[j] = a_start; rm[j] = a_meta;
      if (full) { dcsim_at<double>(c.rec, L.rn_size)[off + j] = a_size; dcsim_at<double>(c.rec, L.rn_f)[off + j] = a_f;
                  dcsim_at<uint32_t>(c.rec, L.rn_jid)[off + j] = a_jid; }
      if constexpr (CAP) { dcsim_at<double>(c.rec, L.rn_done)[off + j] = a_done; dcsim_at<double>(c.rec, L.rn_upd)[off + j] = a_upd; }
    }
  }
  /* earliest remaining finish of DC d, in (t, seq) order */
  const uint32_t mh = dcsim_warp_min_u32(bh);
  int win = -1;
  double wt = DCSIM_INF;
  uint32_t ws = 0xffffffffu;
  if (mh < 0x7ff00000u) {
    const uint32_t ml = dcsim_warp_min_u32(bh == mh ? bl : 0xffffffffu);
    const bool m = (bh == mh) && (bl == ml);
    ws = dcsim_warp_min_u32(m ? bs : 0xffffffffu);
    win = (int)dcsim_pick_u32(m && bs == ws && bi >= 0, (uint32_t)bi);
    wt = dcsim_hilo_f64(mh, ml);
  }
  if (c.lane == 0) {
    CAND_T(c)[CAND_DC0 + d] = wt; CAND_SEQ(c)[CAND_DC0 + d] = ws; DCI(c, DI_FMIN_SLOT)[d] = win;
    c.H->cand_dirty = 1u;
    DCI(c, DI_NRUN)[d] = n1;
    DCF(c, DF_PSUM)[d] = psum;
    dcsim_dequeue_loop<CAP>(c, d, pre, pre_jt); /* appends behind the compacted records */
    dcsim_refresh_power(c, d);
  }
} /* (the event's closing sync follows in dcsim_event_body) */

/* Warp.  Earliest superseded job_finish -> candidate slot CAND_STALE(c). */
DCSIM_DEV void dcsim_rescan_stale(dcsim_ctx_t& c) {
  double t; uint32_t s;
  const int k = dcsim_argmin_ts(dcsim_at<double>(c.blk, c.P->L.st_t), dcsim_at<uint32_t>(c.blk, c.P->L.st_seq),
                                (int)c.H->n_stale, c.lane, &t, &s);
  if (c.lane == 0) {
    CAND_T(c)[CAND_STALE(c)] = k >= 0 ? t : DCSIM_INF;
    CAND_SEQ(c)[CAND_STALE(c)] = k >= 0 ? s : 0xffffffffu;
    c.H->cand_dirty = 1u;
    c.H->smin_slot = (uint32_t)k;
  }
  dcsim_warp_sync();
}

/* Lane 0.  SIM:317-338 _reschedule_job: bank progress at the old frequency, switch, push a new job_finish and
 * leave the old one behind as a stale event. */
DCSIM_DEV void dcsim_reschedule_job(dcsim_ctx_t& c, int d, int slot, double new_f) {
  const dcsim_layout_t& L = c.P->L;
  const int i = d * L.cap_run + slot;
  const uint32_t meta = dcsim_at<uint32_t>(c.rec, L.rn_meta)[i];
  const int g = (int)(meta & 0xffffu), jt = (int)((meta >> 16) & 1u);
  const dcsim_coeffs_t& k = c.P->spec.dc[d].coeffs[jt];
  const double f_old = dcsim_at<double>(c.rec, L.rn_f)[i];
  const double f_cur = f_old != 0.0 ? f_old : DCF(c, DF_CUR_FREQ)[d];
  const double total = dcsim_at<double>(c.rec, L.rn_size)[i];
  const double T0 = dcsim_step_time(g, f_cur, k);
  const double rate = 1.0 / (T0 > 1e-9 ? T0 : 1e-9);
  double dt = c.now - dcsim_at<double>(c.rec, L.rn_upd)[i]; dt = dt > 0.0 ? dt : 0.0;
  const double ud = dcsim_at<double>(c.rec, L.rn_done)[i] + rate * dt;
  const double done = total < ud ? total : ud;
  dcsim_at<double>(c.rec, L.rn_done)[i] = done;
  dcsim_at<double>(c.rec, L.rn_upd)[i] = c.now;
  dcsim_at<double>(c.rec, L.rn_f)[i] = new_f;
  double left = total - done; left = left > 0.0 ? left : 0.0;
  const double T1 = dcsim_step_time(g, new_f, k);
  const double rate_new = 1.0 / (T1 > 1e-9 ? T1 : 1e-9);
  const double finish_in = left / (rate_new > 1e-9 ? rate_new : 1e-9);
  const double t_old = dcsim_at<double>(c.rec, L.rn_t)[i];
  if (!(t_old == DCSIM_INF)) { /* the superseded event stays in the event set */
    const uint32_t ns = c.H->n_stale;
    if ((int)ns >= L.cap_stale) { c.H->status |= DCSIM_ST_STALE_OVERFLOW; }
    else {
      dcsim_at<double>(c.blk, L.st_t)[ns] = t_old;
      dcsim_at<uint32_t>(c.blk, L.st_seq)[ns] = dcsim_at<uint32_t>(c.rec, L.rn_seq)[i];
      c.H->n_stale = ns + 1u;
    }
  }
  const double t_new = c.now + finish_in;
  const bool ok = dcsim_schedulable(c, t_new);
  dcsim_at<double>(c.rec, L.rn_t)[i] = ok ? t_new : DCSIM_INF;
  dcsim_at<uint32_t>(c.rec, L.rn_seq)[i] = ok ? c.seq++ : 0xffffffffu;
  dcsim_at<double>(c.rec, L.rn_pw)[i] = dcsim_task_power(g, new_f, k);
  dcsim_at<double>(c.rec, L.rn_tpt)[i] = 1.0 / T1;
}

/* Lane 0.  SIM:207-315 for algo = cap_greedy (cap_uniform never changes state: SIM:197-203 compares two identical
 * estimates).  Atoms are freq_load_agg.py:44-80's DOWN steps; the UP list is built by the reference and never read. */
DCSIM_DEV void dcsim_control_cap_greedy(dcsim_ctx_t& c) {
  const dcsim_spec_t& sp = c.P->spec;
  const dcsim_layout_t& L = c.P->L;
  double totalP = 0.0;
  for (int d = 0; d < sp.n_dc; ++d) totalP += DCF(c, DF_POWER)[d];
  if (totalP <= sp.power_cap - 5.0) return; /* cap_margin hysteresis, SIM:235-237 */
  double deficit = totalP - sp.power_cap; deficit = deficit > 0.0 ? deficit : 0.0;
  if (deficit <= 1e-6) return;
  double* at_rho = dcsim_at<double>(c.blk, L.at_rho);
  double* at_fto = dcsim_at<double>(c.blk, L.at_fto);
  uint32_t* at_ref = dcsim_at<uint32_t>(c.blk, L.at_ref);
  uint32_t* at_idx = dcsim_at<uint32_t>(c.blk, L.at_idx);
  for (int guard = 10000; deficit > 1e-6 && guard > 0; --guard) {
    int na = 0, n_tasks = 0;
#pragma unroll 1
    for (int d = 0; d < sp.n_dc; ++d) {
      const dcsim_dc_t& cfg = sp.dc[d];
      double lv[DCSIM_MAX_FREQ];
      for (int q = 0; q < cfg.n_freq; ++q) { /* sorted(freq_levels), freq_load_agg.py:45 */
        const double v = cfg.freq_levels[q];
        int r = q;
        while (r > 0 && lv[r - 1] > v) { lv[r] = lv[r - 1]; --r; }
        lv[r] = v;
      }
      const double f_min = lv[0];
      const int n = DCI(c, DI_NRUN)[d];
#pragma unroll 1
      for (int slot = 0; slot < n; ++slot) {
        const int i = d * L.cap_run + slot;
        const uint32_t meta = dcsim_at<uint32_t>(c.rec, L.rn_meta)[i];
        const int g = (int)(meta & 0xffffu), jt = (int)((meta >> 16) & 1u);
        const dcsim_coeffs_t& k = cfg.coeffs[jt];
        const double f_job = dcsim_at<double>(c.rec, L.rn_f)[i];
        const double cur_f = f_job != 0.0 ? f_job : DCF(c, DF_CUR_FREQ)[d];
        if (cur_f <= f_min + 1e-12) continue;
        ++n_tasks;
        int i0 = 0;
        for (int q = 1; q < cfg.n_freq; ++q) {
          const double a = lv[q] - cur_f, b = lv[i0] - cur_f;
          if ((a < 0.0 ? -a : a) < (b < 0.0 ? -b : b)) i0 = q;
        }
        const double T0 = dcsim_step_time(g, lv[i0], k);
        double curV = T0 <= 0.0 ? 0.0 : 1.0 / T0, curP = dcsim_task_power(g, lv[i0], k);
        for (int q = i0; q > 0; --q) {
          const double f_to = lv[q - 1];
          const double T2 = dcsim_step_time(g, f_to, k);
          const double V2 = T2 <= 0.0 ? 0.0 : 1.0 / T2, P2 = dcsim_task_power(g, f_to, k);
          double dV = curV - V2; dV = dV > 0.0 ? dV : 0.0;
          double dP = curP - P2; dP = dP > 0.0 ? dP : 0.0;
          if (dV > 0.0 && dP >= 0.0 && na < L.cap_atoms) {
            at_rho[na] = dP / dV; at_fto[na] = f_to; at_ref[na] = ((uint32_t)d << 16) | (uint32_t)slot;
            ++na;
          }
          curV = V2; curP = P2;
        }
      }
    }
    if (!n_tasks || !na) break;
    for (int a = 0; a < na; ++a) { /* list.sort(key=rho) is stable: insertion sort on (rho, build order) */
      const double r = at_rho[a];
      int q = a;
      while (q > 0 && at_rho[at_idx[q - 1]] > r) { at_idx[q] = at_idx[q - 1]; --q; }
      at_idx[q] = (uint32_t)a;
    }
    bool applied = false;
#pragma unroll 1
    for (int a = 0; a < na; ++a) {
      if (deficit <= 1e-6) break;
      const uint32_t id = at_idx[a];
      const int d = (int)(at_ref[id] >> 16), slot = (int)(at_ref[id] & 0xffffu);
      const double cur_f = dcsim_at<double>(c.rec, L.rn_f)[d * L.cap_run + slot];
      if (at_fto[id] >= cur_f - 1e-12) continue; /* SIM:296 */
      dcsim_reschedule_job(c, d, slot, at_fto[id]);
      applied = true;
      dcsim_resum_power(c, d);
      dcsim_refresh_power(c, d);
      totalP = 0.0;
      for (int e = 0; e < sp.n_dc; ++e) totalP += DCF(c, DF_POWER)[e];
      deficit = totalP - sp.power_cap; deficit = deficit > 0.0 ? deficit : 0.0;
      if (deficit <= 1e-6) break;
    }
    if (!applied) break;
  }
}

/* SIM:929-949 + the :221-225 heuristic of _control.  DC-parallel: one DC per lane.
 * Entered with all prior writes visible; leaves with its own writes visible (trailing sync). */
template <bool CAP>
DCSIM_DEV void dcsim_handle_log(dcsim_ctx_t& c) {
  const dcsim_spec_t& sp = c.P->spec;
  const dcsim_layout_t& L = c.P->L;
  const double interval = sp.log_interval;
  const bool rec = c.is_logged && c.P->rec.cluster != nullptr;
  if constexpr (CAP) { /* SIM:464: _control() precedes _handle_log() */
    if (c.lane == 0) dcsim_control_cap_greedy(c);
    dcsim_warp_sync();
    for (int d = 0; d < sp.n_dc; ++d) dcsim_rescan_dc(c, d); /* finish times may have moved */
    dcsim_rescan_stale(c);
  }
  DCSIM_FOR_EACH_DC(d, c, sp.n_dc) {
    if (sp.control_lower_idle && DCI(c, DI_BUSY)[d] == 0 && sp.dc[d].n_freq > 0) { /* SIM:221-225, before the rows */
      double m = sp.dc[d].freq_levels[0];
      for (int q = 1; q < sp.dc[d].n_freq; ++q) m = sp.dc[d].freq_levels[q] < m ? sp.dc[d].freq_levels[q] : m;
      DCF(c, DF_CUR_FREQ)[d] = m;
    }
    const int n = DCI(c, DI_NRUN)[d];
    const double* tpt = dcsim_at<double>(c.rec, L.rn_tpt) + d * L.cap_run;
    double acc = DCF(c, DF_ACC_UNIT)[d];
    for (int i = 0; i < n; ++i) acc += tpt[i] * interval; /* SIM:941-942, running jobs in dict order */
    DCF(c, DF_ACC_UNIT)[d] = acc;
    if (rec) { /* cluster_log.csv row, SIM:944-948; the rows of one tick are DC-ordered */
      const uint32_t r = c.P->rec.counts[2] + (uint32_t)d;
      if (r < c.P->rec.cluster_cap) {
        const uint32_t* meta = dcsim_at<uint32_t>(c.rec, L.rn_meta) + d * L.cap_run;
        int run_inf = 0;
        for (int i = 0; i < n; ++i) run_inf += ((meta[i] >> 16) & 1u) ? 0 : 1;
        dcsim_cluster_rec_t* o = c.P->rec.cluster + r;
        o->time_s = c.now; o->freq = DCF(c, DF_CUR_FREQ)[d]; o->util_gpu_time = DCF(c, DF_UTIL_TIME)[d];
        o->util_begin_ts = DCF(c, DF_UTIL_BEGIN)[d]; o->acc_job_unit = acc; o->power_w = DCF(c, DF_POWER)[d];
        o->energy_j = DCF(c, DF_ENERGY)[d]; o->dc = d; o->busy = DCI(c, DI_BUSY)[d]; o->run_total = n;
        o->run_inf = run_inf; o->q_inf = dcsim_queue_len(c, d, 0); o->q_train = dcsim_queue_len(c, d, 1);
      }
    }
  }
  if (rec) dcsim_warp_sync(); /* every lane has read counts[2] before lane 0 bumps it */
  if (c.lane == 0) {
    if (rec) c.P->rec.counts[2] += (uint32_t)sp.n_dc;
    const double t = c.now + interval; /* SIM:949 */
    if (dcsim_schedulable(c, t)) { CAND_T(c)[CAND_LOG(c)] = t; CAND_SEQ(c)[CAND_LOG(c)] = c.seq++; }
    else { CAND_T(c)[CAND_LOG(c)] = DCSIM_INF; CAND_SEQ(c)[CAND_LOG(c)] = 0xffffffffu; }
    c.H->cand_dirty = 1u;
  }
} /* (the event's closing sync follows in dcsim_event_body) */

/* ================================================================================================
 * Replica life cycle
 * ============================================================================================== */
/* SIM:31-157, the parts that touch simulation state: zeroed DCs at default_freq, one pending arrival per
 * (ingress, job type) in dict order inf-then-trn (drawn by the pre-pass; here they get the constructor's seqs), then
 * the first log tick. */
DCSIM_DEV void dcsim_replica_init(dcsim_ctx_t& c) {
  const dcsim_spec_t& sp = c.P->spec;
  const dcsim_layout_t& L = c.P->L;
  /* the head only: with every DI_NRUN at 0 no record is ever read before it was written */
  for (int i = c.lane; i < L.rec_off / 4; i += DCSIM_LANES) dcsim_at<uint32_t>(c.blk, 0)[i] = 0u;
  dcsim_warp_sync();
  for (int i = c.lane; i < CAND_N; i += DCSIM_LANES) { CAND_T(c)[i] = DCSIM_INF; CAND_SEQ(c)[i] = 0xffffffffu; }
  DCSIM_FOR_EACH_DC(d, c, sp.n_dc) {
    DCF(c, DF_CUR_FREQ)[d] = sp.dc[d].default_freq; /* models.py:76 */
    DCI(c, DI_FMIN_SLOT)[d] = -1;
    DCF(c, DF_POWER)[d] = (double)sp.dc[d].total_gpus * (sp.dc[d].power_gating ? sp.dc[d].p_sleep : sp.dc[d].p_idle);
  }
  dcsim_warp_sync();
  c.seq = 0u; c.now = 0.0; c.cursor = 0u;
  if (c.lane == 0) {
    const dcsim_arrhdr_t ah = c.P->arr_hdr[c.r];
    c.H->ml_count = ah.ml_count; c.H->status |= ah.status;
    c.H->rng_pos = ah.rng_words; /* every draw of the run happened in the pre-pass */
    for (int s = 0; s < 2 * sp.n_ing; ++s) /* SIM:154-156 */
      if ((ah.first_mask >> s) & 1u) PEND_SEQ(c)[s] = c.seq++;
    const double t = 0.0 + sp.log_interval; /* SIM:157 */
    if (dcsim_schedulable(c, t)) { CAND_T(c)[CAND_LOG(c)] = t; CAND_SEQ(c)[CAND_LOG(c)] = c.seq++; }
    c.H->cand_dirty = 1u;
    c.H->initialized = 1u;
  }
  dcsim_warp_sync();
  dcsim_list_fill(c, 0u, DCSIM_LIST_WINDOW);
  dcsim_list_wait();
}

/* SIM:469-475: util to end_time, then accrue_energy(end_time) WITHOUT power_fn => models.py:82-91. */
DCSIM_DEV void dcsim_replica_tail(dcsim_ctx_t& c) {
  const dcsim_spec_t& sp = c.P->spec;
  const double end = sp.end_time;
  DCSIM_FOR_EACH_DC(d, c, sp.n_dc) {
    const dcsim_dc_t& cfg = sp.dc[d];
    const int busy = DCI(c, DI_BUSY)[d];
    const double last = c.now; /* the latest event's instant: every DC's stamp */
    if (0.0 < last && last < end) DCF(c, DF_UTIL_TIME)[d] += (double)busy * (end - last); /* SIM:471-474 */
    if (last != 0.0) { /* models.py:100-106 with power_fn=None */
      double dt = end - last; dt = dt > 0.0 ? dt : 0.0;
      const double f = DCF(c, DF_CUR_FREQ)[d];
      const double fa = cfg.alpha == 3.0 ? dcsim_cube(f) : pow(f, cfg.alpha);
      const double p_active = (double)busy * (cfg.p_idle + cfg.p_peak * fa);
      const double p_idle = (double)(cfg.total_gpus - busy) * (cfg.power_gating ? cfg.p_sleep : cfg.p_idle);
      DCF(c, DF_ENERGY)[d] += (p_active + p_idle) * dt;
    }
    DCF(c, DF_LAST_T)[d] = end;
  }
  dcsim_warp_sync();
}

/* One popped event (SIM:429-467) of a replica that is `on`: the per-DC accrual with the state before the event, then
 * the handler of the winning candidate slot.  Called by every lane of the warp (see dcsim_event_sync): a replica that
 * is switched off passes through the two synchronisation points and touches nothing.
 *
 * Visibility protocol: the second sync ends every event, so at the next pop-min all shared-memory writes of this one
 * are visible to every lane; inside a handler a (group) sync separates lane 0's part from a lane-parallel step that
 * reads what it wrote.
 *
 * Only the pop-min and these two syncs are event-level.  Making the HANDLERS event-level too (every replica of the
 * warp walks through job_finish, or through the list ring's refill, as soon as one of them has to — so that their
 * collectives also get the full mask) measured 10 % SLOWER (profiles/r02_ab_s16_*): handlers of different replicas
 * are divergent paths of one warp, the scheduler interleaves them, and one replica's L2 round trip hides behind
 * another's arithmetic; a warp-wide sync inside a handler takes that away. */
template <bool CAP, bool RECG>
DCSIM_DEV void dcsim_event_body(dcsim_ctx_t& c, bool on, int win, double t, uint32_t seq, bool tracing, const dcsim_omin_t& om) {
  const dcsim_spec_t& sp = c.P->spec;
  /* SIM:429-437 + models.py:100-106, state before the event.  Every DC's "last" stamp is the previous event's instant
   * (one register for all of them); the first event only stamps (0.0 is the reference's "never touched" sentinel). */
  if (on) {
    if (c.now == 0.0) {
      DCSIM_FOR_EACH_DC(d, c, sp.n_dc) DCF(c, DF_UTIL_BEGIN)[d] = t;
    } else {
      double dt = t - c.now; dt = dt > 0.0 ? dt : 0.0;
      DCSIM_FOR_EACH_DC(d, c, sp.n_dc) {
        DCF(c, DF_UTIL_TIME)[d] += (double)DCI(c, DI_BUSY)[d] * dt;
        DCF(c, DF_ENERGY)[d] += DCF(c, DF_POWER)[d] * dt;
      }
    }
  }
  dcsim_event_sync(); /* every lane has read its candidate / busy / power before lane 0's handler rewrites them */
  dcsim_omin_publish(c, om); /* (before the handler: it may dirty the event set again) */
  if (on) {
    c.now = t;
    /* dispatch on the winning slot itself; the event kind is only spelled out for the (cold) trace */
    if (tracing && c.lane == 0) {
      int kind = KIND_FINISH;
      if (win == CAND_LIST(c)) {
        const uint32_t m = LW_META(c)[c.cursor & (DCSIM_LIST_WINDOW - 1u)];
        kind = (m & ML_XFER) ? KIND_XFER : (int)((m >> 1) & 1u); /* the job type is the stream's low bit */
      } else if (win == CAND_LOG(c)) {
        kind = KIND_LOG;
      }
      const uint32_t row = c.P->rec.counts[0];
      if (row < c.P->rec.trace_cap) { c.P->rec.trace[row].t = t; c.P->rec.trace[row].seq = seq; c.P->rec.trace[row].kind = (uint32_t)kind; }
      c.P->rec.counts[0] = row + 1u;
    }

    if (win == CAND_LIST(c)) {
      dcsim_handle_list<CAP>(c);
    } else if (win < CAND_LIST(c)) {
      dcsim_handle_finish<CAP, RECG>(c, win - CAND_DC0);
    } else if (win == CAND_LOG(c)) {
      if (c.lane == 0) c.H->ev_log++;
      dcsim_handle_log<CAP>(c);
    } else if constexpr (CAP) { /* a superseded job_finish: it advanced the clock and accrued energy, nothing else (SIM:456-461) */
      if (c.lane == 0) {
        c.H->ev_fin++;
        const uint32_t ks = c.H->smin_slot, last = c.H->n_stale - 1u;
        dcsim_at<double>(c.blk, c.P->L.st_t)[ks] = dcsim_at<double>(c.blk, c.P->L.st_t)[last];
        dcsim_at<uint32_t>(c.blk, c.P->L.st_seq)[ks] = dcsim_at<uint32_t>(c.blk, c.P->L.st_seq)[last];
        c.H->n_stale = last;
      }
      dcsim_warp_sync();
      dcsim_rescan_stale(c);
    }
  }
  dcsim_event_sync(); /* the handler's writes (lane 0's mostly) are visible to every lane's next pop-min */
}

/* SIM:423-467: the event loop.  Returns the number of events processed by this call.  `live`: this lane group holds a
 * replica that has not reached end_time yet (false: it only keeps the warp's other replicas company, see below). */
template <bool CAP, bool RECG>
DCSIM_DEV uint32_t dcsim_replica_run(dcsim_ctx_t& c, bool live) {
  const dcsim_spec_t& sp = c.P->spec;
  const uint32_t budget = c.P->budget32; /* per-launch event budget; 0xffffffff = unlimited */
  const bool tracing = c.is_traced && c.P->rec.trace != nullptr;
  uint32_t done_here = 0u;
  bool finished = false;
#if (!defined(DCSIM_HOST_EMU) && DCSIM_LANES < 32) || defined(DCSIM_HOST_UNIFORM_LOOP) /* (the latter: a test-only host build of THIS skeleton) */
  /* Several replicas per warp: the loop is WARP-uniform.  A replica that ends (end_time, event budget, a status bit)
   * is switched off and rides along — through at most the rest of a 16-event chunk of no-ops, then idle as its lanes
   * would be anyway — until every replica of the warp has ended.  That is what lets the pop-min and the two
   * synchronisation points of an event use the constant full member mask (dcsim_event_sync). */
  bool on = live;
  for (;;) {
    /* a capacity overflowed (or a sampler ran away): stop and report, never guess.  Polled every 16 events — every
     * capacity check refuses the write on its own, so a replica that overflowed stays memory-safe until it is seen */
    {
      /* lane 0 hands out the seqs; the packed (seq, slot) reduction of the pop-min needs them below 2^28.  Checked once
       * per chunk with 2^20 of slack (one event pushes a few; the cap controller at most a job_finish per running job) */
      const uint32_t seq0 = dcsim_event_bcast_u32(c.seq, 0);
      if (on && seq0 >= DCSIM_SEQ_LIMIT) { if (c.lane == 0) c.H->status |= DCSIM_ST_SEQ_OVERFLOW; on = false; }
    }
    if (on && c.H->status != 0u) on = false;
    if (!dcsim_event_any(on && done_here < budget)) break;
#pragma unroll 1
    for (int k = 0; k < 16; ++k) {
      if (done_here >= budget) on = false;
      double t = 0.0; uint32_t seq = 0u;
      dcsim_omin_t om;
      const int win = dcsim_argmin_cand(c, om, &t, &seq);
      if (on && (win < 0 || t > sp.end_time)) { finished = true; on = false; } /* `while self.event_q` / SIM:427 */
      dcsim_event_body<CAP, RECG>(c, on, win, t, seq, tracing, om);
      if (on) ++done_here;
    }
  }
#else
  if (!live) return 0u;
  for (;;) {
    /* a capacity overflowed (or a sampler ran away): stop and report, never guess.  Polled every 16 events — every
     * capacity check refuses the write on its own, so a replica that overflowed stays memory-safe until it is seen */
    if (done_here >= budget || c.H->status != 0u) break;
    uint32_t chunk = budget - done_here; chunk = chunk < 16u ? chunk : 16u;
    uint32_t k = 0u;
    for (; k < chunk; ++k) {
      double t; uint32_t seq;
      dcsim_omin_t om;
      const int win = dcsim_argmin_cand(c, om, &t, &seq);
      if (win < 0) { finished = true; break; }         /* `while self.event_q` */
      if (t > sp.end_time) { finished = true; break; } /* SIM:427 */
      dcsim_event_body<CAP, RECG>(c, true, win, t, seq, tracing, om);
    } /* 16-event chunk */
    done_here += k;
    if (finished) break;
  }
#endif
  if (finished && c.H->done == 0u) {
    dcsim_replica_tail(c);
    if (c.lane == 0) c.H->done = 1u;
    dcsim_warp_sync();
  }
  return done_here;
}

/* Writes the replica's row of the summary array (layout: include/dcsim_b200.h). */
DCSIM_DEV void dcsim_write_summary(dcsim_ctx_t& c, double* out) {
  const dcsim_spec_t& sp = c.P->spec;
  const dcsim_hdr_t* H = c.H;
  for (int i = c.lane; i < DCSIM_SUMMARY_K; i += DCSIM_LANES) out[i] = 0.0;
  dcsim_warp_sync();
  if (c.lane == 0) {
    double tot = 0.0;
    for (int d = 0; d < sp.n_dc; ++d) tot += DCF(c, DF_ENERGY)[d];
    out[DCSIM_S_STATUS] = (double)H->status;
    out[DCSIM_S_EVENTS] = (double)H->n_events;
    out[DCSIM_S_JOBS_FINISHED] = (double)(H->n_fin_inf + H->n_fin_trn);
    out[DCSIM_S_JOBS_CREATED] = (double)H->jid;
    out[DCSIM_S_TOTAL_ENERGY_J] = tot;
    out[DCSIM_S_LAT_SUM] = H->lat_sum;
    out[DCSIM_S_LAT_SUM_INF] = H->lat_sum_inf; out[DCSIM_S_FIN_INF] = (double)H->n_fin_inf;
    out[DCSIM_S_LAT_SUM_TRN] = H->lat_sum_trn; out[DCSIM_S_FIN_TRN] = (double)H->n_fin_trn;
    out[DCSIM_S_RNG_WORDS] = (double)H->rng_pos;
    out[DCSIM_S_LAST_T] = H->last_t;
    out[DCSIM_S_SEQ] = (double)H->seq;
    out[DCSIM_S_EV_ARRIVAL] = (double)H->ev_arr; out[DCSIM_S_EV_XFER] = (double)H->ev_xfer;
    out[DCSIM_S_EV_FINISH] = (double)H->ev_fin; out[DCSIM_S_EV_LOG] = (double)H->ev_log;
    out[DCSIM_S_DONE] = (double)H->done;
    out[DCSIM_S_MAX_XFER] = 0.0; /* there is no pool of in-flight transfers to size any more */
    out[DCSIM_S_MAX_RUN] = (double)H->max_run;
    out[DCSIM_S_MAX_Q] = (double)H->max_q;
    out[DCSIM_S_UTIL_BEGIN] = DCF(c, DF_UTIL_BEGIN)[0];
  }
  DCSIM_FOR_EACH_DC(d, c, sp.n_dc) {
    double* o = out + DCSIM_S_DC0 + d * DCSIM_S_DC_STRIDE;
    o[DCSIM_SD_ENERGY_J] = DCF(c, DF_ENERGY)[d];
    o[DCSIM_SD_UTIL_GPU_TIME] = DCF(c, DF_UTIL_TIME)[d];
    o[DCSIM_SD_ACC_JOB_UNIT] = DCF(c, DF_ACC_UNIT)[d];
    o[DCSIM_SD_BUSY] = (double)DCI(c, DI_BUSY)[d];
    o[DCSIM_SD_CURRENT_FREQ] = DCF(c, DF_CUR_FREQ)[d];
    o[DCSIM_SD_Q_INF] = (double)dcsim_queue_len(c, d, 0);
    o[DCSIM_SD_Q_TRN] = (double)dcsim_queue_len(c, d, 1);
    o[DCSIM_SD_RUNNING] = (double)DCI(c, DI_NRUN)[d];
  }
}

/* One replica, one launch: (init |) resume -> run -> summary.  `blk` is the working copy of the state
 * block (shared memory on the GPU), already loaded unless `fresh`; `rec` is the base the running-job record offsets
 * apply to (== blk when the records were staged with it, the block's home in HBM when only the head was: RECG). */
template <bool CAP, bool RECG>
DCSIM_DEV uint32_t dcsim_replica_step(const dcsim_kparams_t* P, uint64_t r, char* blk, char* rec, bool fresh, bool ghost = false) {
  dcsim_ctx_t c;
  c.P = P; c.blk = blk; c.rec = rec; c.H = reinterpret_cast<dcsim_hdr_t*>(blk); c.lane = dcsim_lane();
  c.r = (uint32_t)r; /* n_replicas < 2^32 (checked by dcsim_create) */
  c.is_traced = !ghost && ((int64_t)r == P->rec.trace_replica);
  c.is_logged = !ghost && ((int64_t)r == P->rec.log_replica);
  c.is_ghost = ghost;
  if (ghost) { /* a lane group without a replica (the batch's last warp): reads whatever is there, writes nothing */
    c.seq = 0u; c.now = 0.0; c.cursor = 0u;
    return dcsim_replica_run<CAP, RECG>(c, false);
  }
  if (fresh) {
    dcsim_replica_init(c);
  } else { /* resume: hot scalars back into registers */
    c.seq = c.H->seq; c.now = c.H->now; c.cursor = c.H->ml_cursor;
  }
  const uint32_t n = dcsim_replica_run<CAP, RECG>(c, c.H->done == 0u);
  dcsim_list_wait(); /* a refill still in flight lands before the block is staged out (the ring is part of it) */
  if (c.lane == 0) {
    c.H->ev_xfer = c.cursor - c.H->ev_arr; /* every consumed list entry is an arrival or an xfer_done */
    c.H->jid = c.H->ev_arr;                /* SIM:539: one jid per arrival */
    c.H->n_events = c.H->ev_arr + c.H->ev_xfer + c.H->ev_fin + c.H->ev_log; /* every processed event is one of these */
    c.H->seq = c.seq; c.H->now = c.now; c.H->last_t = c.H->n_events ? c.now : 0.0;
    c.H->ml_cursor = c.cursor;
    if (c.H->done == 0u) /* (the tail stamped end_time itself) */
      for (int d = 0; d < P->spec.n_dc; ++d) DCF(c, DF_LAST_T)[d] = c.now;
  }
  dcsim_warp_sync();
  dcsim_write_summary(c, P->summary + r * DCSIM_SUMMARY_K);
  dcsim_warp_sync();
  return n;
}
