/*
 * dcsim_b200.cu — sm_100a kernels and the C-ABI of include/dcsim_b200.h.
 *
 * Kernels
 *   dcsim_arrivals_kernel     one thread per replica: the replica's arrival sequence (instants, routed DCs, size deviates).
 *   dcsim_merge_kernel        one warp per replica: job sizes, xfer_done instants and the merged, time-ordered
 *                             {arrival, xfer_done} list the event loop consumes.
 *   dcsim_advance_kernel      one warp per replica; stages the replica's state block HBM -> shared memory, runs the
 *                             event loop of dcsim_core.cuh, stages it back, writes the summary row.  Instantiated
 *                             over <CAP, MODE> (power-cap controller compiled in / what is staged) and picked per handle.
 *   dcsim_reduce_kernel       [n_replicas][K] summaries -> DCSIM_AGG_K doubles (the only cross-GPU payload).
 *   dcsim_hist_reduce_kernel  per-replica job-latency histograms -> one [2][128] histogram (opt-in).
 *
 * Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -fmad=false (see __graft_entry__.build()).
 * -fmad=false matters: the reference is CPython float arithmetic, one rounding per operation.
 */
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <new>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define DCSIM_ADV_SUFFIX _g32
#include "dcsim_advance_impl.cuh" /* the 32-lanes-per-replica event loop (and dcsim_core.cuh) */

/* the builds with several replicas per warp live in their own translation units (dcsim_advance_g8.cu, _g16.cu) */
cudaError_t dcsim_adv_launch_g16(const dcsim_kparams_t*, unsigned long long*, int, int, int, int, int, cudaStream_t);
cudaError_t dcsim_adv_attrs_g16(int, int, int, int, int, int*, int*, int*);
cudaError_t dcsim_adv_launch_g8(const dcsim_kparams_t*, unsigned long long*, int, int, int, int, int, cudaStream_t);
cudaError_t dcsim_adv_attrs_g8(int, int, int, int, int, int*, int*, int*);
int dcsim_adv_min_ctas_g16(void);
int dcsim_adv_min_ctas_g8(void);

/* Arrival pre-pass: one THREAD per replica draws that replica's whole arrival sequence in the reference's draw order;
 * consecutive threads = consecutive replicas, so all 32 lanes of a warp run the samplers that the event loop would
 * otherwise run on one lane.  Per-thread scratch in shared memory, [slot][thread]: 2*MAX_ING stream clocks (f64),
 * 2*MAX_ING "latest arrival of the stream" indices (u32), DCSIM_TRNG_RING staged random words (u32). */
#define DCSIM_ARRIVALS_THREADS 128
/* 7 resident CTAs per SM (<= 73 registers, <= 32 kB of scratch each): 148 x 7 x 128 = 132 608 threads, so that a batch of
 * 131 072 replicas (BASELINE config 5 per GPU) is still ONE wave of this latency-bound kernel. */
#define DCSIM_ARRIVALS_MIN_CTAS 7
static size_t dcsim_arrivals_scratch_bytes(int n_ing) { /* per CTA: [slot][thread] arrays for 2 * n_ing streams */
  return (size_t)DCSIM_ARRIVALS_THREADS * ((size_t)(2 * n_ing) * (sizeof(double) + sizeof(uint32_t)) + DCSIM_TRNG_RING * sizeof(uint32_t));
}
extern __shared__ __align__(16) double dcsim_arr_scratch[];
template <bool MT>
__global__ void __launch_bounds__(DCSIM_ARRIVALS_THREADS, DCSIM_ARRIVALS_MIN_CTAS) dcsim_arrivals_kernel(const __grid_constant__ dcsim_kparams_t P) {
  const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= P.n_replicas) return;
  const int n_streams = 2 * P.spec.n_ing;
  double* clocks = dcsim_arr_scratch + threadIdx.x;                                             /* [stream][thread] */
  uint32_t* last = reinterpret_cast<uint32_t*>(dcsim_arr_scratch + n_streams * blockDim.x) + threadIdx.x; /* [stream][thread] */
  uint32_t* ring = last + n_streams * blockDim.x;                                               /* [word][thread] */
  dcsim_generate_arrivals<MT>(&P, r, clocks, last, ring, (int)blockDim.x);
}

/* List merge: one WARP per replica (lane-parallel over the replica's arrivals), a sliding window of them in shared memory. */
#define DCSIM_MERGE_THREADS 128
__global__ void __launch_bounds__(DCSIM_MERGE_THREADS) dcsim_merge_kernel(const __grid_constant__ dcsim_kparams_t P) {
  __shared__ dcsim_merge_ring_t rings[DCSIM_MERGE_THREADS / 32];
  const uint64_t r = (uint64_t)blockIdx.x * (DCSIM_MERGE_THREADS / 32) + (threadIdx.x >> 5);
  if (r >= P.n_replicas) return;
  dcsim_merge_arrivals(&P, r, (int)(threadIdx.x & 31u), &rings[threadIdx.x >> 5]);
}

/* Sums the per-replica latency histograms: thread b of every block owns bin b (coalesced 1 KB rows). */
__global__ void dcsim_hist_reduce_kernel(const uint32_t* __restrict__ hist, uint64_t n, unsigned long long* __restrict__ out) {
  unsigned long long acc = 0ull;
  for (uint64_t r = blockIdx.x; r < n; r += gridDim.x) acc += hist[r * (2 * DCSIM_LAT_BINS) + threadIdx.x];
  if (acc) atomicAdd(out + threadIdx.x, acc);
}

/* Aggregates the summaries; every block reduces a slice, then one atomicAdd per component. */
__global__ void dcsim_reduce_kernel(const double* __restrict__ summary, uint64_t n, double* __restrict__ out) {
  double acc[DCSIM_AGG_K];
#pragma unroll
  for (int k = 0; k < DCSIM_AGG_K; ++k) acc[k] = 0.0;
  for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x) {
    const double* s = summary + r * DCSIM_SUMMARY_K;
    const double fin = s[DCSIM_S_JOBS_FINISHED], e = s[DCSIM_S_TOTAL_ENERGY_J];
    const double ml = fin > 0.0 ? s[DCSIM_S_LAT_SUM] / fin : 0.0;
    acc[DCSIM_A_REPLICAS] += 1.0;
    acc[DCSIM_A_FAILED] += (s[DCSIM_S_STATUS] != 0.0 || s[DCSIM_S_DONE] == 0.0) ? 1.0 : 0.0;
    acc[DCSIM_A_EVENTS] += s[DCSIM_S_EVENTS];
    acc[DCSIM_A_JOBS] += fin;
    acc[DCSIM_A_ENERGY] += e;
    acc[DCSIM_A_ENERGY_SQ] += e * e;
    acc[DCSIM_A_LAT_SUM] += s[DCSIM_S_LAT_SUM];
    acc[DCSIM_A_MEANLAT_SUM] += ml;
    acc[DCSIM_A_MEANLAT_SQ] += ml * ml;
    acc[DCSIM_A_RNG_WORDS] += s[DCSIM_S_RNG_WORDS];
    acc[DCSIM_A_RUNNING] += (s[DCSIM_S_STATUS] == 0.0 && s[DCSIM_S_DONE] == 0.0) ? 1.0 : 0.0;
  }
#pragma unroll
  for (int k = 0; k < DCSIM_AGG_K; ++k) {
    double v = acc[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31u) == 0u && v != 0.0) atomicAdd(out + k, v);
  }
}

/* ================================================================================================
 * C-ABI
 * ============================================================================================== */
struct dcsim {
  dcsim_spec_t spec;
  dcsim_layout_t L;
  uint64_t n_replicas, seed0;
  int device, sm_count, warps_per_cta, ctas, smem_bytes, regs, resident_warps;
  int lanes; /* lanes per replica of the advance kernel picked for this handle: 32, 16 or 8 */
  cudaStream_t stream, own_stream;
  char* d_state;
  char* d_queues;
  double* d_summary;
  double* h_summary_pinned; /* page-locked host mirror of d_summary, allocated on first use (dcsim_fetch_summary_host) */
  unsigned long long* d_events;
  double* d_agg;                 /* DCSIM_AGG_K doubles: scratch of dcsim_all_done */
  unsigned long long* d_hist_out; /* [2][DCSIM_LAT_BINS]: scratch of dcsim_fetch_latency_histogram */
  uint32_t* d_counts;
  dcsim_trace_rec_t* d_trace;
  dcsim_job_rec_t* d_jobs;
  dcsim_cluster_rec_t* d_cluster;
  uint32_t trace_cap, jobs_cap, cluster_cap;
  uint32_t jobs_alloc, cluster_alloc; /* rows the log buffers can hold (kept across set_logging calls) */
  int want_job_log;                   /* layout the NEXT batch needs; applied lazily by ensure_layout() */
  int64_t trace_replica, log_replica;
  int launches;
  int arrivals_ready, mode; /* mode: DCSIM_MODE_* of the advance kernel for this handle's layout */
  double* d_arr_t;
  double* d_arr_raw;
  uint32_t* d_arr_meta;
  uint32_t* d_arr_pred;
  double* d_arr_tx;
  uint32_t* d_arr_fin;
  double* d_ml_t;
  double* d_ml_aux;
  uint32_t* d_ml_meta;
  dcsim_arrhdr_t* d_arr_hdr;
  double max_transfer;
  uint32_t* d_hist;
  uint32_t* d_mt; /* [624][n_replicas] Mersenne Twister states, rng_kind == DCSIM_RNG_MT19937 only */
  int rng_kind;
  uint32_t cap_arr;
  unsigned long long events_seen;
  char err[512];
};

static thread_local char g_create_err[512] = "";
#ifdef DCSIM_DEVICE_TEST_HOOKS
static double g_test_time_quantum = 0.0; /* TEST-ONLY builds: dcsim_test_set_time_quantum */
#endif

static int set_err(dcsim_t* h, int code, const char* fmt, const char* a = "", long long b = 0) {
  char* dst = h ? h->err : g_create_err;
  snprintf(dst, 512, fmt, a, b);
  return code;
}

#define CUDA_TRY(h, call)                                                                  \
  do {                                                                                     \
    cudaError_t e_ = (call);                                                               \
    if (e_ != cudaSuccess)                                                                 \
      return set_err(h, e_ == cudaErrorMemoryAllocation ? DCSIM_E_NOMEM : DCSIM_E_CUDA,    \
                     "CUDA error: %s (line %lld)", cudaGetErrorString(e_), (long long)__LINE__); \
  } while (0)

extern "C" {

size_t dcsim_sizeof_spec(void) { return sizeof(dcsim_spec_t); }
uint32_t dcsim_abi_version(void) { return DCSIM_ABI_VERSION; }
int dcsim_summary_k(void) { return DCSIM_SUMMARY_K; }

static int validate_spec(const dcsim_spec_t* sp) {
  if (sp->magic != DCSIM_SPEC_MAGIC) return set_err(NULL, DCSIM_E_INVALID, "spec: bad magic%s%lld");
  if (sp->abi_version != DCSIM_ABI_VERSION) return set_err(NULL, DCSIM_E_INVALID, "spec: ABI version mismatch%s%lld");
  if (sp->spec_bytes != sizeof(dcsim_spec_t)) return set_err(NULL, DCSIM_E_INVALID, "spec: struct size mismatch (producer says %s%lld bytes)", "", sp->spec_bytes);
  if (sp->n_dc < 1 || sp->n_dc > DCSIM_MAX_DC || sp->n_ing < 1 || sp->n_ing > DCSIM_MAX_ING)
    return set_err(NULL, DCSIM_E_INVALID, "spec: n_dc / n_ing out of range%s%lld");
  if (!(sp->log_interval > 0.0)) return set_err(NULL, DCSIM_E_INVALID, "spec: log_interval must be > 0%s%lld");
  if (sp->policy_name != DCSIM_POLICY_ENERGY_AWARE && sp->policy_name != DCSIM_POLICY_PERF_FIRST)
    return set_err(NULL, DCSIM_E_INVALID, "Unknown policy name%s%lld"); /* policy.py:41 */
  for (int k = 0; k < 2; ++k) {
    const dcsim_arrival_t* a = &sp->arr[k];
    if (a->mode < DCSIM_ARR_OFF || a->mode > DCSIM_ARR_SINUSOID) return set_err(NULL, DCSIM_E_INVALID, "Unknown mode%s%lld"); /* arrivals.py:33 */
    if (a->mode == DCSIM_ARR_SINUSOID && !(a->rate > 0.0 && a->period > 0.0))
      return set_err(NULL, DCSIM_E_INVALID, "sinusoid arrivals need rate > 0 and period > 0%s%lld");
    if (a->mode == DCSIM_ARR_SINUSOID && (a->amp > 1.0 || a->amp < -1.0))
      return set_err(NULL, DCSIM_E_INVALID, "sinusoid arrivals with |amp| > 1 never terminate in the reference (arrivals.py:41-45)%s%lld");
  }
  for (int d = 0; d < sp->n_dc; ++d) {
    const dcsim_dc_t* c = &sp->dc[d];
    if (c->total_gpus < 0 || c->n_freq < 1 || c->n_freq > DCSIM_MAX_FREQ)
      return set_err(NULL, DCSIM_E_INVALID, "spec: DC %s%lld has bad total_gpus / n_freq", "", d);
    if (c->total_gpus > 65535) /* a running record packs the job's GPU count into 16 bits */
      return set_err(NULL, DCSIM_E_INVALID, "spec: DC %s%lld has more than 65535 GPUs", "", d);
  }
  if (sp->cap_arrivals < 0 || (uint32_t)sp->cap_arrivals >= DCSIM_MAX_ARRIVALS)
    return set_err(NULL, DCSIM_E_INVALID, "spec: cap_arrivals must be below 2^24 (%s%lld given)", "", sp->cap_arrivals);
  if (sp->algo < DCSIM_ALGO_DEFAULT || sp->algo > DCSIM_ALGO_CAP_GREEDY)
    return set_err(NULL, DCSIM_E_UNSUPPORTED, "spec: unknown algo id %s%lld", "", sp->algo);
  return DCSIM_OK;
}

/* Launch geometry for the handle's current state-block layout: lanes per replica (32 / 16 / 8), what is staged (whole
 * block / head only / nothing), warps per CTA, shared memory.
 *   DCSIM_GROUP=32|16|8     forces the lanes per replica (default: see pick below);
 *   DCSIM_RECORDS=shared|global forces the whole-block / head-only staging (A/B runs). */
typedef cudaError_t (*dcsim_adv_launch_fn)(const dcsim_kparams_t*, unsigned long long*, int, int, int, int, int, cudaStream_t);
typedef cudaError_t (*dcsim_adv_attrs_fn)(int, int, int, int, int, int*, int*, int*);
static dcsim_adv_launch_fn adv_launch_for(int lanes) { return lanes == 8 ? dcsim_adv_launch_g8 : (lanes == 16 ? dcsim_adv_launch_g16 : dcsim_adv_launch_g32); }
static dcsim_adv_attrs_fn adv_attrs_for(int lanes) { return lanes == 8 ? dcsim_adv_attrs_g8 : (lanes == 16 ? dcsim_adv_attrs_g16 : dcsim_adv_attrs_g32); }
static int min_ctas_for(int lanes) { return lanes == 8 ? dcsim_adv_min_ctas_g8() : (lanes == 16 ? dcsim_adv_min_ctas_g16() : dcsim_adv_min_ctas_g32()); }

static int resident_warps_for(int bytes_per_warp, int smem_optin, int smem_sm, int max_warps, int* wpc_out) {
  /* warps per CTA: whichever of 4 / 2 / 1 keeps the most warps resident (each CTA also reserves 1 KB of shared
   * memory and an SM holds at most 32 CTAs); small state blocks end up at 4 x 8 CTAs, large ones at 1 or 2 */
  int wpc = 0, best_warps = 0;
  for (int cand = DCSIM_MAX_WARPS_PER_CTA; cand >= 1; cand >>= 1) {
    const long long per_cta = (long long)cand * bytes_per_warp;
    if (per_cta > smem_optin) continue;
    int ctas = (int)(smem_sm / (per_cta + 1024));
    if (ctas > 32) ctas = 32;
    int warps = ctas * cand;
    if (warps > max_warps) warps = max_warps; /* register bound */
    if (warps > best_warps) { best_warps = warps; wpc = cand; }
  }
  *wpc_out = wpc;
  return best_warps;
}

static cudaError_t size_launch(dcsim_t* h) {
  cudaError_t e;
  int smem_optin = 0, smem_sm = 0;
  if ((e = cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device)) != cudaSuccess) return e;
  if ((e = cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, h->device)) != cudaSuccess) return e;
  /* Lanes per replica.  Four replicas per warp share everything warp-wide in an event (pop-min, DC sweep, the lane-0
   * handler's issue slots) and pay whenever the event set fits one round of 8 lanes: up to 5 DCs (n_dc finish slots +
   * list + log + stale).  Measured with the event-level pop-min (profiles/r02_ab_s17_*): 4 DC x 64 +35 % over the
   * 32-lane build, debug n=2 +34 %, joint_nf / carbon_cost (up to 64 running jobs per DC: a job_finish walks them 8
   * at a time) +2..3 %; 8 DC x 256 (two slots per lane, all 8 lanes in the sweep) -10 %: it keeps the whole warp. */
  int lanes = h->spec.n_dc <= 5 ? 8 : 32;
  if (lanes == 8) {
    /* ... unless four blocks per warp leave the SM with hardly more resident REPLICAS than one per warp would (very
     * large heads: the power-cap controller's pools — cap_greedy 4 x 64: 12 vs 14 replicas per SM, and the 32-lane
     * build is 1.6x faster there, profiles/r02_ab_s19_*; the bandit's tables: 52 vs 32, 8 lanes 18 % faster) */
    int w8 = 0, w32 = 0, unused = 0;
    const int bytes8 = 4 * h->L.rec_off, bytes32 = h->L.rec_off; /* head-staged: the smallest footprint of each */
    w8 = resident_warps_for(bytes8, smem_optin, smem_sm, min_ctas_for(8) * DCSIM_MAX_WARPS_PER_CTA, &unused);
    w32 = resident_warps_for(bytes32, smem_optin, smem_sm, min_ctas_for(32) * DCSIM_MAX_WARPS_PER_CTA, &unused);
    if (2 * (4 * w8) < 3 * w32) lanes = 32; /* fewer than 1.5x the replicas per SM */
  }
  { const char* g = getenv("DCSIM_GROUP"); if (g) { const int v = atoi(g); if (v == 8 || v == 16 || v == 32) lanes = v; } }
  const int rpw = 32 / lanes; /* replicas per warp */
  const int max_warps = min_ctas_for(lanes) * DCSIM_MAX_WARPS_PER_CTA;
  int wpc_full = 0, wpc_head = 0;
  const int warps_full = resident_warps_for(rpw * h->L.total_bytes, smem_optin, smem_sm, max_warps, &wpc_full);
  const int warps_head = resident_warps_for(rpw * h->L.rec_off, smem_optin, smem_sm, max_warps, &wpc_head);
  const char* force = getenv("DCSIM_RECORDS");
  int mode, wpc, bytes;
  if (wpc_full >= 1 && (warps_full >= warps_head || (force && force[0] == 's')) && !(force && force[0] == 'g' && wpc_head >= 1)) {
    mode = DCSIM_MODE_STAGED; wpc = wpc_full; bytes = h->L.total_bytes;   /* records staged with the rest */
  } else if (wpc_head >= 1) {
    mode = DCSIM_MODE_HEAD; wpc = wpc_head; bytes = h->L.rec_off;          /* records stay in HBM/L2 */
  } else { /* not even the head fits a CTA's shared memory: run in place out of HBM/L2 */
    mode = DCSIM_MODE_INPLACE; wpc = DCSIM_MAX_WARPS_PER_CTA; bytes = 0;
  }
  h->lanes = lanes;
  h->mode = mode;
  h->warps_per_cta = wpc;
  h->smem_bytes = wpc * rpw * bytes;
  const uint64_t per_cta = (uint64_t)wpc * (uint64_t)rpw;
  h->ctas = (int)((h->n_replicas + per_cta - 1) / per_cta);
  int blocks_per_sm = 0, min_ctas = 0;
  if ((e = adv_attrs_for(lanes)(h->L.cap_stale != 0, h->mode, wpc * 32, h->smem_bytes, smem_optin, &h->regs, &blocks_per_sm, &min_ctas)) != cudaSuccess) return e;
  h->resident_warps = blocks_per_sm * wpc;
  return cudaSuccess;
}

/* job_log.csv needs size / f / jid in the running records; switching it on or off re-lays the state block out. */
static int relayout(dcsim_t* h, int job_log) {
  dcsim_layout_t L;
  dcsim_make_layout(&h->spec, &L, job_log);
  if (L.lean == h->L.lean) return DCSIM_OK;
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->L = L;
  CUDA_TRY(h, size_launch(h));
  if (h->d_state) { cudaFree(h->d_state); h->d_state = NULL; }
  const size_t state_bytes = (size_t)h->n_replicas * (size_t)h->L.total_bytes;
  CUDA_TRY(h, cudaMalloc(&h->d_state, state_bytes));
  CUDA_TRY(h, cudaMemsetAsync(h->d_state, 0, state_bytes, h->stream));
  return DCSIM_OK;
}

int dcsim_create(const void* spec_blob, size_t spec_bytes, uint64_t n_replicas, uint64_t base_seed,
                 uint64_t first_replica_id, int device, dcsim_t** out) {
  if (!out) return set_err(NULL, DCSIM_E_INVALID, "create: out is NULL%s%lld");
  *out = NULL;
  if (!spec_blob || spec_bytes != sizeof(dcsim_spec_t))
    return set_err(NULL, DCSIM_E_INVALID, "create: spec blob must be %s%lld bytes", "", (long long)sizeof(dcsim_spec_t));
  if (n_replicas == 0) return set_err(NULL, DCSIM_E_INVALID, "create: n_replicas must be > 0%s%lld");
  if (n_replicas > 0xffffffffull) /* the event loop keeps the local replica index in 32 bits */
    return set_err(NULL, DCSIM_E_INVALID, "create: n_replicas must be below 2^32 per handle%s%lld");
  dcsim_spec_t sp;
  memcpy(&sp, spec_blob, sizeof(sp));
  int rc = validate_spec(&sp);
  if (rc != DCSIM_OK) return rc;

  dcsim_t* h = new (std::nothrow) dcsim();
  if (!h) return set_err(NULL, DCSIM_E_NOMEM, "create: host allocation failed%s%lld");
  memset(h, 0, sizeof(*h));
  h->spec = sp;
  dcsim_make_layout(&h->spec, &h->L, /*job_log=*/0);
  h->cap_arr = (uint32_t)(h->spec.cap_arrivals > 0 ? h->spec.cap_arrivals : 16384);
  for (int i = 0; i < h->spec.n_ing; ++i)
    for (int d = 0; d < h->spec.n_dc; ++d)
      for (int jt = 0; jt < 2; ++jt) {
        const double v = h->spec.transfer_s[i][d][jt];
        if (v == v && v < 1e300 && v > h->max_transfer) h->max_transfer = v; /* finite ones only */
      }
  h->n_replicas = n_replicas;
  h->seed0 = base_seed + first_replica_id;
  h->device = device;
  h->trace_replica = -1;
  h->log_replica = -1;

#define CREATE_TRY(call)                                                                  \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) {                                                              \
      rc = set_err(NULL, e_ == cudaErrorMemoryAllocation ? DCSIM_E_NOMEM : DCSIM_E_CUDA,  \
                   "CUDA error in create: %s (line %lld)", cudaGetErrorString(e_), (long long)__LINE__); \
      dcsim_destroy(h);                                                                   \
      return rc;                                                                          \
    }                                                                                     \
  } while (0)

  CREATE_TRY(cudaSetDevice(device));
  CREATE_TRY(cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device));
  CREATE_TRY(size_launch(h));
  CREATE_TRY(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  h->stream = h->own_stream;
  const size_t state_bytes = (size_t)n_replicas * (size_t)h->L.total_bytes;
  if (h->L.queue_bytes >= (1ull << 32)) /* the event loop addresses inside one replica's FIFOs with 32 bits */
  {
    rc = set_err(NULL, DCSIM_E_INVALID, "create: one replica's FIFO queues exceed 4 GB (cap_q_inf / cap_q_trn too large)%s%lld");
    dcsim_destroy(h);
    return rc;
  }
  const size_t queue_bytes = (size_t)n_replicas * (size_t)h->L.queue_bytes;
  CREATE_TRY(cudaMalloc(&h->d_state, state_bytes));
  CREATE_TRY(cudaMalloc(&h->d_queues, queue_bytes ? queue_bytes : 16));
  CREATE_TRY(cudaMalloc(&h->d_summary, (size_t)n_replicas * DCSIM_SUMMARY_K * sizeof(double)));
  {
    const size_t ne = (size_t)n_replicas * (size_t)h->cap_arr;
    CREATE_TRY(cudaMalloc(&h->d_arr_t, ne * sizeof(double)));
    CREATE_TRY(cudaMalloc(&h->d_arr_raw, ne * sizeof(double)));
    CREATE_TRY(cudaMalloc(&h->d_arr_meta, ne * sizeof(uint32_t)));
    CREATE_TRY(cudaMalloc(&h->d_arr_pred, ne * sizeof(uint32_t)));
    CREATE_TRY(cudaMalloc(&h->d_arr_tx, ne * sizeof(double)));
    CREATE_TRY(cudaMalloc(&h->d_arr_fin, ne * sizeof(uint32_t)));
    CREATE_TRY(cudaMalloc(&h->d_ml_t, 2 * ne * sizeof(double)));
    CREATE_TRY(cudaMalloc(&h->d_ml_aux, 2 * ne * sizeof(double)));
    CREATE_TRY(cudaMalloc(&h->d_ml_meta, 2 * ne * sizeof(uint32_t)));
    CREATE_TRY(cudaMalloc(&h->d_arr_hdr, (size_t)n_replicas * sizeof(dcsim_arrhdr_t)));
  }
  CREATE_TRY(cudaMalloc(&h->d_events, sizeof(unsigned long long)));
  CREATE_TRY(cudaMalloc(&h->d_agg, DCSIM_AGG_K * sizeof(double)));
  CREATE_TRY(cudaMalloc(&h->d_hist_out, 2 * DCSIM_LAT_BINS * sizeof(unsigned long long)));
  CREATE_TRY(cudaMalloc(&h->d_counts, 4 * sizeof(uint32_t)));
  CREATE_TRY(cudaMemsetAsync(h->d_state, 0, state_bytes, h->stream)); /* hdr.initialized == 0 => fresh replica */
  CREATE_TRY(cudaMemsetAsync(h->d_summary, 0, (size_t)n_replicas * DCSIM_SUMMARY_K * sizeof(double), h->stream));
  CREATE_TRY(cudaMemsetAsync(h->d_events, 0, sizeof(unsigned long long), h->stream));
  CREATE_TRY(cudaMemsetAsync(h->d_counts, 0, 4 * sizeof(uint32_t), h->stream));
  CREATE_TRY(cudaStreamSynchronize(h->stream));
#undef CREATE_TRY
  *out = h;
  return DCSIM_OK;
}

int dcsim_reset(dcsim_t* h, uint64_t base_seed, uint64_t first_replica_id) {
  if (!h) return DCSIM_E_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  /* hdr.initialized == 0 marks a fresh replica; the FIFOs need no clearing (head == tail == 0) */
  CUDA_TRY(h, cudaMemsetAsync(h->d_state, 0, (size_t)h->n_replicas * (size_t)h->L.total_bytes, h->stream));
  CUDA_TRY(h, cudaMemsetAsync(h->d_counts, 0, 4 * sizeof(uint32_t), h->stream));
  if (h->d_hist) CUDA_TRY(h, cudaMemsetAsync(h->d_hist, 0, (size_t)h->n_replicas * 2 * DCSIM_LAT_BINS * sizeof(uint32_t), h->stream));
  h->seed0 = base_seed + first_replica_id;
  h->arrivals_ready = 0;
  h->launches = 0; /* a reset batch is "fresh": recorders may be re-targeted before its first advance */
  return DCSIM_OK;
}

int dcsim_set_stream(dcsim_t* h, void* cuda_stream) {
  if (!h) return DCSIM_E_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->stream = cuda_stream ? (cudaStream_t)cuda_stream : h->own_stream;
  return DCSIM_OK;
}

int dcsim_set_trace(dcsim_t* h, uint64_t replica, uint32_t capacity) {
  if (!h) return DCSIM_E_INVALID;
  if (h->launches) return set_err(h, DCSIM_E_STATE, "set_trace must precede the first advance%s%lld");
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (h->d_trace) { cudaFree(h->d_trace); h->d_trace = NULL; }
  h->trace_cap = 0; h->trace_replica = -1;
  if (capacity == 0) return DCSIM_OK;
  if (replica >= h->n_replicas) return set_err(h, DCSIM_E_INVALID, "set_trace: replica out of range%s%lld");
  CUDA_TRY(h, cudaMalloc(&h->d_trace, (size_t)capacity * sizeof(dcsim_trace_rec_t)));
  h->trace_cap = capacity; h->trace_replica = (int64_t)replica;
  return DCSIM_OK;
}

int dcsim_set_logging(dcsim_t* h, uint64_t replica, uint32_t job_capacity, uint32_t cluster_capacity) {
  if (!h) return DCSIM_E_INVALID;
  if (h->launches) return set_err(h, DCSIM_E_STATE, "set_logging must precede the first advance%s%lld");
  CUDA_TRY(h, cudaSetDevice(h->device));
  h->jobs_cap = h->cluster_cap = 0; h->log_replica = -1;
  h->want_job_log = 0; /* the state block is re-laid out (if at all) by the batch's first launch: a caller that
                          switches logging off and on again between batches pays for neither */
  if (replica >= h->n_replicas && (job_capacity || cluster_capacity))
    return set_err(h, DCSIM_E_INVALID, "set_logging: replica out of range%s%lld");
  if (job_capacity == 0 && cluster_capacity == 0) return DCSIM_OK;
  if (job_capacity > h->jobs_alloc) { /* buffers only ever grow; a smaller request reuses them */
    if (h->d_jobs) { cudaFree(h->d_jobs); h->d_jobs = NULL; h->jobs_alloc = 0; }
    CUDA_TRY(h, cudaMalloc(&h->d_jobs, (size_t)job_capacity * sizeof(dcsim_job_rec_t)));
    h->jobs_alloc = job_capacity;
  }
  if (cluster_capacity > h->cluster_alloc) {
    if (h->d_cluster) { cudaFree(h->d_cluster); h->d_cluster = NULL; h->cluster_alloc = 0; }
    CUDA_TRY(h, cudaMalloc(&h->d_cluster, (size_t)cluster_capacity * sizeof(dcsim_cluster_rec_t)));
    h->cluster_alloc = cluster_capacity;
  }
  h->jobs_cap = job_capacity; h->cluster_cap = cluster_capacity; h->log_replica = (int64_t)replica;
  h->want_job_log = job_capacity != 0;
  return DCSIM_OK;
}

static void fill_kparams(const dcsim_t* h, dcsim_kparams_t* P, uint64_t max_events) {
  memset(P, 0, sizeof(*P));
  P->spec = h->spec;
  P->L = h->L;
  P->rec.trace = h->d_trace; P->rec.jobs = h->jobs_cap ? h->d_jobs : NULL; P->rec.cluster = h->cluster_cap ? h->d_cluster : NULL; P->rec.counts = h->d_counts;
  P->rec.trace_cap = h->trace_cap; P->rec.jobs_cap = h->jobs_cap; P->rec.cluster_cap = h->cluster_cap;
  P->rec.trace_replica = h->trace_replica; P->rec.log_replica = h->log_replica;
  P->n_replicas = h->n_replicas;
  P->seed0 = h->seed0;
  P->max_events = max_events;
  P->budget32 = (max_events == 0ull || max_events > 0xfffffffeull) ? 0xffffffffu : (uint32_t)max_events;
  P->state = h->d_state; P->queues = h->d_queues; P->summary = h->d_summary;
  P->end_eps = h->spec.end_time + 1e-9; /* SIM:161 */
  P->arr_t = h->d_arr_t; P->arr_raw = h->d_arr_raw; P->arr_meta = h->d_arr_meta; P->arr_pred = h->d_arr_pred;
  P->arr_tx = h->d_arr_tx; P->arr_fin = h->d_arr_fin;
  P->ml_t = h->d_ml_t; P->ml_aux = h->d_ml_aux; P->ml_meta = h->d_ml_meta;
  P->arr_hdr = h->d_arr_hdr; P->cap_arr = h->cap_arr;
  P->max_transfer = h->max_transfer;
#ifdef DCSIM_DEVICE_TEST_HOOKS
  /* a rounded-up xfer_done instant may lie up to one quantum past t + transfer_s: the merge window must reach that far */
  P->test_time_quantum = g_test_time_quantum;
  P->max_transfer += g_test_time_quantum;
#endif
  P->lat_hist = h->d_hist;
  P->mt_state = h->d_mt;
}

int dcsim_prepare(dcsim_t* h) {
  if (!h) return DCSIM_E_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (h->launches == 0) { const int rc0 = relayout(h, h->want_job_log); if (rc0 != DCSIM_OK) return rc0; }
  if (h->arrivals_ready) return DCSIM_OK;
  dcsim_kparams_t P;
  fill_kparams(h, &P, 0);
  const int nb = (int)((h->n_replicas + DCSIM_ARRIVALS_THREADS - 1) / DCSIM_ARRIVALS_THREADS);
  const size_t scratch = dcsim_arrivals_scratch_bytes(h->spec.n_ing);
  if (h->rng_kind == DCSIM_RNG_MT19937) dcsim_arrivals_kernel<true><<<nb, DCSIM_ARRIVALS_THREADS, scratch, h->stream>>>(P);
  else dcsim_arrivals_kernel<false><<<nb, DCSIM_ARRIVALS_THREADS, scratch, h->stream>>>(P);
  CUDA_TRY(h, cudaGetLastError());
  const int wpb = DCSIM_MERGE_THREADS / 32;
  dcsim_merge_kernel<<<(int)((h->n_replicas + wpb - 1) / wpb), DCSIM_MERGE_THREADS, 0, h->stream>>>(P);
  CUDA_TRY(h, cudaGetLastError());
  h->arrivals_ready = 1;
  h->launches += 2;
  return DCSIM_OK;
}

int dcsim_advance(dcsim_t* h, uint64_t max_events_per_replica, uint64_t* total_events_out) {
  if (!h) return DCSIM_E_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (h->launches == 0) { const int rc0 = relayout(h, h->want_job_log); if (rc0 != DCSIM_OK) return rc0; }
  int rc = dcsim_prepare(h); /* once per (re)seeded batch: the arrival lists of all replicas */
  if (rc != DCSIM_OK) return rc;
  dcsim_kparams_t P;
  fill_kparams(h, &P, max_events_per_replica);
  CUDA_TRY(h, adv_launch_for(h->lanes)(&P, h->d_events, h->L.cap_stale != 0, h->mode, h->ctas, h->warps_per_cta * 32, h->smem_bytes, h->stream));
  h->launches++;
  if (total_events_out) {
    unsigned long long total = 0;
    CUDA_TRY(h, cudaMemcpyAsync(&total, h->d_events, sizeof(total), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    *total_events_out = (uint64_t)(total - h->events_seen);
    h->events_seen = total;
  }
  return DCSIM_OK;
}

int dcsim_fetch_summary(dcsim_t* h, double* out, size_t out_bytes) {
  if (!h || !out) return DCSIM_E_INVALID;
  const size_t need = (size_t)h->n_replicas * DCSIM_SUMMARY_K * sizeof(double);
  if (out_bytes < need) return set_err(h, DCSIM_E_INVALID, "fetch_summary: buffer too small (need %s%lld bytes)", "", (long long)need);
  if (!h->launches) return set_err(h, DCSIM_E_STATE, "fetch_summary before the first advance%s%lld");
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaMemcpyAsync(out, h->d_summary, need, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return DCSIM_OK;
}

int dcsim_fetch_summary_host(dcsim_t* h, const double** host_ptr_out) {
  if (!h || !host_ptr_out) return DCSIM_E_INVALID;
  *host_ptr_out = NULL;
  if (!h->launches) return set_err(h, DCSIM_E_STATE, "fetch_summary_host before the first advance%s%lld");
  CUDA_TRY(h, cudaSetDevice(h->device));
  const size_t need = (size_t)h->n_replicas * DCSIM_SUMMARY_K * sizeof(double);
  if (!h->h_summary_pinned) CUDA_TRY(h, cudaHostAlloc(&h->h_summary_pinned, need, cudaHostAllocDefault));
  CUDA_TRY(h, cudaMemcpyAsync(h->h_summary_pinned, h->d_summary, need, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  *host_ptr_out = h->h_summary_pinned;
  return DCSIM_OK;
}

int dcsim_summary_device_ptr(dcsim_t* h, void** dev_ptr_out) {
  if (!h || !dev_ptr_out) return DCSIM_E_INVALID;
  *dev_ptr_out = h->d_summary;
  return DCSIM_OK;
}

int dcsim_all_done(dcsim_t* h, int* done_out) {
  if (!h || !done_out) return DCSIM_E_INVALID;
  *done_out = 0;
  if (!h->launches) return DCSIM_OK;
  CUDA_TRY(h, cudaSetDevice(h->device));
  double* agg = h->d_agg; /* allocated once per handle: the chunked-resume loop calls this after every chunk */
  int rc = dcsim_reduce_summary(h, agg);
  double host[DCSIM_AGG_K];
  if (rc == DCSIM_OK) {
    cudaError_t e = cudaMemcpyAsync(host, agg, sizeof(host), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    if (e != cudaSuccess) rc = set_err(h, DCSIM_E_CUDA, "CUDA error: %s%lld", cudaGetErrorString(e));
  }
  if (rc != DCSIM_OK) return rc;
  /* a replica that stopped on a capacity overflow never finishes, so "done" = nothing is still running */
  *done_out = host[DCSIM_A_RUNNING] == 0.0;
  return DCSIM_OK;
}

int dcsim_reduce_summary(dcsim_t* h, double* dev_out) {
  if (!h || !dev_out) return DCSIM_E_INVALID;
  if (!h->launches) return set_err(h, DCSIM_E_STATE, "reduce_summary before the first advance%s%lld");
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, cudaMemsetAsync(dev_out, 0, DCSIM_AGG_K * sizeof(double), h->stream));
  int blocks = (int)((h->n_replicas + 255) / 256);
  if (blocks > 4 * h->sm_count) blocks = 4 * h->sm_count;
  dcsim_reduce_kernel<<<blocks, 256, 0, h->stream>>>(h->d_summary, h->n_replicas, dev_out);
  CUDA_TRY(h, cudaGetLastError());
  return DCSIM_OK;
}

/* The run's only collective for callers that own an NCCL communicator (C / C++ hosts; Python callers use
 * dcsim_reduce_summary + torch.distributed).  NCCL is resolved at run time from whatever the process has loaded (or
 * libnccl.so.2), so the library carries no link-time dependency on a particular NCCL build. */
typedef int (*dcsim_nccl_allreduce_fn)(const void*, void*, size_t, int /*ncclDataType_t*/, int /*ncclRedOp_t*/, void* /*ncclComm_t*/, cudaStream_t);
int dcsim_allreduce_summary(dcsim_t* h, void* nccl_comm, double* out) {
  if (!h || !out) return DCSIM_E_INVALID;
  if (!nccl_comm) return set_err(h, DCSIM_E_INVALID, "allreduce_summary: nccl_comm is NULL%s%lld");
  static dcsim_nccl_allreduce_fn fn = NULL;
  if (!fn) {
    void* sym = dlsym(RTLD_DEFAULT, "ncclAllReduce");
    if (!sym) {
      void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
      if (lib) sym = dlsym(lib, "ncclAllReduce");
    }
    if (!sym) return set_err(h, DCSIM_E_UNSUPPORTED, "allreduce_summary: no NCCL in this process (ncclAllReduce not found)%s%lld");
    fn = (dcsim_nccl_allreduce_fn)sym;
  }
  int rc = dcsim_reduce_summary(h, h->d_agg);
  if (rc != DCSIM_OK) return rc;
  const int nccl_rc = fn(h->d_agg, h->d_agg, DCSIM_AGG_K, /*ncclFloat64*/ 8, /*ncclSum*/ 0, nccl_comm, h->stream);
  if (nccl_rc != 0) return set_err(h, DCSIM_E_CUDA, "allreduce_summary: ncclAllReduce failed with code %s%lld", "", (long long)nccl_rc);
  CUDA_TRY(h, cudaMemcpyAsync(out, h->d_agg, DCSIM_AGG_K * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return DCSIM_OK;
}

int dcsim_set_rng(dcsim_t* h, int rng_kind) {
  if (!h) return DCSIM_E_INVALID;
  if (rng_kind != DCSIM_RNG_PHILOX && rng_kind != DCSIM_RNG_MT19937) return set_err(h, DCSIM_E_INVALID, "set_rng: unknown rng kind %s%lld", "", (long long)rng_kind);
  if (h->launches) return set_err(h, DCSIM_E_STATE, "set_rng must precede the first advance%s%lld");
  CUDA_TRY(h, cudaSetDevice(h->device));
  if (rng_kind == DCSIM_RNG_MT19937 && !h->d_mt)
    CUDA_TRY(h, cudaMalloc(&h->d_mt, (size_t)h->n_replicas * DCSIM_MT_N * sizeof(uint32_t)));
  h->rng_kind = rng_kind;
  return DCSIM_OK;
}

int dcsim_enable_latency_histogram(dcsim_t* h) {
  if (!h) return DCSIM_E_INVALID;
  if (h->d_hist) return DCSIM_OK;
  if (h->launches) return set_err(h, DCSIM_E_STATE, "enable_latency_histogram must precede the first advance%s%lld");
  CUDA_TRY(h, cudaSetDevice(h->device));
  const size_t bytes = (size_t)h->n_replicas * 2 * DCSIM_LAT_BINS * sizeof(uint32_t);
  CUDA_TRY(h, cudaMalloc(&h->d_hist, bytes));
  CUDA_TRY(h, cudaMemsetAsync(h->d_hist, 0, bytes, h->stream));
  return DCSIM_OK;
}

int dcsim_fetch_latency_histogram(dcsim_t* h, uint64_t* out, size_t out_bytes) {
  if (!h || !out) return DCSIM_E_INVALID;
  if (!h->d_hist) return set_err(h, DCSIM_E_STATE, "latency histogram not enabled (dcsim_enable_latency_histogram)%s%lld");
  const size_t need = 2 * DCSIM_LAT_BINS * sizeof(uint64_t);
  if (out_bytes < need) return set_err(h, DCSIM_E_INVALID, "fetch_latency_histogram: buffer too small (need %s%lld bytes)", "", (long long)need);
  if (!h->launches) return set_err(h, DCSIM_E_STATE, "fetch_latency_histogram before the first advance%s%lld");
  CUDA_TRY(h, cudaSetDevice(h->device));
  unsigned long long* d_out = h->d_hist_out;
  cudaError_t e = cudaMemsetAsync(d_out, 0, need, h->stream);
  if (e == cudaSuccess) {
    int blocks = 8 * h->sm_count;
    if ((uint64_t)blocks > h->n_replicas) blocks = (int)h->n_replicas;
    dcsim_hist_reduce_kernel<<<blocks, 2 * DCSIM_LAT_BINS, 0, h->stream>>>(h->d_hist, h->n_replicas, d_out);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, need, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return set_err(h, DCSIM_E_CUDA, "CUDA error: %s%lld", cudaGetErrorString(e));
  return DCSIM_OK;
}

int dcsim_recorder_counts(dcsim_t* h, uint32_t* out3) {
  if (!h || !out3) return DCSIM_E_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  uint32_t counts[4];
  CUDA_TRY(h, cudaMemcpyAsync(counts, h->d_counts, sizeof(counts), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  out3[0] = counts[0]; out3[1] = counts[1]; out3[2] = counts[2];
  return DCSIM_OK;
}

static int fetch_records(dcsim_t* h, const void* dev, size_t rec_bytes, uint32_t dev_cap, int which, void* out,
                         uint32_t capacity, uint32_t* n_out) {
  if (!h || !n_out) return DCSIM_E_INVALID;
  *n_out = 0;
  if (!dev) return DCSIM_OK;
  CUDA_TRY(h, cudaSetDevice(h->device));
  uint32_t counts[4];
  CUDA_TRY(h, cudaMemcpyAsync(counts, h->d_counts, sizeof(counts), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  uint32_t n = counts[which] < dev_cap ? counts[which] : dev_cap;
  if (n > capacity) n = capacity;
  if (n && out) {
    CUDA_TRY(h, cudaMemcpyAsync(out, dev, (size_t)n * rec_bytes, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  }
  *n_out = n;
  return DCSIM_OK;
}

int dcsim_fetch_trace(dcsim_t* h, dcsim_trace_rec_t* out, uint32_t capacity, uint32_t* n_out) {
  return fetch_records(h, h ? h->d_trace : NULL, sizeof(dcsim_trace_rec_t), h ? h->trace_cap : 0, 0, out, capacity, n_out);
}
int dcsim_fetch_job_log(dcsim_t* h, dcsim_job_rec_t* out, uint32_t capacity, uint32_t* n_out) {
  return fetch_records(h, h && h->jobs_cap ? h->d_jobs : NULL, sizeof(dcsim_job_rec_t), h ? h->jobs_cap : 0, 1, out, capacity, n_out);
}
int dcsim_fetch_cluster_log(dcsim_t* h, dcsim_cluster_rec_t* out, uint32_t capacity, uint32_t* n_out) {
  return fetch_records(h, h && h->cluster_cap ? h->d_cluster : NULL, sizeof(dcsim_cluster_rec_t), h ? h->cluster_cap : 0, 2, out, capacity, n_out);
}

int dcsim_launch_info(dcsim_t* h, dcsim_launch_info_t* out) {
  if (!h || !out) return DCSIM_E_INVALID;
  memset(out, 0, sizeof(*out));
  out->warps_per_cta = h->warps_per_cta; out->ctas = h->ctas; out->smem_bytes_per_cta = h->smem_bytes;
  out->regs_per_thread = h->regs; out->resident_warps_per_sm = h->resident_warps; out->sm_count = h->sm_count;
  out->cap_xfer = (h->L.xring_mask + 1) / 2; out->cap_run = h->L.cap_run; out->cap_q_inf = h->L.cap_q[0]; out->cap_q_trn = h->L.cap_q[1];
  out->kernel_launches = h->launches;
  out->hbm_bytes_state = (uint64_t)h->n_replicas * (uint64_t)h->L.total_bytes;
  out->hbm_bytes_queues = (uint64_t)h->n_replicas * h->L.queue_bytes;
  out->arrivals_prepass = 1;
  /* per arrival: pre-pass output 24 B + merge scratch 12 B + two list entries of 20 B */
  out->hbm_bytes_arrivals = (uint64_t)h->n_replicas * ((uint64_t)h->cap_arr * 76ull + sizeof(dcsim_arrhdr_t));
  out->staging_mode = h->mode; out->state_block_bytes = h->L.total_bytes;
  out->staged_bytes_per_replica = h->warps_per_cta ? h->smem_bytes / (h->warps_per_cta * (32 / h->lanes)) : 0;
  out->lanes_per_replica = h->lanes;
  return DCSIM_OK;
}

const char* dcsim_last_error(const dcsim_t* h) { return h ? h->err : g_create_err; }

#ifdef DCSIM_DEVICE_TEST_HOOKS
/* TEST-ONLY (builds made with -DDCSIM_DEVICE_TEST_HOOKS, never the product library): every launch from now on rounds
 * arrival and xfer_done instants up to a multiple of `q` (0 = off), like the oracle's and the host build's hook, so that
 * same-instant events are common on the device too. */
void dcsim_test_set_time_quantum(double q) { g_test_time_quantum = q; }
#endif

void dcsim_destroy(dcsim_t* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->own_stream) { cudaStreamSynchronize(h->stream); }
  cudaFree(h->d_state); cudaFree(h->d_queues); cudaFree(h->d_summary); cudaFree(h->d_events); cudaFree(h->d_counts);
  cudaFree(h->d_trace); cudaFree(h->d_jobs); cudaFree(h->d_cluster);
  cudaFree(h->d_hist); cudaFree(h->d_agg); cudaFree(h->d_hist_out);
  if (h->h_summary_pinned) cudaFreeHost(h->h_summary_pinned);
  cudaFree(h->d_mt);
  cudaFree(h->d_arr_t); cudaFree(h->d_arr_raw); cudaFree(h->d_arr_meta); cudaFree(h->d_arr_pred); cudaFree(h->d_arr_tx);
  cudaFree(h->d_arr_fin); cudaFree(h->d_ml_t); cudaFree(h->d_ml_aux); cudaFree(h->d_ml_meta); cudaFree(h->d_arr_hdr);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

} /* extern "C" */
