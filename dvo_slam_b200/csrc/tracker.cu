// tracker.cu -- dvo::DenseTracker::match() (dvo_core/src/dense_tracking.cpp:131-376) for a batch of
// independent frame pairs, all state on the device.
//
// Per Gauss-Newton iteration the reference makes five passes over the points
// (computeResidualsSse, computeWeightsSse, computeScaleSse, computeCompleteDataLogLikelihood and the
// normal-equation loop, dense_tracking.cpp:271-343).  Precision P_k is a global reduction that the
// log-likelihood and J^T W J depend on, so there are exactly two data-parallel stages (stages.cuh):
//   stage A: warp/interpolate/residual/occlusion test, Student-t weight from P_{k-1}, pairwise scale sums
//   stage B: the same residuals again plus gradients, log-likelihood terms and the 21+6 normal-equation
//            coefficients with W = w*P_k
// each followed by a small per-pair step (pair_mid_warp: P_k; pair_end_cta: accept test, 6x6 LDL^T
// solve, SE(3) update, termination logic).  Both stages read their inputs from shared-memory tiles that a
// producer warp fills with bulk asynchronous copies (TMA unit) through an mbarrier pipeline; nothing but
// per-row / per-strip summaries is written.  A batch that fills the GPU runs ALL levels inside ONE persistent
// cooperative launch (k_level_persistent: a coarse segment with one CTA per pair, then slices of the fine levels
// with squads of g, 2g and 4g CTAs); small batches use one launch per level; the test hooks (residual image,
// linearize) run the same kernel for one pair and one iteration.  All sums above an image row are taken in an
// order fixed by the level's geometry, so every plan returns the same bits.
#include "common.cuh"
#include "stages.cuh"

#include <cstdio>
#include <cstring>
#include <limits>
#include <cmath>
#include <cstdlib>
#include <algorithm>

namespace dvo_b200 {

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kEndWarps = 4;   // warps that sum the level's strip partials in pair_end_cta

struct LevelLaunch {
  int w, h, n, pitch;
  int nbands, nstrips;
  int level_index;   // position in Result.Statistics.Levels
  int level_id;      // pyramid level
  int max_iterations;
  int first_level;   // 1 for the coarsest level of the match
  int use_initial_estimate;
  double precision, mu;
};

// ------------------------------------------------------------------------------------------------
// per-pair helpers
// ------------------------------------------------------------------------------------------------
__device__ void prepare_iteration(PairState& st, const PairLevel& pl) {
  // dense_tracking.cpp:259-263
  st.inc = se3_exp(st.x);
  st.initial_old = st.initial;
  st.initial = se3_mul(se3_inverse(st.inc), st.initial);
  st.estimate_old = st.estimate;
  st.estimate = se3_mul(st.inc, st.estimate);
  double T[16];
  se3_matrix(st.estimate, T);
  // KT = K * float(T)[0:3,:] in float, reference operation order (dense_tracking_impl.cpp:142-152)
  for (int j = 0; j < 4; ++j) {
    float t0 = (float)T[j], t1 = (float)T[4 + j], t2 = (float)T[8 + j];
    st.kt[j] = __fadd_rn(__fmul_rn(pl.cfx, t0), __fmul_rn(pl.cox, t2));
    st.kt[4 + j] = __fadd_rn(__fmul_rn(pl.cfy, t1), __fmul_rn(pl.coy, t2));
    st.kt[8 + j] = t2;
  }
}

__device__ void log_iteration(dvo_b200_iteration_stats* ilog, int max_log, int pair, PairState& st, int it_id, int level_id,
                              bool with_increment) {
  if (!ilog || st.iter_log_count >= max_log) { st.iter_log_count++; return; }
  dvo_b200_iteration_stats& e = ilog[(size_t)pair * max_log + st.iter_log_count++];
  e.level = level_id;
  e.id = it_id;
  e.valid_constraints = st.n;
  e.tdist_log_likelihood = st.nll_cur;
  for (int i = 0; i < 4; ++i) e.tdist_precision[i] = (double)st.precision[i];
  e.prior_log_likelihood = st.prior_cur;
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  for (int i = 0; i < 6; ++i) e.increment[i] = with_increment ? st.x[i] : nan;
  for (int i = 0; i < 36; ++i) e.information[i] = with_increment ? st.A_done[i] : nan;
}

// Start of a pyramid level for one pair (dense_tracking.cpp:137-150, 205-210, 238): run by one thread of the squad that
// owns the pair, before the level's first iteration.
__device__ void level_begin(PairState& st, const PairLevel& pl, const double* T_init, int pair, const LevelLaunch& lp) {
  if (lp.first_level) {
    // dense_tracking.cpp:137-150: first increment is the given guess
    st.inc = (lp.use_initial_estimate && T_init) ? se3_from_matrix(T_init + (size_t)pair * 16) : se3_identity();
    st.initial = st.inc; st.initial_old = st.inc;
    st.estimate = se3_identity(); st.estimate_old = se3_identity();
    st.num_levels = 0; st.num_iterations_total = 0; st.iter_log_count = 0;
  }
  // dense_tracking.cpp:205-210
  st.precision[0] = st.precision[1] = st.precision[2] = st.precision[3] = 0.f;
  st.iteration = 0;
  st.error = 1.7976931348623157e308;
  st.last_error = st.error;
  st.have_done = 0;
  st.termination = -1;
  st.level_active = 1;
  st.phase_ok = 0;
  LevelSummary& ls = st.levels[lp.level_index];
  ls.id = lp.level_id; ls.termination = -1;
  ls.max_valid_pixels = pl.max_valid_pixels;
  ls.valid_pixels = pl.rsel[0];
  ls.num_iterations = 0; ls.has_inc = 0; ls.last_n = 0; ls.last_inc_n = -1;
  ls.last_inc_nll = __longlong_as_double(0x7ff8000000000000LL);
  st.num_levels = lp.level_index + 1;
  se3_log(st.inc, st.x);  // dense_tracking.cpp:238
  prepare_iteration(st, pl);
}

// The pair descriptors of all levels and the initial estimates are written by the host into pinned memory; this kernel
// reads them over PCIe (unified addressing) into device memory, which keeps the upload off the H2D copy engine, where it
// would queue behind a bulk image upload of another context.
__global__ void k_stage_words(const uint4* __restrict__ src, uint4* __restrict__ dst, size_t n16) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n16) dst[i] = src[i];
}

// The enqueue-only alignment never waits for the level kernels, and the next launch zeroes a launch's error flag: the flag
// is folded right after each launch into a pinned word that the next synchronisation reads.
__global__ void k_fold_flag(const int* __restrict__ flag, int* __restrict__ accum) {
  const int v = *flag;
  if (v) *accum = v;
}

// one warp per pair: combine the strip summaries of the level in order -> covariance -> P_k (dense_tracking.cpp:276-295).
// e: the level's nstrips strip summaries; strip_base: nstrips + 1 exclusive prefixes of their valid counts (output).
__device__ __noinline__ void pair_mid_warp(PairState& st, int pair, const double* e, int* strip_base, int nstrips, int* active,
                                           const LevelLaunch& lp, dvo_b200_iteration_stats* ilog, int max_log, SegCombineSmem& sm) {
  const int lane = threadIdx.x & 31;
  const SegT<double> all = combine_strip_exports_warp(e, nstrips, strip_base, sm);
  if (lane == 0) {
    long long n = all.n;
    st.n = n;
    st.n_keep = (n / 50) * 50;
    LevelSummary& ls = st.levels[lp.level_index];
    ls.num_iterations += 1;   // level_stats.Iterations.push_back (dense_tracking.cpp:249)
    ls.last_n = n;
    st.num_iterations_total += 1;
    if (n < 6) {
      // dense_tracking.cpp:276-284
      st.initial = st.initial_old; st.estimate = st.estimate_old;
      st.termination = DVO_B200_TERM_TOO_FEW_CONSTRAINTS;
      st.phase_ok = 0;
      st.nll_cur = 0; st.prior_cur = 0;
      log_iteration(ilog, max_log, pair, st, st.iteration, lp.level_id, false);
      // post-loop checks of dense_tracking.cpp:359-363 still apply
      double m = 0; bool nanx = false;
      for (int i = 0; i < 6; ++i) { m = fmax(m, fabs(st.x[i])); nanx |= st.x[i] != st.x[i]; }
      if (!nanx && m <= lp.precision) st.termination = DVO_B200_TERM_INCREMENT_TOO_SMALL;
      if (st.iteration >= lp.max_iterations) st.termination = DVO_B200_TERM_ITERATIONS_EXCEEDED;
      ls.termination = st.termination;
      ls.has_inc = ls.num_iterations >= 2;   // HasIterationWithIncrement (dense_tracking_config.cpp:138-143)
      if (st.termination != DVO_B200_TERM_TOO_FEW_CONSTRAINTS) ls.has_inc = ls.num_iterations >= 1;
      st.have_done = (st.termination == DVO_B200_TERM_TOO_FEW_CONSTRAINTS) ? -1 : st.have_done;
      st.level_active = 0;
      if (active) atomicSub(active, 1);
    } else {
      // tail term for odd n, normaliser 1/(n-3) (dense_tracking_impl.cpp:596), symmetric 2x2
      double c[3];
      bool tail = ((n - 1) & 1) == 0;
      double s = 1.0 / (double)(n - 3);
      for (int k = 0; k < 3; ++k) c[k] = (all.S0[k] + (tail ? all.wl * all.ol[k] : 0.0)) * s;
      float C0 = (float)c[0], C1 = (float)c[1], C3 = (float)c[2];
      // precision = covariance.inverse() (Eigen 2x2 inverse, dense_tracking.cpp:295), float, unfused
      float det = __fsub_rn(__fmul_rn(C0, C3), __fmul_rn(C1, C1));
      float invdet = __fdiv_rn(1.0f, det);
      for (int i = 0; i < 4; ++i) st.precision_prev[i] = st.precision[i];
      st.precision[0] = __fmul_rn(C3, invdet);
      st.precision[1] = __fmul_rn(-C1, invdet);
      st.precision[2] = __fmul_rn(-C1, invdet);
      st.precision[3] = __fmul_rn(C0, invdet);
      st.phase_ok = 1;
    }
  }
  __syncwarp();
}

// End of an iteration (dense_tracking.cpp:297-363): add the level's strip partials, log-likelihood, accept test, solve,
// pose update, termination.  Every thread of the CTA calls; thread 0 does the scalar part in two steps:
//   critical : everything the other CTAs of the squad wait for -- the new K*T and iteration flag, or
//              level_active = 0 -- followed by `release` (the squad barrier of the persistent kernel);
//   deferred : Revertable bookkeeping, statistics, the iteration log.  It finishes before this CTA arrives at
//              the squad's next barrier, so the next P_k / end step (run by whichever CTA arrives last) sees it.
struct PairEndSmem {
  double part[kEndWarps][32];
};

template <typename Release>
__device__ __noinline__ void pair_end_cta(PairState& st, const PairLevel& pl, int pair, const double* partial, int ntiles,
                                             int* active, const LevelLaunch& lp, dvo_b200_iteration_stats* ilog, int max_log,
                                             PairEndSmem& sm, Release release, unsigned long long* tcrit = nullptr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned long long tc0 = 0;
  if (tcrit && threadIdx.x == 0) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(tc0));
  unsigned long long tph = tc0;
  // developer timing: ns per sub-phase of the end step into tcrit[k], the critical part into tcrit[7]
  auto phase = [&](int k) {
    if (tcrit) { unsigned long long tn; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(tn)); atomicAdd(tcrit + k, tn - tph); tph = tn; }
  };
  {   // fp64 sum of the level's strip partials in a fixed order: warp q takes strips q, q+4, ... with independent loads in flight
    double v = 0.0;
    if (lane < kNormalValues && warp < kEndWarps) {
      const double* p = partial + lane;
      int t = warp;
      for (; t + 3 * kEndWarps < ntiles; t += 4 * kEndWarps) {
        const double a0 = __ldcg(p + (size_t)t * kNormalValues);
        const double a1 = __ldcg(p + (size_t)(t + kEndWarps) * kNormalValues);
        const double a2 = __ldcg(p + (size_t)(t + 2 * kEndWarps) * kNormalValues);
        const double a3 = __ldcg(p + (size_t)(t + 3 * kEndWarps) * kNormalValues);
        v += a0; v += a1; v += a2; v += a3;
      }
      for (; t < ntiles; t += kEndWarps) v += __ldcg(p + (size_t)t * kNormalValues);
    }
    if (warp < kEndWarps) sm.part[warp][lane] = v;
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  double vals[kNormalValues];
#pragma unroll
  for (int i = 0; i < kNormalValues; ++i) {
    double v = sm.part[0][i];
#pragma unroll
    for (int q = 1; q < kEndWarps; ++q) v += sm.part[q][i];
    vals[i] = v;
  }
  phase(0);   // partial sums

  // ---- critical ----
  const float P0 = st.precision[0], P1 = st.precision[1], P2 = st.precision[2], P3 = st.precision[3];
  // computeCompleteDataLogLikelihood: 0.5 n log det P - 3.5 sum log(1 + 0.2 d), returned as float
  const float det = __fsub_rn(__fmul_rn(P0, P3), __fmul_rn(P1, P2));
  const float logdet = (float)log((double)det);
  const float ll = (float)(0.5 * (double)st.n * (double)logdet - 0.5 * (5.0 + 2.0) * vals[0]);
  double li[6] = {0, 0, 0, 0, 0, 0};
  double sq = 0;
  if (lp.mu != 0.0) {                              // mu == 0: prior term and the mu*log(initial) shift vanish
    se3_log(st.initial, li);
    for (int i = 0; i < 6; ++i) sq += li[i] * li[i];
  }
  phase(1);   // state loads, log, se3_log
  const double last_error = st.error;              // dense_tracking.cpp:306-307
  const double error = -(double)ll;
  const bool accept = error < last_error;          // dense_tracking.cpp:312
  double A[36], bvec[6], x[6];
  {
    int k = 1;
    for (int i = 0; i < 6; ++i)
      for (int j = i; j < 6; ++j) { A[i * 6 + j] = vals[k]; A[j * 6 + i] = vals[k]; ++k; }
    for (int i = 0; i < 6; ++i) bvec[i] = vals[22 + i];
  }
  int iteration = st.iteration;
  const int it_id = iteration;                     // IterationStats.Id = itctx_.Iteration before the increment (dense_tracking.cpp:251)
  if (accept) {
    double As[36], bs[6];
    for (int i = 0; i < 36; ++i) As[i] = A[i];
    for (int i = 0; i < 6; ++i) { As[i * 6 + i] += lp.mu; bs[i] = bvec[i] + lp.mu * li[i]; }   // lines 345-346
    ldlt_solve6(As, bs, x);                                                                    // line 347
    iteration += 1;                                                                            // line 353
  } else {
    for (int i = 0; i < 6; ++i) x[i] = st.x[i];
  }
  phase(2);   // accept test, LDL^T
  double m = 0; bool nanx = false;
  for (int i = 0; i < 6; ++i) { m = fmax(m, fabs(x[i])); nanx |= x[i] != x[i]; }
  const bool big = !nanx && m > lp.precision;
  const bool exceeded = iteration >= lp.max_iterations;
  const bool level_done = !(accept && big && !exceeded);                                       // line 357
  SE3d inc, estimate_new;
  if (!level_done) {
    // dense_tracking.cpp:259-263 for the next iteration: estimate = exp(x) * estimate, then K * float(T)
    inc = se3_exp(x);
    estimate_new = se3_mul(inc, st.estimate);
    double T[16];
    se3_matrix(estimate_new, T);
    for (int j = 0; j < 4; ++j) {   // reference operation order (dense_tracking_impl.cpp:142-152)
      const float t0 = (float)T[j], t1 = (float)T[4 + j], t2 = (float)T[8 + j];
      st.kt[j] = __fadd_rn(__fmul_rn(pl.cfx, t0), __fmul_rn(pl.cox, t2));
      st.kt[4 + j] = __fadd_rn(__fmul_rn(pl.cfy, t1), __fmul_rn(pl.coy, t2));
      st.kt[8 + j] = t2;
    }
    st.iteration = iteration;
  } else {
    st.level_active = 0;
  }
  phase(3);   // exp, pose product, K*T
  if (tcrit) { unsigned long long tc1; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(tc1)); atomicAdd(tcrit + 7, tc1 - tc0); }
  release();
  phase(4);   // release

  // ---- deferred ----
  LevelSummary& ls = st.levels[lp.level_index];
  st.ll = ll;
  st.nll_cur = -(double)ll;
  st.prior_cur = lp.mu * sq;                       // dense_tracking.cpp:302
  st.last_error = last_error;
  st.error = error;
  for (int i = 0; i < 36; ++i) st.A[i] = A[i];
  for (int i = 0; i < 6; ++i) st.b[i] = bvec[i];
  if (!accept) {
    st.initial = st.initial_old; st.estimate = st.estimate_old;   // dense_tracking.cpp:314-321
    st.termination = DVO_B200_TERM_LOG_LIKELIHOOD_DECREASED;
    log_iteration(ilog, max_log, pair, st, it_id, lp.level_id, false);
  } else {
    for (int i = 0; i < 6; ++i) st.x[i] = x[i];
    for (int i = 0; i < 36; ++i) st.A_done[i] = A[i];
    for (int i = 0; i < 6; ++i) st.A_done[i * 6 + i] += lp.mu;
    st.nll_done = st.nll_cur; st.prior_done = st.prior_cur; st.have_done = 1;
    ls.last_inc_n = st.n; ls.last_inc_nll = st.nll_cur;
    log_iteration(ilog, max_log, pair, st, it_id, lp.level_id, true);
    st.iteration = iteration;
  }
  if (level_done) {
    if (!nanx && m <= lp.precision) st.termination = DVO_B200_TERM_INCREMENT_TOO_SMALL;       // line 359
    if (exceeded) st.termination = DVO_B200_TERM_ITERATIONS_EXCEEDED;                         // line 362
    ls.termination = st.termination;
    int need = (st.termination == DVO_B200_TERM_LOG_LIKELIHOOD_DECREASED ||
                st.termination == DVO_B200_TERM_TOO_FEW_CONSTRAINTS) ? 2 : 1;
    ls.has_inc = ls.num_iterations >= need;
    if (active) atomicSub(active, 1);
  } else {
    st.inc = inc;
    st.initial_old = st.initial;
    st.initial = se3_mul(se3_inverse(inc), st.initial);
    st.estimate_old = st.estimate;
    st.estimate = estimate_new;
  }
  phase(5);   // deferred bookkeeping
}

// ------------------------------------------------------------------------------------------------
// The persistent cooperative level kernel.
//
// The grid is num_sms x C CTAs (C = resident CTAs per SM, 2 with ~93 KB of shared memory each) of 8 warps.  CTAs are
// grouped into squads of g CTAs; a squad owns ONE frame pair at a time, CTA r of the squad the strips r, r+g, r+2g, ...
// (kTileH image rows each), and runs all its Gauss-Newton iterations on the segment's levels inside the kernel:
//   stage A over the CTA's tiles -> per-row scale summaries -> per-strip summaries (fp64) -> squad barrier, the last
//   CTA to arrive combines the level's strips and computes P_k (pair_mid_warp) -> stage B -> per-row sums -> per-strip
//   sums (fp64) -> squad barrier, the last CTA adds the level's strips, tests the log-likelihood, solves the 6x6
//   system and updates the pose (pair_end_cta) -> next iteration,
// then takes the next pair from a global queue.  The two resident CTAs of an SM belong to different squads, so
// one squad's barrier wait is hidden by the other.
// ------------------------------------------------------------------------------------------------
struct SquadState {
  int pair;
  unsigned arrive;
  unsigned phase;
  int pad_[29];   // one 128-byte line per squad
};

struct LevelTail {      // shared memory after the tile pipeline
  SegCombineSmem comb;
  PairEndSmem end;
  int s_flag[2];
};
constexpr size_t kLevelSmemBytes = sizeof(TilePipe) + sizeof(LevelTail);

// One segment of a launch: a group of consecutive pyramid levels that a squad of g CTAs walks a pair through.  A launch
// has one segment, or two (the coarse levels with one CTA per pair, then the fine levels with squads of g CTAs) that the
// grid runs back to back WITHOUT a grid-wide barrier: a CTA that finds the coarse queue empty moves on to the fine
// segment, and fine squads take their pairs from a ring of pairs whose coarse levels are done (`ready`).
constexpr int kMaxSeg = 4;   // segments of one launch: the coarse levels, then up to three slices of the fine levels
struct Segment {
  const PairLevel* pls;   // descriptors of this segment's levels: [level][pair]
  float* row_exports;     // per squad: h segment summaries (one per image row)
  int* row_base;          // per squad: h exclusive prefixes of valid counts, relative to the owning CTA's first row
  double* strip_exports;  // per squad: one scale summary per strip (kStripExportDoubles)
  int* strip_base;        // per squad: nstrips + 1 exclusive prefixes of the strips' valid counts
  float* row_partial;     // per squad: kNormalValues per image row (stage B)
  double* strip_partial;  // per squad: kNormalValues per strip, the strip's rows summed in fp64
  SquadState* squads;
  int* queue;             // next pair (first segment) / next slot of this segment's ready ring (later segments of a fused launch)
  int* ready;             // fused launch, segments >= 1: ring of (pair + 1) whose coarse levels are done, 0 = not yet written
  int* ready_tail;
  int* arrivals;          // CTAs that have entered this segment (squads of segments >= 1 form in order of arrival)
  int cyclic;             // 1: CTA r of a squad takes strips r, r + g, ...; 0: contiguous ranges of strips_per_cta strips
  int pair_begin;         // segments >= 1 of a fused launch own the pairs [pair_begin, pair_begin + npairs_seg)
  int npairs_seg;         // pairs handed out by this segment's queue
  unsigned long long* dbg2;  // optional (timing build): {tiles, inexact tiles, skipped tiles, rounds, rounds of inexact tiles, max / min CTA lifetime}
  unsigned long long* dbg;   // optional: ns spent per CTA in {stage A, stage B, wait A, wait B, mid, end, queue, total}
  int nlev;               // pyramid levels of the segment (coarse to fine)
  int g, nsquads;
  int strips_per_cta[kMaxLevels];
  LevelLaunch lp[kMaxLevels];
};

struct PersistentArgs {
  PairState* states;
  int* error_flag;
  dvo_b200_iteration_stats* ilog;
  int max_log;
  const double* T_init;   // per pair 4x4 (device memory) or nullptr
  int skip_begin;         // test hook: the pair state was placed by k_set_state
  float* dump;            // test hook: seven record planes of the (single) pair, or nullptr
  int npairs;
  int nseg;               // 1, or >= 2 = fused launch: coarse segment + slices of the fine levels
  Segment seg[kMaxSeg];
};

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// returns true in every thread of the CTA that arrived last at barrier episode `episode`
__device__ __forceinline__ bool squad_arrive(SquadState* sq, unsigned episode, int g, int* s_flag) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned old = atomicAdd(&sq->arrive, 1u);
    int last = old == (episode + 1u) * (unsigned)g - 1u;
    if (last) __threadfence();
    s_flag[0] = last;
  }
  __syncthreads();
  return s_flag[0] != 0;
}
__device__ __forceinline__ void squad_release(SquadState* sq, unsigned episode) {
  __threadfence();
  atomicExch(&sq->phase, episode + 1u);
}
__device__ __forceinline__ void squad_wait(SquadState* sq, unsigned episode, int* error_flag) {
  if (threadIdx.x == 0) {
    unsigned spins = 0;
    while (ld_acquire_u32(&sq->phase) < episode + 1u) {
      __nanosleep(100);
      if (((++spins) & 4095u) == 0u) {
        if (*reinterpret_cast<volatile int*>(error_flag)) break;
        if (spins > (1u << 25)) { atomicExch(error_flag, 1); break; }   // ~ seconds: never hang the GPU
      }
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kCtaThreads, 2)
k_level_persistent(const __grid_constant__ PersistentArgs a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  TilePipe& tp = *reinterpret_cast<TilePipe*>(smem_raw);
  LevelTail& lt = *reinterpret_cast<LevelTail*>(smem_raw + sizeof(TilePipe));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&tp.full[i], 1); mbar_init(&tp.empty[i], kConsumerWarps); }
    mbar_fence_init();
  }
  __syncthreads();
  unsigned tile_count = 0;      // tiles staged / consumed by this CTA since the kernel started
  const bool fused = a.nseg >= 2;
#define DVO_TICK() do { if (timing) t0 = global_ns(); } while (0)
#define DVO_TOCK(slot) do { if (timing) { t1 = global_ns(); t_acc[slot] += t1 - t0; t0 = t1; } } while (0)

#pragma unroll 1
  for (int si = 0; si < a.nseg; ++si) {
  const Segment& S = a.seg[si];
  // Squads of the second segment of a fused launch form in ORDER OF ARRIVAL: the CTAs leave the first segment at very
  // different times (1 or 2 coarse pairs each, 3..40 iterations per level), and a squad made of neighbouring block indices
  // would wait for its slowest member (measured: 24 % of the fine segment's CTA time).
  int cta_index = blockIdx.x;
  if (fused && si >= 1) {
    if (threadIdx.x == 0) lt.s_flag[1] = atomicAdd(S.arrivals, 1);
    __syncthreads();
    cta_index = lt.s_flag[1];
    __syncthreads();
  }
  const int squad = cta_index / S.g, rank = cta_index - squad * S.g;
  if (squad >= S.nsquads) continue;   // leftover CTAs of this segment
  SquadState* sq = S.squads + squad;
  int hmax = 0;
  for (int li = 0; li < S.nlev; ++li) hmax = max(hmax, S.lp[li].h);
  float* row_exports = S.row_exports + (size_t)squad * hmax * kSegExportFloats;
  int* row_base = S.row_base + (size_t)squad * hmax;
  const int smax = (hmax + kTileH - 1) / kTileH;      // strips of the tallest level of the segment
  double* strip_exports = S.strip_exports + (size_t)squad * smax * kStripExportDoubles;
  int* strip_base = S.strip_base + (size_t)squad * (smax + 1);
  float* row_partial = S.row_partial + (size_t)squad * hmax * kNormalValues;
  double* strip_partial = S.strip_partial + (size_t)squad * smax * kNormalValues;
  unsigned episode = 0;
  unsigned long long t_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, t0 = 0, t1 = 0;
  const bool timing = S.dbg != nullptr && threadIdx.x == 0;
  PipeTiming tm;
#ifdef DVO_PIPE_TIMING
  tm.on = S.dbg != nullptr && lane == 0 && (warp == 0 || warp == kConsumerWarps);   // one consumer warp and the producer
#endif
  const unsigned long long t_start = timing ? global_ns() : 0;

  for (;;) {
    DVO_TICK();
    // ---- take the next pair from the queue (the last CTA to arrive does it for the squad) ----
    if (squad_arrive(sq, episode, S.g, lt.s_flag)) {
      if (threadIdx.x == 0) {
        int p = atomicAdd(S.queue, 1);
        if (p >= S.npairs_seg) p = -1;
        else if (fused && si >= 1) {
          // slot p of this segment's ready ring: filled by the CTA that finishes the coarse levels of one of the
          // segment's pairs (every pair is pushed exactly once, so every slot < npairs_seg is eventually written)
          unsigned spins = 0;
          int v;
          while ((v = (int)ld_acquire_u32(reinterpret_cast<const unsigned*>(S.ready + p))) == 0) {
            __nanosleep(200);
            if (((++spins) & 4095u) == 0u) {
              if (*reinterpret_cast<volatile int*>(a.error_flag)) break;
              if (spins > (1u << 24)) { atomicExch(a.error_flag, 1); break; }
            }
          }
          p = v - 1;
        }
        sq->pair = p;
        squad_release(sq, episode);
      }
    } else {
      squad_wait(sq, episode, a.error_flag);
    }
    __syncthreads();
    ++episode;
    DVO_TOCK(6);
    const int pair = __ldcg(&sq->pair);
    if (pair < 0 || *reinterpret_cast<volatile int*>(a.error_flag)) break;
    PairState& st = a.states[pair];

    // ---- the squad walks its pair through the levels of this launch, coarse to fine ----
    for (int li = 0; li < S.nlev; ++li) {
    const LevelLaunch& lp = S.lp[li];
    const PairLevel pl = S.pls[(size_t)li * a.npairs + pair];
    LevelGeom geo;
    geo.w = lp.w; geo.h = lp.h; geo.n = lp.n; geo.pitch = lp.pitch; geo.nbands = lp.nbands; geo.nstrips = lp.nstrips;
    if (S.cyclic) {   // CTA r takes strips r, r + g, r + 2g, ...: every CTA of the squad samples the whole image
      const int g_eff = min(S.g, lp.nstrips);
      geo.strip0 = min(rank, lp.nstrips); geo.strip_step = g_eff;
      geo.nmine = rank < g_eff ? (lp.nstrips - rank + g_eff - 1) / g_eff : 0;
    } else {          // contiguous ranges
      geo.strip0 = min(rank * S.strips_per_cta[li], lp.nstrips); geo.strip_step = 1;
      geo.nmine = min(geo.strip0 + S.strips_per_cta[li], lp.nstrips) - geo.strip0;
    }
    if (!a.skip_begin) {   // DenseTracker::match, start of a level: the last CTA to arrive initialises the pair's level state
      if (squad_arrive(sq, episode, S.g, lt.s_flag)) {
        if (threadIdx.x == 0) {
          level_begin(st, pl, a.T_init, pair, lp);
          squad_release(sq, episode);
        }
      } else {
        squad_wait(sq, episode, a.error_flag);
      }
      __syncthreads();
      ++episode;
      DVO_TOCK(6);
    }

    for (;;) {
      // ---- stage A ----
      {
        StageConsts c;
        load_stage_consts(st, pl, lp.w, lp.h, false, c);
        const long long ts0 = DVO_CLOCK(tm);
        stage_a_run(tp, pl, geo, c, row_exports, tile_count, a.error_flag, tm);
        DVO_ADD(tm, rounds_a, DVO_CLOCK(tm) - ts0);
      }
      __syncthreads();
      // this CTA's strips: the rows of a strip in order -> the strip's summary (one thread per strip); row_base: rank of each
      // row's first point inside its strip
      for (int j = threadIdx.x; j < geo.nmine; j += kCtaThreads) {
        const int sj = geo.strip0 + j * geo.strip_step;
        combine_strip_rows(row_exports, sj * kTileH, min(sj * kTileH + kTileH, lp.h), row_base, strip_exports + (size_t)sj * kStripExportDoubles);
      }
      DVO_TOCK(0);
      if (squad_arrive(sq, episode, S.g, lt.s_flag)) {
        DVO_TOCK(2);
        if (warp == 0) {
          pair_mid_warp(st, pair, strip_exports, strip_base, lp.nstrips, nullptr, lp, a.ilog, a.max_log, lt.comb);
          if (lane == 0) squad_release(sq, episode);
        }
        __syncthreads();
        DVO_TOCK(4);
      } else {
        squad_wait(sq, episode, a.error_flag);
        DVO_TOCK(2);
      }
      __syncthreads();
      ++episode;
      if (!__ldcg(&st.level_active) || *reinterpret_cast<volatile int*>(a.error_flag)) break;   // too few constraints

      // ---- stage B ----
      {
        StageConsts c;
        load_stage_consts(st, pl, lp.w, lp.h, true, c);
        StageBConsts cb;
        load_stage_b_consts(st, cb);
        const long long n_keep = __ldcg(&st.n_keep);
        RecordDump dump;
        dump.planes = a.dump; dump.n = lp.n;
        const long long ts0 = DVO_CLOCK(tm);
        if (a.dump) stage_b_run<true>(tp, pl, geo, c, cb, row_base, strip_base, n_keep, dump, row_partial, tile_count, a.error_flag, tm);
        else stage_b_run<false>(tp, pl, geo, c, cb, row_base, strip_base, n_keep, dump, row_partial, tile_count, a.error_flag, tm);
        DVO_ADD(tm, rounds_b, DVO_CLOCK(tm) - ts0);
      }
      __syncthreads();
      // the rows of each of this CTA's strips, in order, in fp64: one thread per (strip, value)
      for (int it = threadIdx.x; it < geo.nmine * kNormalValues; it += kCtaThreads) {
        const int j = it / kNormalValues, i = it - j * kNormalValues;
        const int sj = geo.strip0 + j * geo.strip_step;
        const int nrow = min(kTileH, lp.h - sj * kTileH);
        const float* rp = row_partial + (size_t)sj * kTileH * kNormalValues + i;
        float r[kTileH];
#pragma unroll
        for (int k = 0; k < kTileH; ++k) r[k] = k < nrow ? __ldcg(rp + (size_t)k * kNormalValues) : 0.f;   // independent loads
        double v = 0.0;
#pragma unroll
        for (int k = 0; k < kTileH; ++k) v += (double)r[k];      // a missing row adds an exact zero
        strip_partial[(size_t)sj * kNormalValues + i] = v;
      }
      DVO_TOCK(1);
      if (squad_arrive(sq, episode, S.g, lt.s_flag)) {
        DVO_TOCK(3);
        pair_end_cta(st, pl, pair, strip_partial, lp.nstrips, nullptr, lp, a.ilog, a.max_log, lt.end, [&] { squad_release(sq, episode); }, S.dbg2 ? S.dbg2 + 64 : nullptr);
        __syncthreads();
        DVO_TOCK(5);
      } else {
        squad_wait(sq, episode, a.error_flag);
        DVO_TOCK(3);
      }
      __syncthreads();
      ++episode;
      if (!__ldcg(&st.level_active) || *reinterpret_cast<volatile int*>(a.error_flag)) break;
    }
    if (*reinterpret_cast<volatile int*>(a.error_flag)) break;
    }   // levels
    if (fused && si == 0 && threadIdx.x == 0) {   // this pair's coarse levels are done: hand it to the fine squads (g == 1 here)
      // The fine segments own fixed ranges of the pair index (not of the order of arrival), so which squad size a pair
      // gets -- and with it the rounding of its sums -- does not depend on timing.
      int k = 1;
      while (k + 1 < a.nseg && pair >= a.seg[k + 1].pair_begin) ++k;
      __threadfence();
      const int slot = atomicAdd(a.seg[k].ready_tail, 1);
      asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(a.seg[k].ready + slot), "r"(pair + 1) : "memory");
    }
  }
  if (timing) {
    t_acc[7] = global_ns() - t_start;
    for (int i = 0; i < 8; ++i) atomicAdd(S.dbg + i, t_acc[i]);
  }
#ifdef DVO_PIPE_TIMING
  if (tm.on) {   // cycles: consumer warp 0 {stage A, wait full A, stage B, wait full B}, producer {descriptor, wait empty}
    if (warp == 0) { atomicAdd(S.dbg + 8, tm.rounds_a); atomicAdd(S.dbg + 9, tm.wait_full_a); atomicAdd(S.dbg + 10, tm.rounds_b); atomicAdd(S.dbg + 11, tm.wait_full_b); }
    else { atomicAdd(S.dbg + 12, tm.produce); atomicAdd(S.dbg + 13, tm.wait_empty); atomicAdd(S.dbg + 14, tm.rounds_a); atomicAdd(S.dbg + 15, tm.rounds_b); }
    if (warp == 0) { atomicAdd(S.dbg2 + 3, tm.rounds); atomicAdd(S.dbg2 + 4, tm.slow_rounds); }
    else { atomicAdd(S.dbg2 + 0, tm.tiles); atomicAdd(S.dbg2 + 1, tm.tiles_inexact); atomicAdd(S.dbg2 + 2, tm.tiles_skipped); }
  }
  if (timing) { atomicMax(S.dbg2 + 5, t_acc[7]); atomicMin(S.dbg2 + 6, t_acc[7]); }
#endif
  }   // segments
#undef DVO_TICK
#undef DVO_TOCK
}

// Result assembly (dense_tracking.cpp:368-373)
__global__ void k_finalize(PairState* states, dvo_b200_result* results, int npairs) {
  int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= npairs) return;
  PairState& st = states[p];
  dvo_b200_result& r = results[p];
  const double nan = __longlong_as_double(0x7ff8000000000000LL);
  se3_matrix(se3_inverse(st.estimate), r.transformation);
  // last_iteration = Iterations[size-1] unless LogLikelihoodDecreased (then size-2).  With
  // TooFewConstraints on the last level, or no completed iteration, the reference reads an
  // uninitialised / out-of-range element (SURVEY Q24); defined here as NaN so Result::isNaN() fires.
  bool ok = st.have_done == 1 && st.termination != DVO_B200_TERM_TOO_FEW_CONSTRAINTS;
  for (int i = 0; i < 36; ++i) r.information[i] = ok ? st.A_done[i] * 0.008 * 0.008 : nan;
  r.log_likelihood = ok ? st.nll_done + st.prior_done : nan;
  r.num_levels = st.num_levels;
  r.num_iterations_total = st.num_iterations_total;
  for (int l = 0; l < kMaxLevels; ++l) {
    dvo_b200_level_stats& o = r.levels[l];
    if (l < st.num_levels) {
      const LevelSummary& s = st.levels[l];
      o.id = s.id; o.termination = s.termination; o.max_valid_pixels = s.max_valid_pixels;
      o.valid_pixels = s.valid_pixels; o.num_iterations = s.num_iterations;
      o.has_iteration_with_increment = s.has_inc; o.last_valid_constraints = s.last_n;
      o.last_increment_valid_constraints = s.last_inc_n; o.last_increment_log_likelihood = s.last_inc_nll;
    } else {
      o.id = -1; o.termination = -1; o.max_valid_pixels = 0; o.valid_pixels = 0; o.num_iterations = 0;
      o.has_iteration_with_increment = 0; o.last_valid_constraints = 0; o.last_increment_valid_constraints = -1;
      o.last_increment_log_likelihood = nan;
    }
  }
}

// test hook: place a fixed transform / precision / iteration flag into the state (no exp/log chain)
__global__ void k_set_state(PairState* states, const PairLevel* pls, const double* T, const float* prev_precision,
                            int use_weights, LevelLaunch lp) {
  PairState& st = states[0];
  const PairLevel& pl = pls[0];
  st.estimate = se3_from_matrix(T); st.estimate_old = st.estimate;
  st.initial = se3_identity(); st.initial_old = st.initial; st.inc = se3_identity();
  for (int i = 0; i < 6; ++i) st.x[i] = 0;
  st.iteration = use_weights ? 1 : 0;
  for (int i = 0; i < 4; ++i) st.precision[i] = use_weights ? prev_precision[i] : 0.f;
  st.error = 1.7976931348623157e308; st.last_error = st.error;
  st.level_active = 1; st.phase_ok = 0; st.have_done = 0; st.termination = -1;
  st.num_levels = 1; st.num_iterations_total = 0; st.iter_log_count = 0;
  LevelSummary& ls = st.levels[0];
  ls.id = lp.level_id; ls.num_iterations = 0; ls.valid_pixels = pl.rsel[0]; ls.max_valid_pixels = pl.max_valid_pixels;
  double Tm[16];
  se3_matrix(st.estimate, Tm);
  // take the matrix exactly as given (the round trip through the quaternion is not bit exact)
  for (int j = 0; j < 4; ++j) {
    float t0 = (float)T[j], t1 = (float)T[4 + j], t2 = (float)T[8 + j];
    st.kt[j] = __fadd_rn(__fmul_rn(pl.cfx, t0), __fmul_rn(pl.cox, t2));
    st.kt[4 + j] = __fadd_rn(__fmul_rn(pl.cfy, t1), __fmul_rn(pl.coy, t2));
    st.kt[8 + j] = t2;
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
inline int level_flag_slot(int li) { return li < 8 ? li : 7; }
template <typename T>
int grow(dvo_b200_ctx* ctx, T*& ptr, size_t& cap, size_t need) {
  if (need <= cap) return 0;
  if (ptr) { cudaStreamSynchronize(ctx->stream); cudaFree(ptr); ptr = nullptr; cap = 0; }
  DVO_CUDA(ctx, cudaMalloc((void**)&ptr, need * sizeof(T)));
  cap = need;
  return 0;
}

struct ScratchNeed {
  size_t row_export_floats = 0, row_base_ints = 0, strip_export_doubles = 0, strip_base_ints = 0, row_partial_floats = 0,
         strip_partial_doubles = 0, squads = 0;
  size_t dump_floats = 0;
};

int ensure_workspace(dvo_b200_ctx* ctx, int npairs, const ScratchNeed& need, int max_log_per_pair) {
  Workspace& ws = ctx->ws;
  if ((size_t)npairs > ws.cap_pairs) {
    if (ws.d_pair_level) { cudaStreamSynchronize(ctx->stream); cudaFree(ws.d_pair_level); cudaFree(ws.d_state); }
    ws.d_pair_level = nullptr; ws.d_state = nullptr; ws.cap_pairs = 0;
    DVO_CUDA(ctx, cudaMalloc((void**)&ws.d_pair_level, sizeof(PairLevel) * npairs + 16));   // k_stage_words copies whole 16-byte words
    DVO_CUDA(ctx, cudaMalloc((void**)&ws.d_state, sizeof(PairState) * npairs));
    ws.cap_pairs = npairs;
  }
  int rc;
  if ((rc = grow(ctx, ws.d_row_exports, ws.cap_row_exports, need.row_export_floats))) return rc;
  if ((rc = grow(ctx, ws.d_row_base, ws.cap_row_base, need.row_base_ints))) return rc;
  if ((rc = grow(ctx, ws.d_strip_exports, ws.cap_strip_exports, need.strip_export_doubles))) return rc;
  if ((rc = grow(ctx, ws.d_strip_base, ws.cap_strip_base, need.strip_base_ints))) return rc;
  if ((rc = grow(ctx, ws.d_row_partial, ws.cap_row_partial, need.row_partial_floats))) return rc;
  if ((rc = grow(ctx, ws.d_strip_partial, ws.cap_strip_partial, need.strip_partial_doubles))) return rc;
  if ((rc = grow(ctx, ws.d_squads, ws.cap_squads, need.squads * sizeof(SquadState)))) return rc;
  if ((rc = grow(ctx, ws.d_dump, ws.cap_dump, need.dump_floats))) return rc;
  if (!ws.h_active) DVO_CUDA(ctx, cudaMallocHost((void**)&ws.h_active, sizeof(int) * 8));
  if (!ws.h_flag_accum) {
    DVO_CUDA(ctx, cudaMallocHost((void**)&ws.h_flag_accum, sizeof(int)));
    *ws.h_flag_accum = 0;
  }
  if (max_log_per_pair > 0) {
    size_t n = (size_t)npairs * max_log_per_pair;
    if ((rc = grow(ctx, ws.d_iter_log, ws.cap_iter_log, n))) return rc;
  }
  return 0;
}

int ensure_geometry(dvo_b200_ctx* ctx) {
  if (ctx->num_sms != 0) return 0;
  cudaDeviceProp prop;
  DVO_CUDA(ctx, cudaGetDeviceProperties(&prop, ctx->device));
  DVO_CUDA(ctx, cudaFuncSetAttribute(k_level_persistent, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kLevelSmemBytes));
  int per_sm = 0;
  DVO_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_level_persistent, kCtaThreads, kLevelSmemBytes));
  if (per_sm < 1) return set_error(ctx, DVO_B200_ERR_CUDA, "persistent kernel does not fit on an SM");
  ctx->ctas_per_sm = per_sm;
  ctx->num_sms = prop.multiProcessorCount;
  return 0;
}

// How a group of consecutive pyramid levels is spread over the persistent grid: one launch walks every pair through the
// group's levels (coarse to fine) inside the kernel.
struct GroupPlan {
  int first_li, nlev;   // levels [first_li, first_li + nlev) of the match (index 0 = coarsest)
  int g;                // CTAs per squad
  int nsquads;          // squads in the grid
  int strips_per_cta[kMaxLevels];
  int pair_begin, npairs;   // the pairs this segment's queue hands out (a slice of the batch for the fine segments of a fused launch)
};

// Squad size for one level on its own.  A squad of g CTAs gives each CTA spc = ceil(nstrips / g) strips.  Small squads keep
// many pairs in flight and amortise the two barriers and the serial P_k / solve sections of an iteration over more tiles
// per CTA; but the batch is processed in waves of nsquads pairs, and a last wave that is mostly empty wastes more than
// that.  Pairs are handed out from a queue, so a level takes about (pairs per squad + tail) x time per pair, where the
// tail (pairs that need two or three times the mean number of iterations) is worth a bit more than one pair and the time
// per pair goes with (tiles per CTA + per-iteration overhead in tile units).
int level_squad_size(int nstrips, int nbands, int grid, int npairs) {
  const char* env = getenv("DVO_B200_STRIPS_PER_CTA");     // developer override (experiments)
  const int forced_spc = env ? atoi(env) : 0;
  const double overhead_tiles = 20.0;   // per stage: squad barrier + serial step + pipeline fill, in tile-times (fitted: g = 2..5 within 1 % at batch 512, g >= 6 and g = 1 slower)
  int best_g = 1;
  double best_cost = -1.0;
  for (int spc = 1; spc <= nstrips; ++spc) {
    const int g = (nstrips + spc - 1) / spc;
    if (g > grid) continue;
    if (spc > 1 && (nstrips + spc - 2) / (spc - 1) == g) continue;   // same g as the previous spc: more work per CTA, nothing gained
    const int nsquads = std::min(grid / g, std::max(npairs, 1));
    const double per_squad = (double)npairs / nsquads;
    double cost = (std::max(per_squad, 1.0) + (npairs > nsquads ? 1.2 : 0.0)) * ((double)spc * nbands + overhead_tiles);
    if (forced_spc > 0) cost = std::abs(spc - forced_spc);
    if (best_cost < 0 || cost < best_cost - 1e-9) { best_cost = cost; best_g = g; }
  }
  return best_g;
}

// Levels small enough for one CTA per pair (no squad barriers at all) form one group: a CTA takes a pair from the queue and
// runs it through all of them, so a pair that needs many iterations on one coarse level delays nobody.  The remaining
// (fine) levels form a second group with the squad size of the finest level; a squad likewise walks its pair through both.
// With few pairs every level gets its own launch and the squad size that minimises its latency.
int plan_groups(const dvo_b200_pyramid* ref, int first, int last, int grid, int npairs, GroupPlan* out) {
  const int nlev = first - last + 1;
  int g_level[kMaxLevels];
  for (int li = 0; li < nlev; ++li) {
    const LevelInfo& L = ref->L[first - li];
    g_level[li] = level_squad_size(L.nstrips, L.nbands, grid, npairs);
  }
  int ngroups = 0;
  const bool walk = npairs >= grid / 4 && !getenv("DVO_B200_NO_WALK");
  const int coarse_tiles = getenv("DVO_B200_COARSE_TILES") ? atoi(getenv("DVO_B200_COARSE_TILES")) : 110;   // levels up to 320x240 (105 tiles): one CTA per pair; env = developer override
  for (int li = 0; li < nlev;) {
    GroupPlan& G = out[ngroups++];
    G.first_li = li; G.nlev = 1; G.g = g_level[li];
    if (walk) {
      const LevelInfo& L0 = ref->L[first - li];
      const bool coarse = L0.nstrips * L0.nbands <= coarse_tiles;
      if (coarse) G.g = 1;
      while (li + G.nlev < nlev) {
        const LevelInfo& Ln = ref->L[first - (li + G.nlev)];
        const bool coarse_n = Ln.nstrips * Ln.nbands <= coarse_tiles;
        if (coarse_n != coarse) break;
        if (!coarse) G.g = g_level[li + G.nlev];      // the finest level of the group decides
        G.nlev++;
      }
    }
    if (const char* fg = getenv("DVO_B200_FINE_G")) {     // developer override (experiments): squad size of the non-coarse groups
      const LevelInfo& L0 = ref->L[first - li];
      if (L0.nstrips * L0.nbands > coarse_tiles && atoi(fg) > 0) G.g = std::min(atoi(fg), grid);
    }
    for (int k = 0; k < G.nlev; ++k) {
      const LevelInfo& L = ref->L[first - (li + k)];
      const int g_eff = std::min(G.g, L.nstrips);
      G.strips_per_cta[k] = (L.nstrips + g_eff - 1) / g_eff;
    }
    G.nsquads = std::min(grid / G.g, std::max(npairs, 1));
    G.pair_begin = 0; G.npairs = npairs;
    li += G.nlev;
  }
  return ngroups;
}

int check_batch(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int n, dvo_b200_pyramid* const* refs,
                dvo_b200_pyramid* const* curs) {
  if (!cfg || n <= 0 || !refs || !curs) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match: null argument");
  if (cfg->first_level < cfg->last_level || cfg->last_level < 0 || cfg->first_level >= kMaxLevels)
    return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match: config not sane (FirstLevel >= LastLevel >= 0 required)");
  if (cfg->max_iterations_per_level < 0) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match: max iterations < 0");
  for (int i = 0; i < n; ++i) {
    if (!refs[i] || !curs[i]) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match: null pyramid");
    // a pyramid built on another ctx's stream: order this stream after its build
    for (const dvo_b200_pyramid* p : {refs[i], curs[i]})
      if (p->slab && p->slab->pool != ctx->pool && p->slab->ready) cudaStreamWaitEvent(ctx->stream, p->slab->ready, 0);
    if (refs[i]->levels <= cfg->first_level || curs[i]->levels <= cfg->first_level)
      return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "match: pyramid has fewer levels than FirstLevel+1");
    if (refs[i]->L[0].w != refs[0]->L[0].w || refs[i]->L[0].h != refs[0]->L[0].h ||
        curs[i]->L[0].w != refs[0]->L[0].w || curs[i]->L[0].h != refs[0]->L[0].h)
      return set_error(ctx, DVO_B200_ERR_SHAPE_MISMATCH, "match: all pyramids of a batch must share width/height");
  }
  return 0;
}

void fill_pair_levels(PairLevel* h, int n, dvo_b200_pyramid* const* refs, dvo_b200_pyramid* const* curs, int level) {
  for (int i = 0; i < n; ++i) {
    const dvo_b200_pyramid* r = refs[i];
    const dvo_b200_pyramid* c = curs[i];
    const LevelInfo& rl = r->L[level];
    const LevelInfo& cl = c->L[level];
    PairLevel& q = h[i];
    const size_t plane = (size_t)rl.pitch * rl.h;
    q.r0 = r->planes + rl.rec_off; q.r1 = q.r0;
    q.rmask = r->sel_mask + rl.mask_off;
    q.rsel = r->sel_info + 2 * level;
    q.rtmpl = r->tmpl + rl.tmpl_off;
    q.rrange = r->tile_range + rl.range_off;
    q.c0 = c->planes + cl.plane_off; q.c3 = q.c0 + plane;
    q.cfx = cl.fx; q.cfy = cl.fy; q.cox = cl.ox; q.coy = cl.oy;
    // PointSelection::getMaximumNumberOfPoints (point_selection.cpp:68-71)
    q.max_valid_pixels = (long long)(size_t)((double)r->L[0].n * pow(0.25, (double)level));
  }
}

// The same descriptors against separate selections (refs[i] = sels[i]->pyr): tile records, mask and {S, last} come from
// the selection, template and tile depth ranges from its pyramid.
void fill_pair_levels_selected(PairLevel* h, int n, dvo_b200_pyramid* const* refs, dvo_b200_selection* const* sels,
                               dvo_b200_pyramid* const* curs, int level) {
  fill_pair_levels(h, n, refs, curs, level);
  for (int i = 0; i < n; ++i) {
    const dvo_b200_selection* s = sels[i];
    PairLevel& q = h[i];
    q.r0 = s->rec + s->rec_off[level]; q.r1 = q.r0;
    q.rmask = s->mask + refs[i]->L[level].mask_off;
    q.rsel = s->sel_info + 2 * level;
  }
}

LevelLaunch make_level_launch(const LevelInfo& L, const dvo_b200_config* cfg, int li, int level) {
  LevelLaunch lp;
  lp.w = L.w; lp.h = L.h; lp.n = L.n; lp.pitch = L.pitch; lp.nbands = L.nbands; lp.nstrips = L.nstrips;
  lp.level_index = li; lp.level_id = level; lp.max_iterations = cfg->max_iterations_per_level;
  lp.first_level = li == 0; lp.use_initial_estimate = cfg->use_initial_estimate;
  lp.precision = cfg->precision; lp.mu = cfg->mu;
  return lp;
}

// scratch of one launch = the sum over its segments (they are live at the same time); the workspace keeps the maximum
ScratchNeed segment_need(int hmax, const GroupPlan& pl) {
  ScratchNeed s;
  s.row_export_floats = (size_t)pl.nsquads * hmax * kSegExportFloats;
  s.row_base_ints = (size_t)pl.nsquads * hmax;
  const size_t smax = (size_t)(hmax + kTileH - 1) / kTileH;
  s.strip_export_doubles = (size_t)pl.nsquads * smax * kStripExportDoubles;
  s.strip_base_ints = (size_t)pl.nsquads * (smax + 1);
  s.row_partial_floats = (size_t)pl.nsquads * hmax * kNormalValues;
  s.strip_partial_doubles = (size_t)pl.nsquads * smax * kNormalValues;
  s.squads = (size_t)pl.nsquads;
  return s;
}
void add_launch_need(ScratchNeed& need, int nseg, const int* hmax, const GroupPlan* plans, int npairs) {
  ScratchNeed sum;
  for (int s = 0; s < nseg; ++s) {
    const ScratchNeed q = segment_need(hmax[s], plans[s]);
    sum.row_export_floats += q.row_export_floats; sum.row_base_ints += q.row_base_ints; sum.strip_export_doubles += q.strip_export_doubles;
    sum.strip_base_ints += q.strip_base_ints; sum.row_partial_floats += q.row_partial_floats;
    sum.strip_partial_doubles += q.strip_partial_doubles; sum.squads += q.squads;
  }
  sum.squads += 1 + ((size_t)npairs * sizeof(int) + sizeof(SquadState) - 1) / sizeof(SquadState);   // counters + ready ring
  need.row_export_floats = std::max(need.row_export_floats, sum.row_export_floats);
  need.row_base_ints = std::max(need.row_base_ints, sum.row_base_ints);
  need.strip_export_doubles = std::max(need.strip_export_doubles, sum.strip_export_doubles);
  need.strip_base_ints = std::max(need.strip_base_ints, sum.strip_base_ints);
  need.row_partial_floats = std::max(need.row_partial_floats, sum.row_partial_floats);
  need.strip_partial_doubles = std::max(need.strip_partial_doubles, sum.strip_partial_doubles);
  need.squads = std::max(need.squads, sum.squads);
}

// Enqueue one persistent launch of nseg (1 or 2) segments; squad states, queues, the ready ring and the error flag are
// zeroed first.  lps / d_pls: per segment.  `flag_out` receives the device address of the launch's error flag.
int launch_segments(dvo_b200_ctx* ctx, int nseg, const LevelLaunch (*lps)[kMaxLevels], const GroupPlan* plans, const int* hmax,
                    const PairLevel* const* d_pls, const double* d_Tinit, int npairs, int max_log, float* dump, int skip_begin,
                    int group_index, int** flag_out) {
  Workspace& ws = ctx->ws;
  cudaStream_t st = ctx->stream;
  size_t nsq = 0;
  for (int s = 0; s < nseg; ++s) nsq += plans[s].nsquads;
  const size_t ring_states = ((size_t)npairs * sizeof(int) + sizeof(SquadState) - 1) / sizeof(SquadState);
  DVO_CUDA(ctx, cudaMemsetAsync(ws.d_squads, 0, sizeof(SquadState) * (nsq + 1 + ring_states), st));
  PersistentArgs pa;
  pa.states = ws.d_state;
  SquadState* squads = reinterpret_cast<SquadState*>(ws.d_squads);
  int* counters = reinterpret_cast<int*>(squads + nsq);      // one zeroed 128-byte line: {queue[4], ready tail[4], arrivals[4], error flag}
  int* ring = reinterpret_cast<int*>(squads + nsq + 1);      // npairs slots: the ready rings of the fine segments, by pair range
  pa.error_flag = counters + 3 * kMaxSeg;
  pa.ilog = ws.d_iter_log; pa.max_log = max_log;
  pa.T_init = d_Tinit; pa.skip_begin = skip_begin;
  pa.dump = dump;
  pa.npairs = npairs; pa.nseg = nseg;
  ScratchNeed off;
  size_t sq_off = 0;
  for (int s = 0; s < nseg; ++s) {
    Segment& S = pa.seg[s];
    const GroupPlan& plan = plans[s];
    S.pls = d_pls[s];
    S.row_exports = ws.d_row_exports + off.row_export_floats; S.row_base = ws.d_row_base + off.row_base_ints;
    S.strip_exports = ws.d_strip_exports + off.strip_export_doubles; S.strip_base = ws.d_strip_base + off.strip_base_ints;
    S.row_partial = ws.d_row_partial + off.row_partial_floats; S.strip_partial = ws.d_strip_partial + off.strip_partial_doubles;
    S.squads = squads + sq_off;
    S.queue = counters + s; S.ready_tail = counters + kMaxSeg + s; S.arrivals = counters + 2 * kMaxSeg + s;
    S.pair_begin = plan.pair_begin; S.npairs_seg = plan.npairs;
    S.cyclic = getenv("DVO_B200_CONTIGUOUS") ? 0 : 1;          // developer switch (results are identical either way)
    S.ready = ring + plan.pair_begin;
    const int slot = std::min(group_index + s, 7);
    S.dbg = ctx->d_dbg ? ctx->d_dbg + 16 * slot : nullptr;
    S.dbg2 = ctx->d_dbg ? ctx->d_dbg + 128 + 8 * slot : nullptr;
    S.nlev = plan.nlev; S.g = plan.g; S.nsquads = plan.nsquads;
    for (int k = 0; k < kMaxLevels; ++k) {
      S.strips_per_cta[k] = k < plan.nlev ? plan.strips_per_cta[k] : 0;
      if (k < plan.nlev) S.lp[k] = lps[s][k];
    }
    const ScratchNeed q = segment_need(hmax[s], plan);
    off.row_export_floats += q.row_export_floats; off.row_base_ints += q.row_base_ints; off.strip_export_doubles += q.strip_export_doubles;
    off.strip_base_ints += q.strip_base_ints; off.row_partial_floats += q.row_partial_floats; off.strip_partial_doubles += q.strip_partial_doubles;
    sq_off += plan.nsquads;
  }
  {
    ProfScope prof(ctx, 0);
    ProfScope prof_level(ctx, 8 + std::min(group_index, 7));
    void* args[] = {&pa};
    DVO_CUDA(ctx, cudaLaunchCooperativeKernel((const void*)k_level_persistent, dim3(ctx->num_sms * ctx->ctas_per_sm),
                                              dim3(kCtaThreads), args, kLevelSmemBytes, st));
    ctx->launches++;
  }
  *flag_out = pa.error_flag;
  return 0;
}

// A pinned slot of at least `bytes` for the pair descriptors of one enqueued call.  Waits only if the ring has wrapped onto
// a slot whose k_stage_words has not run yet; growing the slots (a larger batch than before) waits for all of them.
int acquire_desc_slot(dvo_b200_ctx* ctx, size_t bytes, int* slot) {
  if (bytes > ctx->desc_slot_bytes) {
    for (int i = 0; i < dvo_b200_ctx::kDescSlots; ++i) {
      if (ctx->desc_staged[i]) DVO_CUDA(ctx, cudaEventSynchronize(ctx->desc_staged[i]));
      if (ctx->h_desc[i]) cudaFreeHost(ctx->h_desc[i]);
      ctx->h_desc[i] = nullptr;
    }
    ctx->desc_slot_bytes = 0;
    for (int i = 0; i < dvo_b200_ctx::kDescSlots; ++i) {
      DVO_CUDA(ctx, cudaMallocHost(&ctx->h_desc[i], bytes));
      if (!ctx->desc_staged[i]) DVO_CUDA(ctx, cudaEventCreateWithFlags(&ctx->desc_staged[i], cudaEventDisableTiming));
    }
    ctx->desc_slot_bytes = bytes;
  }
  const int i = ctx->desc_next;
  ctx->desc_next = (i + 1) % dvo_b200_ctx::kDescSlots;
  if (cudaEventQuery(ctx->desc_staged[i]) == cudaErrorNotReady) DVO_CUDA(ctx, cudaEventSynchronize(ctx->desc_staged[i]));
  cudaGetLastError();
  *slot = i;
  return 0;
}

}  // namespace

int tracker_match_batch(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, int n, dvo_b200_pyramid* const* refs,
                        dvo_b200_pyramid* const* curs, const double* T_init, dvo_b200_result* h_results,
                        void* d_results_user, dvo_b200_iteration_stats* iter_stats, int max_iter_stats, bool enqueue,
                        dvo_b200_selection* const* sels) {
  int rc = check_batch(ctx, cfg, n, refs, curs);
  if (rc) return rc;
  if (sels)   // a selection built on another ctx's stream: order this stream after its build
    for (int i = 0; i < n; ++i)
      if (sels[i]->slab && sels[i]->slab->pool != ctx->pool && sels[i]->slab->ready) cudaStreamWaitEvent(ctx->stream, sels[i]->slab->ready, 0);
  cudaStream_t st = ctx->stream;
  Workspace& ws = ctx->ws;
  const int last = cfg->last_level, first = cfg->first_level;
  const int max_log = iter_stats ? max_iter_stats : 0;
  if ((rc = ensure_geometry(ctx))) return rc;
  const int nlev = first - last + 1;
  const int grid = ctx->num_sms * ctx->ctas_per_sm;
  GroupPlan groups[kMaxLevels];
  const int ngroups = plan_groups(refs[0], first, last, grid, n, groups);
  int hmaxs[kMaxLevels];
  for (int gi = 0; gi < ngroups; ++gi) {
    hmaxs[gi] = 0;
    for (int k = 0; k < groups[gi].nlev; ++k) hmaxs[gi] = std::max(hmaxs[gi], refs[0]->L[first - (groups[gi].first_li + k)].h);
  }
  // A coarse group (one CTA per pair) followed by a fine group runs as ONE launch of two segments: no grid-wide barrier and
  // no launch boundary between them, so the CTAs that run out of coarse pairs start on fine pairs while the long coarse
  // pairs are still iterating.
  const bool fuse = ngroups == 2 && groups[0].g == 1 && !getenv("DVO_B200_NO_FUSE");
  // Fused launch: the fine group is cut into up to three slices of the pair index with squads of g, 2g and 4g CTAs.  Pairs
  // come off a queue, so with one squad size the launch ends with most squads idle while a few finish pairs that need two
  // or three times the mean number of iterations (measured at batch 512: 16 % of the CTA time).  The last pairs of the
  // batch, which also leave the coarse segment last, therefore go to wider squads that finish a pair in a half / a quarter
  // of the time; the slice a pair belongs to is fixed by its index, so results do not depend on timing.
  GroupPlan segs[kMaxSeg];
  int seg_hmax[kMaxSeg];
  int nseg = 1;
  if (fuse) {
    segs[0] = groups[0]; seg_hmax[0] = hmaxs[0];
    const GroupPlan& F = groups[1];
    int min_strips = 1 << 30;
    for (int k = 0; k < F.nlev; ++k) min_strips = std::min(min_strips, refs[0]->L[first - (F.first_li + k)].nstrips);
    int counts[3] = {n, 0, 0};
    {
      int c2 = 0, c3 = 0;
      const int g2 = 2 * F.g, g3 = 4 * F.g;
      if (g2 <= min_strips && g2 <= grid) c2 = (int)(1.8 * (grid / g2) + 0.5);
      if (c2 && g3 <= min_strips && g3 <= grid) c3 = (int)(1.8 * (grid / g3) + 0.5);
      if (const char* e = getenv("DVO_B200_TAIL")) {       // developer override: "c2,c3" pairs for the 2g and 4g slices
        int a2 = 0, a3 = 0;
        if (sscanf(e, "%d,%d", &a2, &a3) >= 1) { c2 = (g2 <= min_strips && g2 <= grid) ? a2 : 0; c3 = (c2 && g3 <= min_strips && g3 <= grid) ? a3 : 0; }
      }
      const int keep = 2 * (grid / F.g);                     // the first slice keeps at least two pairs per squad
      if (n - c2 - c3 < keep) c3 = 0;
      if (n - c2 < keep) c2 = 0;
      counts[0] = n - c2 - c3; counts[1] = c2; counts[2] = c3;
    }
    int begin = 0;
    for (int k = 0; k < 3; ++k) {
      if (counts[k] <= 0) continue;
      GroupPlan& G = segs[nseg];
      G = F;
      G.g = F.g << k;
      for (int j = 0; j < G.nlev; ++j) {
        const LevelInfo& L = refs[0]->L[first - (G.first_li + j)];
        const int g_eff = std::min(G.g, L.nstrips);
        G.strips_per_cta[j] = (L.nstrips + g_eff - 1) / g_eff;
      }
      G.pair_begin = begin; G.npairs = counts[k];
      G.nsquads = std::min(grid / G.g, std::max(counts[k], 1));
      seg_hmax[nseg] = hmaxs[1];
      begin += counts[k];
      ++nseg;
    }
  }
  ScratchNeed need;
  if (fuse) add_launch_need(need, nseg, seg_hmax, segs, n);
  else for (int gi = 0; gi < ngroups; ++gi) add_launch_need(need, 1, hmaxs + gi, groups + gi, n);
  rc = ensure_workspace(ctx, n * nlev, need, max_log);     // d_pair_level holds the descriptors of every level
  if (rc) return rc;

  // selection masks for non-default thresholds (PointSelection caches per pyramid, point_selection.cpp:100-113)
  // (not for separate selections: their predicate decides, as in match(PointSelection&, ...), dense_tracking.cpp:131-135)
  if (!sels)
    for (int i = 0; i < n; ++i)
      if ((rc = pyramid_reselect(ctx, refs[i], cfg->intensity_derivative_threshold, cfg->depth_derivative_threshold))) return rc;

  // Pair descriptors of every level and the initial estimates go into the pinned stage once; one small kernel copies
  // them to device memory (reads over PCIe: no H2D copy-engine work, no host round trip between the launches below).
  // The enqueue variant takes the initial estimates from the caller's device memory and stages only the descriptors, in
  // a slot of the descriptor ring.
  const size_t desc_bytes = (sizeof(PairLevel) * (size_t)n * nlev + 15) / 16 * 16;
  const bool have_init = cfg->use_initial_estimate && T_init;
  const size_t init_bytes = have_init && !enqueue ? sizeof(double) * 16 * (size_t)n : 0;
  PairLevel* h_desc = nullptr;
  int slot = 0;
  if (enqueue) {
    if ((rc = acquire_desc_slot(ctx, desc_bytes, &slot))) return rc;
    h_desc = (PairLevel*)ctx->h_desc[slot];
  } else {
    if ((rc = ensure_stage(ctx, 0, desc_bytes + init_bytes))) return rc;
    if ((rc = grow(ctx, ws.d_tinit, ws.cap_tinit, (size_t)16 * n))) return rc;
    DVO_CUDA(ctx, cudaStreamSynchronize(st));   // previous use of the pinned stage has drained
    fold_level_flags(ctx);                      // flags of an earlier call whose results stayed on the device
    h_desc = (PairLevel*)ctx->h_stage;
    if (have_init) std::memcpy((char*)ctx->h_stage + desc_bytes, T_init, init_bytes);
  }
  for (int level = first, li = 0; level >= last; --level, ++li) {
    if (sels) fill_pair_levels_selected(h_desc + (size_t)li * n, n, refs, sels, curs, level);
    else fill_pair_levels(h_desc + (size_t)li * n, n, refs, curs, level);
  }
  ctx->h2d_bytes += desc_bytes + init_bytes;
  {
    ProfScope prof(ctx, 2);
    const size_t n16 = desc_bytes / 16;
    k_stage_words<<<(unsigned)((n16 + 255) / 256), 256, 0, st>>>((const uint4*)h_desc, (uint4*)ws.d_pair_level, n16);
    ctx->launches++;
    if (init_bytes) {
      const size_t m16 = init_bytes / 16;
      k_stage_words<<<(unsigned)((m16 + 255) / 256), 256, 0, st>>>((const uint4*)((char*)ctx->h_stage + desc_bytes), (uint4*)ws.d_tinit, m16);
      ctx->launches++;
    }
  }
  if (enqueue) DVO_CUDA(ctx, cudaEventRecord(ctx->desc_staged[slot], st));
  else for (int i = 0; i < 8; ++i) ws.h_active[i] = 0;
  const double* d_tinit = !have_init ? nullptr : enqueue ? T_init : ws.d_tinit;
  // after each launch its error flag goes to pinned memory: into the per-level slots checked when this call (or the next
  // synchronisation) waits, or -- enqueue -- folded into the word the next synchronisation reads
  auto keep_flag = [&](int launch, int* flag) -> int {
    if (enqueue) {
      k_fold_flag<<<1, 1, 0, st>>>(flag, ws.h_flag_accum);
      ctx->launches++;
      return 0;
    }
    DVO_CUDA(ctx, cudaMemcpyAsync(&ws.h_active[level_flag_slot(launch)], flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    return 0;
  };

  if (max_log > 0) DVO_CUDA(ctx, cudaMemsetAsync(ws.d_iter_log, 0, sizeof(dvo_b200_iteration_stats) * (size_t)n * max_log, st));
  LevelLaunch lps[kMaxLevels][kMaxLevels];
  const PairLevel* d_pls[kMaxLevels];
  for (int gi = 0; gi < ngroups; ++gi) {
    const GroupPlan& G = groups[gi];
    for (int k = 0; k < G.nlev; ++k) {
      const int li = G.first_li + k, level = first - li;
      lps[gi][k] = make_level_launch(refs[0]->L[level], cfg, li, level);
    }
    d_pls[gi] = ws.d_pair_level + (size_t)G.first_li * n;
  }
  const int nlaunch = fuse ? 1 : ngroups;
  if (fuse) {
    LevelLaunch seg_lps[kMaxSeg][kMaxLevels];
    const PairLevel* seg_pls[kMaxSeg];
    for (int sgi = 0; sgi < nseg; ++sgi) {
      const int gi = sgi == 0 ? 0 : 1;
      for (int k = 0; k < groups[gi].nlev; ++k) seg_lps[sgi][k] = lps[gi][k];
      seg_pls[sgi] = d_pls[gi];
    }
    int* flag = nullptr;
    if ((rc = launch_segments(ctx, nseg, seg_lps, segs, seg_hmax, seg_pls, d_tinit, n, max_log, nullptr, 0, 0, &flag)))
      return rc;
    if ((rc = keep_flag(0, flag))) return rc;
  } else {
    for (int gi = 0; gi < nlaunch; ++gi) {
      int* flag = nullptr;
      if ((rc = launch_segments(ctx, 1, lps + gi, groups + gi, hmaxs + gi, d_pls + gi, d_tinit, n, max_log, nullptr, 0, gi, &flag)))
        return rc;
      if ((rc = keep_flag(gi, flag))) return rc;
    }
  }
  // results
  dvo_b200_result* d_res = (dvo_b200_result*)d_results_user;
  if (!d_res) {
    size_t bytes = sizeof(dvo_b200_result) * n;
    if ((rc = ensure_stage(ctx, bytes, 0))) return rc;
    d_res = (dvo_b200_result*)ctx->d_stage;
  }
  {
    ProfScope prof(ctx, 2);
    k_finalize<<<(n + 63) / 64, 64, 0, st>>>(ws.d_state, d_res, n);
    ctx->launches++;
  }
  DVO_CUDA(ctx, cudaGetLastError());
  if (!enqueue) ctx->pending_level_flags = nlaunch;   // checked at the next synchronisation point (device-results variant)
  if (h_results) {
    size_t bytes = sizeof(dvo_b200_result) * n;
    if (bytes > ctx->h_results_bytes) {
      if (ctx->h_results) cudaFreeHost(ctx->h_results);
      ctx->h_results = nullptr; ctx->h_results_bytes = 0;
      DVO_CUDA(ctx, cudaMallocHost(&ctx->h_results, bytes));
      ctx->h_results_bytes = bytes;
    }
    DVO_CUDA(ctx, cudaMemcpyAsync(ctx->h_results, d_res, bytes, cudaMemcpyDeviceToHost, st));
    if (iter_stats) {
      DVO_CUDA(ctx, cudaMemcpyAsync(iter_stats, ws.d_iter_log, sizeof(dvo_b200_iteration_stats) * (size_t)n * max_log,
                                    cudaMemcpyDeviceToHost, st));
      ctx->d2h_bytes += sizeof(dvo_b200_iteration_stats) * (size_t)n * max_log;
    }
    DVO_CUDA(ctx, cudaStreamSynchronize(st));
    std::memcpy(h_results, ctx->h_results, bytes);
    ctx->d2h_bytes += bytes;
    return check_level_flags(ctx);
  }
  return 0;
}

// The persistent kernels report a barrier / transaction timeout through a flag copied to pinned memory after every level.
// fold_level_flags moves a reported code of the pending levels into the accumulated word, so that a call which reuses the
// per-level slots does not lose it; check_level_flags reports (and clears) the accumulated code.  Both run after the
// stream has been synchronised.
void fold_level_flags(dvo_b200_ctx* ctx) {
  Workspace& ws = ctx->ws;
  const int nl = ctx->pending_level_flags;
  ctx->pending_level_flags = 0;
  if (!ws.h_active) return;
  for (int li = 0; li < nl && li < 8; ++li)
    if (ws.h_active[li] != 0) {
      if (ws.h_flag_accum && *ws.h_flag_accum == 0) *ws.h_flag_accum = ws.h_active[li];
      ws.h_active[li] = 0;
    }
}

int check_level_flags(dvo_b200_ctx* ctx) {
  Workspace& ws = ctx->ws;
  fold_level_flags(ctx);
  if (!ws.h_flag_accum || *ws.h_flag_accum == 0) return 0;
  const int code = *ws.h_flag_accum;
  *ws.h_flag_accum = 0;
  return set_error(ctx, DVO_B200_ERR_CUDA, code == 2 ? "persistent level kernel: bulk-copy transaction timed out"
                                                     : "persistent level kernel: squad barrier timed out");
}

void tracker_release(dvo_b200_ctx* ctx) {
  for (int i = 0; i < dvo_b200_ctx::kDescSlots; ++i) {
    if (ctx->h_desc[i]) cudaFreeHost(ctx->h_desc[i]);
    if (ctx->desc_staged[i]) cudaEventDestroy(ctx->desc_staged[i]);
    ctx->h_desc[i] = nullptr; ctx->desc_staged[i] = nullptr;
  }
  ctx->desc_slot_bytes = 0;
  if (ctx->ws.h_flag_accum) cudaFreeHost(ctx->ws.h_flag_accum);
  ctx->ws.h_flag_accum = nullptr;
}

// Test hooks (dvo_b200_residual_image, dvo_b200_linearize): ONE Gauss-Newton iteration of the level kernel for one
// pair at a fixed transform: stage A, P_k, stage B (optionally dumping the residual records), end step.
int tracker_linearize(dvo_b200_ctx* ctx, const dvo_b200_config* cfg, dvo_b200_pyramid* ref, dvo_b200_pyramid* cur,
                      int level, const double* T, int use_weights, const float* prev_precision, int64_t* count,
                      float* precision_out, float* ll_out, double* A_out, double* b_out, float* planes7) {
  dvo_b200_config c = *cfg;
  c.first_level = level; c.last_level = level;
  dvo_b200_pyramid* refs[1] = {ref};
  dvo_b200_pyramid* curs[1] = {cur};
  int rc = check_batch(ctx, &c, 1, refs, curs);
  if (rc) return rc;
  if (!T) return set_error(ctx, DVO_B200_ERR_INVALID_ARGUMENT, "linearize: T is null");
  cudaStream_t st = ctx->stream;
  Workspace& ws = ctx->ws;
  const LevelInfo& L = ref->L[level];
  if ((rc = ensure_geometry(ctx))) return rc;
  GroupPlan plan;
  {
    GroupPlan tmp[kMaxLevels];
    plan_groups(ref, level, level, ctx->num_sms * ctx->ctas_per_sm, 1, tmp);
    plan = tmp[0];
    ScratchNeed need;
    const int hm = L.h;
    add_launch_need(need, 1, &hm, &plan, 1);
    if (planes7) need.dump_floats = 7 * (size_t)L.n;
    if ((rc = ensure_workspace(ctx, 1, need, 0))) return rc;
  }
  if ((rc = pyramid_reselect(ctx, ref, cfg->intensity_derivative_threshold, cfg->depth_derivative_threshold))) return rc;
  LevelLaunch lp = make_level_launch(L, &c, 0, level);
  lp.max_iterations = use_weights ? 2 : 1;    // k_set_state starts at iteration 1 / 0: exactly one iteration runs
  lp.first_level = 1; lp.use_initial_estimate = 0; lp.precision = 0.0; lp.mu = 0.0;
  if ((rc = ensure_stage(ctx, 1024, sizeof(PairLevel) + 1024))) return rc;
  DVO_CUDA(ctx, cudaStreamSynchronize(st));
  fill_pair_levels((PairLevel*)ctx->h_stage, 1, refs, curs, level);
  DVO_CUDA(ctx, cudaMemcpyAsync(ws.d_pair_level, ctx->h_stage, sizeof(PairLevel), cudaMemcpyHostToDevice, st));
  DVO_CUDA(ctx, cudaStreamSynchronize(st));
  fold_level_flags(ctx);
  std::memcpy(ctx->h_stage, T, sizeof(double) * 16);
  float pp[4] = {0, 0, 0, 0};
  if (use_weights && prev_precision) std::memcpy(pp, prev_precision, sizeof(pp));
  std::memcpy((char*)ctx->h_stage + 128, pp, sizeof(pp));
  DVO_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage, ctx->h_stage, 256, cudaMemcpyHostToDevice, st));
  ctx->h2d_bytes += sizeof(PairLevel) + 256;
  k_set_state<<<1, 1, 0, st>>>(ws.d_state, ws.d_pair_level, (const double*)ctx->d_stage,
                               (const float*)((char*)ctx->d_stage + 128), use_weights, lp);
  ctx->launches += 1;
  int* flag = nullptr;
  ws.h_active[0] = 0;
  LevelLaunch lps[1][kMaxLevels];
  lps[0][0] = lp;
  const int hm = L.h;
  const PairLevel* d_pls[1] = {ws.d_pair_level};
  if ((rc = launch_segments(ctx, 1, lps, &plan, &hm, d_pls, nullptr, 1, 0, planes7 ? ws.d_dump : nullptr, 1, 0, &flag))) return rc;
  DVO_CUDA(ctx, cudaMemcpyAsync(&ws.h_active[0], flag, sizeof(int), cudaMemcpyDeviceToHost, st));
  DVO_CUDA(ctx, cudaGetLastError());
  PairState* hs = nullptr;
  if ((rc = ensure_stage(ctx, 0, sizeof(PairState) + 64))) return rc;
  hs = (PairState*)ctx->h_stage;
  DVO_CUDA(ctx, cudaMemcpyAsync(hs, ws.d_state, sizeof(PairState), cudaMemcpyDeviceToHost, st));
  DVO_CUDA(ctx, cudaStreamSynchronize(st));
  ctx->pending_level_flags = 1;
  if ((rc = check_level_flags(ctx))) return rc;
  if (count) *count = hs->n;
  if (precision_out) std::memcpy(precision_out, hs->precision, sizeof(float) * 4);
  if (ll_out) *ll_out = hs->ll;
  if (A_out) std::memcpy(A_out, hs->A, sizeof(double) * 36);
  if (b_out) std::memcpy(b_out, hs->b, sizeof(double) * 6);
  if (planes7) {
    // {ei, ez, gx, gy, hx, hy, z_ref}; invalid -> NaN in every plane
    DVO_CUDA(ctx, cudaMemcpy(planes7, ws.d_dump, sizeof(float) * 7 * (size_t)L.n, cudaMemcpyDeviceToHost));
    ctx->d2h_bytes += sizeof(float) * 7 * (size_t)L.n;
  }
  return 0;
}

}  // namespace dvo_b200
