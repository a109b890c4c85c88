// acransac_fused.cu -- the whole a-contrario RANSAC of one image pair inside ONE persistent CTA.
// COMPILED WITH --fmad=false (regard3d_b200/build.py), like acransac_kernels.cu.
//
// Replaces the per-pair body of ImageCollectionGeometricFilter::Robust_model_estimation(GeometricFilter_{F,E,H}Matrix_AC
// (4.0, 2048), ...) (src/R3DComputeMatches.cpp:2099-2115, :2169-2171, :2215-2219); upstream semantics: SURVEY.md A.4-A.6.
//
// Round 1 ran ACRANSAC as ~25 host<->device rounds (samples drawn on the host, two kernels, state machine replayed on
// the host): 54 % of the filter's time was host work and every hypothesis paid a shared-memory sort of its residuals.
// Here a CTA owns a pair from the first sample to the final inlier list:
//   * the sample stream is drawn on the device (acransac_rng.cuh: mt19937 + libstdc++'s uniform_int_distribution,
//     self-checked against the host's <random> at r3d_create());
//   * kBatch iterations are drawn / solved / scored speculatively, then the state machine is replayed in order; an
//     improving model ("event") replaces the sampling pool and discards the speculative tail (generator rewound);
//   * scoring is two-tier.  Tier 1, one warp per model: M residuals -> count of those <= the precision bound and a
//     geometric histogram of them (exponent + 5 mantissa bits); with e_(k) >= the lower edge of the bin that holds
//     rank k, LB = min_k NFA_k(lower edge) is a rigorous lower bound of the model's best NFA (every operation of
//     the NFA formula is monotone under rounding).  Tier 2, the whole CTA, only when LB < minNFA (the model may
//     improve on the best so far): compaction + bitonic sort + the exact NFA scan of round 1.  After the first few
//     models of a pair almost every hypothesis is settled by tier 1 -- no sort.
// The decisions taken are exactly those of the sequential algorithm: tier 1 only skips work whose outcome
// (nfa >= minNFA: "not better") is already certain.
#include "acransac_device.cuh"
#include "acransac_rng.cuh"

#include <random>
#include <type_traits>

namespace r3d {

namespace {

constexpr int kFThreads = 256;
constexpr int kFWarps = kFThreads / 32;
constexpr int kBatch = 24;            // most iterations drawn, solved and tier-1-scored ahead (the batch grows with the
                                      // number of iterations since the last pool replacement: 4, 5, ... kBatch)
constexpr double kApproxRel = 1e-9;   // relative accuracy of the tier-1 residuals (see approx_error)
constexpr int kBins = 1024;           // tier-1 histogram: binades split in 32 (exponent + 5 mantissa bits)
constexpr int kHistStride = kBins + kBins / 32;  // bin b lives at b + (b >> 5): a lane that owns 32 consecutive bins
                                                 // walks them without bank conflicts
__device__ __forceinline__ uint32_t bin_slot(uint32_t b) { return b + (b >> 5); }
constexpr int kBinShift = 52 - 5;

template <int MODEL>
struct BatchBuf {                     // one speculative batch of RANSAC iterations
  Mt19937 snap;                       // generator state before the batch's first draw
  double models[kBatch][ac_max_models(MODEL)][9];
  double lb[kBatch][ac_max_models(MODEL)];
  uint32_t cnt[kBatch][ac_max_models(MODEL)];      // residuals that may be <= the bound (upper count)
  uint32_t cnt_lo[kBatch][ac_max_models(MODEL)];   // residuals that certainly are (lower count)
  uint32_t nm[kBatch];
  uint32_t sample[kBatch][8];
  uint32_t used[kBatch];              // generator outputs consumed up to and including iteration b of the batch
  uint32_t B;                         // iterations in the batch
};

template <int MODEL>
struct FusedSmem {                    // fixed part of the shared memory (the sort / histogram region follows)
  Mt19937 rng;
  BatchBuf<MODEL> q[2];               // the batch being scored / replayed and the one warp 0 prepares meanwhile
  double la[kHistStride];             // logalpha of every bin's lower edge (at bin_slot(b))
  double bestF[9];
  double s_nfa[kFWarps];
  uint32_t s_k[kFWarps];
  uint32_t gcnt[2 * (kFWarps - 1)];   // per model of the tier-1 group: upper / lower count
  uint32_t s_count;
  uint32_t work;
};

template <int MODEL>
__device__ __forceinline__ double model_error(const double* F, const double2 a, const double2 b) {
  return MODEL == 0 ? sym_epi_error(F, a.x, a.y, b.x, b.y)
                    : MODEL == 1 ? asym_error(F, a.x, a.y, b.x, b.y) : epi_dist_error(F, a.x, a.y, b.x, b.y);
}

// ---- tier-1 residuals: fused multiply-adds, one reciprocal instead of IEEE divisions ---------------------------
// Tier 1 only BOUNDS the exact computation, so it need not reproduce the reference's rounding.  approx_bounds()
// returns an interval [*lo, *hi] that contains the residual the tier-2 / CPU code computes (the same rational
// function of the same inputs, rounded differently):
//   * the cancelling term (x2^T F x1 for the epipolar errors, x2 - H x1 for the transfer error) carries an ABSOLUTE
//     error eta = 64 ulp x (largest model entry) x (2 R + 1)^2, R = the pair's largest |coordinate|: both evaluations
//     stay within that of the exact value (<= 12 roundings of terms bounded by that magnitude);
//   * everything else is cancellation-free: relative error <= kApproxRel (2^-53 per operation; the reciprocal is
//     rcp.approx + one Newton step, ~2^-40).
// Degenerate inputs (reciprocal argument outside [1e-280, 1e280], NaN) give [0, +inf): "may or may not be an inlier".
__device__ __forceinline__ double rcp_fast(double x, bool* ok) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = __fma_rn(r, __fma_rn(-x, r, 1.0), r);
  const double ax = fabs(x);
  if (!(ax > 1e-280 && ax < 1e280)) *ok = false;
  return r;
}

template <int MODEL>
__device__ __forceinline__ void approx_bounds(const double* F, double eta, const double2 a, const double2 b, double* lo, double* hi) {
  bool ok = true;
  double l, h;
  if (MODEL == 1) {  // asymmetric transfer error of a homography: |x2 - (H x1)_xy / (H x1)_w|^2
    const double hx = __fma_rn(F[0], a.x, __fma_rn(F[1], a.y, F[2]));
    const double hy = __fma_rn(F[3], a.x, __fma_rn(F[4], a.y, F[5]));
    const double hw = __fma_rn(F[6], a.x, __fma_rn(F[7], a.y, F[8]));
    const double iw = rcp_fast(hw, &ok);
    const double ex = fabs(__fma_rn(-hx, iw, b.x)), ey = fabs(__fma_rn(-hy, iw, b.y));
    // eta bounds the absolute error of hx, hy, hw; propagated through the quotient (|hw| >> eta or the point is flagged)
    const double aiw = fabs(iw);
    const double q = eta * aiw;                                  // relative error of hw
    if (!(q < 1e-3)) ok = false;
    const double dx = eta * aiw + fabs(hx * iw) * q * 1.01 + 4e-16 * (fabs(b.x) + fabs(hx * iw));
    const double dy = eta * aiw + fabs(hy * iw) * q * 1.01 + 4e-16 * (fabs(b.y) + fabs(hy * iw));
    const double lx = fmax(ex - dx, 0.0), ly = fmax(ey - dy, 0.0), ux = ex + dx, uy = ey + dy;
    l = __fma_rn(lx, lx, ly * ly) * (1.0 - kApproxRel);
    h = __fma_rn(ux, ux, uy * uy) * (1.0 + kApproxRel);
  } else {
    const double Fx0 = __fma_rn(F[0], a.x, __fma_rn(F[1], a.y, F[2]));
    const double Fx1 = __fma_rn(F[3], a.x, __fma_rn(F[4], a.y, F[5]));
    const double Fx2 = __fma_rn(F[6], a.x, __fma_rn(F[7], a.y, F[8]));
    const double y = fabs(__fma_rn(b.x, Fx0, __fma_rn(b.y, Fx1, Fx2)));
    const double A = __fma_rn(Fx0, Fx0, Fx1 * Fx1);
    double K;  // the cancellation-free factor
    if (MODEL == 2) {
      K = rcp_fast(A, &ok);                                      // one-sided epipolar distance: y^2 / A
    } else {
      const double Fty0 = __fma_rn(F[0], b.x, __fma_rn(F[3], b.y, F[6]));
      const double Fty1 = __fma_rn(F[1], b.x, __fma_rn(F[4], b.y, F[7]));
      const double B = __fma_rn(Fty0, Fty0, Fty1 * Fty1);
      K = 0.25 * (A + B) * rcp_fast(A * B, &ok);                 // (1/A + 1/B) / 4
    }
    const double yl = fmax(y - eta, 0.0), yh = y + eta;
    l = yl * yl * K * (1.0 - kApproxRel);
    h = yh * yh * K * (1.0 + kApproxRel);
  }
  if (!ok || !(l <= h)) {  // also catches NaN
    l = 0.0;
    h = DBL_MAX * 2.0;
  }
  *lo = l;
  *hi = h;
}

}  // namespace

size_t acransac_fused_smem_bytes(int model, uint32_t cap, bool huge) {
  const size_t fixed = model == 0 ? sizeof(FusedSmem<0>) : (model == 1 ? sizeof(FusedSmem<1>) : sizeof(FusedSmem<2>));
  const size_t hist = (size_t)kFWarps * kBins * sizeof(uint32_t);
  const size_t sortb = huge ? 0 : (size_t)cap * 8;  // residual values; the index array of the inlier sort is global
  const size_t pool = huge ? 0 : (size_t)cap * 2;   // 16-bit pool entries
  return ((fixed + 15) & ~(size_t)15) + std::max(hist, sortb) + pool;
}

// exact count of the residuals <= the precision bound (the classic-RANSAC phase needs it exactly; tier 1 brackets it)
template <int MODEL>
__device__ uint32_t exact_count(const AcPair& pr, const double2* __restrict__ p1, const double2* __restrict__ p2, const double* Fm,
                                uint32_t* s_count) {
  if (threadIdx.x == 0) *s_count = 0;
  __syncthreads();
  uint32_t c = 0;
  for (uint32_t i = threadIdx.x; i < pr.M; i += blockDim.x)
    if (model_error<MODEL>(Fm, p1[i], p2[i]) <= pr.max_thr) ++c;
  for (int o = 16; o >= 1; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31u) == 0 && c) atomicAdd(s_count, c);
  __syncthreads();
  c = *s_count;
  __syncthreads();
  return c;
}

// One persistent CTA per image pair.  order[]: the pairs of this launch (one size class), largest first.
// Shared memory: the fixed block, then one region used by tier 1 (a histogram per warp) and by tier 2 (the residual
// values being sorted), then the sampling pool (16-bit entries).  g_si: `cap` uint32 per CTA, the index array of the
// (rare) inlier sorts.  HUGE: values and pool too live in global scratch (g_se / g_pool) -- the slow-but-correct path
// for pairs with more putative matches than shared memory can sort.
template <int MODEL, bool HUGE>
__global__ void __launch_bounds__(kFThreads, MODEL == 2 ? 1 : 2) k_acransac_fused(
    const AcPair* __restrict__ pairs, const uint32_t* __restrict__ order, uint32_t n_order, uint32_t* __restrict__ work_counter,
    const double2* __restrict__ x1, const double2* __restrict__ x2, const float* __restrict__ logc_n,
    const float* __restrict__ logc_k, uint32_t cap, uint32_t max_iter, double* __restrict__ g_se, uint32_t* __restrict__ g_si,
    uint32_t* __restrict__ g_pool, const uint2* __restrict__ matches, uint2* __restrict__ out_matches,
    AcFusedOut* __restrict__ out, double* __restrict__ out_F) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr uint32_t NS = ac_min_samples(MODEL), MAXM = ac_max_models(MODEL);
  typedef typename std::conditional<HUGE, uint32_t, uint16_t>::type PoolT;
  const double mult_error = MODEL == 1 ? 1.0 : 0.5;
  FusedSmem<MODEL>& S = *reinterpret_cast<FusedSmem<MODEL>*>(smem_raw);
  unsigned char* region = smem_raw + ((sizeof(FusedSmem<MODEL>) + 15) & ~(size_t)15);
  uint32_t* hist_all = reinterpret_cast<uint32_t*>(region);                 // tier 1: kFWarps x kBins
  const size_t hist_bytes = (size_t)kFWarps * kBins * 4;
  const size_t region_bytes = HUGE ? hist_bytes : ((size_t)cap * 8 > hist_bytes ? (size_t)cap * 8 : hist_bytes);
  double* se = HUGE ? g_se + (size_t)blockIdx.x * cap : reinterpret_cast<double*>(region);   // tier 2 (aliases hist)
  uint32_t* si = g_si + (size_t)blockIdx.x * cap;
  PoolT* pool = HUGE ? reinterpret_cast<PoolT*>(g_pool + (size_t)blockIdx.x * cap) : reinterpret_cast<PoolT*>(region + region_bytes);
  const uint32_t tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;

  for (;;) {
    __syncthreads();
    if (tid == 0) S.work = atomicAdd(work_counter, 1u);
    __syncthreads();
    const uint32_t wk = S.work;
    if (wk >= n_order) break;
    const uint32_t pair_id = order[wk];
    const AcPair pr = pairs[pair_id];
    const uint32_t M = pr.M;
    const float* lcn = logc_n + pr.tbl_ofs;
    const double2* p1 = x1 + pr.pt_ofs;
    const double2* p2 = x2 + pr.pt_ofs;

    // ---- per-pair set-up: sampling pool, generator, bin edges, coordinate bound --------------------------------
    double rmax = 0.0;
    for (uint32_t i = tid; i < M; i += kFThreads) {
      pool[i] = (PoolT)i;
      const double2 a = p1[i], b = p2[i];
      rmax = fmax(rmax, fmax(fmax(fabs(a.x), fabs(a.y)), fmax(fabs(b.x), fabs(b.y))));
    }
    for (int o = 16; o >= 1; o >>= 1) rmax = fmax(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
    if (lane == 0) S.s_nfa[warp] = rmax;
    // bin(e) = clamp((bits(e) >> kBinShift) - bin_base, 0, kBins - 1): the precision bound falls in the top bin
    const long long thr_key = __double_as_longlong(pr.max_thr) >> kBinShift;
    const long long bin_base = thr_key - (kBins - 1);
    for (uint32_t b = tid; b < (uint32_t)kBins; b += kFThreads) {
      const long long kb = bin_base + (long long)b;
      const double lo = (b == 0 || kb <= 0) ? 0.0 : __longlong_as_double(kb << kBinShift);
      S.la[bin_slot(b)] = pr.logalpha0 + mult_error * dm::log10_det(lo + (double)FLT_EPSILON);
    }
    if (tid == 0) mt_seed(S.rng);
    __syncthreads();
    for (uint32_t wv = 0; wv < (uint32_t)kFWarps; ++wv) rmax = fmax(rmax, S.s_nfa[wv]);
    const double coord_span = (2.0 * rmax + 1.0) * (2.0 * rmax + 1.0);
    // ACRANSAC state, replicated in the registers of every thread (updated identically from shared data)
    uint32_t iter = 0, nIterReserve = max_iter / 10, nIter = max_iter - nIterReserve;
    bool ac_mode = !(pr.max_thr < DBL_MAX);  // bACRansacMode = (precision == infinity)
    double minNFA = DBL_MAX * 2.0, errorMax = DBL_MAX * 2.0;
    uint32_t best_k = 0, pool_size = M, since_event = 0;
    bool have_inliers = false;
    uint32_t n_exact = 0, n_models = 0, n_events = 0;
    __syncthreads();

    // ---- producer (warp 0): draw the next `Bq` samples and solve them into batch buffer q -------------------
    // UniformSample = a partial Fisher-Yates on the pool, sequential by nature (lane 0); the minimal solvers of the
    // batch then run one per lane.  Called either ahead of time (while warps 1.. score the previous batch) or, after a
    // pool replacement invalidated that speculation, with the whole CTA waiting.
    auto produce = [&](BatchBuf<MODEL>& Q, uint32_t Bq, uint32_t psize) {
      {
        uint32_t* dst = reinterpret_cast<uint32_t*>(&Q.snap);
        const uint32_t* src = reinterpret_cast<const uint32_t*>(&S.rng);
        for (uint32_t i = lane; i < sizeof(Mt19937) / 4; i += 32) dst[i] = src[i];
      }
      __syncwarp();
      if (lane == 0) {
        uint32_t used = 0;
        const uint32_t last_idx = psize - 1;
        for (uint32_t b = 0; b < Bq; ++b) {
          for (uint32_t i = 0; i < NS; ++i) {
            const uint32_t r = uniform_u32(S.rng, i, last_idx, &used);
            const PoolT t = pool[i]; pool[i] = pool[r]; pool[r] = t;
          }
          for (uint32_t i = 0; i < NS; ++i) Q.sample[b][i] = pool[i];
          Q.used[b] = used;
        }
        Q.B = Bq;
      }
      __syncwarp();
      if (lane < Bq) {
        double models[9 * MAXM];
        int nm;
        if (MODEL == 2) {
          double b1[15], b2[15], Es[90];
          for (int t = 0; t < 5; ++t) {
            const double2 a = p1[Q.sample[lane][t]];
            const double2 b = p2[Q.sample[lane][t]];
            bearing(pr.K, a.x, a.y, b1 + 3 * t);
            bearing(pr.K + 3, b.x, b.y, b2 + 3 * t);
          }
          nm = fp::five_point(b1, b2, Es);
          for (int mi = 0; mi < nm; ++mi) fundamental_from_essential(Es + 9 * mi, pr.K, pr.K + 3, models + 9 * mi);
        } else {
          double s1[14], s2[14];
          for (uint32_t t = 0; t < NS; ++t) {
            const double2 a = p1[Q.sample[lane][t]];
            const double2 b = p2[Q.sample[lane][t]];
            s1[2 * t] = a.x; s1[2 * t + 1] = a.y;
            s2[2 * t] = b.x; s2[2 * t + 1] = b.y;
          }
          nm = MODEL == 0 ? seven_point(s1, s2, models) : four_point(s1, s2, models);
        }
        Q.nm[lane] = (uint32_t)nm;
        for (int mi = 0; mi < nm; ++mi)
          for (int t = 0; t < 9; ++t) Q.models[lane][mi][t] = models[9 * mi + t];
      }
      __syncwarp();
    };
    // speculation depth: short right after a pool replacement (improving models come in bursts), longer later
    auto batch_size = [&](uint32_t since, uint32_t remaining) { return min(min((uint32_t)kBatch, 4u + since), remaining); };

    uint32_t cur = 0;
    bool have_cur = false;  // q[cur] holds drawn + solved iterations that continue the sequence at `iter`
    while (iter < nIter) {
      if (!have_cur) {  // (re)start the pipeline: nothing was prepared ahead, or a pool replacement discarded it
        if (warp == 0) produce(S.q[cur], batch_size(since_event, nIter - iter), pool_size);
        __syncthreads();
      }
      BatchBuf<MODEL>& Q = S.q[cur];
      const uint32_t B = Q.B;
      // ---- phase A: warps 1.. score batch `cur` (tier 1); warp 0 prepares the batch after it, assuming that the
      //      replay of `cur` will not replace the pool (if it does, the work is thrown away and the generator rewound)
      const uint32_t ahead = nIter - iter > B ? batch_size(since_event + B, nIter - iter - B) : 0u;
      if (warp == 0) {
        if (ahead) produce(S.q[cur ^ 1u], ahead, pool_size);
      } else {
        // Tier 1, points outer / models inner: the consumer warps split the pair's points, each point is loaded ONCE
        // and scored against a group of kGroup models (their matrices are broadcast reads from shared memory), so the
        // loop is bound by the fp64 pipe instead of by the latency of re-streaming the points for every model.
        constexpr uint32_t kGroup = kFWarps - 1;                 // models per group = consumer warps (one LB scan each)
        constexpr uint32_t kConsumers = (kFWarps - 1) * 32;
        const uint32_t cw = warp - 1, ctid = tid - 32;
        // the batch's models as a flat list (iteration b, model mi) -- every consumer thread walks it identically
        uint32_t n_models_batch = 0;
        for (uint32_t b = 0; b < B; ++b) n_models_batch += Q.nm[b];
        // the histograms alias the tier-2 sort buffer: clear them once per batch, every scan clears its own afterwards
        for (uint32_t i = ctid; i < kGroup * (uint32_t)kHistStride; i += kConsumers) hist_all[i] = 0;
        if (ctid < 2 * kGroup) S.gcnt[ctid] = 0;
        asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory");
        for (uint32_t g0 = 0; g0 < n_models_batch; g0 += kGroup) {
          const uint32_t gn = min(kGroup, n_models_batch - g0);
          // locate the group's models
          uint32_t gb[kGroup], gm[kGroup];
          {
            uint32_t seen = 0, k = 0;
            for (uint32_t b = 0; b < B && k < gn; ++b) {
              const uint32_t nmb = Q.nm[b];
              if (seen + nmb <= g0) { seen += nmb; continue; }
              for (uint32_t mi = (g0 > seen ? g0 - seen : 0u); mi < nmb && k < gn; ++mi) { gb[k] = b; gm[k] = mi; ++k; }
              seen += nmb;
            }
          }
          double eta[kGroup];
          for (uint32_t k = 0; k < gn; ++k) {
            const double* Fm = &Q.models[gb[k]][gm[k]][0];
            double fmax_abs = 0.0;
            for (int t = 0; t < 9; ++t) fmax_abs = fmax(fmax_abs, fabs(Fm[t]));
            eta[k] = 7.2e-15 * fmax_abs * coord_span;            // 64 ulp x the largest term of x2^T F x1 (or H x1)
          }
          uint32_t c_hi[kGroup], c_lo[kGroup];
          for (uint32_t k = 0; k < kGroup; ++k) { c_hi[k] = 0; c_lo[k] = 0; }
          for (uint32_t i = ctid; i < M; i += kConsumers) {
            const double2 a = p1[i], b2 = p2[i];
#pragma unroll
            for (uint32_t k = 0; k < kGroup; ++k) {
              if (k >= gn) break;
              double elo, ehi;
              approx_bounds<MODEL>(&Q.models[gb[k]][gm[k]][0], eta[k], a, b2, &elo, &ehi);
              if (elo <= pr.max_thr) {  // may be an inlier of the precision bound
                long long bin = (__double_as_longlong(elo) >> kBinShift) - bin_base;
                bin = bin < 0 ? 0 : (bin > kBins - 1 ? kBins - 1 : bin);
                atomicAdd(&hist_all[k * kHistStride + bin_slot((uint32_t)bin)], 1u);
                ++c_hi[k];
                if (ehi <= pr.max_thr) ++c_lo[k];
              }
            }
          }
#pragma unroll
          for (uint32_t k = 0; k < kGroup; ++k) {
            if (k >= gn) break;
            uint32_t h = c_hi[k], l = c_lo[k];
            for (int o = 16; o >= 1; o >>= 1) {
              h += __shfl_xor_sync(0xffffffffu, h, o);
              l += __shfl_xor_sync(0xffffffffu, l, o);
            }
            if (lane == 0) { atomicAdd(&S.gcnt[2 * k], h); atomicAdd(&S.gcnt[2 * k + 1], l); }
          }
          asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory");
          if (cw < gn) {  // one warp per model of the group: lower bound of its best NFA from its histogram
            uint32_t* hist = hist_all + (size_t)cw * kHistStride + lane * 33u;  // this lane's 32 consecutive bins
            const double* lab = S.la + lane * 33u;
            const uint32_t ch = S.gcnt[2 * cw], cl = S.gcnt[2 * cw + 1];
            double lbv = DBL_MAX * 2.0;
            if (ch > NS) {
              uint32_t tot = 0;
#pragma unroll 8
              for (uint32_t j = 0; j < 32; ++j) tot += hist[j];
              uint32_t incl = tot;
              for (int o = 1; o < 32; o <<= 1) {
                const uint32_t u = __shfl_up_sync(0xffffffffu, incl, o);
                if ((int)lane >= o) incl += u;
              }
              uint32_t run = incl - tot;  // lower bounds in the bins before this lane's
              // Ranks (run, run + v] live in a bin with lower edge e_b.  With e_(k) the true k-th smallest residual: at
              // least k of the lower bounds are <= e_(k), so the k-th smallest LOWER BOUND is <= e_(k), hence
              //   NFA_k >= g_b(k) = loge0 + la[b] (k - NS) + logc_n[k] + logc_k[k];
              // extra ranks (c_hi >= c) only lower the minimum.  log10 C(n, k) and log10 C(k, NS) are concave in k and
              // the rest of g_b is linear, so over the ranks of one bin g_b is smallest at one of the two end ranks --
              // for the exact binomials.  The float tables differ from them by at most tbl_err (accumulated by
              // k_ac_tables while it sums), which the bound gives back twice over.
              for (uint32_t j = 0; j < 32; ++j) {
                const uint32_t v = hist[j];
                if (v) {
                  const uint32_t ka = max(run + 1, NS + 1), kb = run + v;
                  if (ka <= kb) {
                    const double la = lab[j];
                    const double ga = la * (double)(ka - NS) + ((double)lcn[ka] + (double)logc_k[ka]);
                    const double gb2 = la * (double)(kb - NS) + ((double)lcn[kb] + (double)logc_k[kb]);
                    lbv = fmin(lbv, fmin(ga, gb2));
                  }
                  run += v;
                  hist[j] = 0;
                }
              }
              for (int o = 16; o >= 1; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, lbv, o);
                lbv = ov < lbv ? ov : lbv;
              }
              lbv += pr.loge0;
              // table error (see above), then a few ulp for the (unproven) monotonicity of log10_det at its
              // range-reduction seams
              lbv -= 2.0 * (double)lcn[M + 1] + 1e-4;
              lbv = lbv - 1e-9 * (1.0 + fabs(lbv));
            } else {
#pragma unroll 8
              for (uint32_t j = 0; j < 32; ++j) hist[j] = 0;
            }
            __syncwarp();  // every lane has read the group counters before lane 0 clears them (racecheck: intra-warp hazard)
            if (lane == 0) {
              Q.cnt[gb[cw]][gm[cw]] = ch; Q.cnt_lo[gb[cw]][gm[cw]] = cl; Q.lb[gb[cw]][gm[cw]] = lbv;
              S.gcnt[2 * cw] = 0; S.gcnt[2 * cw + 1] = 0;
            }
          }
          asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory");  // cleared histograms and counters: next group
        }
      }
      __syncthreads();
      // ---- phase B: replay the ACRANSAC state machine over the batch (uniform control flow) ---------------------
      uint32_t consumed = B;
      bool event = false;
      for (uint32_t it = 0; it < B; ++it) {
        bool better = false;
        const uint32_t nm = Q.nm[it];
        for (uint32_t mi = 0; mi < nm; ++mi) {
          ++n_models;
          double Fm[9];
          if (!ac_mode) {  // classic-RANSAC phase: the exact number of residuals within the bound decides the switch
            uint32_t c = Q.cnt_lo[it][mi];
            if (c != Q.cnt[it][mi] && (double)c <= 2.5 * NS && (double)Q.cnt[it][mi] > 2.5 * NS) {
              for (int t = 0; t < 9; ++t) Fm[t] = Q.models[it][mi][t];
              c = exact_count<MODEL>(pr, p1, p2, Fm, &S.s_count);
            }
            if ((double)c > 2.5 * NS) ac_mode = true;
          }
          if (ac_mode && Q.lb[it][mi] < minNFA) {  // the model may improve on the best one: exact NFA (tier 2)
            ++n_exact;
            for (int t = 0; t < 9; ++t) Fm[t] = Q.models[it][mi][t];
            const uint32_t c = residuals_sorted<MODEL, false>(pr, x1, x2, Fm, se, si, cap, &S.s_count);
            const NfaBest r = nfa_scan_sorted<MODEL>(pr, se, c, lcn, logc_k, S.s_nfa, S.s_k);
            if (r.nfa < minNFA) {
              better = true;
              minNFA = r.nfa;
              errorMax = r.err;
              best_k = r.k;
              have_inliers = true;
              if (tid < 9) S.bestF[tid] = Fm[tid];
            }
          }
        }
        const uint32_t iter_abs = iter + it;
        if ((better && minNFA < 0) || (iter_abs + 1 == nIter && nIterReserve)) {
          if (!have_inliers) {
            ++nIter;
            --nIterReserve;
          } else {
            event = true;
            consumed = it + 1;
            break;
          }
        }
      }
      iter += consumed;
      since_event = event ? 0u : since_event + consumed;
      // ---- pool replacement: draw the next samples among the best model's inliers; whatever was drawn after
      //      iteration `consumed - 1` (the tail of this batch, the batch prepared ahead) never happened ----------------
      if (event) {
        ++n_events;
        __syncthreads();  // bestF
        double Fm[9];
        for (int t = 0; t < 9; ++t) Fm[t] = S.bestF[t];
        const uint32_t c = residuals_sorted<MODEL, true>(pr, x1, x2, Fm, se, si, cap, &S.s_count);
        pool_size = best_k < c ? best_k : c;
        for (uint32_t i = tid; i < pool_size; i += kFThreads) pool[i] = (PoolT)si[i];
        if (nIterReserve) {
          nIter = iter + nIterReserve;
          nIterReserve = 0;
        }
        {  // rewind the generator to the end of iteration `consumed - 1`
          uint32_t* dst = reinterpret_cast<uint32_t*>(&S.rng);
          const uint32_t* src = reinterpret_cast<const uint32_t*>(&Q.snap);
          for (uint32_t i = tid; i < sizeof(Mt19937) / 4; i += kFThreads) dst[i] = src[i];
          __syncthreads();
          if (tid == 0)
            for (uint32_t u = 0; u < Q.used[consumed - 1]; ++u) (void)mt_next(S.rng);
        }
        __syncthreads();
        have_cur = false;
      } else {
        have_cur = ahead != 0;  // the batch prepared ahead continues the sequence
        cur ^= 1u;
        __syncthreads();        // warp 0's batch is complete (phase A barrier) and nobody reads the old one any more
      }
    }

    // ---- result: "if (minNFA >= 0) vec_inliers.clear()"; the inlier list in residual order ------------------
    uint32_t n_out = 0;
    if (have_inliers && minNFA < 0) {
      __syncthreads();
      double Fm[9];
      for (int t = 0; t < 9; ++t) Fm[t] = S.bestF[t];
      const uint32_t c = residuals_sorted<MODEL, true>(pr, x1, x2, Fm, se, si, cap, &S.s_count);
      n_out = best_k < c ? best_k : c;
      for (uint32_t i = tid; i < n_out; i += kFThreads) out_matches[pr.pt_ofs + i] = matches[pr.pt_ofs + si[i]];
    }
    // the winning model (relative poses; nullptr for the filter): F = K2^-T E K1^-1 of the best 5-point E, zeros
    // when no model was kept
    if constexpr (MODEL == 2) {
      if (out_F != nullptr && tid < 9) out_F[(size_t)pair_id * 9 + tid] = have_inliers ? S.bestF[tid] : 0.0;
    }
    if (tid == 0) {
      AcFusedOut o;
      o.minNFA = minNFA;
      o.errorMax = errorMax;
      o.n_inliers = n_out;
      o.iterations = iter;
      o.exact_scores = n_exact;
      o.models = n_models;
      o.events = n_events;
      o.pad_ = 0;
      out[pair_id] = o;
    }
  }
}

template <int MODEL, bool HUGE>
static int launch_fused_t(r3d_ctx* ctx, DeviceWorker& w, const AcPair* pairs, const uint32_t* order, uint32_t n_order,
                          uint32_t* work_counter, const double2* x1, const double2* x2, const float* logc_n, const float* logc_k,
                          uint32_t cap, uint32_t max_iter, double* g_se, uint32_t* g_si, uint32_t* g_pool, const uint2* matches,
                          uint2* out_matches, AcFusedOut* out, double* out_F, uint32_t grid) {
  const size_t smem = acransac_fused_smem_bytes(MODEL, cap, HUGE);
  R3D_CUDA_TRY(ctx, cudaFuncSetAttribute(k_acransac_fused<MODEL, HUGE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_acransac_fused<MODEL, HUGE><<<grid, kFThreads, smem, w.stream>>>(pairs, order, n_order, work_counter, x1, x2, logc_n, logc_k,
                                                                      cap, max_iter, g_se, g_si, g_pool, matches, out_matches, out, out_F);
  R3D_CUDA_TRY(ctx, cudaGetLastError());
  return R3D_OK;
}

int acransac_fused_ctas_per_sm(int model, uint32_t cap, bool huge) {
  const size_t smem = acransac_fused_smem_bytes(model, cap, huge);
  const size_t per_sm = 227 * 1024;
  int n = (int)(per_sm / (smem + 1024));
  if (n < 1) n = 1;
  const int by_regs = model == 2 ? 1 : 2;  // __launch_bounds__ of the kernel
  return n < by_regs ? n : by_regs;
}

int launch_acransac_fused(r3d_ctx* ctx, DeviceWorker& w, int model, bool huge, const AcPair* pairs, const uint32_t* order,
                          uint32_t n_order, uint32_t* work_counter, const double2* x1, const double2* x2, const float* logc_n,
                          const float* logc_k, uint32_t cap, uint32_t max_iter, double* g_se, uint32_t* g_si, uint32_t* g_pool,
                          const uint2* matches, uint2* out_matches, AcFusedOut* out, double* out_F, uint32_t grid) {
  if (!n_order) return R3D_OK;
  if (out_F != nullptr && model != 2) return fail(ctx, R3D_ERR_INVALID, "launch_acransac_fused: the winning-model output needs the E model");
#define R3D_FUSED_CASE(MD, HG)                                                                                          \
  if (model == MD && huge == HG)                                                                                        \
    return launch_fused_t<MD, HG>(ctx, w, pairs, order, n_order, work_counter, x1, x2, logc_n, logc_k, cap, max_iter, \
                                  g_se, g_si, g_pool, matches, out_matches, out, out_F, grid);
  R3D_FUSED_CASE(0, false) R3D_FUSED_CASE(0, true) R3D_FUSED_CASE(1, false) R3D_FUSED_CASE(1, true)
  R3D_FUSED_CASE(2, false) R3D_FUSED_CASE(2, true)
#undef R3D_FUSED_CASE
  return fail(ctx, R3D_ERR_INVALID, "launch_acransac_fused: unknown model");
}

// ---- the restated sample stream against this process's <random> -------------------------------------------------
bool rng_selftest() {
  static int cached = -1;
  if (cached >= 0) return cached == 1;
  std::mt19937 ref;
  Mt19937* mine = new Mt19937;
  mt_seed(*mine);
  bool ok = true;
  // pool sizes as ACRANSAC sees them, tiny and huge ranges, the full range
  const uint32_t sizes[] = {8, 9, 17, 100, 1000, 4097, 65536, 1000003, 0x7fffffffu, 0xfffffff0u};
  for (int round = 0; round < 400 && ok; ++round) {
    for (uint32_t sz : sizes) {
      for (uint32_t i = 0; i < 7 && i < sz; ++i) {
        std::uniform_int_distribution<uint32_t> d(i, sz - 1);
        uint32_t used = 0;
        if (d(ref) != uniform_u32(*mine, i, sz - 1, &used)) { ok = false; break; }
      }
      if (!ok) break;
    }
    std::uniform_int_distribution<uint32_t> full(0u, 0xffffffffu);
    uint32_t used = 0;
    if (ok && full(ref) != uniform_u32(*mine, 0u, 0xffffffffu, &used)) ok = false;
  }
  // both generators must also sit at the same position afterwards
  if (ok) {
    uint32_t a = (uint32_t)ref();
    if (a != mt_next(*mine)) ok = false;
  }
  delete mine;
  cached = ok ? 1 : 0;
  return ok;
}

}  // namespace r3d
