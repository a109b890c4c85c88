// acransac_host.cu -- host orchestration of the AC-RANSAC fundamental filter (r3d_filter_pairs).
//
// Replaces ImageCollectionGeometricFilter::Robust_model_estimation(GeometricFilter_FMatrix_AC(4.0,
// 2048), putatives, false) + Get_geometric_matches() (src/R3DComputeMatches.cpp:2099-2115).
//
// ACRANSAC (SURVEY.md A.5) is sequential per pair: the sampling pool shrinks to the inlier set after
// every improving model.  Between two pool replacements, however, the sample sequence depends only
// on (RNG state, pool) -- not on the data.  So every active pair draws a batch of samples ahead on
// the host (with the very std::mt19937 / uniform_int_distribution code of the CPU path -- the
// distribution algorithm is implementation-defined, never re-implemented on the device), ALL
// pairs' hypotheses are solved and scored in two launches, and a per-pair sequential scan replays
// the state machine, discarding the speculative tail after a pool replacement.
#include "acransac.cuh"
#include "acransac_rng.cuh"
#include "detmath.cuh"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <memory>
#include <numeric>
#include <random>

namespace r3d {

namespace {

double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

struct PairState {
  uint32_t src;  // index in the putative map
  uint32_t I, J, M;
  uint32_t pt_ofs, tbl_ofs;
  // ACRANSAC state
  std::vector<uint32_t> vec_index;
  std::unique_ptr<std::mt19937[]> rngs;  // [0] generator (default seed), [1] its snapshot: host-round path only (5 KB)
  uint32_t iter = 0, nIter = 0, nIterReserve = 0;
  bool ac_mode = false;
  double minNFA = std::numeric_limits<double>::infinity();
  double errorMax = std::numeric_limits<double>::infinity();
  bool have_inliers = false;       // vec_inliers non-empty in the reference's sense
  std::vector<uint32_t> inliers;   // host copy of the best model's inlier list (sorted by residual)
  uint32_t best_k = 0;
  // per-round bookkeeping
  uint32_t hyp_ofs = 0, hyp_n = 0;
  std::vector<uint32_t> swap_log;  // 7 swap targets per drawn iteration (undo log of the partial Fisher-Yates)
  uint32_t since_event = 0;
  bool best_changed = false, event = false;
  uint32_t best_hyp = 0, best_model = 0;
  bool done = false;
};

// rand_sampling.hpp UniformSample(num_samples, rng, &vec_index, &sample)
inline void uniform_sample7(uint32_t ns, std::mt19937& rng, std::vector<uint32_t>& vec_index, uint32_t* sample, uint32_t* log7) {
  const uint32_t last_idx = (uint32_t)vec_index.size() - 1;
  for (uint32_t i = 0; i < ns; ++i) {
    std::uniform_int_distribution<uint32_t> distribution(i, last_idx);
    const uint32_t sample_idx = distribution(rng);
    std::swap(vec_index[i], vec_index[sample_idx]);
    log7[i] = sample_idx;
  }
  for (uint32_t i = 0; i < ns; ++i) sample[i] = vec_index[i];
}
// advance the generator exactly like uniform_sample7 does, without touching the pool
inline void skip_sample7(uint32_t ns, std::mt19937& rng, uint32_t pool_size) {
  const uint32_t last_idx = pool_size - 1;
  for (uint32_t i = 0; i < ns; ++i) {
    std::uniform_int_distribution<uint32_t> distribution(i, last_idx);
    (void)distribution(rng);
  }
}

// device scratch out of the worker's size-bucketed pool (context.cu): no cudaMalloc / cudaFree per call --
// both synchronise the device and cost up to a second per call on multi-GPU boxes.  Everything that
// touches these buffers is ordered on w.stream, so a released block may be handed out again at once.
template <typename T>
struct DevBuf {
  DeviceWorker* w;
  T* p = nullptr;
  size_t cap = 0;
  explicit DevBuf(DeviceWorker& worker) : w(&worker) {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { if (p) pool_release(*w, p); }
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) pool_release(*w, p);
    p = nullptr;
    cap = 0;
    const size_t c = n + n / 2 + 64;
    p = (T*)pool_alloc(*w, c * sizeof(T));
    if (!p) return cudaErrorMemoryAllocation;
    cap = c;
    return cudaSuccess;
  }
};

std::vector<uint32_t> st_src(const std::vector<PairState>& st) {
  std::vector<uint32_t> v(st.size());
  for (size_t a = 0; a < st.size(); ++a) v[a] = st[a].src;
  return v;
}

}  // namespace

// Relative poses (r3d_relative_poses): what the essential AC-RANSAC leaves on the device feeds k_relpose on the same
// stream, before the one synchronisation; the per-pair results land in out[] (indexed by pair of the putative map)
struct RelposeIo {
  const AcPointSrc* d_src = nullptr;  // positions and intrinsics of each pair's views (set by filter_pairs_model)
  r3d_relative_pose* out = nullptr;
};

namespace {

// The device-resident ACRANSAC (acransac_fused.cu): the pairs are cut into size classes (shared-memory sort capacity
// 1024 ... 16384 putative matches; beyond that the "huge" class sorts in global scratch), one persistent launch per
// class, largest pairs first; ONE synchronisation, then the inlier lists come back through pinned staging.
// rp != nullptr (essential model): the relative-pose kernel runs after the AC-RANSAC launches.
int run_fused(r3d_ctx* ctx, DeviceWorker& w, int model, uint32_t max_iter, const r3d_matches* put, const std::vector<uint32_t>& src,
              const std::vector<AcPair>& hpairs, const AcPair* d_pairs, const double2* d_x1, const double2* d_x2,
              const uint2* d_match, const float* d_logc_n, const float* d_logc_k, uint32_t pt_total, uint32_t sizeSample,
              double t_begin, r3d_filter_timing& T, std::vector<std::vector<r3d_indmatch>>& result, RelposeIo* rp) {
  const uint32_t n = (uint32_t)hpairs.size();
  constexpr int kClasses = 6;  // caps 1024, 2048, 4096, 8192, 16384, huge
  std::vector<uint32_t> order[kClasses];
  uint32_t huge_maxM = 0;
  for (uint32_t a = 0; a < n; ++a) {
    const uint32_t M = hpairs[a].M;
    int c = 0;
    while (c < 5 && (1024u << c) < M) ++c;
    if (M > 16384u) { c = 5; huge_maxM = std::max(huge_maxM, M); }
    order[c].push_back(a);
  }
  std::vector<uint32_t> horder;
  uint32_t class_ofs[kClasses + 1] = {0};
  for (int c = 0; c < kClasses; ++c) {
    std::stable_sort(order[c].begin(), order[c].end(), [&](uint32_t x, uint32_t y) { return hpairs[x].M > hpairs[y].M; });
    class_ofs[c] = (uint32_t)horder.size();
    horder.insert(horder.end(), order[c].begin(), order[c].end());
  }
  class_ofs[kClasses] = (uint32_t)horder.size();
  DevBuf<uint32_t> d_order(w), d_work(w), d_si(w), d_pool(w);
  DevBuf<double> d_se(w);
  DevBuf<AcFusedOut> d_out(w);
  DevBuf<uint2> d_outm(w);
  R3D_CUDA_TRY(ctx, d_order.ensure(horder.size()));
  R3D_CUDA_TRY(ctx, d_work.ensure(kClasses));
  R3D_CUDA_TRY(ctx, d_out.ensure(n));
  R3D_CUDA_TRY(ctx, d_outm.ensure(pt_total));
  DevBuf<double> d_F(w);
  DevBuf<RelposeDev> d_rp(w);
  DevBuf<unsigned long long> d_keys(w);
  DevBuf<uint8_t> d_mask(w);
  if (rp) {
    R3D_CUDA_TRY(ctx, d_F.ensure((size_t)n * 9));
    R3D_CUDA_TRY(ctx, d_rp.ensure(n));
    R3D_CUDA_TRY(ctx, d_keys.ensure(pt_total));
    R3D_CUDA_TRY(ctx, d_mask.ensure(pt_total));
  }
  R3D_CUDA_TRY(ctx, cudaMemcpyAsync(d_order.p, horder.data(), horder.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, w.stream));
  R3D_CUDA_TRY(ctx, cudaMemsetAsync(d_work.p, 0, kClasses * sizeof(uint32_t), w.stream));
  cudaEvent_t ev[3];
  for (auto& e : ev) R3D_CUDA_TRY(ctx, cudaEventCreate(&e));
  struct EvGuard { cudaEvent_t* e; ~EvGuard() { for (int i = 0; i < 3; ++i) cudaEventDestroy(e[i]); } } evg{ev};
  R3D_CUDA_TRY(ctx, cudaEventRecord(ev[0], w.stream));
  // launch geometry of every class first: the scratch buffers are shared by the launches (same stream) and must not move
  uint32_t caps[kClasses] = {0}, grids[kClasses] = {0};
  size_t si_need = 0, huge_need = 0;
  for (int c = 0; c < kClasses; ++c) {
    const uint32_t cnt = class_ofs[c + 1] - class_ofs[c];
    if (!cnt) continue;
    const bool huge = c == 5;
    uint32_t cap = 1024u << c;
    if (huge) {
      cap = 32768;
      while (cap < huge_maxM) cap <<= 1;
    }
    uint32_t grid = std::min<uint32_t>(cnt, (uint32_t)w.sm_count * (uint32_t)acransac_fused_ctas_per_sm(model, cap, huge));
    if (huge) grid = std::min<uint32_t>(grid, (uint32_t)w.sm_count);
    caps[c] = cap;
    grids[c] = grid;
    si_need = std::max(si_need, (size_t)grid * cap);
    if (huge) huge_need = (size_t)grid * cap;
  }
  R3D_CUDA_TRY(ctx, d_si.ensure(si_need));
  if (huge_need) {
    R3D_CUDA_TRY(ctx, d_se.ensure(huge_need));
    R3D_CUDA_TRY(ctx, d_pool.ensure(huge_need));
  }
  for (int c = kClasses - 1; c >= 0; --c) {  // the long-running classes first
    const uint32_t cnt = class_ofs[c + 1] - class_ofs[c];
    if (!cnt) continue;
    int rc = launch_acransac_fused(ctx, w, model, c == 5, d_pairs, d_order.p + class_ofs[c], cnt, d_work.p + c, d_x1, d_x2, d_logc_n,
                                   d_logc_k, caps[c], max_iter, d_se.p, d_si.p, d_pool.p, d_match, d_outm.p, d_out.p,
                                   rp ? d_F.p : nullptr, grids[c]);
    if (rc) return rc;
    T.kernel_launches += 1;
  }
  R3D_CUDA_TRY(ctx, cudaEventRecord(ev[1], w.stream));
  std::vector<RelposeDev> hrp;
  if (rp) {
    int rc = launch_relpose(ctx, w, d_pairs, rp->d_src, n, d_out.p, d_F.p, d_outm.p, d_keys.p, d_mask.p, d_rp.p);
    if (rc) return rc;
    T.kernel_launches += 1;
    R3D_CUDA_TRY(ctx, cudaEventRecord(ev[2], w.stream));
    hrp.resize(n);
    R3D_CUDA_TRY(ctx, cudaMemcpyAsync(hrp.data(), d_rp.p, (size_t)n * sizeof(RelposeDev), cudaMemcpyDeviceToHost, w.stream));
  }
  std::vector<AcFusedOut> hout(n);
  R3D_CUDA_TRY(ctx, cudaMemcpyAsync(hout.data(), d_out.p, (size_t)n * sizeof(AcFusedOut), cudaMemcpyDeviceToHost, w.stream));
  R3D_CUDA_TRY(ctx, cudaStreamSynchronize(w.stream));
  float ms = 0.f, ms_total = 0.f;
  cudaEventElapsedTime(&ms, ev[0], ev[1]);
  T.ms_score = ms;
  if (rp) {
    cudaEventElapsedTime(&ms_total, ev[0], ev[2]);
    for (uint32_t a = 0; a < n; ++a) {  // RelativePose_Info of every pair that ran
      const AcFusedOut& o = hout[a];
      const RelposeDev& d = hrp[a];
      r3d_relative_pose& r = rp->out[src[a]];
      r.min_nfa = o.minNFA;
      if (!(o.minNFA < 0) || !((double)o.n_inliers > sizeSample * 2.5)) continue;
      r.found_residual_precision = std::sqrt(o.errorMax);
      r.n_inliers = o.n_inliers;
      std::memcpy(r.essential, d.E, sizeof(r.essential));
      if (d.n_front == 0) continue;  // no candidate puts a point in front of both cameras
      r.valid = 1;
      r.n_front = d.n_front;
      std::memcpy(r.rotation, d.R, sizeof(r.rotation));
      std::memcpy(r.translation, d.t, sizeof(r.translation));
      std::memcpy(r.center, d.C, sizeof(r.center));
      r.median_angle_deg = d.median_angle_deg;
    }
  }
  T.ms_solve = 0.0;
  T.rounds = 1;
  for (const AcFusedOut& o : hout) T.hypotheses += o.iterations;
  if (getenv("R3D_DEBUG_TIMING")) {
    uint64_t ex = 0, mo = 0, evs = 0;
    for (const AcFusedOut& o : hout) { ex += o.exact_scores; mo += o.models; evs += o.events; }
    fprintf(stderr, "[r3d] fused filter: %u pairs, kernel %.2f ms, %llu iterations, %llu models, %llu exact (%.2f %%), %llu events\n", n, ms,
            (unsigned long long)T.hypotheses, (unsigned long long)mo, (unsigned long long)ex, 100.0 * (double)ex / (double)std::max<uint64_t>(mo, 1),
            (unsigned long long)evs);
  }
  const double t_after_kernel = now_ms();
  // ---- inlier lists back: chunks of whole pairs through two pinned staging buffers, copied out by the host pool ----
  // GeometricFilter_*Matrix_AC::Robust_estimation keeps the pair iff #inliers > MINIMUM_SAMPLES * 2.5
  const size_t kStageElems = (size_t)4 << 20;  // 32 MB of (i, j) per buffer
  if (w.h_fstage_cap < kStageElems) {
    for (void*& hp : w.h_fstage) {
      if (hp) cudaFreeHost(hp);
      hp = nullptr;
      R3D_CUDA_TRY(ctx, cudaMallocHost(&hp, kStageElems * sizeof(uint2)));
    }
    w.h_fstage_cap = kStageElems;
  }
  struct Chunk { uint32_t a0, a1; size_t lo, hi; };
  std::vector<Chunk> chunks;
  {  // pairs are laid out in pt_ofs order (a ascending)
    uint32_t a = 0;
    while (a < n) {
      Chunk c{a, a, hpairs[a].pt_ofs, hpairs[a].pt_ofs};
      while (c.a1 < n && ((size_t)hpairs[c.a1].pt_ofs + hpairs[c.a1].M - c.lo <= kStageElems || c.a1 == c.a0)) {
        c.hi = (size_t)hpairs[c.a1].pt_ofs + hpairs[c.a1].M;
        ++c.a1;
      }
      chunks.push_back(c);
      a = c.a1;
    }
  }
  std::vector<uint2> big;  // a single pair larger than the staging buffer
  cudaEvent_t cev[2];
  for (auto& e : cev) R3D_CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  struct EvGuard2 { cudaEvent_t* e; ~EvGuard2() { for (int i = 0; i < 2; ++i) cudaEventDestroy(e[i]); } } evg2{cev};
  auto issue = [&](size_t ci) -> cudaError_t {
    const Chunk& c = chunks[ci];
    if (c.hi - c.lo > kStageElems) return cudaSuccess;  // handled synchronously below
    // only the inlier prefix of each pair is meaningful, but one contiguous copy beats thousands of small ones
    cudaError_t e = cudaMemcpyAsync(w.h_fstage[ci & 1], d_outm.p + c.lo, (c.hi - c.lo) * sizeof(uint2), cudaMemcpyDeviceToHost, w.stream);
    if (e != cudaSuccess) return e;
    return cudaEventRecord(cev[ci & 1], w.stream);
  };
  if (!chunks.empty()) R3D_CUDA_TRY(ctx, issue(0));
  for (size_t ci = 0; ci < chunks.size(); ++ci) {
    const Chunk& c = chunks[ci];
    const uint2* base;
    if (c.hi - c.lo > kStageElems) {
      big.resize(c.hi - c.lo);
      R3D_CUDA_TRY(ctx, cudaMemcpy(big.data(), d_outm.p + c.lo, (c.hi - c.lo) * sizeof(uint2), cudaMemcpyDeviceToHost));
      base = big.data();
    } else {
      R3D_CUDA_TRY(ctx, cudaEventSynchronize(cev[ci & 1]));
      base = (const uint2*)w.h_fstage[ci & 1];
    }
    if (ci + 1 < chunks.size()) R3D_CUDA_TRY(ctx, issue(ci + 1));  // the other buffer: free since chunk ci - 1 was consumed
    parallel_for(ctx->host_threads, c.a1 - c.a0, [&](size_t k) {
      const uint32_t a = c.a0 + (uint32_t)k;
      const AcFusedOut& o = hout[a];
      if (!(o.minNFA < 0) || !((double)o.n_inliers > sizeSample * 2.5)) return;
      const r3d_indmatch* sp = (const r3d_indmatch*)(base + (hpairs[a].pt_ofs - c.lo));
      result[src[a]].assign(sp, sp + o.n_inliers);
    });
  }
  (void)put;
  if (getenv("R3D_DEBUG_TIMING"))
    fprintf(stderr, "[r3d] fused filter total %.2f ms (kernel %.2f, results back %.2f)\n", now_ms() - t_begin, T.ms_score, now_ms() - t_after_kernel);
  T.ms_device_total = rp ? (double)ms_total : T.ms_score;
  T.ms_host = now_ms() - t_begin - T.ms_device_total;
  return R3D_OK;
}

}  // namespace

// pairs [p0, p1) of the putative map on worker w; result (sized by the caller to the whole map) is indexed by pair
int filter_pairs_model(r3d_ctx* ctx, DeviceWorker& w, int model, double precision_px, uint32_t max_iter, const r3d_matches* put,
                   const r3d_view_info* views, uint32_t n_views, uint64_t p0, uint64_t p1, r3d_filter_timing& T,
                   std::vector<std::vector<r3d_indmatch>>& result, RelposeIo* rp = nullptr) {
  R3D_CUDA_TRY(ctx, cudaSetDevice(w.device));
  T = r3d_filter_timing{};
  const double t_begin = now_ms();
  const uint32_t sizeSample = ac_min_samples(model), MAX_MODELS = ac_max_models(model);  // Kernel::MINIMUM_SAMPLES / MAX_MODELS

  // ---- per pair set-up (kernel adaptor of SURVEY.md A.5: normalisation, logalpha0, tables) ----
  std::vector<PairState> st;
  std::vector<AcPair> hpairs;
  std::vector<AcPointSrc> hsrc;
  uint64_t n_match_total = 0, n_table_total = 0;  // (i, j) of every putative match / logc_n entries, pair after pair
  uint32_t maxM = 0;
  {
    uint64_t pt_total = 0, tbl_total = 0;
    for (uint64_t p = p0; p < p1; ++p) {
      const uint32_t I = put->pairs[2 * p], J = put->pairs[2 * p + 1];
      const uint32_t M = (uint32_t)put->per[p].size();
      if (M <= sizeSample) continue;  // ACRANSAC returns at once: nData <= MINIMUM_SAMPLES
      if (I >= n_views || J >= n_views) return fail(ctx, R3D_ERR_INVALID, "r3d_filter_pairs: view id outside views[]");
      // GeometricFilter_EMatrix_AC::Robust_estimation returns false without two valid pinhole intrinsics
      if (model == 2 && (!(views[I].focal > 0.0) || !(views[J].focal > 0.0))) continue;
      auto vi = w.views.find(I), vj = w.views.find(J);
      if (vi == w.views.end() || vj == w.views.end() || !vi->second.has_xy || !vj->second.has_xy)
        return fail(ctx, R3D_ERR_INVALID, "r3d_filter_pairs: positions of a view were not uploaded");
      PairState s;
      s.src = (uint32_t)p; s.I = I; s.J = J; s.M = M;
      s.pt_ofs = (uint32_t)pt_total;
      s.tbl_ofs = (uint32_t)tbl_total;
      pt_total += M;
      tbl_total += M + 2;  // logc_n[0..M] and the table's error bound (k_ac_tables)
      maxM = std::max(maxM, M);
      st.push_back(std::move(s));
    }
    if (st.empty()) return R3D_OK;
    if (pt_total > 0xfffffff0ull) return fail(ctx, R3D_ERR_UNSUPPORTED, "r3d_filter_pairs: too many putative matches in one call");
    n_match_total = pt_total;
    n_table_total = tbl_total;
    hsrc.resize(st.size());
    hpairs.resize(st.size());
  }
  // the persistent per-pair kernel draws the sample stream on the device; it needs the restated
  // std::uniform_int_distribution to agree with this process's <random> (acransac_rng.cuh)
  const bool use_fused = rng_selftest() && !getenv("R3D_FILTER_HOST_ROUNDS");
  if (rp && !use_fused)
    return fail(ctx, R3D_ERR_UNSUPPORTED, "r3d_relative_poses: needs the device-resident AC-RANSAC (R3D_FILTER_HOST_ROUNDS is set "
                                          "or the device sample stream failed its self-test)");
  // log-combinatorial tables (float, upstream makelogcombi_n / makelogcombi_k).  logcombi(k,n) is a
  // running float sum over i = 1..min(k,n-k): its partial sums ARE the entries for smaller k, so one
  // O(n) pass reproduces the upstream O(n^2) table bit for bit.
  std::vector<float> vlog10(maxM + 2);
  for (uint32_t k = 0; k <= maxM + 1; ++k) vlog10[k] = std::log10((float)k);
  std::vector<float> hlogc_k(maxM + 1, 0.f);
  for (uint32_t n = 0; n <= maxM; ++n) {
    uint32_t k = sizeSample;
    if (k >= n) { hlogc_k[n] = 0.f; continue; }
    if (n - k < k) k = n - k;
    float r = 0.f;
    for (uint32_t i = 1; i <= k; ++i) r += vlog10[n - i + 1] - vlog10[i];
    hlogc_k[n] = r;
  }
  std::atomic<int> bad{0};
  const double t_pairs0 = now_ms();
  parallel_for(ctx->host_threads, st.size(), [&](size_t a) {
    PairState& s = st[a];
    const uint64_t p = s.src;
    const uint32_t M = s.M;
    const ViewDev& vi = w.views.find(s.I)->second;
    const ViewDev& vj = w.views.find(s.J)->second;
    const int wI = (int)views[s.I].width, hI = (int)views[s.I].height, wJ = (int)views[s.J].width, hJ = (int)views[s.J].height;
    // the essential adaptor keeps pixel coordinates (normalizer = identity)
    const double s1 = model == 2 ? 1.0 : 1.0 / std::sqrt((double)(wI * hI));
    const double s2 = model == 2 ? 1.0 : 1.0 / std::sqrt((double)(wJ * hJ));
    const double c1x = model == 2 ? 0.0 : (double)(-.5f * wI) * s1, c1y = model == 2 ? 0.0 : -.5 * hI * s1;
    const double c2x = model == 2 ? 0.0 : (double)(-.5f * wJ) * s2, c2y = model == 2 ? 0.0 : -.5 * hJ * s2;
    // the matched positions are looked up, promoted to double and normalised on the device (k_ac_points):
    // the host only ships the (i, j) list
    static_assert(sizeof(r3d_indmatch) == sizeof(uint2), "IndMatch layout");
    AcPointSrc& ps = hsrc[a];
    ps.xyI = vi.d_xy; ps.xyJ = vj.d_xy;
    ps.s1 = s1; ps.c1x = c1x; ps.c1y = c1y; ps.s2 = s2; ps.c2x = c2x; ps.c2y = c2y;
    ps.nI = vi.n; ps.nJ = vj.n; ps.identity = model == 2 ? 1u : 0u; ps.pad_ = 0;
    AcPair ap;
    ap.pt_ofs = s.pt_ofs; ap.M = M; ap.tbl_ofs = s.tbl_ofs; ap.pad_ = 0;
    const double precision = precision_px * precision_px;  // upper_bound_precision = Square(dPrecision)
    ap.max_thr = precision * s2 * s2;
    if (model == 0) {  // point-to-line
      const double D = std::sqrt((double)wJ * (double)wJ + (double)hJ * (double)hJ);
      const double Aarea = (double)wJ * (double)hJ;
      ap.logalpha0 = dm::log10_det(2.0 * D / Aarea / s2);
    } else if (model == 2) {  // ACKernelAdaptorEssential: log10(2 D / A * .5), pixel units
      const double D = std::sqrt((double)wJ * (double)wJ + (double)hJ * (double)hJ);
      const double Aarea = (double)wJ * (double)hJ;
      ap.logalpha0 = dm::log10_det(2.0 * D / Aarea * .5);
    } else {           // point-to-point
      ap.logalpha0 = dm::log10_det(R3D_PI / ((double)wJ * (double)hJ) / (s2 * s2));
    }
    ap.loge0 = dm::log10_det((double)MAX_MODELS * (double)(M - sizeSample));
    ap.K[0] = views[s.I].focal; ap.K[1] = views[s.I].ppx; ap.K[2] = views[s.I].ppy;
    ap.K[3] = views[s.J].focal; ap.K[4] = views[s.J].ppx; ap.K[5] = views[s.J].ppy;
    hpairs[a] = ap;
    if (!use_fused) {  // state of the host-round path only
      s.rngs.reset(new std::mt19937[2]);
      s.vec_index.resize(M);
      std::iota(s.vec_index.begin(), s.vec_index.end(), 0u);
    }
    s.nIterReserve = max_iter / 10;
    s.nIter = max_iter - s.nIterReserve;
    s.ac_mode = (precision == std::numeric_limits<double>::infinity());
  });
  (void)bad;
  if (getenv("R3D_DEBUG_TIMING"))
    fprintf(stderr, "[r3d] filter set-up: pair scan %.2f ms, per-pair tables + match copy %.2f ms\n", t_pairs0 - t_begin, now_ms() - t_pairs0);
  uint32_t cap = 32;
  while (cap < maxM) cap <<= 1;
  if (!use_fused && (size_t)cap * 12 > 200 * 1024)
    return fail(ctx, R3D_ERR_UNSUPPORTED, "r3d_filter_pairs: more than 16384 putative matches in one pair (host-round path)");

  // ---- device buffers -------------------------------------------------------------------------
  DevBuf<AcPair> d_pairs(w);
  DevBuf<double2> d_x1(w), d_x2(w);
  DevBuf<AcPointSrc> d_src(w);
  DevBuf<uint2> d_match(w);
  DevBuf<uint32_t> d_bad(w);
  DevBuf<float> d_logc_n(w), d_logc_k(w), d_vlog10(w);
  DevBuf<AcHyp> d_hyp(w);
  DevBuf<double> d_F(w);
  DevBuf<uint32_t> d_nm(w), d_inl(w);
  DevBuf<AcScore> d_score(w);
  DevBuf<AcInlierReq> d_req(w);
  R3D_CUDA_TRY(ctx, d_pairs.ensure(hpairs.size()));
  R3D_CUDA_TRY(ctx, d_x1.ensure(n_match_total));
  R3D_CUDA_TRY(ctx, d_x2.ensure(n_match_total));
  R3D_CUDA_TRY(ctx, d_src.ensure(hsrc.size()));
  R3D_CUDA_TRY(ctx, d_match.ensure(n_match_total));
  R3D_CUDA_TRY(ctx, d_bad.ensure(1));
  R3D_CUDA_TRY(ctx, d_logc_n.ensure(n_table_total));
  R3D_CUDA_TRY(ctx, d_vlog10.ensure(vlog10.size()));
  R3D_CUDA_TRY(ctx, d_logc_k.ensure(hlogc_k.size()));
  R3D_CUDA_TRY(ctx, cudaMemcpyAsync(d_pairs.p, hpairs.data(), hpairs.size() * sizeof(AcPair), cudaMemcpyHostToDevice, w.stream));
  R3D_CUDA_TRY(ctx, cudaMemcpyAsync(d_src.p, hsrc.data(), hsrc.size() * sizeof(AcPointSrc), cudaMemcpyHostToDevice, w.stream));
  // the putative (i, j) lists: gathered by the host pool into two pinned staging buffers, chunk by chunk, while the
  // previous chunk is on its way to the device (a pageable 800 MB source at C3 would move at a fraction of the link)
  {
    const size_t kStageElems = (size_t)4 << 20;  // 32 MB of (i, j) per buffer
    if (w.h_fstage_cap < kStageElems) {
      for (void*& hp : w.h_fstage) {
        if (hp) cudaFreeHost(hp);
        hp = nullptr;
        R3D_CUDA_TRY(ctx, cudaMallocHost(&hp, kStageElems * sizeof(uint2)));
      }
      w.h_fstage_cap = kStageElems;
    }
    cudaEvent_t uev[2];
    for (auto& e : uev) R3D_CUDA_TRY(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    struct UevGuard { cudaEvent_t* e; ~UevGuard() { for (int i = 0; i < 2; ++i) cudaEventDestroy(e[i]); } } uevg{uev};
    size_t a0 = 0, chunk_no = 0;
    while (a0 < st.size()) {
      size_t a1 = a0;
      const size_t lo = hpairs[a0].pt_ofs;
      size_t hi = lo;
      while (a1 < st.size() && ((size_t)hpairs[a1].pt_ofs + hpairs[a1].M - lo <= kStageElems || a1 == a0)) {
        hi = (size_t)hpairs[a1].pt_ofs + hpairs[a1].M;
        ++a1;
      }
      if (hi - lo > kStageElems) {  // one pair larger than the staging buffer: straight from its (pageable) span
        R3D_CUDA_TRY(ctx, cudaMemcpyAsync(d_match.p + lo, put->per[st[a0].src].data(), (hi - lo) * sizeof(uint2), cudaMemcpyHostToDevice, w.stream));
        R3D_CUDA_TRY(ctx, cudaStreamSynchronize(w.stream));
      } else {
        const int buf = (int)(chunk_no & 1);
        if (chunk_no >= 2) R3D_CUDA_TRY(ctx, cudaEventSynchronize(uev[buf]));  // the copy that last read this buffer is done
        uint2* stage = (uint2*)w.h_fstage[buf];
        parallel_for(ctx->host_threads, a1 - a0, [&](size_t k) {
          const size_t a = a0 + k;
          std::memcpy(stage + (hpairs[a].pt_ofs - lo), put->per[st[a].src].data(), (size_t)hpairs[a].M * sizeof(uint2));
        });
        R3D_CUDA_TRY(ctx, cudaMemcpyAsync(d_match.p + lo, stage, (hi - lo) * sizeof(uint2), cudaMemcpyHostToDevice, w.stream));
        R3D_CUDA_TRY(ctx, cudaEventRecord(uev[buf], w.stream));
        ++chunk_no;
      }
      a0 = a1;
    }
  }
  R3D_CUDA_TRY(ctx, cudaMemsetAsync(d_bad.p, 0, sizeof(uint32_t), w.stream));
  {
    int rcp = launch_ac_points(ctx, w, d_pairs.p, d_src.p, (uint32_t)hpairs.size(), d_match.p, d_x1.p, d_x2.p, d_bad.p);
    if (rcp) return rcp;
    uint32_t hbad = 0;
    R3D_CUDA_TRY(ctx, cudaMemcpyAsync(&hbad, d_bad.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, w.stream));
    R3D_CUDA_TRY(ctx, cudaStreamSynchronize(w.stream));
    if (hbad) return fail(ctx, R3D_ERR_INVALID, "r3d_filter_pairs: match index out of range");
    T.kernel_launches += 1;
  }
  // logc_n tables: float prefix sums over the host's log10 table, one thread per pair in the upstream order
  R3D_CUDA_TRY(ctx, cudaMemcpyAsync(d_vlog10.p, vlog10.data(), vlog10.size() * sizeof(float), cudaMemcpyHostToDevice, w.stream));
  {
    int rct = launch_ac_tables(ctx, w, d_pairs.p, (uint32_t)hpairs.size(), d_vlog10.p, d_logc_n.p);
    if (rct) return rct;
    T.kernel_launches += 1;
  }
  R3D_CUDA_TRY(ctx, cudaMemcpyAsync(d_logc_k.p, hlogc_k.data(), hlogc_k.size() * sizeof(float), cudaMemcpyHostToDevice, w.stream));

  if (getenv("R3D_DEBUG_TIMING")) fprintf(stderr, "[r3d] filter host set-up + point upload: %.2f ms\n", now_ms() - t_begin);
  if (use_fused) {
    if (rp) rp->d_src = d_src.p;
    return run_fused(ctx, w, model, max_iter, put, st_src(st), hpairs, d_pairs.p, d_x1.p, d_x2.p, d_match.p, d_logc_n.p, d_logc_k.p,
                     (uint32_t)n_match_total, sizeSample, t_begin, T, result, rp);
  }

  cudaEvent_t ev[3];
  for (auto& e : ev) R3D_CUDA_TRY(ctx, cudaEventCreate(&e));
  struct EvGuard { cudaEvent_t* e; ~EvGuard() { for (int i = 0; i < 3; ++i) cudaEventDestroy(e[i]); } } evg{ev};

  std::vector<AcHyp> hhyp;
  std::vector<AcScore> hscore;
  std::vector<uint32_t> hnm, hinl;
  std::vector<AcInlierReq> hreq;
  std::vector<uint32_t> active(st.size());
  std::iota(active.begin(), active.end(), 0u);
  const uint32_t kMaxHypPerRound = 1u << 18;
  // per-round loops are short (microseconds per pair): a handful of threads beats spawning one per core
  const int round_threads = std::min(ctx->host_threads, 8);

  double tm_setup = now_ms() - t_begin, tm_sample = 0, tm_gpu_wait = 0, tm_scan = 0, tm_inl = 0, tm_tail = 0;
  while (!active.empty()) {
    T.rounds++;
    double tq = now_ms();
    // ---- 1. draw a batch of samples ahead for every active pair -----------------------------
    uint32_t budget = std::max<uint32_t>(8u, kMaxHypPerRound / (uint32_t)active.size());
    uint32_t Htot = 0;
    for (uint32_t a : active) {
      PairState& s = st[a];
      uint32_t B = std::min<uint32_t>(std::max<uint32_t>(8u, 2u * s.since_event), 128u);
      B = std::min(B, budget);
      B = std::min(B, s.nIter - s.iter);
      s.hyp_ofs = Htot;
      s.hyp_n = B;
      Htot += B;
    }
    hhyp.resize(Htot);
    parallel_for(round_threads, active.size(), [&](size_t ai) {
      const uint32_t a = active[ai];
      PairState& s = st[a];
      s.rngs[1] = s.rngs[0];
      s.swap_log.resize((size_t)s.hyp_n * 7);
      for (uint32_t b = 0; b < s.hyp_n; ++b) {
        AcHyp& h = hhyp[s.hyp_ofs + b];
        h.pair = a;
        uniform_sample7(sizeSample, s.rngs[0], s.vec_index, h.sample, &s.swap_log[(size_t)b * 7]);
      }
    });
    tm_sample += now_ms() - tq; tq = now_ms();
    const uint32_t H = (uint32_t)hhyp.size();
    T.hypotheses += H;
    R3D_CUDA_TRY(ctx, d_hyp.ensure(H));
    R3D_CUDA_TRY(ctx, d_F.ensure((size_t)H * 9 * MAX_MODELS));
    R3D_CUDA_TRY(ctx, d_nm.ensure(H));
    R3D_CUDA_TRY(ctx, d_score.ensure((size_t)H * MAX_MODELS));
    R3D_CUDA_TRY(ctx, cudaMemcpyAsync(d_hyp.p, hhyp.data(), (size_t)H * sizeof(AcHyp), cudaMemcpyHostToDevice, w.stream));
    // ---- 2. solve + score on the device -------------------------------------------------------
    R3D_CUDA_TRY(ctx, cudaEventRecord(ev[0], w.stream));
    int rc = launch_f7_solve(ctx, w, model, d_pairs.p, d_x1.p, d_x2.p, d_hyp.p, H, d_F.p, d_nm.p);
    if (rc) return rc;
    R3D_CUDA_TRY(ctx, cudaEventRecord(ev[1], w.stream));
    rc = launch_f7_score(ctx, w, model, d_pairs.p, d_x1.p, d_x2.p, d_hyp.p, H, d_F.p, d_nm.p, d_logc_n.p, d_logc_k.p, cap, d_score.p);
    if (rc) return rc;
    R3D_CUDA_TRY(ctx, cudaEventRecord(ev[2], w.stream));
    T.kernel_launches += 2;
    hscore.resize((size_t)H * MAX_MODELS);
    hnm.resize(H);
    R3D_CUDA_TRY(ctx, cudaMemcpyAsync(hscore.data(), d_score.p, (size_t)H * MAX_MODELS * sizeof(AcScore), cudaMemcpyDeviceToHost, w.stream));
    R3D_CUDA_TRY(ctx, cudaMemcpyAsync(hnm.data(), d_nm.p, (size_t)H * sizeof(uint32_t), cudaMemcpyDeviceToHost, w.stream));
    R3D_CUDA_TRY(ctx, cudaStreamSynchronize(w.stream));
    float ms;
    cudaEventElapsedTime(&ms, ev[0], ev[1]); T.ms_solve += ms;
    cudaEventElapsedTime(&ms, ev[1], ev[2]); T.ms_score += ms;
    const double t_host0 = now_ms();
    tm_gpu_wait += now_ms() - tq; tq = now_ms();
    // ---- 3. replay the ACRANSAC state machine over the batch ----------------------------------
    parallel_for(round_threads, active.size(), [&](size_t ai) {
      PairState& s = st[active[ai]];
      s.best_changed = false;
      s.event = false;
      uint32_t consumed = s.hyp_n;
      for (uint32_t it = 0; it < s.hyp_n; ++it) {
        const uint32_t h = s.hyp_ofs + it;
        bool better = false;
        for (uint32_t mi = 0; mi < hnm[h]; ++mi) {
          const AcScore& sc = hscore[(size_t)h * MAX_MODELS + mi];
          if (!s.ac_mode && (double)sc.count > 2.5 * sizeSample) s.ac_mode = true;
          if (s.ac_mode && sc.nfa < s.minNFA) {
            better = true;
            s.minNFA = sc.nfa;
            s.errorMax = sc.err;
            s.best_k = sc.k;
            s.best_hyp = h;
            s.best_model = mi;
            s.best_changed = true;
            s.have_inliers = true;
          }
        }
        const uint32_t iter_abs = s.iter + it;
        if ((better && s.minNFA < 0) || (iter_abs + 1 == s.nIter && s.nIterReserve)) {
          if (!s.have_inliers) {
            ++s.nIter;
            --s.nIterReserve;
          } else {
            s.event = true;
            consumed = it + 1;
            break;
          }
        }
      }
      if (consumed < s.hyp_n) {  // discard the speculative tail: undo its swaps, replay the generator
        for (uint32_t b = s.hyp_n; b-- > consumed;)
          for (int i = (int)sizeSample - 1; i >= 0; --i) std::swap(s.vec_index[i], s.vec_index[s.swap_log[(size_t)b * 7 + i]]);
        s.rngs[0] = s.rngs[1];
        for (uint32_t b = 0; b < consumed; ++b) skip_sample7(sizeSample, s.rngs[0], (uint32_t)s.vec_index.size());
      }
      s.iter += consumed;
      s.since_event = s.event ? 0 : s.since_event + consumed;
    });
    hreq.clear();
    uint32_t inl_total = 0;
    for (uint32_t a : active) {
      PairState& s = st[a];
      if (s.best_changed) {  // the best model's inlier list is needed now (event) or possibly later
        AcInlierReq rq;
        rq.pair = a; rq.k = s.best_k; rq.out_ofs = inl_total; rq.hyp_model = s.best_hyp * MAX_MODELS + s.best_model;
        hreq.push_back(rq);
        inl_total += s.best_k;
      }
    }
    tm_scan += now_ms() - tq; tq = now_ms();
    // ---- 4. fetch the inlier lists of the new best models --------------------------------------
    if (!hreq.empty()) {
      // the F matrices of this round are still on the device (d_F); the kernel reads them there
      R3D_CUDA_TRY(ctx, d_req.ensure(hreq.size()));
      R3D_CUDA_TRY(ctx, d_inl.ensure(inl_total));
      R3D_CUDA_TRY(ctx, cudaMemcpyAsync(d_req.p, hreq.data(), hreq.size() * sizeof(AcInlierReq), cudaMemcpyHostToDevice, w.stream));
      rc = launch_f7_inliers(ctx, w, model, d_pairs.p, d_x1.p, d_x2.p, d_req.p, (uint32_t)hreq.size(), d_F.p, cap, d_inl.p);
      if (rc) return rc;
      T.kernel_launches += 1;
      hinl.resize(inl_total);
      R3D_CUDA_TRY(ctx, cudaMemcpyAsync(hinl.data(), d_inl.p, (size_t)inl_total * sizeof(uint32_t), cudaMemcpyDeviceToHost, w.stream));
      R3D_CUDA_TRY(ctx, cudaStreamSynchronize(w.stream));
      for (const AcInlierReq& rq : hreq) {
        PairState& s = st[rq.pair];
        s.inliers.assign(hinl.begin() + rq.out_ofs, hinl.begin() + rq.out_ofs + rq.k);
      }
    }
    tm_inl += now_ms() - tq; tq = now_ms();
    // ---- 5. pool replacement, termination ---------------------------------------------------------
    std::vector<uint32_t> next;
    for (uint32_t a : active) {
      PairState& s = st[a];
      if (s.event) {
        s.vec_index = s.inliers;  // ACRANSAC optimisation: draw samples among the best inlier set
        if (s.nIterReserve) {
          s.nIter = s.iter + s.nIterReserve;  // (iter + 1 + nIterReserve with the 0-based loop index)
          s.nIterReserve = 0;
        }
      }
      if (s.iter < s.nIter) next.push_back(a);
      else s.done = true;
    }
    active.swap(next);
    T.ms_host += now_ms() - t_host0;
    tm_tail += now_ms() - tq;
  }
  if (getenv("R3D_DEBUG_TIMING"))
    fprintf(stderr, "[r3d] filter: setup %.1f sample %.1f gpu+copies %.1f scan %.1f inliers %.1f tail %.1f ms, rounds %llu\n", tm_setup,
            tm_sample, tm_gpu_wait, tm_scan, tm_inl, tm_tail, (unsigned long long)T.rounds);
  // ---- result: GeometricFilter_FMatrix_AC::Robust_estimation keeps the pair iff #inliers > 7*2.5 ----
  for (const PairState& s : st) {
    if (!(s.minNFA < 0)) continue;  // "if (minNFA >= 0) vec_inliers.clear()"
    if (!(s.inliers.size() > sizeSample * 2.5)) continue;
    auto& out = result[s.src];
    out.reserve(s.inliers.size());
    for (uint32_t idx : s.inliers) out.push_back(put->per[s.src][idx]);
  }
  T.ms_device_total = T.ms_solve + T.ms_score;
  T.ms_host = now_ms() - t_begin - T.ms_device_total;
  return R3D_OK;
}

}  // namespace r3d

using namespace r3d;

// Diagnostics (host only): 1 when the device-side restatement of std::mt19937 + std::uniform_int_distribution
// (acransac_rng.cuh) reproduces this process's <random>, i.e. when the filter runs fully on the device.
extern "C" int r3d_debug_rng_selftest(void) { return rng_selftest() ? 1 : 0; }

namespace {

// image pairs are independent: cut the map into contiguous ranges of equal putative-match counts, one per device
// of the context (every device holds all positions), no collective -- the same rule as r3d_match_pairs.
// run(worker, p0, p1, timing) filters pairs [p0, p1); the context's filter timing becomes the slowest device's.
template <typename Run>
int shard_pairs(r3d_ctx* ctx, const r3d_matches* putative, Run run) {
  const uint64_t P_all = putative->pairs.size() / 2;
  const size_t nw = ctx->workers.size();
  std::vector<uint64_t> cut(nw + 1, 0);
  {
    std::vector<double> cost(P_all + 1, 0.0);
    for (uint64_t p = 0; p < P_all; ++p) cost[p + 1] = cost[p] + (double)putative->per[p].size() + 1.0;
    for (size_t k = 1; k < nw; ++k)
      cut[k] = std::min<uint64_t>(P_all, (uint64_t)(std::lower_bound(cost.begin(), cost.end(), cost[P_all] * (double)k / (double)nw) - cost.begin()));
    cut[nw] = P_all;
  }
  std::vector<int> rcs(nw, R3D_OK);
  std::vector<r3d_filter_timing> tms(nw);
  if (nw == 1) {
    rcs[0] = run(ctx->workers[0], (uint64_t)0, P_all, tms[0]);
  } else {
    std::vector<std::thread> th;
    for (size_t k = 0; k < nw; ++k)
      th.emplace_back([&, k]() { rcs[k] = run(ctx->workers[k], cut[k], cut[k + 1], tms[k]); });
    for (auto& t : th) t.join();
  }
  for (int rc : rcs)
    if (rc) return rc;
  r3d_filter_timing sum{};
  for (const r3d_filter_timing& t : tms) {
    sum.ms_solve = std::max(sum.ms_solve, t.ms_solve);
    sum.ms_score = std::max(sum.ms_score, t.ms_score);
    sum.ms_device_total = std::max(sum.ms_device_total, t.ms_device_total);
    sum.ms_host = std::max(sum.ms_host, t.ms_host);
    sum.kernel_launches += t.kernel_launches;
    sum.hypotheses += t.hypotheses;
    sum.rounds = std::max(sum.rounds, t.rounds);
  }
  ctx->filter_timing = sum;
  return R3D_OK;
}

// the pairs that kept inliers, in map order (pairs whose estimation failed disappear from the map)
r3d_matches* inlier_map(const r3d_matches* putative, std::vector<std::vector<r3d_indmatch>>& res) {
  r3d_matches* m = new r3d_matches();
  const uint64_t P = putative->pairs.size() / 2;
  for (uint64_t p = 0; p < P; ++p) {
    if (res[p].empty()) continue;
    m->push(putative->pairs[2 * p], putative->pairs[2 * p + 1], std::move(res[p]));
  }
  return m;
}

}  // namespace

extern "C" int r3d_filter_pairs(r3d_ctx* ctx, int model, double precision_px, uint32_t max_iter, const r3d_matches* putative,
                                const r3d_view_info* views, uint32_t n_views, r3d_matches** out) {
  if (!ctx || !putative || !views || !out) return fail(ctx, R3D_ERR_INVALID, "r3d_filter_pairs: bad arguments");
  *out = nullptr;
  if (model != R3D_MODEL_F && model != R3D_MODEL_H && model != R3D_MODEL_E)
    return fail(ctx, R3D_ERR_INVALID, "r3d_filter_pairs: unknown model");
  const int internal = model == R3D_MODEL_F ? 0 : (model == R3D_MODEL_H ? 1 : 2);
  std::vector<std::vector<r3d_indmatch>> res(putative->pairs.size() / 2);
  const int rc = shard_pairs(ctx, putative, [&](DeviceWorker& w, uint64_t p0, uint64_t p1, r3d_filter_timing& T) {
    return filter_pairs_model(ctx, w, internal, precision_px, max_iter, putative, views, n_views, p0, p1, T, res);
  });
  if (rc) return rc;
  *out = inlier_map(putative, res);
  return R3D_OK;
}

extern "C" int r3d_relative_poses(r3d_ctx* ctx, const r3d_matches* matches, const r3d_view_info* views, uint32_t n_views,
                                  double precision_px, uint32_t max_iter, r3d_relative_pose* out, r3d_matches** inliers) {
  if (!ctx || !matches || !views || !out) return fail(ctx, R3D_ERR_INVALID, "r3d_relative_poses: bad arguments");
  if (inliers) *inliers = nullptr;
  if (!(precision_px > 0.0)) return fail(ctx, R3D_ERR_INVALID, "r3d_relative_poses: precision_px must be > 0 (or +inf)");
  const uint64_t P = matches->pairs.size() / 2;
  for (uint64_t p = 0; p < P; ++p) {  // pairs that never reach the estimation keep this: invalid, nothing found
    r3d_relative_pose& r = out[p];
    std::memset(&r, 0, sizeof(r));
    r.I = matches->pairs[2 * p];
    r.J = matches->pairs[2 * p + 1];
    r.min_nfa = std::numeric_limits<double>::infinity();
    r.found_residual_precision = std::numeric_limits<double>::infinity();
  }
  std::vector<std::vector<r3d_indmatch>> res(P);
  const int rc = shard_pairs(ctx, matches, [&](DeviceWorker& w, uint64_t p0, uint64_t p1, r3d_filter_timing& T) {
    RelposeIo io;
    io.out = out;
    return filter_pairs_model(ctx, w, 2, precision_px, max_iter, matches, views, n_views, p0, p1, T, res, &io);
  });
  if (rc) return rc;
  if (inliers) *inliers = inlier_map(matches, res);
  return R3D_OK;
}
