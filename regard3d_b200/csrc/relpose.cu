// relpose.cu -- relative pose of every image pair from its essential AC-RANSAC result, one CTA per pair.
// COMPILED WITH --fmad=false (regard3d_b200/build.py), like acransac_fused.cu.
//
// Replaces the part of openMVG::sfm::robustRelativePose that follows ACRANSAC -- RelativePoseFromEssential /
// estimate_Rt_fromE (MotionFromEssential, TriangulateDLT of every inlier under the four candidates, cheirality count,
// std::max_element) -- plus the median triangulation angle AutomaticInitialPairChoice scores a pair with.  Upstream
// semantics: SURVEY.md A.9.  The AC-RANSAC itself is k_acransac_fused<2> on the same stream, which leaves the
// winning model (as the F = K2^-T E K1^-1 it scored), the AcFusedOut record and the inlier (i, j) list of every pair
// on the device.
//
// k_relpose, per CTA: thread 0 forms E = K2^T F K1 (the winning 5-point E up to rounding) and takes its SVD (4 candidates, shared memory); the threads split the inliers: bearings, 4 DLT
// triangulations and 8 depth tests each, integer block reductions of the 4 counts (deterministic); then the angle of
// every inlier in front under the chosen candidate; then an exact MSD radix select (8 passes of 8 bits over the bit
// patterns of the non-negative angles, keys in global scratch -- any pair size) of the n_front/2-th smallest angle.
#include "acransac_device.cuh"
#include "relpose_math.cuh"

namespace r3d {

namespace {

constexpr int kRThreads = 256;
constexpr unsigned long long kNotFront = ~0ull;  // key of an inlier not in front: above every angle's bit pattern

__device__ __forceinline__ void pair_bearings(const AcPair& pr, const AcPointSrc& ps, uint2 m, double* b1, double* b2) {
  const float2 a = ps.xyI[m.x], b = ps.xyJ[m.y];  // the essential adaptor works on pixel positions (identity)
  bearing(pr.K, (double)a.x, (double)a.y, b1);
  bearing(pr.K + 3, (double)b.x, (double)b.y, b2);
}

__global__ void __launch_bounds__(kRThreads) k_relpose(const AcPair* __restrict__ pairs, const AcPointSrc* __restrict__ src,
                                                       const AcFusedOut* __restrict__ ac, const double* __restrict__ Fall,
                                                       const uint2* __restrict__ inl, unsigned long long* __restrict__ keys,
                                                       uint8_t* __restrict__ mask, RelposeDev* __restrict__ out) {
  __shared__ double sE[9], sR[2][9], su3[3];
  __shared__ uint32_t s_cnt[4], s_hist[256], s_k;
  __shared__ unsigned long long s_prefix;
  const uint32_t a = blockIdx.x, tid = threadIdx.x;
  const AcPair pr = pairs[a];
  const AcFusedOut o = ac[a];
  // robustRelativePose fails at once when ACRANSAC kept fewer than MINIMUM_SAMPLES * 2.5 inliers (0 when minNFA >= 0)
  const uint32_t n = (o.minNFA < 0.0 && (double)o.n_inliers > 5 * 2.5) ? o.n_inliers : 0u;
  if (n == 0) {
    if (tid == 0) {
      RelposeDev r = {};
      out[a] = r;
    }
    return;
  }
  const AcPointSrc ps = src[a];
  const uint2* pin = inl + pr.pt_ofs;
  unsigned long long* pkeys = keys + pr.pt_ofs;
  uint8_t* pmask = mask + pr.pt_ofs;
  if (tid == 0) {
    rp::essential_from_fundamental(Fall + (size_t)a * 9, pr.K, pr.K + 3, sE);
    rp::motion_from_essential(sE, sR[0], sR[1], su3);
  }
  if (tid < 4) s_cnt[tid] = 0;
  __syncthreads();

  // ---- cheirality: every inlier under the four candidates -------------------------------------------------------
  uint32_t c[4] = {0, 0, 0, 0};
  for (uint32_t k = tid; k < n; k += kRThreads) {
    double b1[3], b2[3];
    pair_bearings(pr, ps, pin[k], b1, b2);
    uint32_t bits = 0;
#pragma unroll
    for (int cand = 0; cand < 4; ++cand) {
      const double* R = sR[cand >> 1];
      const double t[3] = {(cand & 1) ? -su3[0] : su3[0], (cand & 1) ? -su3[1] : su3[1], (cand & 1) ? -su3[2] : su3[2]};
      double X[3];
      rp::triangulate_dlt(R, t, b1, b2, X);
      if (X[2] > 0.0 && rp::depth(R, t, X) > 0.0) {  // Depth(I, 0, X) > 0 && Depth(R, t, X) > 0
        bits |= 1u << cand;
        ++c[cand];
      }
    }
    pmask[k] = (uint8_t)bits;
  }
#pragma unroll
  for (int cand = 0; cand < 4; ++cand) {
    uint32_t v = c[cand];
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    if ((tid & 31u) == 0 && v) atomicAdd(&s_cnt[cand], v);
  }
  __syncthreads();
  int best = 0;  // std::max_element: the first maximum
  for (int cand = 1; cand < 4; ++cand)
    if (s_cnt[cand] > s_cnt[best]) best = cand;
  const uint32_t n_front = s_cnt[best];
  if (n_front == 0) {  // robustRelativePose fails; E is still reported
    if (tid == 0) {
      RelposeDev r = {};
      for (int i = 0; i < 9; ++i) r.E[i] = sE[i];
      out[a] = r;
    }
    return;
  }
  const double* R = sR[best >> 1];
  const double sg = (best & 1) ? -1.0 : 1.0;
  const double t[3] = {sg * su3[0], sg * su3[1], sg * su3[2]};

  // ---- triangulation angle of every inlier in front under the chosen candidate ----------------------------------
  for (uint32_t k = tid; k < n; k += kRThreads) {
    unsigned long long key = kNotFront;
    if (pmask[k] & (1u << best)) {
      double b1[3], b2[3];
      pair_bearings(pr, ps, pin[k], b1, b2);
      key = (unsigned long long)__double_as_longlong(rp::ray_angle_deg(R, b1, b2));  // >= 0: bits order like values
    }
    pkeys[k] = key;
  }
  __syncthreads();

  // ---- the (n_front / 2)-th smallest angle (0-based, std::nth_element): MSD radix select --------------------------
  unsigned long long prefix = 0, known = 0;
  uint32_t rank = n_front / 2;
  for (int shift = 56; shift >= 0; shift -= 8) {
    s_hist[tid] = 0;  // kRThreads == 256 bins
    __syncthreads();
    for (uint32_t k = tid; k < n; k += kRThreads) {
      const unsigned long long key = pkeys[k];
      if ((key & known) == prefix) atomicAdd(&s_hist[(uint32_t)(key >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (tid == 0) {
      uint32_t below = 0, d = 0;
      for (; d < 255u; ++d) {
        if (below + s_hist[d] > rank) break;
        below += s_hist[d];
      }
      s_prefix = prefix | ((unsigned long long)d << shift);
      s_k = rank - below;
    }
    __syncthreads();
    prefix = s_prefix;
    rank = s_k;
    known |= 0xffull << shift;
    __syncthreads();
  }

  if (tid == 0) {
    RelposeDev r;
    for (int i = 0; i < 9; ++i) r.E[i] = sE[i];
    for (int i = 0; i < 9; ++i) r.R[i] = R[i];
    for (int i = 0; i < 3; ++i) r.t[i] = t[i];
    for (int i = 0; i < 3; ++i) r.C[i] = -((R[i] * t[0] + R[3 + i] * t[1]) + R[6 + i] * t[2]);  // C = -R^T t
    r.median_angle_deg = __longlong_as_double((long long)prefix);
    r.n_front = n_front;
    r.pad_ = 0;
    out[a] = r;
  }
}

static_assert(kRThreads == 256, "one histogram bin per thread");

}  // namespace

int launch_relpose(r3d_ctx* ctx, DeviceWorker& w, const AcPair* pairs, const AcPointSrc* src, uint32_t n_pairs,
                   const AcFusedOut* ac, const double* F, const uint2* inl, unsigned long long* keys, uint8_t* mask,
                   RelposeDev* out) {
  if (!n_pairs) return R3D_OK;
  k_relpose<<<n_pairs, kRThreads, 0, w.stream>>>(pairs, src, ac, F, inl, keys, mask, out);
  R3D_CUDA_TRY(ctx, cudaGetLastError());
  return R3D_OK;
}

}  // namespace r3d
