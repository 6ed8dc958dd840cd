// robust_pose.cu — the pieces of RobustPoseEstimator.estimate_pose (robust_pose_estimator.py:89-251) that sit
// around the batched RANSAC stages: the displacement median behind the adaptive threshold and the parallax
// statistics, the n-point homography refit on the H-RANSAC winner's inliers, and the decision stage
// (decompose_homography, per-branch diagnostics and score, model selection, stability gates).
//   * displacement_median_kernel: one CTA per pair.  The float32 norm of every selected displacement is
//     recomputed from the correspondences in each pass (no scratch buffer, any count) and the order statistics
//     are found by an exact 4 x 8-bit radix select on the bit patterns (non-negative floats order like their
//     bit patterns).  Bit-identical to np.median(np.linalg.norm(pts2 - pts1, axis=1)) on float32 inputs.
//   * refit_homography_kernel: one CTA per pair, the structure of refit_essential_kernel (pose.cu): fixed-order
//     reductions, the 9x9 Gram matrix of the DLT rows in float64, warp-cooperative parallel-order Jacobi.
//   * robust_pose_decide_kernel: one CTA per pair; lane 0 makes the decision, the CTA writes the selected
//     model's inlier flags and, given a record sink, the pair's pose record (include/b2s.h).
#include "common.cuh"

namespace b2s {

constexpr int kMedThreads = 256;
constexpr int kHRefitThreads = 256;
constexpr int kDecideThreads = 128;

struct Mat3Arg {   // a 3x3 matrix passed by value
  double m[9];
};

// |pts2 - pts1| in float32, every operation rounded on its own (np.linalg.norm: (d * d) summed, then sqrt)
__device__ __forceinline__ uint32_t displacement_bits(const float4 c) {
  const float dx = __fsub_rn(c.z, c.x), dy = __fsub_rn(c.w, c.y);
  return __float_as_uint(__fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy))));
}

// np.clip(x, lo, hi) == minimum(maximum(x, lo), hi): NaN propagates, lo > hi gives hi
__device__ __forceinline__ double np_clip(double x, double lo, double hi) {
  const double y = (x < lo) ? lo : x;
  return (y > hi) ? hi : y;
}

// the k-th smallest (0-based) selected displacement, as its bit pattern
__device__ uint32_t radix_select(const float4* __restrict__ cp, const uint8_t* __restrict__ mp, int M, int k,
                                 uint32_t* s_hist, int* s_pick) {
  const int tid = threadIdx.x;
  uint32_t prefix = 0u, pmask = 0u;
  for (int shift = 24; shift >= 0; shift -= 8) {
    for (int i = tid; i < 256; i += kMedThreads) s_hist[i] = 0u;
    __syncthreads();
    for (int m = tid; m < M; m += kMedThreads) {
      if (mp && mp[m] == 0) continue;
      const uint32_t b = displacement_bits(cp[m]);
      if ((b & pmask) == prefix) atomicAdd(&s_hist[(b >> shift) & 255u], 1u);
    }
    __syncthreads();
    if (tid == 0) {
      int acc = 0, bin = 0;
      for (; bin < 255; ++bin) {
        if (acc + (int)s_hist[bin] > k) break;
        acc += (int)s_hist[bin];
      }
      s_pick[0] = bin;
      s_pick[1] = acc;
    }
    __syncthreads();
    k -= s_pick[1];
    prefix |= (uint32_t)s_pick[0] << shift;
    pmask |= 255u << shift;
    __syncthreads();
  }
  return prefix;
}

__global__ void __launch_bounds__(kMedThreads) displacement_median_kernel(
    const float4* __restrict__ corr, const int32_t* __restrict__ c_off, const int32_t* __restrict__ c_count,
    const uint8_t* __restrict__ mask, const b2s_robust_pose_config* __restrict__ cfg, int n_cfg,
    float* __restrict__ median_out, double* __restrict__ th_out, double* __restrict__ th2_out) {
  __shared__ uint32_t s_hist[256];
  __shared__ int s_pick[2];
  __shared__ int s_n, s_nan;
  const int pair = blockIdx.x, tid = threadIdx.x;
  const int M = max(c_count[pair], 0);   // a negative count is the selection kernel's overflow flag: no model
  const float4* cp = corr + c_off[pair];
  const uint8_t* mp = mask ? mask + c_off[pair] : nullptr;
  if (tid == 0) s_n = 0, s_nan = 0;
  __syncthreads();
  int n = 0, nan = 0;
  for (int m = tid; m < M; m += kMedThreads) {
    if (mp && mp[m] == 0) continue;
    ++n;
    nan |= isnan(__uint_as_float(displacement_bits(cp[m]))) ? 1 : 0;
  }
  if (n) atomicAdd(&s_n, n);
  if (nan) atomicOr(&s_nan, 1);
  __syncthreads();
  n = s_n;
  float med;
  if (n == 0) {
    med = 0.0f;                                                       // _median_parallax of an empty selection
  } else if (s_nan) {
    med = __uint_as_float(0x7FC00000u);                               // np.median propagates NaN
  } else if (n & 1) {
    med = __uint_as_float(radix_select(cp, mp, M, n >> 1, s_hist, s_pick));
  } else {
    const float a = __uint_as_float(radix_select(cp, mp, M, (n >> 1) - 1, s_hist, s_pick));
    const float b = __uint_as_float(radix_select(cp, mp, M, n >> 1, s_hist, s_pick));
    med = __fdiv_rn(__fadd_rn(a, b), 2.0f);                           // np.mean of the two middle float32 values
  }
  if (tid != 0) return;
  if (median_out) median_out[pair] = med;
  if (cfg) {
    const b2s_robust_pose_config& c = cfg[n_cfg == 1 ? 0 : pair];
    double th;
    if (n == 0) {
      th = np_clip(c.base_ransac_threshold, c.min_ransac_threshold, c.max_ransac_threshold);
    } else {
      const double scale = np_clip(__ddiv_rn((double)med, 25.0), 0.5, 2.0);
      th = np_clip(__dmul_rn(c.base_ransac_threshold, scale), c.min_ransac_threshold, c.max_ransac_threshold);
    }
    if (th_out) th_out[pair] = th;
    if (th2_out) th2_out[pair] = __dmul_rn(th, th);
  }
}

// ---- n-point normalised DLT (homography.py:118-142) ------------------------------------------------------

// Sum of N per-thread values over the CTA in a fixed order (warp butterfly, then the warps in order); every
// thread gets the same total.
template <int N>
__device__ __forceinline__ void cta_sum(double (&v)[N], double (*s_part)[N]) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < N; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xFFFFFFFFu, v[k], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < N; ++k) s_part[warp][k] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < N; ++k) {
    double t = 0.0;
    for (int w = 0; w < kHRefitThreads / 32; ++w) t += s_part[w][k];
    v[k] = t;
  }
  __syncthreads();
}

__device__ __forceinline__ double finite_or_zero(double x) { return isfinite(x) ? x : 0.0; }   // np.nan_to_num(A, 0, 0, 0)

__global__ void __launch_bounds__(kHRefitThreads) refit_homography_kernel(
    const float4* __restrict__ corr, const int32_t* __restrict__ c_off, const int32_t* __restrict__ c_count,
    const uint8_t* __restrict__ mask, double* __restrict__ H_out, int32_t* __restrict__ n_used) {
  constexpr int kWarps = kHRefitThreads / 32;
  __shared__ double s_p5[kWarps][5];
  __shared__ double s_p2[kWarps][2];
  __shared__ double s_part[kWarps][45];
  __shared__ double s_M[9][9], s_V[9][9];
  const int pair = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int M = max(c_count[pair], 0);
  const float4* cp = corr + c_off[pair];
  const uint8_t* mp = mask ? mask + c_off[pair] : nullptr;
  // Hartley centroid of both point sets
  double c5[5] = {0.0, 0.0, 0.0, 0.0, 0.0};
  for (int m = tid; m < M; m += kHRefitThreads) {
    if (mp && mp[m] == 0) continue;
    const float4 c = cp[m];
    c5[0] += (double)c.x, c5[1] += (double)c.y, c5[2] += (double)c.z, c5[3] += (double)c.w, c5[4] += 1.0;
  }
  cta_sum<5>(c5, s_p5);
  const int total = (int)c5[4];
  double* ho = H_out + (size_t)pair * 9;
  if (total < 4) {
    if (tid < 9) ho[tid] = 0.0;
    if (tid == 0 && n_used) n_used[pair] = total;
    return;
  }
  const double inv_n = 1.0 / c5[4];
  const double csx = c5[0] * inv_n, csy = c5[1] * inv_n, cdx = c5[2] * inv_n, cdy = c5[3] * inv_n;
  // RMS distance from the centroid
  double v2[2] = {0.0, 0.0};
  for (int m = tid; m < M; m += kHRefitThreads) {
    if (mp && mp[m] == 0) continue;
    const float4 c = cp[m];
    const double ax = (double)c.x - csx, ay = (double)c.y - csy, bx = (double)c.z - cdx, by = (double)c.w - cdy;
    v2[0] += ax * ax + ay * ay;
    v2[1] += bx * bx + by * by;
  }
  cta_sum<2>(v2, s_p2);
  const double ss = sqrt(2.0) / sqrt(v2[0] * inv_n), sd = sqrt(2.0) / sqrt(v2[1] * inv_n);
  // Gram matrix of the 2n DLT rows (upper triangle, 45 entries)
  double acc[45];
#pragma unroll
  for (int k = 0; k < 45; ++k) acc[k] = 0.0;
  for (int m = tid; m < M; m += kHRefitThreads) {
    if (mp && mp[m] == 0) continue;
    const float4 c = cp[m];
    const double x = ((double)c.x - csx) * ss, y = ((double)c.y - csy) * ss;
    const double u = ((double)c.z - cdx) * sd, v = ((double)c.w - cdy) * sd;
    const double a[9] = {finite_or_zero(-x), finite_or_zero(-y), -1.0, 0.0, 0.0, 0.0,
                         finite_or_zero(u * x), finite_or_zero(u * y), finite_or_zero(u)};
    const double b[9] = {0.0, 0.0, 0.0, finite_or_zero(-x), finite_or_zero(-y), -1.0,
                         finite_or_zero(v * x), finite_or_zero(v * y), finite_or_zero(v)};
    int k = 0;
#pragma unroll
    for (int i = 0; i < 9; ++i)
#pragma unroll
      for (int j = i; j < 9; ++j) acc[k] = fma(a[i], a[j], fma(b[i], b[j], acc[k])), ++k;
  }
#pragma unroll
  for (int k = 0; k < 45; ++k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xFFFFFFFFu, acc[k], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 45; ++k) s_part[warp][k] = acc[k];
  }
  __syncthreads();
  if (tid < 45) {
    double t = 0.0;
    for (int w = 0; w < kWarps; ++w) t += s_part[w][tid];
    int i = 0, rem = tid;
    while (rem >= 9 - i) rem -= 9 - i, ++i;
    const int j = i + rem;
    s_M[i][j] = t;
    s_M[j][i] = t;
  }
  if (tid < 81) s_V[tid / 9][tid % 9] = (tid / 9 == tid % 9) ? 1.0 : 0.0;
  __syncthreads();
  if (warp != 0) return;
  if (lane == 0 && n_used) n_used[pair] = total;
  // eigenvector of the smallest eigenvalue: the parallel-order Jacobi of refit_essential_kernel (pose.cu)
  __shared__ int s_rot;
  __shared__ double s_c4[4], s_s4[4];
  __shared__ int s_p4[4], s_q4[4];
  for (int sweep = 0; sweep < 30; ++sweep) {
    if (lane == 0) s_rot = 0;
    __syncwarp();
    for (int r = 0; r < 9; ++r) {
      if (lane < 4) {
        const int a = (r + lane + 1) % 9, b2 = (r + 9 - (lane + 1)) % 9;
        const int p = min(a, b2), q = max(a, b2);
        const double apq = s_M[p][q], app = s_M[p][p], aqq = s_M[q][q];
        double c = 1.0, sn = 0.0;
        if (fabs(apq) > 1.0e-17 * sqrt(fabs(app * aqq)) && apq != 0.0) {
          const double theta = (aqq - app) / (2.0 * apq);
          const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(fma(theta, theta, 1.0)));
          c = rsqrt(fma(t, t, 1.0));
          sn = t * c;
          s_rot = 1;
        }
        s_c4[lane] = c, s_s4[lane] = sn, s_p4[lane] = p, s_q4[lane] = q;
      }
      __syncwarp();
      for (int task = lane; task < 36; task += 32) {
        const int j = task / 9, k = task - 9 * j, p = s_p4[j], q = s_q4[j];
        const double c = s_c4[j], sn = s_s4[j];
        if (sn != 0.0) {
          const double mkp = s_M[k][p], mkq = s_M[k][q];
          s_M[k][p] = c * mkp - sn * mkq;
          s_M[k][q] = sn * mkp + c * mkq;
          const double vkp = s_V[k][p], vkq = s_V[k][q];
          s_V[k][p] = c * vkp - sn * vkq;
          s_V[k][q] = sn * vkp + c * vkq;
        }
      }
      __syncwarp();
      for (int task = lane; task < 36; task += 32) {
        const int j = task / 9, k = task - 9 * j, p = s_p4[j], q = s_q4[j];
        const double c = s_c4[j], sn = s_s4[j];
        if (sn != 0.0) {
          const double mpk = s_M[p][k], mqk = s_M[q][k];
          s_M[p][k] = c * mpk - sn * mqk;
          s_M[q][k] = sn * mpk + c * mqk;
        }
      }
      __syncwarp();
    }
    if (s_rot == 0) break;
  }
  if (lane == 0) {
    int best = 0;
    for (int k = 1; k < 9; ++k) best = (s_M[k][k] < s_M[best][best]) ? k : best;
    double n[9];
    for (int k = 0; k < 9; ++k) n[k] = s_V[k][best];
    // H = T_dst^-1 Hn T_src, T = [s 0 -s c; 0 s -s c; 0 0 1]  (homography.py:141), then H / H[2][2]
    double M1[9];
    for (int r = 0; r < 3; ++r) {
      M1[3 * r + 0] = n[3 * r + 0] * ss;
      M1[3 * r + 1] = n[3 * r + 1] * ss;
      M1[3 * r + 2] = fma(-ss * csx, n[3 * r + 0], fma(-ss * csy, n[3 * r + 1], n[3 * r + 2]));
    }
    const double isd = 1.0 / sd;
    double Hm[9];
    for (int c = 0; c < 3; ++c) {
      Hm[c] = fma(isd, M1[c], cdx * M1[6 + c]);
      Hm[3 + c] = fma(isd, M1[3 + c], cdy * M1[6 + c]);
      Hm[6 + c] = M1[6 + c];
    }
    const double r22 = 1.0 / Hm[8];
    for (int k = 0; k < 9; ++k) ho[k] = Hm[k] * r22;
  }
}

// ---- decision stage ---------------------------------------------------------------------------------------

// Orthogonal polar factor of a 3x3 matrix (= U V^T of its SVD, unique for a non-singular matrix) by the
// Newton iteration X <- (X + X^-T) / 2, quadratically convergent; false for a singular or non-finite input.
__device__ bool polar_factor3(const double (&A)[9], double (&X)[9]) {
#pragma unroll
  for (int k = 0; k < 9; ++k) X[k] = A[k];
  bool last = false;
  for (int it = 0; it < 100; ++it) {
    double c[9];
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
        c[3 * i + j] = X[3 * i1 + j1] * X[3 * i2 + j2] - X[3 * i1 + j2] * X[3 * i2 + j1];   // cofactors: X^-T = c / det
      }
    const double det = X[0] * c[0] + X[1] * c[1] + X[2] * c[2];
    if (!(fabs(det) > 0.0) || !isfinite(det)) return false;
    const double id = 1.0 / det;
    double diff = 0.0, nrm = 0.0;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const double y = 0.5 * (X[k] + c[k] * id);
      diff += (y - X[k]) * (y - X[k]);
      nrm += y * y;
      X[k] = y;
    }
    if (last) break;
    if (diff <= 1e-20 * nrm) last = true;   // one more step after convergence reaches the rounding level
  }
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 9; ++k) ok &= (bool)isfinite(X[k]);
  return ok;
}

// decompose_homography (homography.py:59-78): Kinv h1 normalisation, [r1 r2 r1 x r2], polar factor
__device__ bool decompose_homography_dev(const double* __restrict__ H, const double (&ki)[9], double (&R)[9], double (&t)[3]) {
  double k1[3], k2[3], k3[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    k1[r] = ki[3 * r] * H[0] + ki[3 * r + 1] * H[3] + ki[3 * r + 2] * H[6];
    k2[r] = ki[3 * r] * H[1] + ki[3 * r + 1] * H[4] + ki[3 * r + 2] * H[7];
    k3[r] = ki[3 * r] * H[2] + ki[3 * r + 1] * H[5] + ki[3 * r + 2] * H[8];
  }
  const double norm = sqrt(k1[0] * k1[0] + k1[1] * k1[1] + k1[2] * k1[2]);
  double r1[3], r2[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) r1[r] = k1[r] / norm, r2[r] = k2[r] / norm, t[r] = k3[r] / norm;
  const double r3[3] = {r1[1] * r2[2] - r1[2] * r2[1], r1[2] * r2[0] - r1[0] * r2[2], r1[0] * r2[1] - r1[1] * r2[0]};
  const double A[9] = {r1[0], r2[0], r3[0], r1[1], r2[1], r3[1], r1[2], r2[2], r3[2]};
  bool ok = true;
#pragma unroll
  for (int k = 0; k < 9; ++k) ok &= (bool)isfinite(A[k]);   // np.linalg.svd raises on a non-finite matrix
  return ok && polar_factor3(A, R);
}

__device__ __forceinline__ double norm3(const double (&t)[3]) { return sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]); }

__global__ void __launch_bounds__(kDecideThreads) robust_pose_decide_kernel(
    const int32_t* __restrict__ c_off, const int32_t* __restrict__ c_count, const int32_t* __restrict__ e_best_h,
    const int32_t* __restrict__ e_inliers, const uint8_t* __restrict__ e_mask, const double* __restrict__ e_R,
    const double* __restrict__ e_t, const int32_t* __restrict__ e_votes, const float* __restrict__ e_median,
    const float* __restrict__ all_median, const double* __restrict__ th, const int32_t* __restrict__ h_best_h,
    const int32_t* __restrict__ h_inliers, const uint8_t* __restrict__ h_mask, const double* __restrict__ H_fit,
    const Mat3Arg Kinv, const b2s_robust_pose_config* __restrict__ cfg, int n_cfg,
    b2s_pose_result* __restrict__ results, uint8_t* __restrict__ out_mask, int mask_stride, const b2s_record_sink sink) {
  __shared__ int s_src;   // 0: essential mask, 1: homography mask, -1: zeros
  const int pair = blockIdx.x, tid = threadIdx.x;
  const int M = max(c_count[pair], 0);
  if (tid == 0) {
    const b2s_robust_pose_config& c = cfg[n_cfg == 1 ? 0 : pair];
    b2s_pose_result r = {};
    r.e_best_h = r.h_best_h = -1;
    r.e_inliers = r.h_inliers = -1;
    r.match_count = M;
    r.threshold = th[pair];
    int src = -1;
    if (M < c.min_matches) {
      r.outcome = B2S_POSE_ERR_MATCHES;
    } else if (M < 8) {
      r.outcome = B2S_POSE_ERR_EIGHT;
    } else {
      r.e_best_h = e_best_h[pair];
      r.e_inliers = e_inliers[pair];
      double te[3] = {e_t[pair * 3], e_t[pair * 3 + 1], e_t[pair * 3 + 2]};
      const double ne = norm3(te);
      if (r.e_best_h < 0 || r.e_inliers < 8) {
        r.outcome = B2S_POSE_ERR_ESSENTIAL;
      } else if (ne == 0.0) {
        r.outcome = B2S_POSE_ERR_TRANSLATION;
        r.method = B2S_POSE_METHOD_ESSENTIAL;
      } else {
        // essential branch (_estimate_essential): the cheirality count is the K7 vote of the picked candidate
        const int32_t* v = e_votes + pair * 4;
        int win = 0;
        for (int k = 1; k < 4; ++k) win = (v[k] > v[win]) ? k : win;
        const int e_inl = r.e_inliers, ch = v[win];
        const double ratio_e = (double)e_inl / (double)max(M, 1), par_e = (double)e_median[pair];
        const double chr_e = (double)ch / (double)max(e_inl, 1);
        const double score_e = __dmul_rn(__dmul_rn(c.essential_bias, ratio_e), c.min_parallax > par_e ? c.min_parallax : par_e);
        r.score_essential = score_e;
        // homography branch (_estimate_homography)
        r.h_best_h = h_best_h[pair];
        r.h_inliers = h_inliers[pair];
        double Rh[9], th_[3];
        const double ki[9] = {Kinv.m[0], Kinv.m[1], Kinv.m[2], Kinv.m[3], Kinv.m[4], Kinv.m[5], Kinv.m[6], Kinv.m[7], Kinv.m[8]};
        if (r.h_best_h < 0 || r.h_inliers < 4 || !decompose_homography_dev(H_fit + (size_t)pair * 9, ki, Rh, th_)) {
          r.outcome = B2S_POSE_ERR_HOMOGRAPHY;
        } else if (norm3(th_) == 0.0) {
          r.outcome = B2S_POSE_ERR_TRANSLATION;
          r.method = B2S_POSE_METHOD_HOMOGRAPHY;
        } else {
          const int h_inl = r.h_inliers;
          const double ratio_h = (double)h_inl / (double)max(M, 1), par_h = (double)all_median[pair];
          const double score_h = __dmul_rn(__dmul_rn(c.homography_bias, ratio_h), c.min_parallax > par_h ? c.min_parallax : par_h);
          r.score_homography = score_h;
          const bool use_h = score_h > score_e;          // max([essential, homography]): the first maximum wins
          if (use_h) {
            const double nh = norm3(th_);
            r.method = B2S_POSE_METHOD_HOMOGRAPHY;
            r.inliers = h_inl, r.cheirality_inliers = h_inl;
            r.inlier_ratio = ratio_h, r.median_parallax = par_h, r.cheirality_ratio = 1.0, r.score = score_h;
            for (int k = 0; k < 9; ++k) r.R[k] = Rh[k];
            for (int k = 0; k < 3; ++k) r.t[k] = th_[k] / nh;
          } else {
            r.method = B2S_POSE_METHOD_ESSENTIAL;
            r.inliers = e_inl, r.cheirality_inliers = ch;
            r.inlier_ratio = ratio_e, r.median_parallax = par_e, r.cheirality_ratio = chr_e, r.score = score_e;
            for (int k = 0; k < 9; ++k) r.R[k] = e_R[(size_t)pair * 9 + k];
            for (int k = 0; k < 3; ++k) r.t[k] = te[k] / ne;
          }
          src = r.method;
          // _apply_stability_gates, in the reference's order
          int gate = B2S_GATE_NONE;
          if (r.inliers < c.min_inliers) gate = B2S_GATE_LOW_INLIER_COUNT;
          else if (r.inlier_ratio < c.min_inlier_ratio) gate = B2S_GATE_LOW_INLIER_RATIO;
          else if (r.median_parallax < c.min_parallax) gate = B2S_GATE_LOW_PARALLAX;
          else if (!use_h && r.cheirality_inliers < c.min_cheirality_inliers) gate = B2S_GATE_CHEIRALITY_INLIERS;
          else if (!use_h && r.cheirality_ratio < c.min_cheirality_ratio) gate = B2S_GATE_CHEIRALITY_RATIO;
          r.gate = gate;
          r.outcome = gate == B2S_GATE_NONE ? B2S_POSE_ESTIMATE : B2S_POSE_GATE_FAILED;
        }
      }
    }
    results[pair] = r;
    s_src = src;
  }
  __syncthreads();
  const int src = s_src;
  const uint8_t* from = src == 0 ? e_mask : (src == 1 ? h_mask : nullptr);
  const int off = c_off[pair];
  for (int m = tid; m < M; m += kDecideThreads) out_mask[off + m] = from ? from[off + m] : (uint8_t)0;
  for (int m = M + tid; m < mask_stride; m += kDecideThreads) out_mask[off + m] = 0;   // unused tail of a compact slot
  if (!sink.records) return;
  // The pair's pose record, written by the kernel that holds the answer (no extra launch at the end of the step): this
  // is the send slice of the all-gather / the source of the step's one device->host copy.  The result is read back
  // from `results` (written by thread 0 before the barrier), so the decision keeps its registers.
  uint8_t* rec = sink.records + (size_t)pair * sink.record_bytes;
  const int S = sink.stride, n = min(M, S);
  const b2s_pose_result* r = results + pair;
  if (tid < 16) {
    const int outcome = r->outcome;
    const bool answer = outcome == B2S_POSE_ESTIMATE || outcome == B2S_POSE_GATE_FAILED;
    int32_t v;
    if (tid == 0) v = c_count[pair];                   // the selection count (-1 on overflow)
    else if (tid == 1) v = answer ? (r->method == B2S_POSE_METHOD_HOMOGRAPHY ? r->h_best_h : r->e_best_h) : -1;
    else if (tid == 2) v = r->inliers;
    else if (tid == 3) v = sink.pair_id0 + pair;
    else if (tid < 13) v = __float_as_int((float)r->R[tid - 4]);   // zero for an error outcome
    else v = __float_as_int((float)r->t[tid - 13]);
    reinterpret_cast<int32_t*>(rec)[tid] = v;
  } else if (tid < 16 + B2S_POSE_BLOCK_BYTES / 8) {    // pose block: the 200-byte result, then 56 zero bytes
    const int w = tid - 16;
    reinterpret_cast<uint64_t*>(rec + record_bytes(S))[w] =
        w < B2S_POSE_RESULT_BYTES / 8 ? reinterpret_cast<const uint64_t*>(r)[w] : 0ull;
  }
  uint16_t* rq = reinterpret_cast<uint16_t*>(rec + 64);
  uint16_t* rt = rq + S;
  uint16_t* rd = rt + S;
  uint8_t* rm = reinterpret_cast<uint8_t*>(rd + S);
  const size_t base = (size_t)pair * S;
  for (int k = tid; k < S; k += kDecideThreads) {
    const bool live = k < n;
    rq[k] = live ? (uint16_t)sink.out_q[base + k] : (uint16_t)0;
    rt[k] = live ? (uint16_t)sink.out_t[base + k] : (uint16_t)0;
    rd[k] = live ? (uint16_t)sink.out_d[base + k] : (uint16_t)0;
    rm[k] = (live && from) ? from[off + k] : (uint8_t)0;
  }
  for (size_t k = 64 + 7 * (size_t)S + tid; k < record_bytes(S); k += kDecideThreads) rec[k] = 0;   // every byte is defined
}

}  // namespace b2s

extern "C" {

int b2s_displacement_median_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, const uint8_t* mask,
                                    int n_pairs, const b2s_robust_pose_config* cfg, int n_cfg, float* median_out,
                                    double* th_out, double* th2_out, void* stream) {
  using namespace b2s;
  B2S_REQUIRE(corr && c_off && c_count, "null pointer");
  B2S_REQUIRE(n_pairs >= 0, "negative size");
  B2S_REQUIRE(cfg == nullptr || n_cfg == 1 || n_cfg == n_pairs, "n_cfg must be 1 or n_pairs");
  if (n_pairs == 0) return B2S_OK;
  displacement_median_kernel<<<n_pairs, kMedThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(corr), c_off, c_count, mask, cfg, n_cfg, median_out, th_out, th2_out);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  return B2S_OK;
}

int b2s_refit_homography_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, const uint8_t* mask,
                                 int n_pairs, double* H_out, int32_t* n_used, void* stream) {
  using namespace b2s;
  B2S_REQUIRE(corr && c_off && c_count && H_out, "null pointer");
  B2S_REQUIRE(n_pairs >= 0, "negative size");
  if (n_pairs == 0) return B2S_OK;
  refit_homography_kernel<<<n_pairs, kHRefitThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(corr), c_off, c_count, mask, H_out, n_used);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  return B2S_OK;
}

static int robust_pose_decide(const int32_t* c_off, const int32_t* c_count, int n_pairs, const int32_t* e_best_h,
                              const int32_t* e_inliers, const uint8_t* e_mask, const double* e_R, const double* e_t,
                              const int32_t* e_votes, const float* e_median, const float* all_median, const double* th,
                              const int32_t* h_best_h, const int32_t* h_inliers, const uint8_t* h_mask, const double* H_fit,
                              const double* Kinv_host, const b2s_robust_pose_config* cfg, int n_cfg,
                              b2s_pose_result* results, uint8_t* out_mask, int mask_stride, const b2s_record_sink* sink,
                              void* stream) {
  using namespace b2s;
  B2S_REQUIRE(c_off && c_count && e_best_h && e_inliers && e_mask && e_R && e_t && e_votes && e_median && all_median && th &&
                  h_best_h && h_inliers && h_mask && H_fit && cfg && results && out_mask, "null pointer");
  B2S_REQUIRE(n_pairs >= 0, "negative size");
  B2S_REQUIRE(n_cfg == 1 || n_cfg == n_pairs, "n_cfg must be 1 or n_pairs");
  b2s_record_sink sk{};
  if (sink && sink->records) {
    B2S_REQUIRE(sink->out_q && sink->out_t && sink->out_d && sink->stride > 0, "record sink: selection outputs and stride required");
    B2S_REQUIRE(sink->record_bytes >= pose_record_bytes(sink->stride) && (sink->record_bytes & 15u) == 0 &&
                    ((uintptr_t)sink->records & 15u) == 0,
                "record sink: record_bytes (%zu) must be >= b2s_pose_record_bytes(stride) = %zu and 16-byte aligned",
                sink->record_bytes, pose_record_bytes(sink->stride));
    sk = *sink;
  }
  if (n_pairs == 0) return B2S_OK;
  Mat3Arg Kinv;
  for (int i = 0; i < 9; ++i) Kinv.m[i] = Kinv_host ? Kinv_host[i] : ((i % 4 == 0) ? 1.0 : 0.0);
  robust_pose_decide_kernel<<<n_pairs, kDecideThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      c_off, c_count, e_best_h, e_inliers, e_mask, e_R, e_t, e_votes, e_median, all_median, th, h_best_h, h_inliers,
      h_mask, H_fit, Kinv, cfg, n_cfg, results, out_mask, mask_stride, sk);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  return B2S_OK;
}

int b2s_robust_pose_decide(const int32_t* c_off, const int32_t* c_count, int n_pairs, const int32_t* e_best_h,
                           const int32_t* e_inliers, const uint8_t* e_mask, const double* e_R, const double* e_t,
                           const int32_t* e_votes, const float* e_median, const float* all_median, const double* th,
                           const int32_t* h_best_h, const int32_t* h_inliers, const uint8_t* h_mask, const double* H_fit,
                           const double* Kinv_host, const b2s_robust_pose_config* cfg, int n_cfg,
                           b2s_pose_result* results, uint8_t* out_mask, int mask_stride, void* stream) {
  return robust_pose_decide(c_off, c_count, n_pairs, e_best_h, e_inliers, e_mask, e_R, e_t, e_votes, e_median, all_median, th,
                            h_best_h, h_inliers, h_mask, H_fit, Kinv_host, cfg, n_cfg, results, out_mask, mask_stride, nullptr,
                            stream);
}

int b2s_robust_pose_decide_records(const int32_t* c_off, const int32_t* c_count, int n_pairs, const int32_t* e_best_h,
                                   const int32_t* e_inliers, const uint8_t* e_mask, const double* e_R, const double* e_t,
                                   const int32_t* e_votes, const float* e_median, const float* all_median, const double* th,
                                   const int32_t* h_best_h, const int32_t* h_inliers, const uint8_t* h_mask,
                                   const double* H_fit, const double* Kinv_host, const b2s_robust_pose_config* cfg, int n_cfg,
                                   b2s_pose_result* results, uint8_t* out_mask, int mask_stride, const b2s_record_sink* sink,
                                   void* stream) {
  return robust_pose_decide(c_off, c_count, n_pairs, e_best_h, e_inliers, e_mask, e_R, e_t, e_votes, e_median, all_median, th,
                            h_best_h, h_inliers, h_mask, H_fit, Kinv_host, cfg, n_cfg, results, out_mask, mask_stride, sink,
                            stream);
}

}  // extern "C"
