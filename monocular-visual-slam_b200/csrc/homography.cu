// homography.cu — K5/K6: batched RANSAC homography hypotheses (SURVEY.md §8f next-row #3).
//
// Replaces the body of the Python loop of ransac_homography
// (/root/reference/homography.py:192-211): the 4-point normalised DLT (dlt_homography,
// :131-142, with Hartley normalisation :118-125), the symmetric transfer error of every
// correspondence (:195-205) and the sequential best / early-exit bookkeeping (:207-211), for
// thousands of hypotheses and many frame pairs per launch.  float64 like the reference.
// The 8x9 DLT system goes through the same Householder null-vector routine as the 8-point
// essential-matrix solver (linalg.cuh); H is de-normalised and scaled to H[2][2] = 1, which
// also removes the sign / scale freedom of the null vector.
#include "linalg.cuh"

namespace b2s {

constexpr int kHomThreads = 128;

// inverse of a 3x3 matrix by the adjugate (the reference calls np.linalg.inv, :198)
__device__ __forceinline__ void inv3(const double (&h)[9], double (&o)[9]) {
  const double c0 = fma(h[4], h[8], -h[5] * h[7]);
  const double c1 = fma(h[5], h[6], -h[3] * h[8]);
  const double c2 = fma(h[3], h[7], -h[4] * h[6]);
  const double det = fma(h[0], c0, fma(h[1], c1, h[2] * c2));
  const double r = 1.0 / det;
  o[0] = c0 * r;
  o[1] = fma(h[2], h[7], -h[1] * h[8]) * r;
  o[2] = fma(h[1], h[5], -h[2] * h[4]) * r;
  o[3] = c1 * r;
  o[4] = fma(h[0], h[8], -h[2] * h[6]) * r;
  o[5] = fma(h[2], h[3], -h[0] * h[5]) * r;
  o[6] = c2 * r;
  o[7] = fma(h[1], h[6], -h[0] * h[7]) * r;
  o[8] = fma(h[0], h[4], -h[1] * h[3]) * r;
}

// symmetric transfer error < th (homography.py:195-206); NaN -> outlier
__device__ __forceinline__ bool transfer_inlier(const double (&h)[9], const double (&g)[9], double x, double y, double u,
                                                double v, double th) {
  const double pw = fma(h[6], x, fma(h[7], y, h[8]));
  const double px = fma(h[0], x, fma(h[1], y, h[2])) / pw;
  const double py = fma(h[3], x, fma(h[4], y, h[5])) / pw;
  const double qw = fma(g[6], u, fma(g[7], v, g[8]));
  const double qx = fma(g[0], u, fma(g[1], v, g[2])) / qw;
  const double qy = fma(g[3], u, fma(g[4], v, g[5])) / qw;
  const double e1 = sqrt(fma(px - u, px - u, (py - v) * (py - v)));
  const double e2 = sqrt(fma(qx - x, qx - x, (qy - y) * (qy - y)));
  return e1 + e2 < th;
}

// ---- K5: 4-point DLT, one thread per hypothesis ----------------------------------------
__global__ void __launch_bounds__(kHomThreads) homography_dlt_kernel(
    const float4* __restrict__ corr, const int32_t* __restrict__ c_off, const int32_t* __restrict__ c_count, int H,
    const int32_t* __restrict__ samples_in, uint64_t seed, const int32_t* __restrict__ pair_ids, int pair_id0,
    int32_t* __restrict__ samples_out, double* __restrict__ H_out) {
  const int pair = blockIdx.y;
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  const int M = max(c_count[pair], 0);   // a negative count is the selection kernel's overflow flag: no model
  const float4* cp = corr + c_off[pair];
  double* ho = H_out + ((size_t)pair * H + h) * 9;
  int idx[4];
  if (samples_in) {
    for (int k = 0; k < 4; ++k) idx[k] = samples_in[((size_t)pair * H + h) * 4 + k];
  } else if (M >= 4) {
    draw_distinct<4>(seed, pair_ids ? pair_ids[pair] : pair_id0 + pair, h, M, idx);   // keyed by the GLOBAL pair id
  } else {
    for (int k = 0; k < 4; ++k) idx[k] = 0;
  }
  if (samples_out)
    for (int k = 0; k < 4; ++k) samples_out[((size_t)pair * H + h) * 4 + k] = idx[k];
  bool ok = M >= 4;
  for (int k = 0; k < 4; ++k) ok &= (idx[k] >= 0 && idx[k] < M);
  if (!ok) {
    for (int k = 0; k < 9; ++k) ho[k] = 0.0;
    return;
  }
  double sx[4], sy[4], dx[4], dy[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float4 c = cp[idx[k]];
    sx[k] = c.x, sy[k] = c.y, dx[k] = c.z, dy[k] = c.w;
  }
  // Hartley normalisation of the two 4-point sets (homography.py:118-125)
  const double csx = 0.25 * ((sx[0] + sx[1]) + (sx[2] + sx[3])), csy = 0.25 * ((sy[0] + sy[1]) + (sy[2] + sy[3]));
  const double cdx = 0.25 * ((dx[0] + dx[1]) + (dx[2] + dx[3])), cdy = 0.25 * ((dy[0] + dy[1]) + (dy[2] + dy[3]));
  double vs = 0.0, vd = 0.0;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    vs += fma(sx[k] - csx, sx[k] - csx, (sy[k] - csy) * (sy[k] - csy));
    vd += fma(dx[k] - cdx, dx[k] - cdx, (dy[k] - cdy) * (dy[k] - cdy));
  }
  const double ss = sqrt(2.0) / sqrt(0.25 * vs), sd = sqrt(2.0) / sqrt(0.25 * vd);   // inf for coincident points, as in the reference
  double A[8][9];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const double x = ss * (sx[k] - csx), y = ss * (sy[k] - csy), u = sd * (dx[k] - cdx), v = sd * (dy[k] - cdy);
    A[2 * k][0] = -x;  A[2 * k][1] = -y;  A[2 * k][2] = -1.0;
    A[2 * k][3] = 0.0; A[2 * k][4] = 0.0; A[2 * k][5] = 0.0;
    A[2 * k][6] = u * x; A[2 * k][7] = u * y; A[2 * k][8] = u;
    A[2 * k + 1][0] = 0.0; A[2 * k + 1][1] = 0.0; A[2 * k + 1][2] = 0.0;
    A[2 * k + 1][3] = -x;  A[2 * k + 1][4] = -y;  A[2 * k + 1][5] = -1.0;
    A[2 * k + 1][6] = v * x; A[2 * k + 1][7] = v * y; A[2 * k + 1][8] = v;
  }
  double n[9];
  null_vector_8x9(A, n);
  // H = T_dst^-1 Hn T_src with T = [s 0 -s c; 0 s -s c; 0 0 1]  (homography.py:141)
  double M1[9];  // Hn T_src
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    M1[3 * r + 0] = n[3 * r + 0] * ss;
    M1[3 * r + 1] = n[3 * r + 1] * ss;
    M1[3 * r + 2] = fma(-ss * csx, n[3 * r + 0], fma(-ss * csy, n[3 * r + 1], n[3 * r + 2]));
  }
  const double isd = 1.0 / sd;
  double Hm[9];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    Hm[c] = fma(isd, M1[c], cdx * M1[6 + c]);
    Hm[3 + c] = fma(isd, M1[3 + c], cdy * M1[6 + c]);
    Hm[6 + c] = M1[6 + c];
  }
  const double r22 = 1.0 / Hm[8];
#pragma unroll
  for (int k = 0; k < 9; ++k) ho[k] = Hm[k] * r22;
}

// ---- K6: transfer-error scoring, one thread per hypothesis -----------------------------
constexpr int kHomChunk = 1024;

__global__ void __launch_bounds__(kHomThreads) homography_score_kernel(
    const float4* __restrict__ corr, const int32_t* __restrict__ c_off, const int32_t* __restrict__ c_count,
    const double* __restrict__ Hm, int H, double th_all, const double* __restrict__ th_pp, int32_t* __restrict__ counts) {
  struct alignas(16) P4 { double x, y, u, v; };
  __shared__ P4 s_p[kHomChunk];
  const int pair = blockIdx.y;
  const int h = blockIdx.x * kHomThreads + threadIdx.x;
  const int M = max(c_count[pair], 0);   // a negative count is the selection kernel's overflow flag: no model
  const float4* cp = corr + c_off[pair];
  const double th = th_pp ? th_pp[pair] : th_all;
  const bool live = h < H;
  double hm[9], gi[9];
  {
    const double* hp = Hm + ((size_t)pair * H + (live ? h : 0)) * 9;
#pragma unroll
    for (int k = 0; k < 9; ++k) hm[k] = hp[k];
  }
  inv3(hm, gi);
  int count = 0;
  for (int base = 0; base < M; base += kHomChunk) {
    const int n = min(kHomChunk, M - base);
    __syncthreads();
    for (int m = threadIdx.x; m < n; m += kHomThreads) {
      const float4 c = __ldg(cp + base + m);
      s_p[m] = P4{(double)c.x, (double)c.y, (double)c.z, (double)c.w};
    }
    __syncthreads();
#pragma unroll 2
    for (int m = 0; m < n; ++m) {
      const P4 c = s_p[m];
      count += transfer_inlier(hm, gi, c.x, c.y, c.u, c.v, th) ? 1 : 0;
    }
  }
  if (live) counts[(size_t)pair * H + h] = count;
}

// ---- winner selection + inlier mask (same sequential rule as ransac_select_kernel) ------
__global__ void __launch_bounds__(256) homography_select_kernel(
    const int32_t* __restrict__ counts, const float4* __restrict__ corr, const int32_t* __restrict__ c_off,
    const int32_t* __restrict__ c_count, const double* __restrict__ Hm, int H, double th_all,
    const double* __restrict__ th_pp, int32_t* __restrict__ best_h, int32_t* __restrict__ best_count,
    uint8_t* __restrict__ mask) {
  __shared__ int s_early;
  __shared__ unsigned long long s_best;
  __shared__ int s_cnt;
  const int pair = blockIdx.x, tid = threadIdx.x;
  const int M = max(c_count[pair], 0);   // a negative count is the selection kernel's overflow flag: no model
  if (tid == 0) {
    s_early = 0x7FFFFFFF;
    s_best = 0ull;
    s_cnt = 0;
  }
  __syncthreads();
  const double early_thr = 0.8 * (double)M;  // "inliers.size > 0.8 * n" (homography.py:210)
  int early = 0x7FFFFFFF;
  unsigned long long bestk = 0ull;
  for (int h = tid; h < H; h += blockDim.x) {
    const int c = counts[(size_t)pair * H + h];
    if ((double)c > early_thr) early = min(early, h);
    const unsigned long long k = ((unsigned long long)(uint32_t)c << 32) | (uint32_t)(0xFFFFFFFFu - (uint32_t)h);
    bestk = max(bestk, k);
  }
  if (early != 0x7FFFFFFF) atomicMin(&s_early, early);
  atomicMax(&s_best, bestk);
  __syncthreads();
  int win;
  if (s_early != 0x7FFFFFFF) win = s_early;
  else win = ((s_best >> 32) == 0ull) ? -1 : (int)(0xFFFFFFFFu - (uint32_t)(s_best & 0xFFFFFFFFull));
  const float4* cp = corr + c_off[pair];
  uint8_t* mp = mask + c_off[pair];
  int mine = 0;
  if (win >= 0) {
    double hm[9], gi[9];
    const double* hp = Hm + ((size_t)pair * H + win) * 9;
#pragma unroll
    for (int k = 0; k < 9; ++k) hm[k] = hp[k];
    inv3(hm, gi);
    const double th = th_pp ? th_pp[pair] : th_all;
    for (int m = tid; m < M; m += blockDim.x) {
      const float4 c = cp[m];
      const bool in = transfer_inlier(hm, gi, (double)c.x, (double)c.y, (double)c.z, (double)c.w, th);
      mp[m] = in ? 1 : 0;
      mine += in ? 1 : 0;
    }
  } else {
    for (int m = tid; m < M; m += blockDim.x) mp[m] = 0;
  }
  if (mine) atomicAdd(&s_cnt, mine);
  __syncthreads();
  if (tid == 0) {
    best_h[pair] = win;
    best_count[pair] = s_cnt;
  }
}

}  // namespace b2s

extern "C" {

int b2s_homography_dlt_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, int n_pairs, int H,
                               const int32_t* samples_in, uint64_t seed, const int32_t* pair_ids, int pair_id0,
                               int32_t* samples_out, double* H_out, void* stream) {
  using namespace b2s;
  B2S_REQUIRE(corr && c_off && c_count && H_out, "null pointer");
  B2S_REQUIRE(n_pairs >= 0 && H >= 0, "negative size");
  B2S_REQUIRE(n_pairs <= 65535, "n_pairs %d exceeds grid.y limit 65535; split the batch", n_pairs);
  if (n_pairs == 0 || H == 0) return B2S_OK;
  dim3 grid((H + kHomThreads - 1) / kHomThreads, n_pairs);
  homography_dlt_kernel<<<grid, kHomThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(corr), c_off, c_count, H, samples_in, seed, pair_ids, pair_id0, samples_out, H_out);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  return B2S_OK;
}

int b2s_homography_score_batched(const float* corr, const int32_t* c_off, const int32_t* c_count, int n_pairs,
                                 const double* Hm, int H, double th, const double* th_per_pair, int32_t* counts,
                                 void* stream) {
  using namespace b2s;
  B2S_REQUIRE(corr && c_off && c_count && Hm && counts, "null pointer");
  B2S_REQUIRE(n_pairs >= 0 && H >= 0, "negative size");
  B2S_REQUIRE(n_pairs <= 65535, "n_pairs %d exceeds grid.y limit 65535; split the batch", n_pairs);
  if (n_pairs == 0 || H == 0) return B2S_OK;
  dim3 grid((H + kHomThreads - 1) / kHomThreads, n_pairs);
  homography_score_kernel<<<grid, kHomThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<const float4*>(corr), c_off, c_count, Hm, H, th, th_per_pair, counts);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  return B2S_OK;
}

int b2s_homography_select(const int32_t* counts, const float* corr, const int32_t* c_off, const int32_t* c_count,
                          int n_pairs, const double* Hm, int H, double th, const double* th_per_pair, int32_t* best_h,
                          int32_t* best_count, uint8_t* inlier_mask, void* stream) {
  using namespace b2s;
  B2S_REQUIRE(counts && corr && c_off && c_count && Hm && best_h && best_count && inlier_mask, "null pointer");
  B2S_REQUIRE(n_pairs >= 0 && H >= 0, "negative size");
  if (n_pairs == 0) return B2S_OK;
  homography_select_kernel<<<n_pairs, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      counts, reinterpret_cast<const float4*>(corr), c_off, c_count, Hm, H, th, th_per_pair, best_h, best_count,
      inlier_mask);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  return B2S_OK;
}

}  // extern "C"
