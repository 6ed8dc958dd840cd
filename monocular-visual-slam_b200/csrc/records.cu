// records.cu — fixed-size per-pair result records and the candidate ranking of the relocalization sweep.
//
// b2s_pack_records: the hot path ends with per-pair results scattered over seven arrays (match count, winning
// hypothesis, inlier count, R | t, and max_matches x (queryIdx, trainIdx, distance, inlier flag)).  The
// reference hands them back as Python objects (feature_pipeline.py.bak:78-95 -> list[DMatch];
// homography.py:423-438 -> (R, t, inliers, match_count)).  Here one kernel writes them as ONE fixed-size
// record per pair straight into the buffer that leaves the GPU: the send slice of the NCCL all-gather when
// pairs are sharded over GPUs (SURVEY.md 8e: "count, best_h, inlier_count, R|t 12 x f32, matches 500 x
// (u16, u16, u16)"), or the single device->host copy of a step (it was seven).
//
// b2s_rank_pairs: the relocalizer verifies only the best `k` candidates (persistent_map.py:242,
// max_candidates); in the whole-map sweep (BASELINE config #5) the candidates are ranked by cross-check match
// count, ties to the lower frame id (the reference's (-score, frame_id) order, persistent_map.py:236-241).  One
// CTA ranks all pairs and emits the CSR view (c_off, c_count) of the winners' correspondences, so the RANSAC
// kernels run on them without a host round trip.
#include "common.cuh"

namespace b2s {

// record layout: record_bytes / pose_record_bytes (common.cuh)

struct PackParams {
  const int32_t* __restrict__ count;
  const int32_t* __restrict__ count_total;  // optional: header[0] (matches before truncation), default count
  const int32_t* __restrict__ best_h;
  const int32_t* __restrict__ best_count;
  const int32_t* __restrict__ out_q;
  const int32_t* __restrict__ out_t;
  const int32_t* __restrict__ out_d;
  const uint8_t* __restrict__ mask;
  const double* __restrict__ R;
  const double* __restrict__ t;
  const int32_t* __restrict__ pair_ids;  // optional: id written into the header (default pair_id0 + p)
  const int32_t* __restrict__ src_pair;  // optional: record p describes input pair src_pair[p] (ranked candidates)
  int stride, pair_id0;
  uint8_t* __restrict__ records;
  size_t rec_bytes;
};

__global__ void __launch_bounds__(128) pack_records_kernel(const PackParams p) {
  const int r = blockIdx.x, tid = threadIdx.x;
  const int pair = p.src_pair ? p.src_pair[r] : r;
  uint8_t* rec = p.records + (size_t)r * p.rec_bytes;
  int32_t* hdr = reinterpret_cast<int32_t*>(rec);
  const int S = p.stride;
  uint16_t* rq = reinterpret_cast<uint16_t*>(rec + 64);
  uint16_t* rt = rq + S;
  uint16_t* rd = rt + S;
  uint8_t* rm = reinterpret_cast<uint8_t*>(rd + S);
  if (pair < 0) {  // an empty candidate slot
    if (tid < 16) hdr[tid] = tid == 3 ? -1 : 0;
    for (int k = tid; k < S; k += blockDim.x) rq[k] = rt[k] = rd[k] = 0, rm[k] = 0;
    return;
  }
  const int n = max(0, min(p.count[pair], S));
  const int rp = p.src_pair ? r : pair;   // ranked candidates: the RANSAC / pose arrays hold one entry per CANDIDATE
  if (tid < 16) {
    int32_t v = 0;
    if (tid == 0) v = p.count_total ? p.count_total[pair] : p.count[pair];
    else if (tid == 1) v = p.best_h ? p.best_h[rp] : -1;
    else if (tid == 2) v = p.best_count ? p.best_count[rp] : 0;
    else if (tid == 3) v = p.pair_ids ? p.pair_ids[pair] : p.pair_id0 + pair;
    else if (tid < 13) v = p.R ? __float_as_int((float)p.R[(size_t)rp * 9 + (tid - 4)]) : 0;
    else v = p.t ? __float_as_int((float)p.t[(size_t)rp * 3 + (tid - 13)]) : 0;
    hdr[tid] = v;
  }
  const size_t base = (size_t)pair * S;
  for (int k = tid; k < S; k += blockDim.x) {
    const bool live = k < n;
    rq[k] = live ? (uint16_t)p.out_q[base + k] : (uint16_t)0;
    rt[k] = live ? (uint16_t)p.out_t[base + k] : (uint16_t)0;
    rd[k] = live ? (uint16_t)p.out_d[base + k] : (uint16_t)0;
    rm[k] = (live && p.mask) ? p.mask[base + k] : (uint8_t)0;
  }
}

// ---- ranking: the k pairs with the largest score, ties to the lower id ------------------------------
// One CTA, k <= 32 rounds of a block-wide arg-max over the key (score, ~id, ~index), each round looking only
// below the key taken before it: n = 4541 pairs and k = 5 is ~25 us of latency-bound work once per query; not a
// throughput kernel.
struct RankKey {
  unsigned long long hi;  // score << 32 | ~id   (larger score first, then the lower id)
  uint32_t lo;            // ~index             (then the lower position; makes every key unique)
};
__device__ __forceinline__ bool rank_before(const RankKey& a, const RankKey& b) { return a.hi > b.hi || (a.hi == b.hi && a.lo > b.lo); }
__device__ __forceinline__ RankKey rank_shfl(const RankKey& k, int o) {
  RankKey r;
  r.hi = __shfl_xor_sync(0xFFFFFFFFu, k.hi, o);
  r.lo = __shfl_xor_sync(0xFFFFFFFFu, k.lo, o);
  return r;
}

__global__ void __launch_bounds__(1024) rank_pairs_kernel(const int32_t* __restrict__ score, const int32_t* __restrict__ ids,
                                                          const int32_t* __restrict__ sel_count, int n, int k, int stride,
                                                          int32_t* __restrict__ top_idx, int32_t* __restrict__ top_id,
                                                          int32_t* __restrict__ c_off, int32_t* __restrict__ c_count) {
  __shared__ RankKey s_best[32];
  __shared__ RankKey s_last;   // the key taken in the previous round: later rounds only look below it
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int round = 0; round < k; ++round) {
    RankKey best{0ull, 0u};
    bool have = false;
    const RankKey last = s_last;   // (uninitialised in round 0, unused there)
    for (int i = tid; i < n; i += blockDim.x) {
      const int sc = score[i];
      if (sc < 0) continue;
      const uint32_t id = ids ? (uint32_t)ids[i] : (uint32_t)i;
      const RankKey key{((unsigned long long)(uint32_t)sc << 32) | (unsigned long long)(0xFFFFFFFFu - id), 0xFFFFFFFFu - (uint32_t)i};
      if (round > 0 && !rank_before(last, key)) continue;   // already taken (or the one just taken)
      if (!have || rank_before(key, best)) best = key, have = true;
    }
    // invalid lanes carry {0, 0}: below every real key (lo = ~i >= 2^32 - n > 0)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const RankKey v = rank_shfl(best, o);
      if (rank_before(v, best)) best = v;
    }
    if (lane == 0) s_best[warp] = best;
    __syncthreads();
    if (warp == 0) {
      RankKey b = lane < (int)(blockDim.x >> 5) ? s_best[lane] : RankKey{0ull, 0u};
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const RankKey v = rank_shfl(b, o);
        if (rank_before(v, b)) b = v;
      }
      if (lane == 0) {
        const bool found = b.lo != 0u;
        const int i = found ? (int)(0xFFFFFFFFu - b.lo) : -1;
        if (found) s_last = b;
        else s_last = RankKey{0ull, 0u};   // nothing below: every later round is empty too
        top_idx[round] = i;
        if (top_id) top_id[round] = i >= 0 ? (ids ? ids[i] : i) : -1;
        if (c_off) c_off[round] = i >= 0 ? i * stride : 0;
        if (c_count) c_count[round] = (i >= 0 && sel_count) ? max(0, sel_count[i]) : 0;
      }
    }
    __syncthreads();
  }
}

}  // namespace b2s

extern "C" {

size_t b2s_record_bytes(int max_matches) { return b2s::record_bytes(max_matches); }
size_t b2s_pose_record_bytes(int max_matches) { return b2s::pose_record_bytes(max_matches); }

int b2s_pack_records(const int32_t* count, const int32_t* count_total, const int32_t* best_h, const int32_t* best_count, const int32_t* out_q,
                     const int32_t* out_t, const int32_t* out_d, const uint8_t* inlier_mask, const double* R,
                     const double* t, const int32_t* pair_ids, const int32_t* src_pair, int n_records, int stride,
                     int pair_id0, uint8_t* records, size_t record_bytes, void* stream) {
  using namespace b2s;
  B2S_REQUIRE(n_records >= 0 && stride > 0, "bad size");
  B2S_REQUIRE(count && out_q && out_t && out_d && records, "null pointer");
  B2S_REQUIRE(record_bytes >= b2s::record_bytes(stride) && (record_bytes & 15u) == 0 && ((uintptr_t)records & 15u) == 0,
              "record_bytes must be >= b2s_record_bytes(stride) and 16-byte aligned");
  B2S_REQUIRE((R == nullptr) == (t == nullptr), "pass both R and t or neither");
  if (n_records == 0) return B2S_OK;
  PackParams p{count, count_total, best_h, best_count, out_q, out_t, out_d, inlier_mask, R, t, pair_ids, src_pair, stride, pair_id0, records, record_bytes};
  pack_records_kernel<<<n_records, 128, 0, static_cast<cudaStream_t>(stream)>>>(p);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  return B2S_OK;
}

int b2s_rank_pairs(const int32_t* score, const int32_t* ids, const int32_t* sel_count, int n, int k, int stride,
                   int32_t* top_idx, int32_t* top_id, int32_t* c_off, int32_t* c_count, void* stream) {
  using namespace b2s;
  B2S_REQUIRE(score && top_idx, "null pointer");
  B2S_REQUIRE(n >= 0 && n < (1 << 22) && k >= 0 && k <= 32 && stride >= 0, "rank_pairs: n < 2^22, k <= 32");
  if (k == 0) return B2S_OK;
  rank_pairs_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(score, ids, sel_count, n, k, stride, top_idx, top_id, c_off, c_count);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  return B2S_OK;
}

}  // extern "C"
