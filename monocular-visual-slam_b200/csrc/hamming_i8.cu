// hamming_i8.cu — K2: Hamming kNN-2 + column minimum on the 5th-gen tensor cores.
//
// Same contract as K1 (hamming_popc.cu); replaces the same reference calls
// (/root/reference/feature_pipeline.py.bak:68,82,84; homography.py:12-15,21-23).
//
// Hamming as a dense contraction whose result already IS a 16-bit sort key.  Query bits map
// to +-8 (bit b -> 8(1-2b)), train bits to -+8, so a 256-byte dot product is 128*ham - 2^14
// exactly.  One more K-step multiplies a constant "ones" block [1, 64 x8, 0..] (A side, lives
// in shared memory for the whole kernel) with the B-side tile's "index" chunk
// [row mod 128, 64 x4, 0..], adding the tile-local column and cancelling the bias:
//     acc = 128*ham + (row mod 128)            0 <= acc <= 32895, i.e. a 16-bit key.
// Rows past the end of a pair carry zero data and the index chunk [127 x9, 0..], which yields
// acc = 65151: larger than every valid key, still 16 bits — no tail masking in the epilogue.
// Unsigned 16-bit min over keys is the lexicographic (distance, index) minimum = OpenCV's tie
// rule, so the epilogue is tcgen05.ld.pack::16b (two columns per register) followed by packed
// VIMNMX.U16x2 / VIMNMX3.U16x2 only: 1.25 instructions per element for the per-row top-2 and
// 0.25 for the column minimum (the 32-bit-key version needed 2.5 + 0.5).  Once per 128-column
// tile the two packed halves are folded and widened into the global packed key.
// tcgen05.mma kind::i8 (M=128, N=128, K=32 per instruction, int32 accumulators in TMEM)
// produces a 128x128 tile in 9 instructions.
//
// Two products per tile pair so that BOTH reductions are per-thread (a TMEM lane is a
// matrix row and each epilogue thread owns one lane):
//     D1 = Qtile . Ttile^T   lanes = queries,  columns = train rows  -> per-row top-2
//     D2 = Ttile . Qtile^T   lanes = train rows, columns = queries   -> per-column minimum
// Both read the same two shared-memory tiles (K-major, canonical no-swizzle core-matrix
// layout), only the A/B descriptor roles swap.
//
// Pipeline (persistent CTAs, one per SM, 320 threads; work item = (pair, 128-query tile)):
//   warp 0   producer : cp.async.bulk (TMA engine) of pre-expanded 34 KB operand tiles into
//                       a 4-stage ring + a double-buffered query tile, mbarrier expect_tx
//   warp 1   MMA      : one thread issues 18 tcgen05.mma per train tile, tcgen05.commit
//                       releases the smem stage and publishes the TMEM accumulator stage
//   warps 2-9 epilogue: two sets of 4 warps; set e owns TMEM stage e (every other tile pair),
//                       thread = TMEM lane, 4 x tcgen05.ld.32x32b.x32.pack::16b per tile pair
//                       software-pipelined against the packed min/max folds
// TMEM: 2 accumulator stages x (D1 128 cols + D2 128 cols) = 512 columns.
#include "tcgen05.cuh"

namespace b2s {

constexpr int kI8Tile = 128;                      // rows per operand tile
constexpr int kI8Chunks = 17;                     // 16-byte k-chunks per row: 16 data + 1 index
constexpr int kI8ChunkBytes = kI8Tile * 16;       // 2048: one k-chunk of all 128 rows (= LBO)
constexpr int kI8TileBytes = kI8Chunks * kI8ChunkBytes;  // 34 KB
constexpr int kI8Units = kI8Chunks * kI8Tile;     // 16-byte units per tile
constexpr int kI8Stages = 4;
constexpr int kI8Threads = 320;
constexpr uint32_t kKey16Valid = 32896u;          // 16-bit keys below this are real (ham <= 256, col <= 127)
constexpr uint32_t kKey32Pad = 0x7F000000u;       // widened padding / initial keys land at or above this

// ---- pre-pass: 256 bits -> 256 int8 (+-8) + index chunk, UMMA canonical K-major layout
// Tile = 128 rows x 17 k-chunks of 16 bytes.  Unit (row r, k-chunk kc) sits at unit index
// kc*128 + r: 8 rows x 16 B form one 128-byte core matrix, 8-row groups are 128 B apart
// (SBO), k-chunks 2048 B apart (LBO).
__device__ __forceinline__ uint32_t spread4(uint32_t nib, bool train) {
  const uint32_t sp = (nib * 0x00204081u) & 0x01010101u;  // bit i -> byte i (0 or 1)
  // query: +8 / -8 for clear / set;  train: -8 / +8
  return train ? (0xF8F8F8F8u - sp * 0xF0u) : (0x08080808u + sp * 0xF0u);
}

// Unified tiles (single-product kernel): 18 chunks, the same tile serves a frame as query and as
// train operand.  Data: bit clear / set -> +8 / -8 on both sides, so the 8 data K-steps give
// 64 (256 - 2 ham) = 2^14 - 128 ham: the accumulator DEcreases with the distance.  The index K-step
// multiplies the query tile's chunk 17 with the train tile's chunk 16:
//     A (chunk 17) [-1, r, 127, 127, 127, 127, 2, 0..]     B (chunk 16) [c, -1, 127, 127, 127, 6, 1, 0..]
// = -c - r + 3 * 16129 + 762 + 2 = 49151 - c - r, so that  acc = 65535 - (128 ham + c + r) = ~key:
// the COMPLEMENT of the 16-bit key 128 ham + column + row.  The epilogue takes maxima instead of
// minima and complements its few results.  Padding rows are all zero on both sides: acc = 0, below
// every real value (>= 32513), and 65535 = "none" after the complement.
// Otherwise two-product tiles (17 chunks; index chunk [r, 64 x4, 0..], padding rows [127 x9, 0..]).
__global__ void __launch_bounds__(128) expand_pm8_kernel(const uint8_t* __restrict__ desc,
                                                         const int32_t* __restrict__ off,
                                                         const int32_t* __restrict__ src, int tiles_per_pair,
                                                         int train, bool unified, uint4* __restrict__ out,
                                                         const int32_t* __restrict__ blk_rows,
                                                         const int32_t* __restrict__ blk_tile0) {
  // one CTA per (tile, pair), one thread per row: the row's 32 bytes are read once (2 x LDG.128)
  // and its 17 / 18 k-chunks leave as STG.128 that are contiguous across the 128 threads.
  const int chunks = unified ? kI8Chunks + 1 : kI8Chunks;
  const int pair = blockIdx.y, tile = blockIdx.x, r = threadIdx.x;
  // block mode (blk_rows != nullptr): "pair" is a descriptor BLOCK (a frame) shared by several pairs:
  // blk_rows[b] rows starting at input row src[b], expanded once to tiles blk_tile0[b] ...
  const int o = blk_rows ? 0 : off[pair];
  const int n = blk_rows ? blk_rows[pair] : off[pair + 1] - o;
  if (tile * kI8Tile >= n) return;  // tile never read
  const int in0 = src ? src[pair] : o;
  const int row = tile * kI8Tile + r;
  const bool valid = row < n;
  const size_t tile_idx = blk_rows ? (size_t)blk_tile0[pair] + tile : (size_t)pair * tiles_per_pair + tile;
  uint4* dst = out + tile_idx * (size_t)(chunks * kI8Tile) + r;
  uint4 lo = make_uint4(0, 0, 0, 0), hi = lo;
  if (valid) {
    const uint4* p = reinterpret_cast<const uint4*>(desc + (size_t)(in0 + row) * B2S_DESC_BYTES);
    lo = __ldg(p);
    hi = __ldg(p + 1);
  }
  const uint32_t w[8] = {lo.x, lo.y, lo.z, lo.w, hi.x, hi.y, hi.z, hi.w};
#pragma unroll
  for (int kc = 0; kc < 16; ++kc) {
    uint4 v = make_uint4(0, 0, 0, 0);
    if (valid) {
      const uint32_t bits = (w[kc >> 1] >> (16 * (kc & 1))) & 0xFFFFu;   // descriptor bytes 2 kc, 2 kc + 1
      const bool tr = train && !unified;   // unified tiles: one sign for both roles
      v.x = spread4(bits & 15u, tr);
      v.y = spread4((bits >> 4) & 15u, tr);
      v.z = spread4((bits >> 8) & 15u, tr);
      v.w = spread4((bits >> 12) & 15u, tr);
    }
    dst[kc * kI8Tile] = v;
  }
  if (unified) {
    // chunk 16 = index chunk of the row as a TRAIN row (B side; a train slot is then ONE contiguous
    // 34 KB copy), chunk 17 = as a QUERY row (A side); padding rows are all zero
    const uint32_t rr = (uint32_t)r;
    dst[17 * kI8Tile] = valid ? make_uint4(0x7F7F00FFu | (rr << 8), 0x00027F7Fu, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
    dst[16 * kI8Tile] = valid ? make_uint4(0x7F7FFF00u | rr, 0x0001067Fu, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
  } else {
    dst[16 * kI8Tile] = valid ? make_uint4((uint32_t)r | 0x40404000u, 0x00000040u, 0u, 0u)  // [r, 64, 64, 64, 64, 0, ...]
                              : make_uint4(0x7F7F7F7Fu, 0x7F7F7F7Fu, 0x0000007Fu, 0u);      // [127 x9, 0, ...] -> acc = 65151
  }
}

__device__ __forceinline__ void tc_mma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// instruction descriptor: S32 accumulate, signed 8-bit A and B, both K-major, M = 128, N = 128
constexpr uint32_t kIdescI8 = (2u << 4) | (1u << 7) | (1u << 10) | ((128u >> 3) << 17) | ((128u >> 4) << 24);

// The 18 MMAs of one tile pair as ONE asm block: 8 data K-steps + the index K-step into D1
// (A = query tile, B = train tile), the same into D2 with the roles swapped.  After the 14th
// MMA a non-consumed mbarrier.try_wait probes the barrier of the NEXT tile pair; its predicate
// is only read after the last MMA has been queued, so the probe's latency (and the hardware
// sleep until the phase completes) overlaps the MMA stream instead of idling the tensor pipe
// at the tile boundary (~170 clk per blocking wait, b2s_mma_microbench variants 2 vs 3).
// Returns 1 when the next tile pair's barrier phase was seen complete.
__device__ __forceinline__ uint32_t tc_mma_tile_pair(uint32_t d1, uint32_t d2, uint64_t qdesc, uint64_t tdesc,
                                                     uint64_t odesc, uint32_t idesc, uint64_t* next_bar,
                                                     uint32_t next_parity, uint32_t has_next) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred pacc, pnew, pprobe, pdone;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.eq.b32 pacc, 0, 0;\n\t"
      "setp.ne.b32 pnew, 0, 0;\n\t"
      "setp.ne.b32 pprobe, %9, 0;\n\t"
      "setp.ne.b32 pdone, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], %3, %4, %6, pnew;\n\t"
      "add.u64 da, %3, 256;\n\t"
      "add.u64 db, %4, 256;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %6, pacc;\n\t"
      "add.u64 da, %3, 512;\n\t"
      "add.u64 db, %4, 512;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %6, pacc;\n\t"
      "add.u64 da, %3, 768;\n\t"
      "add.u64 db, %4, 768;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %6, pacc;\n\t"
      "add.u64 da, %3, 1024;\n\t"
      "add.u64 db, %4, 1024;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %6, pacc;\n\t"
      "add.u64 da, %3, 1280;\n\t"
      "add.u64 db, %4, 1280;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %6, pacc;\n\t"
      "add.u64 da, %3, 1536;\n\t"
      "add.u64 db, %4, 1536;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %6, pacc;\n\t"
      "add.u64 da, %3, 1792;\n\t"
      "add.u64 db, %4, 1792;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %6, pacc;\n\t"
      "add.u64 db, %4, 2048;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], %5, db, %6, pacc;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%2], %4, %3, %6, pnew;\n\t"
      "add.u64 da, %4, 256;\n\t"
      "add.u64 db, %3, 256;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%2], da, db, %6, pacc;\n\t"
      "add.u64 da, %4, 512;\n\t"
      "add.u64 db, %3, 512;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%2], da, db, %6, pacc;\n\t"
      "add.u64 da, %4, 768;\n\t"
      "add.u64 db, %3, 768;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%2], da, db, %6, pacc;\n\t"
      "add.u64 da, %4, 1024;\n\t"
      "add.u64 db, %3, 1024;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%2], da, db, %6, pacc;\n\t"
      "@pprobe mbarrier.try_wait.parity.shared::cta.b64 pdone, [%7], %8;\n\t"
      "add.u64 da, %4, 1280;\n\t"
      "add.u64 db, %3, 1280;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%2], da, db, %6, pacc;\n\t"
      "add.u64 da, %4, 1536;\n\t"
      "add.u64 db, %3, 1536;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%2], da, db, %6, pacc;\n\t"
      "add.u64 da, %4, 1792;\n\t"
      "add.u64 db, %3, 1792;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%2], da, db, %6, pacc;\n\t"
      "add.u64 db, %3, 2048;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%2], %5, db, %6, pacc;\n\t"
      "selp.u32 %0, 1, 0, pdone;\n\t"
      "}"
      : "=r"(ok)
      : "r"(d1), "r"(d2), "l"(qdesc), "l"(tdesc), "l"(odesc), "r"(idesc), "r"(smem_u32(next_bar)), "r"(next_parity),
        "r"(has_next)
      : "memory");
  return ok;
}


// 64 accumulator columns -> 32 registers: register j = low16(col 2j+1) << 16 | low16(col 2j)
#define TMEM_LD_X32P(taddr, v)                                                                             \
  asm volatile(                                                                                            \
      "tcgen05.ld.sync.aligned.32x32b.x32.pack::16b.b32 "                                                  \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                            \
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"            \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),    \
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),           \
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),         \
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),         \
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])                                                              \
      : "r"(taddr))

// 16 TMEM lanes x 128 accumulator columns -> 32 registers (tools/probes/ld16x256.cu): with gr = lane / 4,
// tc = lane % 4, register j = 4 g + 2 r + b holds row  lane0 + gr + 8 r  and columns
// 16 g + 4 tc + 2 b (low half) and + 1 (high half).  A thread owns whole 4-column groups of TWO rows.
#define TMEM_LD_16X256_X8P(taddr, v)                                                                       \
  asm volatile(                                                                                            \
      "tcgen05.ld.sync.aligned.16x256b.x8.pack::16b.b32 "                                                  \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "                            \
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"            \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),    \
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),           \
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),         \
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),         \
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])                                                              \
      : "r"(taddr))

struct I8Params {
  const uint8_t* __restrict__ qx;  // expanded query tiles  [pair][q_tiles][34 KB]
  const uint8_t* __restrict__ tx;  // expanded train tiles  [pair][t_tiles][34 KB]
  const int32_t* __restrict__ q_off;
  const int32_t* __restrict__ t_off;
  uint32_t* __restrict__ fwd_best;
  uint32_t* __restrict__ fwd_second;
  uint32_t* __restrict__ bwd_best;
  int q_tiles, t_tiles, n_pairs;
  const int32_t* __restrict__ q_xt;  // optional (shared blocks): first expanded tile of each pair's query / train side,
  const int32_t* __restrict__ t_xt;  // both in the ONE unified buffer qx == tx; nullptr = pair * q_tiles / pair * t_tiles
  // single-product kernel only: t_split > 1 cuts every (pair, query block) into t_split work items along the
  // train axis; item `part` writes its rows' top-2 to partial[part * total_nq + row] and a merge kernel folds them
  int t_split;
  int total_nq;
  uint2* __restrict__ partial;
};

// 64 columns (32 packed registers) folded into 2 interleaved packed top-2 chains.  The low and
// the high 16-bit lane of every register are independent streams (even / odd columns).  Two
// registers per step: the two smallest of {best, second, lo, hi} are min(best, lo) and
// min3(second, max(best, lo), hi) — 5 instructions per 4 columns.
__device__ __forceinline__ void fold_top2_p16(const uint32_t (&v)[32], uint32_t (&b)[2], uint32_t (&s)[2]) {
#pragma unroll
  for (int k = 0; k < 32; k += 2) {
    const int c = (k >> 1) & 1;
    const uint32_t lo = __vminu2(v[k], v[k + 1]), hi = __vmaxu2(v[k], v[k + 1]);
    const uint32_t mb = __vmaxu2(b[c], lo);
    b[c] = __vminu2(b[c], lo);
    s[c] = __vimin3_u16x2(s[c], mb, hi);
  }
}
__device__ __forceinline__ void fold_min_p16(const uint32_t (&v)[32], uint32_t (&m)[2]) {
#pragma unroll
  for (int k = 0; k < 32; k += 2) {
    const int c = (k >> 1) & 1;
    m[c] = __vimin3_u16x2(m[c], v[k], v[k + 1]);
  }
}
__device__ __forceinline__ uint32_t swap16(uint32_t x) { return __byte_perm(x, 0, 0x1032); }
// tile-local 16-bit key (ham << 7 | col) -> packed key (ham << 22 | base + col); padding keys
// (>= kKey16Valid) land at or above kKey32Pad and are turned into "none" by the caller
__device__ __forceinline__ uint32_t key16_to_key32(uint32_t k16, uint32_t base) {
  return ((k16 & 0xFF80u) << (kIdxBits - 7)) | (base + (k16 & 127u));
}

// Persistent: gridDim.x CTAs (one per SM) walk the (pair, query tile) work items round-robin.
// TMEM, barriers and the train-tile ring are set up once; the ring and the accumulator stages
// keep cycling across work items (global tile counter g), and the query tile is double
// buffered, so the pipeline never drains between items.
__global__ void __launch_bounds__(kI8Threads, 1) hamming_knn2_i8_kernel(const I8Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_q = smem;                                   // 2 x 34 KB (double-buffered query tile)
  uint8_t* s_t = smem + 2 * kI8TileBytes;                // kI8Stages x 34 KB
  uint8_t* s_ones = smem + (2 + kI8Stages) * kI8TileBytes;  // 2 k-chunks: [1, 64 x8, 0..] | zeros
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_ones + 2 * kI8ChunkBytes);
  uint64_t* b_full = bars;                               // [kI8Stages]
  uint64_t* b_empty = bars + kI8Stages;                  // [kI8Stages]
  uint64_t* b_tfull = bars + 2 * kI8Stages;              // [2]
  uint64_t* b_qempty = bars + 2 * kI8Stages + 6;         // [2]
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 2 * kI8Stages + 8);
  uint2* s_merge = reinterpret_cast<uint2*>(bars + 2 * kI8Stages + 9);  // [128] the two epilogue sets meet here

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_items = p.n_pairs * p.q_tiles;

  // constant A-side operand of the index K-step (the second chunk multiplies whatever follows a
  // tile's index chunk in shared memory by zero)
  for (int i = threadIdx.x; i < 2 * kI8Tile; i += kI8Threads)
    reinterpret_cast<uint4*>(s_ones)[i] =
        (i < kI8Tile) ? make_uint4(0x40404001u, 0x40404040u, 0x00000040u, 0u) : make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> tensor-core reads

  if (threadIdx.x == 0) {
    // full[s] of tile pair g completes when (a) its operand tile(s) have landed (producer
    // expect_tx + TMA complete_tx) AND (b) the four epilogue warps that drained tile pair g-2
    // have released its TMEM stage — ONE wait per tile pair on the MMA thread: every blocking
    // wait there idles the tensor pipe for ~170 clk (b2s_mma_microbench variants 2 vs 3).
    for (int s = 0; s < kI8Stages; ++s) {
      mbar_init(&b_full[s], 5);
      mbar_init(&b_empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&b_tfull[a], 1);
      mbar_init(&b_qempty[a], 1);
      for (int k = 0; k < 4; ++k) mbar_arrive(&b_full[a]);  // tile pairs 0 and 1 find their TMEM stage free
    }
    mbar_fence_init();
  }
  if (warp == 1) {  // TMEM: all 512 columns (1 CTA per SM by shared-memory footprint)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(s_tmem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  // every role walks the same item sequence; items past a pair's last query tile are skipped
  if (warp == 0) {
    // ===== producer =====
    if (lane == 0) {
      uint32_t n = 0, g = 0;  // items seen by this CTA, train tiles streamed by this CTA
      for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
        const int pair = w / p.q_tiles, qt = w - pair * p.q_tiles;
        const int nq = p.q_off[pair + 1] - p.q_off[pair];
        const int nt = p.t_off[pair + 1] - p.t_off[pair];
        if (qt * kI8Tile >= nq || nt == 0) continue;
        const int n_tt = (nt + kI8Tile - 1) / kI8Tile;
        const uint32_t qb = n & 1u;
        const uint8_t* tsrc = p.tx + (size_t)pair * p.t_tiles * kI8TileBytes;
        for (int t = 0; t < n_tt; ++t, ++g) {
          const uint32_t s = g % kI8Stages;
          if (g >= kI8Stages) mbar_wait_bounded(&b_empty[s], ((g / kI8Stages) - 1u) & 1u);
          if (t == 0) {  // the item's query tile rides on the barrier of its first train tile
            if (n >= 2) mbar_wait_bounded(&b_qempty[qb], ((n >> 1) - 1u) & 1u);
            mbar_arrive_expect_tx(&b_full[s], 2 * kI8TileBytes);
            bulk_g2s(s_q + (size_t)qb * kI8TileBytes, p.qx + ((size_t)pair * p.q_tiles + qt) * kI8TileBytes,
                     kI8TileBytes, &b_full[s]);
          } else {
            mbar_arrive_expect_tx(&b_full[s], kI8TileBytes);
          }
          bulk_g2s(s_t + (size_t)s * kI8TileBytes, tsrc + (size_t)t * kI8TileBytes, kI8TileBytes, &b_full[s]);
        }
        ++n;
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (elect_one()) {
      uint32_t n = 0, g = 0;
      bool probed = false;  // the barrier of the coming tile pair was already seen complete
      const uint64_t odesc = make_smem_desc(smem_u32(s_ones));
      for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
        const int pair = w / p.q_tiles, qt = w - pair * p.q_tiles;
        const int nq = p.q_off[pair + 1] - p.q_off[pair];
        const int nt = p.t_off[pair + 1] - p.t_off[pair];
        if (qt * kI8Tile >= nq || nt == 0) continue;
        const int n_tt = (nt + kI8Tile - 1) / kI8Tile;
        const uint32_t qb = n & 1u;
        const uint64_t qdesc = make_smem_desc(smem_u32(s_q + (size_t)qb * kI8TileBytes));
        for (int t = 0; t < n_tt; ++t, ++g) {
          const uint32_t s = g % kI8Stages, a = g & 1u;
          if (!probed)  // operands landed AND TMEM stage a drained (first tile pair, item boundaries, late epilogue)
            mbar_wait_bounded(&b_full[s], (g / kI8Stages) & 1u);
          tc_fence_after();
          const uint64_t tdesc = make_smem_desc(smem_u32(s_t + (size_t)s * kI8TileBytes));
          const uint32_t d1 = tmem_base + a * 256u, d2 = d1 + 128u;
          const uint32_t gn = g + 1u;
          probed = tc_mma_tile_pair(d1, d2, qdesc, tdesc, odesc, kIdescI8, &b_full[gn % kI8Stages],
                                    (gn / kI8Stages) & 1u, (t + 1 < n_tt) ? 1u : 0u) != 0u;
          tc_commit(&b_empty[s]);  // smem stage reusable once these MMAs have read it
          tc_commit(&b_tfull[a]);  // accumulators complete
        }
        tc_commit(&b_qempty[qb]);  // query tile buffer reusable once this item's MMAs have read it
        ++n;
      }
    }
  } else {
    // ===== epilogue: 2 sets of 4 warps; warp%4 = TMEM lane quarter, set e handles tile pairs with g%2 == e =====
    const int quarter = warp & 3;
    const uint32_t eset = (uint32_t)(warp - 2) >> 2;
    const int row = quarter * 32 + lane;  // TMEM lane = tile row
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + eset * 256u;
    uint32_t g = 0;
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      const int pair = w / p.q_tiles, qt = w - pair * p.q_tiles;
      const int qo = p.q_off[pair], nq = p.q_off[pair + 1] - qo;
      const int q0 = qt * kI8Tile;
      if (q0 >= nq) continue;
      const int to = p.t_off[pair], nt = p.t_off[pair + 1] - to;
      if (nt == 0) continue;
      const int n_tt = (nt + kI8Tile - 1) / kI8Tile;
      const int nq_valid = min(kI8Tile, nq - q0);
      uint32_t gbest = kNone, gsecond = kNone;
      for (int t = 0; t < n_tt; ++t, ++g) {
        if ((g & 1u) != eset) continue;
        const int tbase = t * kI8Tile;
        const int nt_valid = min(kI8Tile, nt - tbase);
        mbar_wait_bounded(&b_tfull[eset], (g >> 1) & 1u);
        tc_fence_after();
        uint32_t v0[32], v1[32], v2[32], v3[32];
        uint32_t b[2] = {kNone, kNone}, s2[2] = {kNone, kNone}, m[2] = {kNone, kNone};
        // D1 columns 0-63 | 64-127, D2 columns 0-63 | 64-127: 128 packed registers, all four
        // loads in flight at once, and the TMEM stage goes back to the MMA thread as soon as
        // they have landed — before any of the folding (the stage is held for the load latency
        // only, so the MMA thread's probe of the next barrier finds it complete)
        TMEM_LD_X32P(lane_addr, v0);
        TMEM_LD_X32P(lane_addr + 64u, v1);
        TMEM_LD_X32P(lane_addr + 128u, v2);
        TMEM_LD_X32P(lane_addr + 192u, v3);
        tmem_ld_wait();
        TMEM_REGS_READY(v0);
        TMEM_REGS_READY(v1);
        TMEM_REGS_READY(v2);
        TMEM_REGS_READY(v3);
        tc_fence_before();
        __syncwarp();
        // accumulator stage drained into registers: release it to tile pair g+2 (same stage)
        if (lane == 0) mbar_arrive(&b_full[(g + 2u) % kI8Stages]);
        fold_top2_p16(v0, b, s2);
        fold_top2_p16(v1, b, s2);
        fold_min_p16(v2, m);
        fold_min_p16(v3, m);
        // ---- per-row top-2 of this tile: merge the two chains, then the even / odd halves ----
        {
          const uint32_t bb = __vminu2(b[0], b[1]);
          const uint32_t ss = __vimin3_u16x2(__vmaxu2(b[0], b[1]), s2[0], s2[1]);
          const uint32_t bw = swap16(bb);
          const uint32_t best16 = __vminu2(bb, bw);                          // both halves: tile minimum
          const uint32_t sec16 = __vimin3_u16x2(__vmaxu2(bb, bw), ss, swap16(ss));  // both halves: tile second
          top2_insert(gbest, gsecond, key16_to_key32(best16 & 0xFFFFu, (uint32_t)tbase));
          top2_insert(gbest, gsecond, key16_to_key32(sec16 & 0xFFFFu, (uint32_t)tbase));
        }
        // ---- column minimum: this thread's train row against the 128 queries of the item ----
        {
          const uint32_t mm = __vminu2(m[0], m[1]);
          const uint32_t cm = __vminu2(mm, swap16(mm)) & 0xFFFFu;
          if (row < nt_valid && cm < kKey16Valid) atomicMin(&p.bwd_best[to + tbase + row], key16_to_key32(cm, (uint32_t)q0));
        }
      }
      // the two epilogue sets (even / odd tile pairs) meet in shared memory
      if (eset == 1) s_merge[row] = make_uint2(gbest, gsecond);
      asm volatile("bar.sync 1, 256;" ::: "memory");  // epilogue warps only
      if (eset == 0 && row < nq_valid) {
        const uint2 o = s_merge[row];
        top2_insert(gbest, gsecond, o.x);
        top2_insert(gbest, gsecond, o.y);
        p.fwd_best[qo + q0 + row] = gbest >= kKey32Pad ? kNone : gbest;
        p.fwd_second[qo + q0 + row] = gsecond >= kKey32Pad ? kNone : gsecond;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");  // s_merge free for the next item
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}

// =====================================================================================
// Single-product variant (B2S_VARIANT_I8MMA1): D = Qtile . Ttile^T only.
//
// The two-product kernel above spends half of its tensor time on D^T just to make the column
// minimum a per-thread reduction.  Here the column minimum comes out of D itself: the index
// K-step of the unified tiles adds the ROW as well as the column (see expand_pm8_kernel), so the
// very registers the per-row top-2 is folded from also order a column's entries by (ham, row).
// A thread folds the four rows it holds, a 3-level butterfly over the warp leaves lane L with
// columns 4L..4L+3 over the warp's 32 rows, and the lane widens its four keys and sends them to
// bwd_best with atomicMin — but only those that beat the current value, which it staged before
// waiting for the accumulator (a stale value merely costs a redundant atomic; ~ln(64) of the 64
// candidates per train row and pair survive the filter).
// Work item = (pair, 256-query block, train part): both 128-row sub-tiles stay in shared memory
// while the train tiles stream past once, which halves the L2 -> SM operand traffic (at ~650 clk
// per tile pair 34 KB per tile pair would exceed the L2 slice throughput of the chip).  Four query
// sub-tiles per item (with a 2-stage ring) halve it again but measured 8 % slower on every
// BASELINE shape: the epilogue's ALU pipe, not L2, bounds the kernel (DESIGN section 4).
// Four TMEM stages of 128 columns: tile pair g uses stage g%4 and sub-tile g%2, epilogue set s
// owns stage s (every other train tile of sub-tile s&1), and the two sets of a sub-tile merge
// their running top-2 at the end of the item.  The MMA thread runs up to four tile pairs ahead.
// One barrier per tile pair ("go"): operands landed + TMEM stage drained, probed from inside
// the MMA stream as above.
constexpr int kI8sGo = 16;  // go barriers: the producer runs up to 8 tile pairs ahead of the MMA thread
constexpr int kI8sQTileBytes = (kI8Chunks + 1) * kI8ChunkBytes;  // unified tiles: 18 chunks
constexpr int kI8sThreads = 576;  // producer warp + MMA warp + 16 epilogue warps
constexpr int kI8sSubTiles = 2;   // 128-row query sub-tiles per work item
constexpr int kI8sStages = 4;     // train-tile ring slots
constexpr size_t kI8sSmemBytes = (size_t)kI8sSubTiles * kI8sQTileBytes + (size_t)kI8sStages * kI8TileBytes +
                                 kI8ChunkBytes + 8 * (kI8sGo + 12) + 16 + 4 * kI8Tile * sizeof(uint2) +
                                 16 * 32 * sizeof(uint4);

__device__ __forceinline__ uint32_t tc_mma_tile_single(uint32_t d, uint64_t qdesc, uint64_t tdesc, uint32_t idesc,
                                                       uint64_t* next_bar, uint32_t next_parity, uint32_t has_next) {
  // 8 data K-steps + the index K-step (chunks 16/17 of the query tile x chunk 16 of the train tile)
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred pacc, pnew, pprobe, pdone;\n\t"
      ".reg .b64 da, db;\n\t"
      "setp.eq.b32 pacc, 0, 0;\n\t"
      "setp.ne.b32 pnew, 0, 0;\n\t"
      "setp.ne.b32 pprobe, %7, 0;\n\t"
      "setp.ne.b32 pdone, 0, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], %2, %3, %4, pnew;\n\t"
      "add.u64 da, %2, 256;\n\t"
      "add.u64 db, %3, 256;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %4, pacc;\n\t"
      "add.u64 da, %2, 512;\n\t"
      "add.u64 db, %3, 512;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %4, pacc;\n\t"
      "add.u64 da, %2, 768;\n\t"
      "add.u64 db, %3, 768;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %4, pacc;\n\t"
      "add.u64 da, %2, 1024;\n\t"
      "add.u64 db, %3, 1024;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %4, pacc;\n\t"
      "@pprobe mbarrier.try_wait.parity.shared::cta.b64 pdone, [%5], %6;\n\t"
      "add.u64 da, %2, 1280;\n\t"
      "add.u64 db, %3, 1280;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %4, pacc;\n\t"
      "add.u64 da, %2, 1536;\n\t"
      "add.u64 db, %3, 1536;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %4, pacc;\n\t"
      "add.u64 da, %2, 1792;\n\t"
      "add.u64 db, %3, 1792;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %4, pacc;\n\t"
      "add.u64 da, %2, 2048;\n\t"
      "add.u64 db, %3, 2048;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%1], da, db, %4, pacc;\n\t"
      "selp.u32 %0, 1, 0, pdone;\n\t"
      "}"
      : "=r"(ok)
      : "r"(d), "l"(qdesc), "l"(tdesc), "r"(idesc), "r"(smem_u32(next_bar)), "r"(next_parity), "r"(has_next)
      : "memory");
  return ok;
}

// One butterfly step over N live registers: lanes with up = 1 keep the upper half and send the
// lower one.  The choice is arithmetic, not SEL: every ALU-pipe instruction (SEL, LOP3, PRMT,
// VIMNMX) issues at 64 threads/clk/SM on this part (tools/pipe_rates.py) and so does IMAD on
// the FMA pipe; the epilogue is bound by whichever of the two pipes carries more, so the
// selection goes to the FMA pipe (3 instructions) and only the maximum stays on the ALU pipe.
//   e = a - b;  send = up*e + b  (= up ? a : b);  keep = (-up)*e + a  (= up ? b : a)   (exact mod 2^32)
template <int N>
__device__ __forceinline__ void colmin_step(uint32_t (&y)[16], uint32_t up, uint32_t nup, int lane_mask) {
#pragma unroll
  for (int i = 0; i < N / 2; ++i) {
    uint32_t send, keep;
    if (i % 5 == 4) {
      // every fifth exchange selects on the ALU pipe instead (2 SEL): with ~205 other ALU-pipe and
      // ~77 other FMA-pipe instructions per tile pair this split levels the two pipes
      asm("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %4, 0;\n\tselp.b32 %0, %2, %3, p;\n\tselp.b32 %1, %3, %2, p;\n\t}"
          : "=r"(send), "=r"(keep)
          : "r"(y[i]), "r"(y[i + N / 2]), "r"(up));
    } else {
      asm("{\n\t.reg .u32 e;\n\tsub.u32 e, %2, %3;\n\tmad.lo.u32 %0, %4, e, %3;\n\tmad.lo.u32 %1, %5, e, %2;\n\t}"
          : "=r"(send), "=r"(keep)
          : "r"(y[i]), "r"(y[i + N / 2]), "r"(up), "r"(nup));
    }
    const uint32_t got = __shfl_xor_sync(0xFFFFFFFFu, send, lane_mask);
    y[i] = __vmaxu2(keep, got);
  }
}

// TOP2 = false: the per-row SECOND neighbour is not computed (fwd_second stays "none").  The reference's production
// matcher — BFMatcher(crossCheck=True).match at feature_pipeline.py.bak:82 (cross_check is the default and what
// configs/pipeline/kitti_default.json sets), persistent_map.py:266, keyframe_manager.py:126,141 — never looks at it;
// only the kNN + ratio mode (.bak:84-91) and match_orb_descriptors do.  Dropping the second pass removes 64 of the
// epilogue's ~164 packed min/max instructions per thread and tile pair, and the epilogue's ALU pipe is the kernel's limiter.
template <bool TOP2>
__global__ void __launch_bounds__(kI8sThreads, 1) hamming_knn2_i8s_kernel(const I8Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_q = smem;                                   // 2 x 36 KB: the item's query sub-tiles (18 chunks each)
  uint8_t* s_t = smem + kI8sSubTiles * kI8sQTileBytes;   // kI8sStages x 34 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_t + kI8sStages * kI8TileBytes + kI8ChunkBytes);  // +1 chunk: see below
  uint64_t* b_go = bars;                                 // [kI8sGo]
  uint64_t* b_empty = bars + kI8sGo;                     // [4] one per ring slot
  uint64_t* b_tfull = bars + kI8sGo + 4;                 // [4] one per TMEM stage
  uint64_t* b_qempty = bars + kI8sGo + 8;                // [4] (2 used: one per query sub-tile)
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + kI8sGo + 12);
  uint2* s_merge = reinterpret_cast<uint2*>(s_tmem + 4);  // [2 item parities][2 sub-tiles][128], the two sets of a sub-tile meet here
  uint4* s_cur = reinterpret_cast<uint4*>(s_merge + 4 * kI8Tile);  // [16 epilogue warps][32 lanes]: staged bwd_best values

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q_blocks = (p.q_tiles + kI8sSubTiles - 1) / kI8sSubTiles;
  const int t_split = p.t_split;
  const int n_items = p.n_pairs * q_blocks * t_split;    // item w = ((pair * q_blocks) + qb) * t_split + part

  // the index K-step reads one chunk past the last ring slot (times the query tile's zero chunk):
  // keep that chunk inside the allocation and defined; the query slots' chunk 17 is never loaded
  // and must read as zero
  for (int i = threadIdx.x; i < kI8Tile; i += kI8sThreads) {
    reinterpret_cast<uint4*>(s_t + kI8sStages * kI8TileBytes)[i] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
    for (int sub = 0; sub < kI8sSubTiles; ++sub)
      reinterpret_cast<uint4*>(s_q + sub * kI8sQTileBytes + kI8TileBytes)[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");

  if (threadIdx.x == 0) {
    for (int k = 0; k < kI8sGo; ++k) mbar_init(&b_go[k], 5);  // producer + the 4 warps that drained tile pair g-4
    for (int s = 0; s < 4; ++s) mbar_init(&b_empty[s], 1);
    for (int a = 0; a < 4; ++a) {
      mbar_init(&b_tfull[a], 1);
      for (int k = 0; k < 4; ++k) mbar_arrive(&b_go[a]);  // tile pairs 0..3 find their TMEM stage free
    }
    for (int a = 0; a < 4; ++a) mbar_init(&b_qempty[a], 1);
    mbar_fence_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(s_tmem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  // all roles walk the same items; an item always has 2 (t1 - t0) tile pairs (a trailing sub-tile may
  // be all padding: its MMAs then read stale shared memory and every result is ignored)
#define B2S_I8S_ITEM(w)                                                                          \
  const int part = (w) % t_split, pq = (w) / t_split;                                            \
  const int pair = pq / q_blocks, qb = pq - pair * q_blocks;                                     \
  const int nq = p.q_off[pair + 1] - p.q_off[pair];                                              \
  const int to = p.t_off[pair], nt = p.t_off[pair + 1] - to;                                     \
  const int n_tt = (nt + kI8Tile - 1) / kI8Tile;                                                 \
  const int t0 = (int)(((long long)part * n_tt) / t_split), t1 = (int)(((long long)(part + 1) * n_tt) / t_split); \
  if (qb * kI8sSubTiles * kI8Tile >= nq || t0 >= t1) continue;
  if (warp == 0) {
    // ===== producer =====
    if (lane == 0) {
      uint32_t n = 0, tau = 0;  // items / train tiles seen by this CTA
      for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
        B2S_I8S_ITEM(w)
        (void)to;
        const int q0 = qb * kI8sSubTiles * kI8Tile;
        // unified 18-chunk tiles on both sides: a train slot takes chunks 0..16 (data + its B-side index
        // chunk, one copy), a query slot chunks 0..15 and chunk 17 (its A-side index chunk, two copies
        // once per item)
        const size_t t_tile0 = p.t_xt ? (size_t)p.t_xt[pair] : (size_t)pair * p.t_tiles;
        const size_t q_tile0 = p.q_xt ? (size_t)p.q_xt[pair] : (size_t)pair * p.q_tiles;
        const uint8_t* tsrc = p.tx + t_tile0 * kI8sQTileBytes;
        const uint8_t* qsrc = p.qx + (q_tile0 + (size_t)kI8sSubTiles * qb) * kI8sQTileBytes;
        for (int t = t0; t < t1; ++t, ++tau) {
          const uint32_t s = tau % kI8sStages, g = (uint32_t)kI8sSubTiles * tau;
          if (tau >= (uint32_t)kI8sStages) mbar_wait_bounded(&b_empty[s], ((tau / kI8sStages) - 1u) & 1u);
#pragma unroll
          for (int sub = 0; sub < kI8sSubTiles; ++sub) {
            uint64_t* go = &b_go[(g + (uint32_t)sub) % kI8sGo];
            const bool load_q = t == t0 && q0 + sub * kI8Tile < nq;   // the item's query sub-tile rides on its first tile pair
            const uint32_t t_bytes = sub == 0 ? (uint32_t)kI8TileBytes : 0u;   // the train tile rides on sub-tile 0
            if (load_q) {
              if (n >= 1) mbar_wait_bounded(&b_qempty[sub], (n - 1u) & 1u);
              mbar_arrive_expect_tx(go, (uint32_t)kI8TileBytes + t_bytes);
              uint8_t* qdst = s_q + sub * kI8sQTileBytes;
              const uint8_t* qs = qsrc + (size_t)sub * kI8sQTileBytes;
              bulk_g2s(qdst, qs, 16 * kI8ChunkBytes, go);
              bulk_g2s(qdst + 16 * kI8ChunkBytes, qs + 17 * kI8ChunkBytes, kI8ChunkBytes, go);
            } else if (t_bytes) {
              mbar_arrive_expect_tx(go, t_bytes);
            } else {
              mbar_arrive(go);
            }
            if (t_bytes) bulk_g2s(s_t + (size_t)s * kI8TileBytes, tsrc + (size_t)t * kI8sQTileBytes, kI8TileBytes, go);
          }
        }
        ++n;
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    if (elect_one()) {
      uint32_t g = 0;
      bool probed = false;
      uint64_t qdesc[kI8sSubTiles];
#pragma unroll
      for (int sub = 0; sub < kI8sSubTiles; ++sub) qdesc[sub] = make_smem_desc(smem_u32(s_q + sub * kI8sQTileBytes));
      for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
        B2S_I8S_ITEM(w)
        (void)to;
        for (int t = t0; t < t1; ++t) {
          const uint32_t s = (g / (uint32_t)kI8sSubTiles) % kI8sStages;
          const uint64_t tdesc = make_smem_desc(smem_u32(s_t + (size_t)s * kI8TileBytes));
#pragma unroll
          for (uint32_t sub = 0; sub < (uint32_t)kI8sSubTiles; ++sub, ++g) {
            if (!probed)  // first tile pair, item boundaries, late epilogue or late loads
              mbar_wait_bounded(&b_go[g % kI8sGo], (g / kI8sGo) & 1u);
            tc_fence_after();
            const uint32_t gn = g + 1u;
            const uint32_t more = (sub + 1u < (uint32_t)kI8sSubTiles || t + 1 < t1) ? 1u : 0u;
            probed = tc_mma_tile_single(tmem_base + (g & 3u) * 128u, qdesc[sub], tdesc, kIdescI8,
                                        &b_go[gn % kI8sGo], (gn / kI8sGo) & 1u, more) != 0u;
            if (sub == (uint32_t)kI8sSubTiles - 1u) tc_commit(&b_empty[s]);  // train tile consumed by every sub-tile
            tc_commit(&b_tfull[g & 3u]);                    // accumulator stage complete
            if (t == t1 - 1) tc_commit(&b_qempty[sub]);     // the item's last use of this query sub-tile
          }
        }
      }
    }
  } else {
    // ===== epilogue: 4 sets of 4 warps; set s owns TMEM stage s, i.e. the tile pairs g with g%4 == s
    // (sub-tile s&1, every other train tile); warp%4 = TMEM lane quarter.  Four warps per scheduler
    // instead of two: the per-tile-pair work is a long dependent chain (TMEM load, folds, butterfly)
    // and two warps left the ALU and FMA pipes half idle.  The accumulator is read with
    // tcgen05.ld.16x256b: a thread owns 4 ROWS (gr, gr+8, gr+16, gr+24 of its warp's 32 TMEM lanes,
    // gr = lane/4) x 32 columns (eight 4-column groups, 16 g + 4 (lane%4) ..+3).
    //  * Column minimum: the four rows are folded inside the thread (2 instructions per register) and
    //    only then cross lanes: 3 butterfly levels over 16 registers (14 exchanges) leave lane L holding
    //    columns 4L..4L+3.
    //  * Per-row top-2: 16 registers per row, two rows in lock step (independent dependency chains: with
    //    64 of the 96 registers holding the accumulator ptxas otherwise runs one serial chain at a time
    //    and the epilogue is latency-, not issue-bound); the results of two rows share a register
    //    (row a | row b << 16), the four lanes that share a row merge in that packed form (4 SHFL per
    //    level) and lane%4 = k finishes row k: one running top-2 per thread. =====
    const int quarter = warp & 3;
    const uint32_t set = (uint32_t)(warp - 2) >> 2;
    const uint32_t sub = set & 1u;
    const int gr = lane >> 2, tc = lane & 3;
    const int row = quarter * 32 + gr + 8 * tc;   // the tile-local row this lane keeps the running top-2 of
    const uint32_t row_base = (uint32_t)(quarter * 32 + gr);
    const uint32_t pick = tc == 0 ? 0x3210u : tc == 1 ? 0x1032u : tc == 2 ? 0x7654u : 0x5476u;  // row k = tc -> low half
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quarter * 32) << 16) + set * 128u;
    uint32_t g_item = 0, n = 0;  // first tile pair of the item, items
    for (int w = blockIdx.x; w < n_items; w += gridDim.x) {
      B2S_I8S_ITEM(w)
      const int q0 = qb * kI8sSubTiles * kI8Tile + (int)sub * kI8Tile;   // first query row of this set's sub-tile
      const int rows_valid = max(0, min(kI8Tile, nq - q0));
      const bool staged = (reinterpret_cast<uintptr_t>(p.bwd_best + to) & 15u) == 0;   // cp.async.cg moves 16 aligned bytes
      uint32_t gbest = kNone, gsecond = kNone;
      // this set's tile pairs: g = g_item + 2 (t - t0) + sub with g % 4 == set, i.e. every other train tile;
      // stage `set` has served g / 4 tile pairs before g
      const uint32_t g_end = g_item + (uint32_t)kI8sSubTiles * (uint32_t)(t1 - t0);
      for (uint32_t g = (g_item + 3u - set) / 4u * 4u + set; g < g_end; g += 4u) {
        const int t = t0 + (int)((g - g_item) >> 1);
        const int tbase = t * kI8Tile;
        // current column minima of this lane's 4 train rows (stale is fine: only used to skip atomics).
        // Holding them in registers through the top-2 costs more than it saves (96 registers, 64 of them
        // accumulator), and loading them late leaves the L2 latency exposed (10 % of the epilogue's
        // samples sat on the first compare): cp.async parks them in this lane's shared-memory slot
        // before the accumulator wait.  (.cg needs 16-byte alignment: a pair whose slice of bwd_best does
        // not start on a 16-byte boundary takes the plain loads below.)
        uint4* cur_slot = s_cur + (warp - 2) * 32 + lane;
        if (staged) {
          const int left = nt - tbase - 4 * lane;   // valid rows from this lane's first column on
          const uint32_t nbytes = (uint32_t)(4 * max(0, min(4, left)));
          const uint32_t* src = p.bwd_best + (left > 0 ? to + tbase + 4 * lane : to);
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n\tcp.async.commit_group;"
                       ::"r"(smem_u32(cur_slot)), "l"(src), "r"(nbytes) : "memory");
        }
        mbar_wait_bounded(&b_tfull[set], (g >> 2) & 1u);
        tc_fence_after();
        uint32_t ra[32], rb[32];
        TMEM_LD_16X256_X8P(lane_addr, ra);
        TMEM_LD_16X256_X8P(lane_addr + (16u << 16), rb);
        tmem_ld_wait();
        TMEM_REGS_READY(ra);
        TMEM_REGS_READY(rb);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&b_go[(g + 4u) % kI8sGo]);
        // register i (0..15 = 2 g + b) of the first / second row held by a 32-register load
#define B2S_R0(r, i) (r[4 * ((i) >> 1) + ((i) & 1)])
#define B2S_R1(r, i) (r[4 * ((i) >> 1) + 2 + ((i) & 1)])
        // ---- per-row top-2 of this tile: rows (0, 1) from ra, rows (2, 3) from rb, two rows in lock step ----
        uint32_t pb[2], ps[2];  // packed results: row a in the low half, row b in the high half
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t(&r)[32] = h ? rb : ra;
          // pass 1: minimum per 16-bit lane (even / odd columns of the 4-column groups)
          uint32_t m0 = __vimax3_u16x2(B2S_R0(r, 0), B2S_R0(r, 1), B2S_R0(r, 2));
          uint32_t m1 = __vimax3_u16x2(B2S_R1(r, 0), B2S_R1(r, 1), B2S_R1(r, 2));
#pragma unroll
          for (int i = 3; i < 15; i += 2) {
            m0 = __vimax3_u16x2(m0, B2S_R0(r, i), B2S_R0(r, i + 1));
            m1 = __vimax3_u16x2(m1, B2S_R1(r, i), B2S_R1(r, i + 1));
          }
          const uint32_t bb0 = __vmaxu2(m0, B2S_R0(r, 15)), bb1 = __vmaxu2(m1, B2S_R1(r, 15));
          // fold the even / odd halves of both rows at once: x = (row a even | row b even), y = (.. odd | .. odd)
          const uint32_t x = __byte_perm(bb0, bb1, 0x5410), y = __byte_perm(bb0, bb1, 0x7632);
          pb[h] = __vmaxu2(x, y);
          if constexpr (TOP2) {
            // pass 2: values are unique within a row (or zero padding, never the largest of a real row), so
            // x - best wraps to 0 exactly for the maximum itself and keeps the order of everything below it
            const uint32_t cn0 = __vneg2(bb0), cn1 = __vneg2(bb1);
            uint32_t a00 = 0u, a01 = 0u, a10 = 0u, a11 = 0u;
#pragma unroll
            for (int i = 0; i < 16; i += 2) {
              a00 = __viaddmax_u16x2(B2S_R0(r, i), cn0, a00);
              a10 = __viaddmax_u16x2(B2S_R1(r, i), cn1, a10);
              a01 = __viaddmax_u16x2(B2S_R0(r, i + 1), cn0, a01);
              a11 = __viaddmax_u16x2(B2S_R1(r, i + 1), cn1, a11);
            }
            const uint32_t ss0 = __vadd2(__vmaxu2(a00, a01), bb0);  // second largest per 16-bit lane (mod 2^16 per lane)
            const uint32_t ss1 = __vadd2(__vmaxu2(a10, a11), bb1);
            const uint32_t sx = __byte_perm(ss0, ss1, 0x5410), sy = __byte_perm(ss0, ss1, 0x7632);
            ps[h] = __vimax3_u16x2(__vminu2(x, y), sx, sy);
          }
        }
        // the four lanes that share these rows hold disjoint columns: merge best / second, both row pairs
#pragma unroll
        for (int o = 1; o <= 2; o <<= 1) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const uint32_t ob = __shfl_xor_sync(0xFFFFFFFFu, pb[h], o);
            if constexpr (TOP2) {
              const uint32_t os = __shfl_xor_sync(0xFFFFFFFFu, ps[h], o);
              ps[h] = __vimax3_u16x2(__vminu2(pb[h], ob), ps[h], os);
            }
            pb[h] = __vmaxu2(pb[h], ob);
          }
        }
        // lane%4 = k finishes row k: complement (acc = ~key), then the keys carry + row: take it off before widening
        const uint32_t best16 = ~__byte_perm(pb[0], pb[1], pick) & 0xFFFFu;
        if constexpr (TOP2) {
          const uint32_t sec16 = ~__byte_perm(ps[0], ps[1], pick) & 0xFFFFu;
          top2_insert(gbest, gsecond, key16_to_key32(best16 - (uint32_t)row, (uint32_t)tbase));
          top2_insert(gbest, gsecond, key16_to_key32(sec16 - (uint32_t)row, (uint32_t)tbase));
        } else {
          gbest = min(gbest, key16_to_key32(best16 - (uint32_t)row, (uint32_t)tbase));
        }
        // ---- column minima: the 4 rows inside the thread, then 3 butterfly levels over lane bits 2..4 ----
        uint32_t y[16];
        uint32_t cur[4] = {0u, 0u, 0u, 0u};
#pragma unroll
        for (int i = 0; i < 16; ++i) y[i] = __vmaxu2(__vimax3_u16x2(B2S_R0(ra, i), B2S_R1(ra, i), B2S_R0(rb, i)), B2S_R1(rb, i));
        // current column minima of this lane's 4 train rows (stale is fine: only used to skip atomics):
        // requested here, into the accumulator registers the fold just freed, and consumed after the
        // butterfly (requesting them before the accumulator wait costs 4 registers through the top-2
        // and measured slower: 892 vs 876 clk per tile pair)
        if (!staged) {
          const int nt_valid = min(kI8Tile, nt - tbase);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int c = 4 * lane + k;
            cur[k] = (c < nt_valid) ? __ldcg(&p.bwd_best[to + tbase + c]) : 0u;
          }
        }
        const uint32_t u16 = (lane >> 4) & 1, u8 = (lane >> 3) & 1, u4 = (lane >> 2) & 1;
        colmin_step<16>(y, u16, 0u - u16, 16);
        colmin_step<8>(y, u8, 0u - u8, 8);
        colmin_step<4>(y, u4, 0u - u4, 4);
        // register i of lane L is now position 2 (L/4) + i, i.e. columns 16 (L/4) + 4 (L%4) + 2 i, +1 = 4 L + 2 i, +1
        // acc = 65535 - (128 ham + column + row): complement and take the column off in one subtraction
        // (no borrow between the halves: 65535 - column >= acc)
        const uint32_t cfix = (uint32_t)(4 * lane) * 0x10001u + 0x00010000u;
        y[0] = (0xFFFFFFFFu - cfix) - y[0];
        y[1] = (0xFFFFFFFFu - cfix - 0x00020002u) - y[1];
        if (staged) {
          asm volatile("cp.async.wait_group 0;" ::: "memory");
          const uint4 c4 = *cur_slot;
          cur[0] = c4.x; cur[1] = c4.y; cur[2] = c4.z; cur[3] = c4.w;
        }
#undef B2S_R0
#undef B2S_R1
        const uint32_t cm16[4] = {y[0] & 0xFFFFu, y[0] >> 16, y[1] & 0xFFFFu, y[1] >> 16};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t key = key16_to_key32(cm16[k], (uint32_t)q0);
          // rows_valid == 0: the whole sub-tile is padding and its MMAs read stale shared memory
          if (rows_valid > 0 && cm16[k] < kKey16Valid && key < cur[k]) atomicMin(&p.bwd_best[to + tbase + 4 * lane + k], key);
        }
      }
      g_item = g_end;
      // the two sets of a sub-tile (even / odd train tiles) meet in shared memory; double buffered by
      // item parity, so one named barrier per item is enough
      uint2* mg = s_merge + (((n & 1u) * 2u + sub) << 7);
      if (set >= 2u) mg[row] = make_uint2(gbest, gsecond);
      asm volatile("bar.sync %0, 256;" ::"r"(1u + sub) : "memory");
      if (set < 2u && row < rows_valid) {
        const uint2 o = mg[row];
        top2_insert(gbest, gsecond, o.x);
        top2_insert(gbest, gsecond, o.y);
        const int qo = p.q_off[pair];
        // best-only: gsecond is not a second neighbour (the merge of the two sets above put the larger of their bests there)
        const uint32_t ob = gbest >= kKey32Pad ? kNone : gbest, os = (!TOP2 || gsecond >= kKey32Pad) ? kNone : gsecond;
        if (t_split > 1) {
          p.partial[(size_t)part * p.total_nq + qo + q0 + row] = make_uint2(ob, os);
        } else {
          p.fwd_best[qo + q0 + row] = ob;
          p.fwd_second[qo + q0 + row] = os;
        }
      }
      ++n;
    }
  }

#undef B2S_I8S_ITEM
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
  }
}


// ---- measurement: raw tcgen05.mma kind::i8 issue rate (no epilogue), one CTA per SM ------
// n_dim = 128 or 256; A = 128 rows, B = n_dim rows, both in the canonical no-swizzle layout.
// variant 0: 8 accumulating MMAs per iteration, nothing else.
// variant 1: the K2 issue pattern — 9 MMAs into D1 and 9 into D2 per iteration, no barriers.
// variant 2: variant 1 + the two tcgen05.commit of a tile pair (nobody waits on them).
// variant 3: variant 2 + waiting, before iteration i, for the commit of iteration i-2 (the
//            TMEM-stage dependency of the real kernel with an infinitely fast epilogue).
// variant 4: variant 3 with the wait for iteration i+1 taken after the first 4 MMAs of i.
__global__ void __launch_bounds__(128, 1) mma_rate_kernel(int iters, int n_dim, int variant) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ uint64_t bar, bars2[4];
  __shared__ uint32_t s_tm;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < (3 * kI8TileBytes) / 16; i += blockDim.x)
    reinterpret_cast<uint4*>(smem)[i] = make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u);
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    for (int i = 0; i < 4; ++i) mbar_init(&bars2[i], 1);
    mbar_fence_init();
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&s_tm)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = s_tm;
  if (warp == 1 && lane == 0) {
    const uint64_t adesc = make_smem_desc(smem_u32(smem));
    const uint64_t bdesc = make_smem_desc(smem_u32(smem + kI8TileBytes));
    const uint32_t idesc = (2u << 4) | (1u << 7) | (1u << 10) | (((uint32_t)n_dim >> 3) << 17) | ((128u >> 4) << 24);
    if (variant == 0) {
      for (int it = 0; it < iters; ++it) {
        const uint32_t d = tm + (uint32_t)((it & 1) * 256);
#pragma unroll
        for (int k = 0; k < 8; ++k) tc_mma_i8(d, adesc + (uint64_t)k * 256u, bdesc + (uint64_t)k * 256u, idesc, k > 0);
      }
    } else {
      for (int it = 0; it < iters; ++it) {
        const uint32_t d1 = tm + (uint32_t)((it & 1) * 256), d2 = d1 + 128u;
        if (variant == 3 && it >= 2) mbar_wait_bounded(&bars2[it & 1], ((it >> 1) - 1) & 1);
#pragma unroll
        for (int k = 0; k < 9; ++k) {
          tc_mma_i8(d1, adesc + (uint64_t)(k & 7) * 256u, bdesc + (uint64_t)(k & 7) * 256u, idesc, k > 0);
          if (variant == 4 && k == 3 && it >= 1) mbar_wait_bounded(&bars2[(it + 1) & 1], (((it + 1) >> 1) - 1) & 1);
        }
#pragma unroll
        for (int k = 0; k < 9; ++k) tc_mma_i8(d2, bdesc + (uint64_t)(k & 7) * 256u, adesc + (uint64_t)(k & 7) * 256u, idesc, k > 0);
        if (variant >= 2) {
          tc_commit(&bars2[2 + (it & 1)]);
          tc_commit(&bars2[it & 1]);
        }
      }
    }
    tc_commit(&bar);
    mbar_wait_bounded(&bar, 0);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tm) : "memory");
  }
}

// ---- measurement: TMEM -> register read bandwidth (tcgen05.ld 32x32b.x32), `warps` warps per SM
__global__ void __launch_bounds__(512, 1) tmem_read_kernel(int iters, uint32_t* sink) {
  __shared__ uint32_t s_tm;
  const int warp = threadIdx.x >> 5;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&s_tm)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = s_tm;
  const uint32_t lane_addr = tm + ((uint32_t)((warp & 3) * 32) << 16);
  const int nw = blockDim.x >> 5;
  uint32_t acc = 0;
  for (int it = 0; it < iters; ++it) {
    // the warps sharing a lane quarter split the 512 columns
    const int per = 512 / (nw / 4);
    const int c0 = (warp >> 2) * per;
    for (int c = c0; c < c0 + per; c += 64) {
      uint32_t v0[32], v1[32];
      TMEM_LD_X32(lane_addr + (uint32_t)c, v0);
      TMEM_LD_X32(lane_addr + (uint32_t)c + 32u, v1);
      tmem_ld_wait();
#pragma unroll
      for (int k = 0; k < 32; k += 8) acc ^= v0[k] ^ v1[k];
    }
  }
  if (acc == 0x12345u) sink[0] = acc;
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tm) : "memory");
  }
}

int tmem_read_launch(int iters, int warps, double* bytes_out, uint32_t* sink, cudaStream_t st) {
  B2S_REQUIRE(warps == 4 || warps == 8 || warps == 16, "warps must be 4, 8 or 16");
  tmem_read_kernel<<<sm_count(), warps * 32, 0, st>>>(iters, sink);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  if (bytes_out) *bytes_out = (double)sm_count() * iters * 128.0 * 512.0 * 4.0;
  return B2S_OK;
}

int mma_rate_launch(int iters, int n_dim, double* macs_out, cudaStream_t st) {
  const int variant = n_dim >> 16;  // diagnostics: upper half selects the issue pattern (see mma_rate_kernel)
  n_dim &= 0xFFFF;
  B2S_REQUIRE(n_dim == 128 || n_dim == 256, "n_dim must be 128 or 256");
  B2S_REQUIRE(variant >= 0 && variant <= 4 && (variant == 0 || n_dim == 128), "bad variant");
  const size_t smem = 3 * (size_t)kI8TileBytes;
  B2S_CUDA(cudaFuncSetAttribute(mma_rate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mma_rate_kernel<<<sm_count(), 128, smem, st>>>(iters, n_dim, variant);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  if (macs_out) *macs_out = (double)sm_count() * iters * (variant ? 18.0 : 8.0) * 128.0 * n_dim * 32.0;
  return B2S_OK;
}

// optional CUDA-event pair around the main kernel only (b2s_hamming_kernel_timing): the roofline
// of bench.py is quoted on the tensor-core kernel alone, the pre-pass is reported beside it
static bool g_i8_timing = false;
static cudaEvent_t g_i8_ev[2] = {nullptr, nullptr};
int hamming_i8_timing(int enable, float* last_ms) {
  if (last_ms) {
    *last_ms = -1.0f;
    if (g_i8_ev[0] && g_i8_ev[1]) {
      B2S_CUDA(cudaEventSynchronize(g_i8_ev[1]));
      B2S_CUDA(cudaEventElapsedTime(last_ms, g_i8_ev[0], g_i8_ev[1]));
    }
  }
  if (enable >= 0) {
    g_i8_timing = enable != 0;
    if (g_i8_timing && !g_i8_ev[0]) {
      B2S_CUDA(cudaEventCreate(&g_i8_ev[0]));
      B2S_CUDA(cudaEventCreate(&g_i8_ev[1]));
    }
  }
  return B2S_OK;
}

constexpr size_t kI8SmemBytes =
    (size_t)(2 + kI8Stages) * kI8TileBytes + 2 * kI8ChunkBytes + 8 * (2 * kI8Stages + 9) + 128 * sizeof(uint2);

int hamming_merge_launch(const uint2* partial, int total_nq, int t_split, uint32_t* fwd_best, uint32_t* fwd_second,
                         cudaStream_t st);  // hamming_popc.cu

// Work decomposition of the single-product kernel: the train-axis split.
// A lone 10 000 x 10 000 pair has 40 (pair, 256-query block) items for 148 SMs, a lone 2000 x 2000 pair 8:
// the train axis is then cut into t_split pieces (merged afterwards on the packed keys, like K1's t_split) so
// that whole waves of items cover the machine.
static int plan_i8s(int n_pairs, int max_nq, int max_nt, int t_split_req) {
  const int qt = (max_nq + kI8Tile - 1) / kI8Tile, tt = (max_nt + kI8Tile - 1) / kI8Tile;
  const long sms = sm_count();
  const long base = (long)n_pairs * ((qt + kI8sSubTiles - 1) / kI8sSubTiles);
  int ts = 1;
  if (t_split_req > 0) {
    ts = t_split_req;
  } else if (base > 0 && base < 4 * sms) {
    // waves x (train tiles per item + ~2 tiles of query loads and pipeline fill per item), smallest wins
    long best_cost = -1;
    for (int c = 1; c <= tt && c <= 64; ++c) {
      const long waves = (base * c + sms - 1) / sms;
      const long cost = waves * ((tt + c - 1) / c + 2);
      if (best_cost < 0 || cost < best_cost) {
        best_cost = cost;
        ts = c;
      }
    }
  }
  if (ts > tt) ts = tt;
  if (ts < 1) ts = 1;
  return ts;
}

static size_t partial_bytes(int total_nq, int t_split) {
  return t_split > 1 ? (((size_t)total_nq * t_split * sizeof(uint2) + 127) & ~(size_t)127) : 0;
}

size_t hamming_i8_workspace_bytes(int n_pairs, int total_nq, int max_nq, int max_nt, int t_split) {
  const size_t qt = (size_t)((max_nq + kI8Tile - 1) / kI8Tile), tt = (size_t)((max_nt + kI8Tile - 1) / kI8Tile);
  // sized for the largest layout (unified 18-chunk tiles on both sides) + the partial top-2 of a train-axis split
  return (size_t)n_pairs * (qt + tt) * kI8sQTileBytes + partial_bytes(total_nq, plan_i8s(n_pairs, max_nq, max_nt, t_split));
}

// every key starts as "none".  Three separate memset nodes on purpose: ONE 7 MB memset over the (often
// adjacent) arrays, or a fill kernel, is 1 % faster for a lone step but changed how two steps in flight
// interleave and cost the end-to-end path 8 % (439k -> 403k pairs/s, A/B on one box).
static int clear_keys(uint32_t* fwd_best, uint32_t* fwd_second, uint32_t* bwd_best, int total_nq, int total_nt,
                      cudaStream_t st) {
  if (total_nt > 0) B2S_CUDA(cudaMemsetAsync(bwd_best, 0xFF, sizeof(uint32_t) * (size_t)total_nt, st));
  if (total_nq > 0) {
    B2S_CUDA(cudaMemsetAsync(fwd_best, 0xFF, sizeof(uint32_t) * (size_t)total_nq, st));
    B2S_CUDA(cudaMemsetAsync(fwd_second, 0xFF, sizeof(uint32_t) * (size_t)total_nq, st));
  }
  return B2S_OK;
}

// the single-product kernel: picks the instantiation, opts into its shared memory (per launch: the
// attribute is per device, and a process may drive several), brackets it with the timing events
template <bool TOP2>
static int launch_i8s_inst(const I8Params& p, int grid, cudaStream_t st) {
  static bool attr_set[64] = {false};   // one flag array per instantiation
  if (first_use_on_device(attr_set))
    B2S_CUDA(cudaFuncSetAttribute(hamming_knn2_i8s_kernel<TOP2>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)kI8sSmemBytes));
  hamming_knn2_i8s_kernel<TOP2><<<grid, kI8sThreads, kI8sSmemBytes, st>>>(p);
  return B2S_OK;
}
static int g_i8_last_plan[2] = {0, 0};   // t_split, grid of the most recent launch (diagnostics)
void hamming_i8_last_plan(int* subs, int* t_split, int* grid) {
  if (subs) *subs = kI8sSubTiles;
  if (t_split) *t_split = g_i8_last_plan[0];
  if (grid) *grid = g_i8_last_plan[1];
}
static int launch_i8s(I8Params& p, int t_split, int total_nq, uint8_t* partial_ws, bool need_second, cudaStream_t st) {
  p.t_split = t_split;
  p.total_nq = total_nq;
  p.partial = t_split > 1 ? reinterpret_cast<uint2*>(partial_ws) : nullptr;
  if (t_split > 1)   // parts that own no train tile of a short pair still report "none"
    B2S_CUDA(cudaMemsetAsync(partial_ws, 0xFF, sizeof(uint2) * (size_t)total_nq * t_split, st));
  const long items = (long)((p.q_tiles + kI8sSubTiles - 1) / kI8sSubTiles) * p.n_pairs * t_split;
  const int grid = (int)(items < (long)sm_count() ? items : (long)sm_count());
  g_i8_last_plan[0] = t_split, g_i8_last_plan[1] = grid;
  if (g_i8_timing) B2S_CUDA(cudaEventRecord(g_i8_ev[0], st));
  if (int rc = need_second ? launch_i8s_inst<true>(p, grid, st) : launch_i8s_inst<false>(p, grid, st)) return rc;
  B2S_CUDA(cudaGetLastError());
  if (g_i8_timing) B2S_CUDA(cudaEventRecord(g_i8_ev[1], st));
  note_launch();
  if (t_split > 1) {
    if (int rc2 = hamming_merge_launch(p.partial, total_nq, t_split, p.fwd_best, p.fwd_second, st)) return rc2;
    // best-only: the merge folded the parts' BEST keys into fwd_second; that is not a second neighbour
    if (!need_second) B2S_CUDA(cudaMemsetAsync(p.fwd_second, 0xFF, sizeof(uint32_t) * (size_t)total_nq, st));
  }
  return B2S_OK;
}

int hamming_i8_launch(const uint8_t* q, const uint8_t* t, const int32_t* q_off, const int32_t* t_off,
                      const int32_t* q_src, const int32_t* t_src, int n_pairs, int total_nq, int total_nt, int max_nq,
                      int max_nt, uint32_t* fwd_best, uint32_t* fwd_second, uint32_t* bwd_best, int t_split,
                      void* workspace, size_t workspace_bytes, int single, int need_second, cudaStream_t st) {
  B2S_REQUIRE(n_pairs <= 65535, "n_pairs %d exceeds grid.y limit 65535; split the batch", n_pairs);
  if (int rc = clear_keys(fwd_best, fwd_second, bwd_best, total_nq, total_nt, st)) return rc;  // rows of pairs without train descriptors keep "none"
  if (total_nq == 0 || total_nt == 0 || max_nq == 0 || max_nt == 0) return B2S_OK;
  const int qt = (max_nq + kI8Tile - 1) / kI8Tile, tt = (max_nt + kI8Tile - 1) / kI8Tile;
  const size_t tiles_bytes = (size_t)n_pairs * (qt + tt) * kI8sQTileBytes;
  int split = plan_i8s(n_pairs, max_nq, max_nt, single ? t_split : 1);
  while (split > 1 && tiles_bytes + partial_bytes(total_nq, split) > workspace_bytes) --split;  // shrink rather than fail
  const size_t need = tiles_bytes + partial_bytes(total_nq, single ? split : 1);
  B2S_REQUIRE(workspace != nullptr && workspace_bytes >= need,
              "i8 variant needs %zu workspace bytes (b2s_hamming_workspace_bytes_v), got %zu", need, workspace_bytes);
  B2S_REQUIRE(((uintptr_t)workspace & 127u) == 0, "workspace must be 128-byte aligned");
  const int q_units = (single ? kI8Chunks + 1 : kI8Chunks) * kI8Tile;
  uint8_t* qx = static_cast<uint8_t*>(workspace);
  uint8_t* tx = qx + (size_t)n_pairs * qt * q_units * 16;
  expand_pm8_kernel<<<dim3(qt, n_pairs), 128, 0, st>>>(q, q_off, q_src, qt, 0, single != 0, reinterpret_cast<uint4*>(qx),
                                                       nullptr, nullptr);
  B2S_CUDA(cudaGetLastError());
  expand_pm8_kernel<<<dim3(tt, n_pairs), 128, 0, st>>>(t, t_off, t_src, tt, 1, single != 0, reinterpret_cast<uint4*>(tx),
                                                       nullptr, nullptr);
  B2S_CUDA(cudaGetLastError());
  note_launch(2);
  I8Params p;
  p.qx = qx;
  p.tx = tx;
  p.q_off = q_off;
  p.t_off = t_off;
  p.fwd_best = fwd_best;
  p.fwd_second = fwd_second;
  p.bwd_best = bwd_best;
  p.q_tiles = qt;
  p.t_tiles = tt;
  p.n_pairs = n_pairs;
  p.q_xt = nullptr;
  p.t_xt = nullptr;
  p.t_split = 1;
  p.total_nq = total_nq;
  p.partial = nullptr;
  if (single) return launch_i8s(p, split, total_nq, static_cast<uint8_t*>(workspace) + tiles_bytes, need_second != 0, st);
  static bool attr_set[64] = {false};
  if (first_use_on_device(attr_set))
    B2S_CUDA(cudaFuncSetAttribute(hamming_knn2_i8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kI8SmemBytes));
  const long items = (long)qt * n_pairs;
  const int grid = (int)(items < (long)sm_count() ? items : (long)sm_count());
  if (g_i8_timing) B2S_CUDA(cudaEventRecord(g_i8_ev[0], st));
  hamming_knn2_i8_kernel<<<grid, kI8Threads, kI8SmemBytes, st>>>(p);
  B2S_CUDA(cudaGetLastError());
  if (g_i8_timing) B2S_CUDA(cudaEventRecord(g_i8_ev[1], st));
  note_launch();
  return B2S_OK;
}

size_t hamming_i8_shared_workspace_bytes(int total_tiles, int n_pairs, int total_nq, int max_nq, int max_nt, int t_split) {
  return (size_t)total_tiles * kI8sQTileBytes + partial_bytes(total_nq, plan_i8s(n_pairs, max_nq, max_nt, t_split));
}

// Batches whose pairs share descriptor blocks (frames): every block is expanded ONCE into unified
// tiles, the pairs address them through q_xtile / t_xtile.  Single-product kernel.
int hamming_i8_shared_launch(const uint8_t* desc, const int32_t* blk_row0, const int32_t* blk_rows,
                             const int32_t* blk_tile0, int n_blocks, int total_tiles, int max_block_rows,
                             const int32_t* q_xtile, const int32_t* t_xtile, const int32_t* q_off, const int32_t* t_off,
                             int n_pairs, int total_nq, int total_nt, int max_nq, int max_nt, uint32_t* fwd_best,
                             uint32_t* fwd_second, uint32_t* bwd_best, int t_split, int need_second, void* workspace,
                             size_t workspace_bytes, cudaStream_t st) {
  B2S_REQUIRE(n_blocks <= 65535, "n_blocks %d exceeds grid.y limit 65535; split the batch", n_blocks);
  if (int rc = clear_keys(fwd_best, fwd_second, bwd_best, total_nq, total_nt, st)) return rc;
  if (total_nq == 0 || total_nt == 0 || max_nq == 0 || max_nt == 0 || n_blocks == 0) return B2S_OK;
  const size_t tiles_bytes = (size_t)total_tiles * kI8sQTileBytes;
  int split = plan_i8s(n_pairs, max_nq, max_nt, t_split);
  while (split > 1 && tiles_bytes + partial_bytes(total_nq, split) > workspace_bytes) --split;
  const size_t need = tiles_bytes + partial_bytes(total_nq, split);
  B2S_REQUIRE(workspace != nullptr && workspace_bytes >= need,
              "shared-block Hamming needs %zu workspace bytes (b2s_hamming_shared_workspace_bytes), got %zu", need,
              workspace_bytes);
  B2S_REQUIRE(((uintptr_t)workspace & 127u) == 0, "workspace must be 128-byte aligned");
  const int bt = (max_block_rows + kI8Tile - 1) / kI8Tile;
  uint8_t* x = static_cast<uint8_t*>(workspace);
  expand_pm8_kernel<<<dim3(bt, n_blocks), 128, 0, st>>>(desc, nullptr, blk_row0, 0, 0, true, reinterpret_cast<uint4*>(x),
                                                       blk_rows, blk_tile0);
  B2S_CUDA(cudaGetLastError());
  note_launch();
  I8Params p;
  p.qx = x;
  p.tx = x;
  p.q_off = q_off;
  p.t_off = t_off;
  p.fwd_best = fwd_best;
  p.fwd_second = fwd_second;
  p.bwd_best = bwd_best;
  p.q_tiles = (max_nq + kI8Tile - 1) / kI8Tile;
  p.t_tiles = (max_nt + kI8Tile - 1) / kI8Tile;
  p.n_pairs = n_pairs;
  p.q_xt = q_xtile;
  p.t_xt = t_xtile;
  return launch_i8s(p, split, total_nq, x + tiles_bytes, need_second != 0, st);
}

}  // namespace b2s
