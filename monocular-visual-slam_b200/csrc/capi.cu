// capi.cu — C-ABI glue of libb2s.so: errors, device info, variant dispatch, pipe microbenchmarks.
#include <stdarg.h>
#include <string.h>

#include "common.cuh"

namespace b2s {

static thread_local char g_err[512] = "";
static unsigned long long g_launches = 0;

void note_launch(int n) { __atomic_fetch_add(&g_launches, (unsigned long long)n, __ATOMIC_RELAXED); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what) {
  set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
  return B2S_ERR_CUDA;
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

int hamming_popc_launch(const uint8_t* q, const uint8_t* t, const int32_t* q_off, const int32_t* t_off,
                        const int32_t* q_src, const int32_t* t_src, int n_pairs, int total_nq, int total_nt,
                        int max_nq, int max_nt, uint32_t* fwd_best, uint32_t* fwd_second, uint32_t* bwd_best,
                        int t_split, void* workspace, size_t workspace_bytes, cudaStream_t st);

size_t hamming_i8_workspace_bytes(int n_pairs, int total_nq, int max_nq, int max_nt, int t_split);
int hamming_i8_launch(const uint8_t* q, const uint8_t* t, const int32_t* q_off, const int32_t* t_off,
                      const int32_t* q_src, const int32_t* t_src, int n_pairs, int total_nq, int total_nt, int max_nq,
                      int max_nt, uint32_t* fwd_best, uint32_t* fwd_second, uint32_t* bwd_best, int t_split,
                      void* workspace, size_t workspace_bytes, int single, int need_second, cudaStream_t st);

size_t hamming_i8_shared_workspace_bytes(int total_tiles, int n_pairs, int total_nq, int max_nq, int max_nt, int t_split);
int hamming_i8_shared_launch(const uint8_t* desc, const int32_t* blk_row0, const int32_t* blk_rows,
                             const int32_t* blk_tile0, int n_blocks, int total_tiles, int max_block_rows,
                             const int32_t* q_xtile, const int32_t* t_xtile, const int32_t* q_off, const int32_t* t_off,
                             int n_pairs, int total_nq, int total_nt, int max_nq, int max_nt, uint32_t* fwd_best,
                             uint32_t* fwd_second, uint32_t* bwd_best, int t_split, int need_second, void* workspace,
                             size_t workspace_bytes, cudaStream_t st);
void hamming_i8_last_plan(int* subs, int* t_split, int* grid);

int hamming_i8_timing(int enable, float* last_ms);
int mma_rate_launch(int iters, int n_dim, double* macs_out, cudaStream_t st);
int tmem_read_launch(int iters, int warps, double* bytes_out, uint32_t* sink, cudaStream_t st);

// ---- pipe microbenchmarks: 8 independent chains x 8 unrolled = 64 instructions / iteration ----
template <int WHICH>
__global__ void __launch_bounds__(256) pipe_kernel(int iters, uint32_t* sink) {
  uint32_t x[8];
  double d[8];
  float f[8], g[8];
  unsigned long long p2[8];
  float2 q2[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    x[k] = threadIdx.x * 2654435761u + k * 40503u + blockIdx.x;
    d[k] = 1.0 + 1e-9 * (double)x[k];
    f[k] = 1.0f + 1e-7f * (float)(x[k] & 1023);
    g[k] = 1.0f - 1e-7f * (float)(x[k] & 511);
    p2[k] = ((unsigned long long)__float_as_uint(f[k]) << 32) | __float_as_uint(f[k] * 0.5f);
    q2[k] = make_float2(f[k] * 0.25f, g[k] * 0.125f);
  }
  const uint32_t c1 = blockIdx.x | 1u, c2 = threadIdx.x | 3u;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (WHICH == 0) asm volatile("popc.b32 %0, %0;" : "+r"(x[k]));
        if (WHICH == 1) asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(x[k]) : "r"(c1), "r"(c2));
        if (WHICH == 2) asm volatile("add.u32 %0, %0, %1;" : "+r"(x[k]) : "r"(c1));
        if (WHICH == 3) asm volatile("min.u32 %0, %0, %1;" : "+r"(x[k]) : "r"(c2));
        if (WHICH == 4) asm volatile("fma.rn.f64 %0, %0, %1, %1;" : "+d"(d[k]) : "d"(d[(k + 1) & 7]));
        if (WHICH == 5) asm volatile("fma.rn.f32 %0, %0, %1, %1;" : "+f"(f[k]) : "f"(f[(k + 1) & 7]));
        if (WHICH == 6) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(x[k]) : "r"(c1), "r"(c2));
        if (WHICH == 7) asm volatile("redux.sync.min.s32 %0, %0, 0xffffffff;" : "+r"(x[k]));
        if (WHICH == 8) asm volatile("shfl.sync.bfly.b32 %0, %0, 1, 0x1f, 0xffffffff;" : "+r"(x[k]));
        if (WHICH == 9) x[k] = __vminu2(x[k], c2 + it);                      // VIMNMX.U16x2
        if (WHICH == 10) x[k] = __vimin3_u16x2(x[k], c1 + it, c2);           // VIMNMX3.U16x2
        if (WHICH == 11) x[k] = __viaddmax_u16x2(x[k], c1, c2);              // VIADDMNMX.U16x2
        if (WHICH == 12)  // SEL with a loop-invariant predicate
          asm volatile("{\n\t.reg .pred p;\n\tsetp.gt.u32 p, %2, 5;\n\tselp.b32 %0, %0, %1, p;\n\t}" : "+r"(x[k]) : "r"(c1), "r"(c2));
        if (WHICH == 13) asm volatile("prmt.b32 %0, %0, %1, 0x1032;" : "+r"(x[k]) : "r"(c1));
        if (WHICH == 14) asm volatile("fma.rn.f32x2 %0, %0, %1, %1;" : "+l"(p2[k]) : "l"(p2[(k + 1) & 7]));  // FFMA2: counts as ONE instruction
        if (WHICH == 15) {  // FFMA2 and scalar FFMA alternating (counted as ONE instruction per pair: compare the time with 14)
          asm volatile("fma.rn.f32x2 %0, %0, %1, %1;" : "+l"(p2[k]) : "l"(p2[(k + 1) & 7]));
          asm volatile("fma.rn.f32 %0, %0, %1, %1;" : "+f"(f[k]) : "f"(f[(k + 1) & 7]));
        }
        if (WHICH == 16) {  // one FFMA2 + two scalar FFMA
          asm volatile("fma.rn.f32x2 %0, %0, %1, %1;" : "+l"(p2[k]) : "l"(p2[(k + 1) & 7]));
          asm volatile("fma.rn.f32 %0, %0, %1, %1;" : "+f"(f[k]) : "f"(f[(k + 1) & 7]));
          asm volatile("fma.rn.f32 %0, %0, %1, %1;" : "+f"(g[k]) : "f"(g[(k + 1) & 7]));
        }
        if (WHICH == 17) {  // one FFMA2 + one ALU-pipe add: does the half-rate packed FMA leave its second issue cycle to another pipe?
          asm volatile("fma.rn.f32x2 %0, %0, %1, %1;" : "+l"(p2[k]) : "l"(p2[(k + 1) & 7]));
          asm volatile("add.u32 %0, %0, %1;" : "+r"(x[k]) : "r"(c1));
        }
        if (WHICH == 18) {  // one FFMA2 + two ALU-pipe adds
          asm volatile("fma.rn.f32x2 %0, %0, %1, %1;" : "+l"(p2[k]) : "l"(p2[(k + 1) & 7]));
          asm volatile("add.u32 %0, %0, %1;" : "+r"(x[k]) : "r"(c1));
          asm volatile("add.u32 %0, %0, %1;" : "+r"(x[(k + 3) & 7]) : "r"(c2));
        }
        if (WHICH == 19) {  // FFMA2 with three distinct 64-bit sources (register-file read bandwidth)
          asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(p2[k]) : "l"(p2[(k + 1) & 7]), "l"(p2[(k + 2) & 7]));
        }
        if (WHICH == 20) q2[k] = __ffma2_rn(make_float2(f[k], f[k]), q2[(k + 1) & 7], q2[k]);               // (scalar, pair, pair)
        if (WHICH == 21) q2[k] = __ffma2_rn(make_float2(f[k], f[k]), q2[k], make_float2(g[k], g[k]));       // (scalar, pair, scalar)
        if (WHICH == 22) asm volatile("fma.rn.f32 %0, %0, %1, %2;" : "+f"(f[k]) : "f"(g[k]), "f"(f[(k + 1) & 7]));   // scalar FFMA, three distinct sources
        if (WHICH == 23) q2[k] = __ffma2_rn(q2[k], q2[k], q2[(k + 1) & 7]);                                 // (pair, same pair, pair)
        if (WHICH == 24) q2[k] = __ffma2_rn(make_float2(f[k], f[k]), q2[k], q2[k]);                         // (scalar, pair, same pair)
      }
    }
  }
  uint32_t acc = 0;
#pragma unroll
  for (int k = 0; k < 8; ++k) acc ^= x[k] ^ (uint32_t)__double_as_longlong(d[k]) ^ __float_as_uint(f[k]) ^ (uint32_t)p2[k] ^ (uint32_t)(p2[k] >> 32) ^ __float_as_uint(g[k]) ^ __float_as_uint(q2[k].x) ^ __float_as_uint(q2[k].y);
  if (acc == 0x12345678u) sink[0] = acc;  // keeps the chains alive, practically never taken
}

}  // namespace b2s

extern "C" {

int b2s_abi_version(void) { return B2S_ABI_VERSION; }

unsigned long long b2s_launch_count(void) { return __atomic_load_n(&b2s::g_launches, __ATOMIC_RELAXED); }

const char* b2s_last_error(void) { return b2s::g_err; }

int b2s_device_info(int* sm_count, int* cc_major, int* cc_minor, int* clock_khz) {
  int dev = 0;
  B2S_CUDA(cudaGetDevice(&dev));
  int v = 0;
  if (sm_count) {
    B2S_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev));
    *sm_count = v;
  }
  if (cc_major) {
    B2S_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, dev));
    *cc_major = v;
  }
  if (cc_minor) {
    B2S_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMinor, dev));
    *cc_minor = v;
  }
  if (clock_khz) {
    B2S_CUDA(cudaDeviceGetAttribute(&v, cudaDevAttrClockRate, dev));
    *clock_khz = v;
  }
  return B2S_OK;
}

int b2s_hamming_knn2_batched(const uint8_t* q_desc, const uint8_t* t_desc, const int32_t* q_off,
                             const int32_t* t_off, const int32_t* q_src_row, const int32_t* t_src_row, int n_pairs,
                             int total_nq, int total_nt, int max_nq, int max_nt, uint32_t* fwd_best,
                             uint32_t* fwd_second, uint32_t* bwd_best, int variant, int t_split, void* workspace,
                             size_t workspace_bytes, void* stream) {
  using namespace b2s;
  B2S_REQUIRE(n_pairs >= 0 && total_nq >= 0 && total_nt >= 0 && max_nq >= 0 && max_nt >= 0, "negative size");
  B2S_REQUIRE(max_nq < B2S_MAX_ROWS_PER_PAIR && max_nt < B2S_MAX_ROWS_PER_PAIR,
              "more than 2^22-1 rows in one pair does not fit the packed key");
  if (n_pairs == 0) return B2S_OK;
  B2S_REQUIRE(q_off && t_off && fwd_best && fwd_second && bwd_best, "null pointer");
  B2S_REQUIRE((total_nq == 0 || q_desc) && (total_nt == 0 || t_desc), "null descriptor pointer");
  B2S_REQUIRE((((uintptr_t)q_desc | (uintptr_t)t_desc) & 15u) == 0, "descriptor buffers must be 16-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((variant & ~B2S_HAMMING_BEST_ONLY) == B2S_VARIANT_POPC) {
    return hamming_popc_launch(q_desc, t_desc, q_off, t_off, q_src_row, t_src_row, n_pairs, total_nq, total_nt,
                               max_nq, max_nt, fwd_best, fwd_second, bwd_best, t_split, workspace, workspace_bytes,
                               st);
  }
  const int need_second = !(variant & B2S_HAMMING_BEST_ONLY);
  variant &= ~B2S_HAMMING_BEST_ONLY;
  if (variant == B2S_VARIANT_I8MMA || variant == B2S_VARIANT_I8MMA1) {
    return hamming_i8_launch(q_desc, t_desc, q_off, t_off, q_src_row, t_src_row, n_pairs, total_nq, total_nt, max_nq,
                             max_nt, fwd_best, fwd_second, bwd_best, t_split, workspace, workspace_bytes,
                             variant == B2S_VARIANT_I8MMA1, need_second, st);
  }
  set_error("Hamming variant %d is not built into this library", variant);
  return B2S_ERR_UNSUPPORTED;
}

size_t b2s_hamming_shared_workspace_bytes(int total_tiles, int n_pairs, int total_nq, int max_nq, int max_nt, int t_split) {
  return b2s::hamming_i8_shared_workspace_bytes(total_tiles, n_pairs, total_nq, max_nq, max_nt, t_split);
}

void b2s_hamming_last_plan(int* subs, int* t_split, int* grid) { b2s::hamming_i8_last_plan(subs, t_split, grid); }

int b2s_hamming_knn2_shared(const uint8_t* desc, const int32_t* blk_row0, const int32_t* blk_rows,
                            const int32_t* blk_tile0, int n_blocks, int total_tiles, int max_block_rows,
                            const int32_t* q_xtile, const int32_t* t_xtile, const int32_t* q_off, const int32_t* t_off,
                            int n_pairs, int total_nq, int total_nt, int max_nq, int max_nt, uint32_t* fwd_best,
                            uint32_t* fwd_second, uint32_t* bwd_best, int t_split, int need_second, void* workspace,
                            size_t workspace_bytes, void* stream) {
  using namespace b2s;
  B2S_REQUIRE(n_pairs >= 0 && n_blocks >= 0 && total_tiles >= 0 && total_nq >= 0 && total_nt >= 0 && max_nq >= 0 &&
                  max_nt >= 0 && max_block_rows >= 0, "negative size");
  B2S_REQUIRE(max_nq < B2S_MAX_ROWS_PER_PAIR && max_nt < B2S_MAX_ROWS_PER_PAIR,
              "more than 2^22-1 rows in one pair does not fit the packed key");
  B2S_REQUIRE(n_pairs <= 65535, "n_pairs %d exceeds 65535; split the batch", n_pairs);
  if (n_pairs == 0) return B2S_OK;
  B2S_REQUIRE(desc && blk_row0 && blk_rows && blk_tile0 && q_xtile && t_xtile && q_off && t_off && fwd_best &&
                  fwd_second && bwd_best, "null pointer");
  B2S_REQUIRE(((uintptr_t)desc & 15u) == 0, "descriptor buffer must be 16-byte aligned");
  return hamming_i8_shared_launch(desc, blk_row0, blk_rows, blk_tile0, n_blocks, total_tiles, max_block_rows, q_xtile,
                                  t_xtile, q_off, t_off, n_pairs, total_nq, total_nt, max_nq, max_nt, fwd_best,
                                  fwd_second, bwd_best, t_split, need_second, workspace, workspace_bytes,
                                  static_cast<cudaStream_t>(stream));
}

size_t b2s_hamming_workspace_bytes_v(int variant, int n_pairs, int total_nq, int max_nq, int max_nt, int t_split) {
  variant &= ~B2S_HAMMING_BEST_ONLY;
  if (variant == B2S_VARIANT_I8MMA || variant == B2S_VARIANT_I8MMA1)
    return b2s::hamming_i8_workspace_bytes(n_pairs, total_nq, max_nq, max_nt, variant == B2S_VARIANT_I8MMA1 ? t_split : 1);
  return b2s_hamming_workspace_bytes(total_nq, t_split);
}

int b2s_hamming_kernel_timing(int enable, float* last_ms) { return b2s::hamming_i8_timing(enable, last_ms); }

int b2s_mma_microbench(int iters, int n_dim, double* macs_out, void* stream) {
  return b2s::mma_rate_launch(iters, n_dim, macs_out, static_cast<cudaStream_t>(stream));
}

int b2s_tmem_microbench(int iters, int warps, double* bytes_out, uint32_t* sink, void* stream) {
  return b2s::tmem_read_launch(iters, warps, bytes_out, sink, static_cast<cudaStream_t>(stream));
}

int b2s_pipe_microbench(int which, int iters, int ctas_per_sm, double* ops_out, uint32_t* sink, void* stream) {
  using namespace b2s;
  B2S_REQUIRE(which >= 0 && which <= 24, "which must be 0..24");
  B2S_REQUIRE(iters > 0 && ctas_per_sm > 0 && sink, "bad argument");
  const int grid = sm_count() * ctas_per_sm;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (which) {
    case 0: pipe_kernel<0><<<grid, 256, 0, st>>>(iters, sink); break;
    case 1: pipe_kernel<1><<<grid, 256, 0, st>>>(iters, sink); break;
    case 2: pipe_kernel<2><<<grid, 256, 0, st>>>(iters, sink); break;
    case 3: pipe_kernel<3><<<grid, 256, 0, st>>>(iters, sink); break;
    case 4: pipe_kernel<4><<<grid, 256, 0, st>>>(iters, sink); break;
    case 5: pipe_kernel<5><<<grid, 256, 0, st>>>(iters, sink); break;
    case 7: pipe_kernel<7><<<grid, 256, 0, st>>>(iters, sink); break;
    case 8: pipe_kernel<8><<<grid, 256, 0, st>>>(iters, sink); break;
    case 9: pipe_kernel<9><<<grid, 256, 0, st>>>(iters, sink); break;
    case 10: pipe_kernel<10><<<grid, 256, 0, st>>>(iters, sink); break;
    case 11: pipe_kernel<11><<<grid, 256, 0, st>>>(iters, sink); break;
    case 12: pipe_kernel<12><<<grid, 256, 0, st>>>(iters, sink); break;
    case 13: pipe_kernel<13><<<grid, 256, 0, st>>>(iters, sink); break;
    case 14: pipe_kernel<14><<<grid, 256, 0, st>>>(iters, sink); break;
    case 15: pipe_kernel<15><<<grid, 256, 0, st>>>(iters, sink); break;
    case 17: pipe_kernel<17><<<grid, 256, 0, st>>>(iters, sink); break;
    case 18: pipe_kernel<18><<<grid, 256, 0, st>>>(iters, sink); break;
    case 19: pipe_kernel<19><<<grid, 256, 0, st>>>(iters, sink); break;
    case 20: pipe_kernel<20><<<grid, 256, 0, st>>>(iters, sink); break;
    case 21: pipe_kernel<21><<<grid, 256, 0, st>>>(iters, sink); break;
    case 22: pipe_kernel<22><<<grid, 256, 0, st>>>(iters, sink); break;
    case 23: pipe_kernel<23><<<grid, 256, 0, st>>>(iters, sink); break;
    case 24: pipe_kernel<24><<<grid, 256, 0, st>>>(iters, sink); break;
    case 16: pipe_kernel<16><<<grid, 256, 0, st>>>(iters, sink); break;
    default: pipe_kernel<6><<<grid, 256, 0, st>>>(iters, sink); break;
  }
  B2S_CUDA(cudaGetLastError());
  note_launch();
  if (ops_out) *ops_out = (double)grid * 256.0 * (double)iters * 64.0;
  return B2S_OK;
}

}  // extern "C"
