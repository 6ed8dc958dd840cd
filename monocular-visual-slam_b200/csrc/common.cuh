// common.cuh — shared device/host helpers for libb2s (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/b2s.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libb2s is written for sm_100a (B200) only"
#endif

namespace b2s {

// ---- result records (include/b2s.h) -------------------------------------------
// record = 16 x int32 header | S x u16 queryIdx | S x u16 trainIdx | S x u16 distance | S x u8 inlier | pad to 64 B
__host__ __device__ constexpr size_t record_bytes(int S) { return ((size_t)64 + 7 * (size_t)S + 63) & ~(size_t)63; }
// pose record = record | b2s_pose_result | zero pad to B2S_POSE_BLOCK_BYTES; the pose block starts on a 64-byte
// boundary, so its doubles are aligned
__host__ __device__ constexpr size_t pose_record_bytes(int S) { return record_bytes(S) + B2S_POSE_BLOCK_BYTES; }
static_assert(record_bytes(1) == 128 && record_bytes(500) == 3584 && pose_record_bytes(500) == 3840, "record layout");
static_assert(B2S_POSE_BLOCK_BYTES - B2S_POSE_RESULT_BYTES == 56, "pose block = b2s_pose_result + 56 zero bytes");

// ---- error plumbing (no exceptions across the C ABI) --------------------------
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define B2S_CUDA(call)                                        \
  do {                                                        \
    cudaError_t e__ = (call);                                 \
    if (e__ != cudaSuccess) return b2s::cuda_fail(e__, #call); \
  } while (0)

#define B2S_REQUIRE(cond, ...)       \
  do {                               \
    if (!(cond)) {                   \
      b2s::set_error(__VA_ARGS__);   \
      return B2S_ERR_INVALID;        \
    }                                \
  } while (0)

int sm_count();
// true exactly once per (flag array, current device): function attributes such as the dynamic shared-memory
// opt-in are per device, and one process may drive several GPUs (HammingMatcher(device=...)).  A race between
// host threads only repeats an idempotent call.
inline bool first_use_on_device(bool (&done)[64]) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
  if (done[dev]) return false;
  done[dev] = true;
  return true;
}
void note_launch(int n = 1);  // counts kernels launched by this library (b2s_launch_count)

constexpr uint32_t kNone = 0xFFFFFFFFu;
constexpr int kIdxBits = B2S_IDX_BITS;
constexpr uint32_t kIdxMask = B2S_IDX_MASK;
constexpr uint32_t kInvalidRow = 0x80000000u;  // added to a key: sorts after every valid key, no overflow

// ---- PTX wrappers: mbarrier + 1-D bulk async copy (TMA engine, SASS UBLKCP) ---
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// ---- packed-key top-2 ------------------------------------------------------------
__device__ __forceinline__ void top2_insert(uint32_t& best, uint32_t& second, uint32_t key) {
  uint32_t mx = max(best, key);
  best = min(best, key);
  second = min(second, mx);
}

}  // namespace b2s
