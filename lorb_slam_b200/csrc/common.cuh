// common.cuh — context, error plumbing and device helpers shared by the
// sm_100a kernels behind include/lorb_cuda.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/lorb_cuda.h"

namespace lorb {

void set_error(const char* fmt, ...);

#define LORB_CUDA_TRY(expr)                                                              \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess) {                                                             \
      lorb::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return LORB_ERR_CUDA;                                                              \
    }                                                                                    \
  } while (0)

#define LORB_REQUIRE(cond, msg)                                         \
  do {                                                                  \
    if (!(cond)) {                                                      \
      lorb::set_error("%s:%d: bad argument: %s", __FILE__, __LINE__, msg); \
      return LORB_ERR_ARG;                                              \
    }                                                                   \
  } while (0)

// Grow-only buffer (device or pinned host).  Owned by a ctx; never shrinks so
// steady-state calls allocate nothing.
struct Buf {
  void* p = nullptr;
  size_t cap = 0;
  bool pinned = false;
  int reserve(size_t bytes);
  void release();
  template <typename T>
  T* as() const {
    return reinterpret_cast<T*>(p);
  }
};

struct Dist;  // NCCL state (dist.cu)

}  // namespace lorb

struct lorb_ctx {
  int device = 0;
  int sm_count = 0;
  int smem_optin = 0;  // max dynamic shared memory per block (opt-in)
  cudaStream_t stream = nullptr;
  long long launches = 0;
  // generic scratch: device buffers d[i], pinned host buffers h[i]
  lorb::Buf d[16];
  lorb::Buf h[8];
  // resident descriptor bank + sweep plan (match_bf.cu)
  lorb::Buf bank;
  int bank_n_kf = 0, bank_n_desc = 0;
  lorb::Buf plan_pairs, plan_out;
  int plan_n_pairs = 0, plan_max_a = 0, plan_max_b = 0;
  // tensor-core form of the sweep (match_tc.cu): int8 operand images of the bank, unit list,
  // row / column key scratch
  int sweep_impl = -1;  // LORB_SWEEP_POPC / LORB_SWEEP_TENSOR; -1 = default (env LORB_SWEEP_IMPL)
  lorb::Buf tc_img, tc_units, tc_keys;
  int tc_img_n_kf = 0, tc_img_n_desc = 0;
  long long tc_n_units = 0;
  std::vector<long long> tc_chunk_units;  // first unit of every <= 16384-pair chunk of the plan (+ end)
  size_t tc_keys_rows = 0;
  int proj_coop_blocks[2] = {-1, -1};  // co-resident CTAs of the cooperative claim resolution (match_proj.cu)
  int chol_chain_blocks = -1;          // same for the chain Cholesky (ba_local.cu); -1 = not yet queried
  lorb::Dist* dist = nullptr;
  lorb_ba_loss ba_loss = {LORB_LOSS_TRIVIAL, 0, 1.0};  // robust loss of every BA solve on this ctx
  void* ba_cache = nullptr;  // reusable lorb_ba_problem of the host-buffer BA calls (ba_local.cu)
  cudaStream_t ba_stream2 = nullptr;  // side branch of the large-path build pass (camera rows beside the Schur pairs)
  cudaEvent_t ba_ev[2] = {nullptr, nullptr};
  // cached CUDA graphs of the ORB extractor's detection chain (orb.cu), one per job slot
  void* orb_graph[2] = {nullptr, nullptr};
  cudaStream_t orb_stream2 = nullptr;  // side branch of the extractor graph (capture only)
  cudaEvent_t orb_ev[3] = {nullptr, nullptr, nullptr};
  cudaStream_t orb_stream3 = nullptr;  // second frame of a stereo pair runs its graph here, concurrently
  cudaEvent_t orb_join = nullptr;
  // optional event timing of the library's own kernels (lorb_ctx_profile)
  int prof_on = 0;
  void* prof = nullptr;  // lorb::Prof (ctx.cu)
};

namespace lorb {

inline int dev_reserve(lorb_ctx* c, int slot, size_t bytes) { return c->d[slot].reserve(bytes); }
inline int pin_reserve(lorb_ctx* c, int slot, size_t bytes) {
  c->h[slot].pinned = true;
  return c->h[slot].reserve(bytes);
}

// Event brackets around a kernel (no-ops unless lorb_ctx_profile enabled them).
void prof_begin(lorb_ctx* c, int slot);
void prof_end(lorb_ctx* c, int slot);

#define LORB_TRY(expr)          \
  do {                          \
    int _rc = (expr);           \
    if (_rc != LORB_OK) return _rc; \
  } while (0)

namespace tc {  // match_tc.cu
int bank_expand(lorb_ctx* c);
int plan_build(lorb_ctx* c, const int* pa, const int* pb, int n_pairs);
int launch_sweep(lorb_ctx* c, int kf_base_a, int kf_base_b, int n_pairs, int* out);
}  // namespace tc

// Kernel launch bookkeeping: every launch goes through this so that
// lorb_ctx_launch_count is the bench's "gpu_launches".
#define LORB_LAUNCH(ctx, kernel, grid, block, smem, ...)                   \
  do {                                                                     \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);       \
    (ctx)->launches++;                                                     \
    LORB_CUDA_TRY(cudaGetLastError());                                     \
  } while (0)

// ------------------------------------------------------------ device helpers
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// mbarrier + 1-D TMA bulk copy (cp.async.bulk; SASS UBLKCP) used to stage
// descriptor blocks into shared memory.
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(smem_u32(smem_dst)),
      "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// LOP3 with an explicit truth table (0x96 = a^b^c, 0xE8 = majority).
template <int LUT>
__device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(d) : "r"(a), "r"(b), "r"(c), "n"(LUT));
  return d;
}
// a*b+c on the FMA pipe (IMAD), keeping the ALU pipe for LOP3/VIMNMX.
__device__ __forceinline__ uint32_t imad(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

// 256-bit Hamming distance, plain form: 8 x (XOR, POPC) + adds.
// Same value as reference src/matcher.cpp:369-385 (SWAR popcount there).
__device__ __forceinline__ uint32_t hamming256_popc8(const uint32_t (&q)[8], const uint32_t (&t)[8]) {
  uint32_t s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += __popc(q[i] ^ t[i]);
  return s;
}

// 256-bit Hamming distance, carry-save form: the 8 XOR words are compressed
// with four 3:2 counters (LOP3 0x96 / 0xE8) into ones/ones/twos/fours words so
// only 4 POPC are issued:  d = popc(s3) + popc(x7) + 2*popc(t) + 4*popc(f).
__device__ __forceinline__ uint32_t hamming256_csa(const uint32_t (&q)[8], const uint32_t (&t)[8]) {
  uint32_t x0 = q[0] ^ t[0], x1 = q[1] ^ t[1], x2 = q[2] ^ t[2], x3 = q[3] ^ t[3];
  uint32_t x4 = q[4] ^ t[4], x5 = q[5] ^ t[5], x6 = q[6] ^ t[6], x7 = q[7] ^ t[7];
  uint32_t s1 = lop3<0x96>(x0, x1, x2), c1 = lop3<0xE8>(x0, x1, x2);
  uint32_t s2 = lop3<0x96>(x3, x4, x5), c2 = lop3<0xE8>(x3, x4, x5);
  uint32_t s3 = lop3<0x96>(s1, s2, x6), c3 = lop3<0xE8>(s1, s2, x6);
  uint32_t tw = lop3<0x96>(c1, c2, c3), fo = lop3<0xE8>(c1, c2, c3);
  uint32_t ones = imad((uint32_t)__popc(s3), 1u, (uint32_t)__popc(x7));
  uint32_t d = imad((uint32_t)__popc(tw), 2u, ones);
  return imad((uint32_t)__popc(fo), 4u, d);
}

// Packed (distance, index) keys: distance in the high bits, index in the low
// KEY_IDX_BITS, so that unsigned min() == (smallest distance, then lowest
// index) — exactly OpenCV's first-strict-minimum tie-break on both sides.
constexpr int KEY_IDX_BITS = 20;
constexpr uint32_t KEY_IDX_MASK = (1u << KEY_IDX_BITS) - 1u;
constexpr uint32_t KEY_NONE = 0xFFFFFFFFu;
__device__ __forceinline__ uint32_t make_key(uint32_t dist, uint32_t idx) {
  return imad(dist, 1u << KEY_IDX_BITS, idx);
}

#endif  // __CUDACC__

}  // namespace lorb
