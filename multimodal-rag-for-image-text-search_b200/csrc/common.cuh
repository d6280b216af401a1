// Shared device helpers for the sm_100a scan kernels: orderable top-k keys, mbarrier / bulk-copy /
// TMA / tcgen05 PTX wrappers.  Everything here is hand-written inline PTX for sm_100a; there is no
// other backend.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace mmr {

// ------------------------------------------------------------------------------------------------
// Top-k keys.  One u64 orders (score desc, row asc):  key = orderable(score) << 32 | (~row).
// Larger key = better hit.  key 0 is the "empty slot" sentinel (no finite/inf float maps to 0 in the
// high word).  Row ordinals are local to one resident index (< 2^32 rows per GPU); the shard base is
// added when results are written out as int64.
// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t f32_orderable(float f) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(f + 0.0f);  // -0.0 -> +0.0 so equal scores tie
#else
  f = f + 0.0f;
  uint32_t u;
  memcpy(&u, &f, 4);
#endif
  return u ^ ((u >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__host__ __device__ __forceinline__ float f32_from_orderable(uint32_t o) {
  uint32_t u = o ^ ((o >> 31) ? 0x80000000u : 0xFFFFFFFFu);
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}
__host__ __device__ __forceinline__ uint64_t make_key(float score, uint32_t row) {
  return (uint64_t(f32_orderable(score)) << 32) | uint64_t(0xFFFFFFFFu - row);
}
__host__ __device__ __forceinline__ float key_score(uint64_t key) { return f32_from_orderable(uint32_t(key >> 32)); }
__host__ __device__ __forceinline__ uint32_t key_row(uint64_t key) { return 0xFFFFFFFFu - uint32_t(key); }

// ------------------------------------------------------------------------------------------------
// Switches (DESIGN 6a).  Read ONCE from the environment when the library is loaded; mmr_set_option() changes them
// afterwards (tests, bench).  Nothing on the search path calls getenv.
// ------------------------------------------------------------------------------------------------
struct Options {
  int pdl = 0;            // MMR_PDL=1        pipelined launches (programmatic dependent launch) for K1 / merge_wait
  int enc_fuse_ln = 0;    // MMR_ENC_FUSE_LN     device encoders: LayerNorm folded into the GEMM behind it (gemm_wt_kernel<.., true>):
                          //                     0 = never (default: measured no faster, profiles/r02_encoder_summary.md), 1 = for
                          //                     passes of <= 16 tokens, 2 = whenever the token tile is 64
  int enc_att_mma = 1;    // MMR_ENC_ATT_MMA     device encoders: 1 = the cross-encoder runs attention_mma_kernel (bf16 tensor-core
                          //                     contractions), the query encoders the fp32 kernel (default); 0 = fp32 everywhere;
                          //                     2 = every model from 96 tokens on (measurement)
  int enc_gemm_smem_kb = 100;  // MMR_ENC_GEMM_SMEM_KB  shared-memory budget of one encoder GEMM CTA (ring depth).  100 lets two CTAs
                               //                       share an SM, so one tile's epilogue (the bound: bias / GELU / residual over
                               //                       NT columns per thread) overlaps the other's loads and MMAs: 128 x 128 rerank
                               //                       pairs 1.99 -> 1.45 ms against 200 (profiles/r02_encoder_summary.md)
  int enc_narrow_tiles = 1;    // MMR_ENC_NARROW_TILES=0  encoder GEMMs: token tile by token count only (default: halved for the narrow
                               //                         GEMMs until every SM has two CTAs)
  int inline_query = 1;   // MMR_INLINE_QUERY=0  host-buffer calls always stage the query with an H2D copy (measurement)
  int mailbox = 0;        // MMR_MAILBOX=1       host-buffer calls spin on a flag the kernel writes into the mapped mailbox instead
                          //                     of synchronising the stream (measured no faster: profiles/r02_fixed_cost.json)
};
inline Options& options() {
  static Options o;
  return o;
}

#ifdef __CUDACC__
// ------------------------------------------------------------------------------------------------
// Warp helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t shfl_u64(uint64_t v, int src) {
  uint32_t lo = __shfl_sync(0xffffffffu, uint32_t(v), src);
  uint32_t hi = __shfl_sync(0xffffffffu, uint32_t(v >> 32), src);
  return (uint64_t(hi) << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl_u64_xor(uint64_t v, int mask) {
  uint32_t lo = __shfl_xor_sync(0xffffffffu, uint32_t(v), mask);
  uint32_t hi = __shfl_xor_sync(0xffffffffu, uint32_t(v >> 32), mask);
  return (uint64_t(hi) << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl_up_u64(uint64_t v, int d) {
  uint32_t lo = __shfl_up_sync(0xffffffffu, uint32_t(v), d);
  uint32_t hi = __shfl_up_sync(0xffffffffu, uint32_t(v >> 32), d);
  return (uint64_t(hi) << 32) | lo;
}
__device__ __forceinline__ float warp_allreduce_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------
// Shared-memory addresses, mbarrier, bulk async copy (TMA engine, 1-D, no descriptor)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// global -> shared bulk copy; completion is signalled as `bytes` of transaction on `bar`.
// src and dst must be 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void bulk_g2s_hint(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar,
                                              uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          dst_smem),
      "l"(src), "r"(bytes), "r"(bar), "l"(policy)
      : "memory");
}

__device__ __forceinline__ void lds_v4(uint32_t addr, uint32_t (&r)[4]) {
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void lds_v2(uint32_t addr, uint32_t (&r)[2]) {
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(addr));
}
// Programmatic dependent launch, the always-safe form: the kernel lets its successor be scheduled right away and
// itself waits for its predecessor's completion (and memory flush) before doing anything.  Only launch latency and
// per-CTA setup overlap; data dependencies are untouched.
__device__ __forceinline__ void pdl_chain_prologue() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// The two halves separately: a kernel whose first phase touches nothing its predecessor wrote (barrier init, tensor-memory
// allocation, TMA loads of the index) lets that phase run UNDER the predecessor and waits only in the warps that read the
// predecessor's outputs.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait_prior_grid() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif  // __CUDACC__

}  // namespace mmr
