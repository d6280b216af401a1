// K2x2 -- the tensor-bound variant of K2 on CTA pairs: tcgen05.mma.cta_group::2 (M = 256 queries per pair).
//
// Why: with cta_group::1 every SM reads the whole 128-row index tile from its own shared memory for each MMA
// (64 B/cycle) and TMA writes the same tile in (64 B/cycle): the 128 B/cycle shared-memory port is the ceiling
// (profiles/r01_k2_summary.md).  A CTA pair shares the tile: each CTA loads HALF of it (64 rows), the pair's MMA
// reads both halves, so per-SM shared-memory and L2->SM traffic per flop halve.
//
// Pair layout (cluster of 2 CTAs on one TPC):
//   * CTA rank r owns query tile 2*pair + r: its 128 normalised bf16 queries live in ITS tensor memory (A operand,
//     written with tcgen05.st), its accumulators D[128 x 128] live in ITS tensor memory, its epilogue warps filter
//     ITS queries with K2's epilogue (k2_epilogue).
//   * both CTAs stream the same row tiles; CTA r TMA-loads rows [row0 + 64 r, row0 + 64 r + 64) of each K-slice
//     (8 KB, SWIZZLE_128B) into its own ring.  The loads use .cta_group::2 and signal the LEADER's "full" barrier.
//   * only the leader (rank 0) issues tcgen05.mma.cta_group::2 (M=256, N=128, K=16); tcgen05.commit ... multicast
//     releases the ring slot in both CTAs and publishes the accumulator to both epilogues.
//   * both epilogues release the accumulator by arriving on the leader's "tmem empty" barrier (remote arrive).
#pragma once
#include "scan_umma.cuh"

namespace mmr {

constexpr int K2X_HALF = 64;                 // index rows per CTA per tile
constexpr int K2X_SLICE = K2X_HALF * 128;    // 8 KB: [64 rows x 64 bf16]
constexpr int K2X_MAX_STAGES = 24;
constexpr int K2X_ACC = 2;

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> the same offset in CTA `rank` of the cluster (shared::cluster address)
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// Remote arrive with the default (.release.cta) semantics: the arriving warps publish nothing through ordinary memory
// (tensor-memory reads are ordered by tcgen05.fence::before_thread_sync), and a cluster-scope release costs a full
// memory barrier per arrive -- it was 31 % of all stall samples in the first version (profiles/r01_k2_summary.md).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc_512_2sm(uint32_t dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(512u) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_512_2sm(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(512u) : "memory");
}
// TMA load issued by either CTA of the pair; completion bytes go to the LEADER's mbarrier (peer bit cleared).
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst_smem, const CUtensorMap* map, uint32_t bar, int32_t c0,
                                                int32_t c1) {
  const uint32_t leader_bar = bar & 0xFEFFFFFFu;
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          dst_smem),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma2_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      :
      : "r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive (once every prior MMA of this thread has completed) on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma2_commit_mc(uint32_t bar) {
  const uint16_t mask = 3;
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"(mask)
      : "memory");
}
__host__ __device__ constexpr uint32_t umma_idesc_m256_n128(bool bf16) {
  return (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) | (uint32_t(K2_NT >> 3) << 17) |
         (uint32_t(256 >> 4) << 24);
}

template <bool DUMP>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(K2_THREADS, 1)
scan_umma2_kernel(const __grid_constant__ CUtensorMap tm_x, const UmmaParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  pdl_launch_dependents();   // (as in scan_umma_kernel: only the epilogue warps wait for the previous kernel of the chain)
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int ks = p.ks, nstages = p.nstages, k = p.k;
  const uint32_t rank = cluster_ctarank();
  const bool lead_cta = rank == 0;
  const uint32_t acc_col0 = uint32_t(ks * 32);  // columns [0, D/2) hold this CTA's packed query tile

  const uint32_t st_s = smem_u32(smem);
  uint64_t* lists = reinterpret_cast<uint64_t*>(smem + size_t(nstages) * K2X_SLICE);  // [k][128]
  uint32_t* metas = reinterpret_cast<uint32_t*>(lists + size_t(k) * K2_BM);
  uint64_t* bars = reinterpret_cast<uint64_t*>(metas + K2_BM);
  const uint32_t bar_full = smem_u32(bars);                       // [K2X_MAX_STAGES]  used in the leader
  const uint32_t bar_empty = bar_full + K2X_MAX_STAGES * 8;       // [K2X_MAX_STAGES]  used in both CTAs
  const uint32_t bar_tfull = bar_empty + K2X_MAX_STAGES * 8;      // [K2X_ACC]         used in both CTAs
  const uint32_t bar_tempty = bar_tfull + K2X_ACC * 8;            // [K2X_ACC]         used in the leader
  const uint32_t bar_q = bar_tempty + K2X_ACC * 8;                // [1]               used in the leader
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * K2X_MAX_STAGES + 2 * K2X_ACC + 1);

  const int pair = int(blockIdx.x >> 1);
  const int n_qpairs = (p.n_qtiles + 1) >> 1;
  const int qpair = pair % n_qpairs;
  const int rs = pair / n_qpairs;
  const int qt = qpair * 2 + int(rank);
  const uint32_t nrows = p.row_end - p.row_begin;
  const int ntiles_all = int((nrows + K2_NT - 1) / K2_NT);
  const int ntiles = p.probe_out ? min(ntiles_all, rs + p.probe_tiles * p.n_rslots) : ntiles_all;

  if (threadIdx.x == 0) {
    if ((st_s & 1023u) != 0) __trap();
    for (int s = 0; s < K2X_MAX_STAGES; ++s) {
      mbar_init(bar_full + s * 8, 1);
      mbar_init(bar_empty + s * 8, 1);
    }
    for (int a = 0; a < K2X_ACC; ++a) {
      mbar_init(bar_tfull + a * 8, 1);
      mbar_init(bar_tempty + a * 8, 8);  // 4 epilogue warps x 2 CTAs
    }
    mbar_init(bar_q, 8);
    fence_mbar_init();
    tma_prefetch_desc(&tm_x);
  }
  if (warp == 1) tmem_alloc_512_2sm(smem_u32(tmem_slot));
  tc_fence_before();
  cluster_sync_all();  // barriers of both CTAs are initialised before anyone signals across the pair
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer (both CTAs, own half)
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    for (int t = rs; t < ntiles; t += p.n_rslots) {
      const int32_t row0 = int32_t(p.row_begin + uint32_t(t) * K2_NT + rank * K2X_HALF);
      for (int s = 0; s < ks; ++s) {
        mbar_wait(bar_empty + stage * 8, phase ^ 1u);
        if (leader) {
          if (lead_cta) mbar_arrive_expect_tx(bar_full + stage * 8, 2 * K2X_SLICE);  // both halves land on this barrier
          tma_load_2d_2sm(st_s + stage * K2X_SLICE, &tm_x, bar_full + stage * 8, s * 64, row0);
        }
        __syncwarp();
        if (++stage == nstages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA only)
    if (lead_cta) {
      const bool leader = elect_one();
      const uint32_t idesc = p.idesc;
      mbar_wait(bar_q, 0);
      tc_fence_after();
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (int t = rs; t < ntiles; t += p.n_rslots) {
        mbar_wait(bar_tempty + acc * 8, acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc_col0 + uint32_t(acc) * K2_NT;
        for (int s = 0; s < ks; ++s) {
          mbar_wait(bar_full + stage * 8, phase);
          tc_fence_after();
          const uint64_t b_desc = umma_smem_desc(st_s + stage * K2X_SLICE);
          if (leader) {
#pragma unroll
            for (int kk = 0; kk < 4; ++kk)
              umma2_f16_ts(d_tmem, tmem_base + uint32_t(s * 32 + kk * 8), b_desc + uint64_t(kk * 2), idesc,
                           uint32_t((s | kk) != 0));
            umma2_commit_mc(bar_empty + stage * 8);
          }
          __syncwarp();
          if (++stage == nstages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        if (leader) umma2_commit_mc(bar_tfull + acc * 8);
        __syncwarp();
        if (++acc == K2X_ACC) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: thread = query (both CTAs)
    const int quarter = warp & 3;
    const int qglob = qt * K2_BM + quarter * 32 + lane;
    const bool live = qglob < p.B;
    pdl_wait_prior_grid();
    // stage the (already normalised, bf16) query tile into tensor memory: lane = query, column c = elements 2c, 2c+1
    const uint32_t* qsrc = reinterpret_cast<const uint32_t*>(p.qbf16) + size_t(live ? qglob : 0) * (ks * 32);
    for (int c = 0; c < ks; ++c) {
      uint32_t w[32];
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        uint4 x = live ? *reinterpret_cast<const uint4*>(qsrc + c * 32 + j) : make_uint4(0u, 0u, 0u, 0u);
        w[j] = x.x; w[j + 1] = x.y; w[j + 2] = x.z; w[j + 3] = x.w;
      }
      tmem_st_x32(tmem_base + (uint32_t(quarter * 32) << 16) + uint32_t(c * 32), w);
    }
    tmem_wait_st();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive_cluster(mapa_u32(bar_q, 0));
    k2_epilogue<DUMP, K2X_ACC>(p, qt, rs, ntiles, lists, metas, tmem_base + acc_col0, bar_tfull,
                               [&](int acc) { mbar_arrive_cluster(mapa_u32(bar_tempty + acc * 8, 0)); });
  }
  tc_fence_before();
  cluster_sync_all();  // the peer's shared memory / tensor memory stay alive until the leader's MMAs are done
  if (warp == 1) tmem_dealloc_512_2sm(tmem_base);
}
#endif  // __CUDACC__

// [n_rows, dim] 16-bit row-major -> boxes of [64 rows x 64 elements], 128-byte swizzle (one CTA's half tile)
inline bool umma2_make_map(CUtensorMap* map, const void* base, int64_t n_rows, int dim, bool bf16) {
  mmr_encode_tiled_fn fn = umma_encode_fn();
  if (!fn) return false;
  cuuint64_t gdim[2] = {cuuint64_t(dim), cuuint64_t(n_rows)};
  cuuint64_t gstr[1] = {cuuint64_t(dim) * 2};
  cuuint32_t box[2] = {64, K2X_HALF};
  cuuint32_t estr[2] = {1, 1};
  return fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base),
            gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

inline int umma2_plan_stages(int k, size_t* smem_bytes) {
  const size_t fixed = size_t(k) * K2_BM * 8 + K2_BM * 4 + (2 * K2X_MAX_STAGES + 2 * K2X_ACC + 2) * 8 + 1024;
  int stages = int((size_t(K2_SMEM_LIMIT) - fixed) / K2X_SLICE);
  stages = std::min(stages, K2X_MAX_STAGES);
  if (smem_bytes) *smem_bytes = fixed + size_t(std::max(stages, 0)) * K2X_SLICE;
  return stages;
}

#ifdef __CUDACC__
struct Umma2IndexState {
  bool valid = false;
  const void* rows = nullptr;
  int64_t n_rows = 0;
  CUtensorMap map;
};

// One K2 search: prep queries -> [probe pass -> floor] -> scan (grid = query tiles x row slots) -> per-query merge.  `ws` is
// the K2 slice of the workspace (umma_workspace_bytes).  dump != nullptr runs the raw-score debug variant instead of top-k.
inline int umma_search(UmmaIndexState& st, Umma2IndexState& st2, const void* rows, int64_t n_rows, int dim, int dtype, int sm_count,
                       const float* queries, int B, int k, uint32_t r0, uint32_t r1, int64_t row_base, float* out_s,
                       int64_t* out_r, uint8_t* ws, cudaStream_t stream, std::string& err, float* dump = nullptr,
                       int64_t dump_ld = 0, float* qerr = nullptr) {
  // Kernel, chosen from measurements on B200 (profiles/r01_k2_summary.md): one query tile (B <= 128) is HBM-bound and
  // fastest on single CTAs with both operands in shared memory and 4 accumulators (scan_umma_kernel).  Several query tiles
  // are tensor-bound: CTA pairs (cta_group::2) with the query tile in tensor memory (scan_umma2_kernel) read half the
  // shared memory per MMA and are 5-9 % faster than single CTAs there (B=1024: 8.30 vs 8.72 ms).
  const bool pair = umma_qtiles(B) >= 2;
  size_t smem_bytes = 0;
  const int stages = pair ? umma2_plan_stages(k, &smem_bytes) : umma_plan_stages(dim, k, &smem_bytes);
  // the pair kernel's packed query tile (D/2 columns) and its accumulators share the 512 tensor-memory columns
  if (stages < 2 || (pair && dim / 2 + K2X_ACC * K2_NT > 512)) {
    err = "K2: shared / tensor memory plan does not fit";
    return MMR_ERR_UNSUPPORTED;
  }
  static bool attr_done[64] = {};
  int cur_dev = 0;
  cudaGetDevice(&cur_dev);
  bool& attr_set = attr_done[cur_dev & 63];
  if (!attr_set) {
    cudaFuncSetAttribute(scan_umma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_LIMIT);
    cudaFuncSetAttribute(scan_umma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_LIMIT);
    cudaFuncSetAttribute(scan_umma2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_LIMIT);
    cudaFuncSetAttribute(scan_umma2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, K2_SMEM_LIMIT);
    attr_set = true;
  }
  __nv_bfloat16* qb = reinterpret_cast<__nv_bfloat16*>(ws);
  uint64_t* partial = reinterpret_cast<uint64_t*>(ws + umma_align(size_t(B) * dim * 2));
  const int ctas_max = std::max(sm_count, std::min(umma_qtiles(B), sm_count));
  float* probe = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(partial) + umma_align(size_t(ctas_max) * K2_BM * k * 8));
  float* floor = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(probe) + umma_align(size_t(ctas_max) * K2_BM * 4));
  if (pair) {
    if (!st2.valid || st2.rows != rows || st2.n_rows != n_rows) {
      if (!umma2_make_map(&st2.map, rows, n_rows, dim, dtype == MMR_BF16)) {
        err = "cuTensorMapEncodeTiled failed for the half-tile index map";
        return MMR_ERR_CUDA;
      }
      st2.valid = true;
      st2.rows = rows;
      st2.n_rows = n_rows;
    }
  } else {
    if (!st.valid || st.rows != rows || st.n_rows != n_rows) {
      if (!umma_make_map(&st.map, rows, n_rows, dim, dtype == MMR_BF16)) {
        err = "cuTensorMapEncodeTiled failed for the index";
        return MMR_ERR_CUDA;
      }
      st.valid = true;
      st.rows = rows;
      st.n_rows = n_rows;
    }
    // the query tile is TMA-loaded too (one tile, so one pass below)
    if (!(st.q_valid && st.q_ptr == qb && st.q_rows == B)) {
      if (!umma_make_map(&st.q_map, qb, B, dim, dtype == MMR_BF16)) {
        err = "cuTensorMapEncodeTiled failed for the queries";
        return MMR_ERR_CUDA;
      }
      st.q_valid = true;
      st.q_ptr = qb;
      st.q_rows = B;
    }
  }
  // the scan kernel chosen above: top-k, or raw scores when prm.dump is set
  auto launch_scan = [&](int grid, const UmmaParams& prm) {
    const bool d = prm.dump != nullptr;
    if (pair)
      launch_pdl(d ? scan_umma2_kernel<true> : scan_umma2_kernel<false>, dim3(grid), dim3(K2_THREADS), smem_bytes, stream,
                 st2.map, prm);
    else
      launch_pdl(d ? scan_umma_kernel<true> : scan_umma_kernel<false>, dim3(grid), dim3(K2_THREADS), smem_bytes, stream,
                 st.q_map, st.map, prm);
  };
  if (dtype == MMR_BF16) launch_pdl(prep_queries_kernel<__nv_bfloat16>, dim3((B + 3) / 4), dim3(128), 0, stream, queries, qb, B, dim, qerr);
  else launch_pdl(prep_queries_kernel<__half>, dim3((B + 3) / 4), dim3(128), 0, stream, queries, reinterpret_cast<__half*>(qb), B, dim, qerr);
  int launches = 1;
  const int max_q_per_pass = sm_count * K2_BM;
  for (int q0 = 0; q0 < B; q0 += max_q_per_pass) {
    const int bq = std::min(B - q0, max_q_per_pass);
    UmmaParams p{};
    p.ks = dim / 64;
    p.nstages = stages;
    p.k = k;
    p.B = bq;
    p.row_begin = r0;
    p.row_end = r1;
    p.n_qtiles = umma_qtiles(bq);
    const int64_t ntiles = (int64_t(r1) - r0 + K2_NT - 1) / K2_NT;
    const int n_qpairs = (p.n_qtiles + 1) / 2;
    if (pair) {
      p.n_rslots = int(std::max<int64_t>(1, std::min<int64_t>((sm_count / 2) / n_qpairs, ntiles)));
      p.idesc = umma_idesc_m256_n128(dtype == MMR_BF16);
    } else {
      p.n_rslots = int(std::max<int64_t>(1, std::min<int64_t>(sm_count / p.n_qtiles, ntiles)));
      p.idesc = umma_idesc_m128_n128(dtype == MMR_BF16);
    }
    p.partial = partial;
    p.qbf16 = qb + size_t(q0) * dim;
    p.dump = dump ? dump + int64_t(q0) * dump_ld : nullptr;
    p.dump_ld = dump_ld;
    const int grid = pair ? 2 * n_qpairs * p.n_rslots : p.n_qtiles * p.n_rslots;
    // probe pass: worth it when every CTA streams many tiles (the warm-up it removes is ~k ln(n/k) inserts/thread)
    const int64_t tiles_per_cta = ntiles / p.n_rslots;
    if (!dump && tiles_per_cta >= 8 && p.n_rslots >= k) {
      launches += 2;
      UmmaParams pp = p;
      pp.probe_out = probe;
      pp.probe_tiles = int(std::max<int64_t>(1, std::min<int64_t>(16, tiles_per_cta / 24)));
      launch_scan(grid, pp);
      const int wpb = 4;
      if (k <= 32) launch_pdl(probe_floor_kernel<1>, dim3((bq + wpb - 1) / wpb), dim3(wpb * 32), 0, stream, probe, p.n_qtiles, p.n_rslots, bq, k, floor + q0);
      else launch_pdl(probe_floor_kernel<2>, dim3((bq + wpb - 1) / wpb), dim3(wpb * 32), 0, stream, probe, p.n_qtiles, p.n_rslots, bq, k, floor + q0);
      p.floor = floor + q0;
    }
    launches += dump ? 1 : 2;
    launch_scan(grid, p);
    if (!dump) {
      const int wpb = 4;
      if (k <= 32)
        launch_pdl(merge_partials_kernel<1>, dim3((bq + wpb - 1) / wpb), dim3(wpb * 32), 0, stream, partial, p.n_qtiles,
                   p.n_rslots, bq, k, out_s + size_t(q0) * k, out_r + size_t(q0) * k, row_base);
      else
        launch_pdl(merge_partials_kernel<2>, dim3((bq + wpb - 1) / wpb), dim3(wpb * 32), 0, stream, partial, p.n_qtiles,
                   p.n_rslots, bq, k, out_s + size_t(q0) * k, out_r + size_t(q0) * k, row_base);
    }
  }
  umma_last_launches() = launches;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    err = std::string("K2 launch failed: ") + cudaGetErrorString(e);
    return MMR_ERR_CUDA;
  }
  return MMR_OK;
}
#endif
}  // namespace mmr
