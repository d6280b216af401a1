// K2 -- tensor-core exact scan for query batches: score contraction on tcgen05 / TMEM with the top-k
// selection fused into the accumulator read-back, so scores never touch HBM.
//
// Replaces the same reference call as K1 (LanceDBStore.search_text / search_image,
// app/storage/lancedb_store.py:103-123) when B queries share one row range.
//
// One persistent CTA (192 threads, 1 per SM) owns one 128-query tile and a strided set of 128-row index
// tiles:
//   D[128 queries x 128 rows] (fp32, TMEM) = Q[128 x D] (bf16, shared, resident) . X[128 x D]^T (bf16, TMA-streamed)
//   * warp 0, one lane : TMA producer.  Loads the query tile once (D/64 boxes of 128 x 64, SWIZZLE_128B), then
//                        streams index tiles as D/64 K-slices of 16 KB through an mbarrier ring of nstages.
//   * warp 1, one lane : issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=128, K=16), 4 per K-slice,
//                        commits the slice's "empty" barrier and, per tile, the accumulator's "full" barrier.
//                        (the whole warp allocates / frees the 512 TMEM columns = 4 accumulators of 128 columns.)
//   * warps 2-5        : epilogue.  Thread = one query (TMEM lane).  tcgen05.ld 32 columns at a time, max-tree,
//                        one compare against the thread's k-th best score; the rare winner is inserted into the
//                        thread's private sorted list (shared memory).  No cross-thread traffic.
// Four accumulators let the MMAs of tile t+1..t+3 run under the epilogue of tile t.
// CTA (qt, rs) handles query tile qt and row tiles rs, rs + RS, ...  This kernel serves batches of one query tile
// (B <= 128); larger batches run on CTA pairs (scan_umma2.cuh), which share the same epilogue (k2_epilogue).
// Per-CTA lists go to global memory; merge_partials_kernel reduces them per query.
#pragma once
#include <cuda.h>

#include <cstdlib>
#include <string>
#include <type_traits>

#include "common.cuh"
#include "topk.cuh"

namespace mmr {

constexpr int K2_THREADS = 192;
constexpr int K2_BM = 128;               // queries per tile  (UMMA M, TMEM lanes)
constexpr int K2_NT = 128;               // index rows per tile (UMMA N, TMEM columns per accumulator)
constexpr int K2_SLICE = 128 * 128;      // bytes of one [128 rows x 64 bf16] SWIZZLE_128B box
constexpr int K2_ACC = 4;                // TMEM accumulators (4 x 128 = 512 columns)
constexpr int K2_MAX_STAGES = 13;
constexpr int K2_SMEM_LIMIT = 227 * 1024;

struct UmmaParams {
  int32_t ks;       // D / 64
  int32_t nstages;  // index ring depth
  int32_t k;
  int32_t B;
  uint32_t row_begin, row_end;
  int32_t n_qtiles, n_rslots;
  uint64_t* partial;  // [n_qtiles * n_rslots][128][k]
  const void* qbf16;  // pair kernel: normalised bf16 queries of this launch, [B][D]
  const float* floor; // per query: a proven lower bound of its final k-th best score (nullptr = none)
  float* probe_out;   // probe pass: [n_qtiles * n_rslots][128] best score seen by each CTA (nullptr = real scan)
  int32_t probe_tiles;  // probe pass: row tiles per CTA
  uint32_t idesc;       // tcgen05 instruction descriptor (bf16 or fp16 operands)
  float* dump;        // DUMP mode: raw scores [B][dump_ld]
  int64_t dump_ld;
};

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------- PTX
__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const CUtensorMap* map, uint32_t bar, int32_t c0,
                                            int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                   dst_smem),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}
// One lane of a converged warp (always the same one): the thread that issues TMA / tcgen05.mma / commit.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc_512(uint32_t dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(512u) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_512(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(512u) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T ; bf16 x bf16 -> f32
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// mbarrier arrives once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor for a K-major, SWIZZLE_128B operand tile of [rows x 64 bf16]:
// rows are 128 B apart, 8-row groups 1024 B apart (SBO), LBO unused for swizzled K-major (1), version 1 (sm_100).
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t smem_addr) {
  return uint64_t((smem_addr & 0x3FFFFu) >> 4) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
// Instruction descriptor, kind::f16: D=f32, A=B=bf16 (format 1) or fp16 (format 0), both K-major, M=128, N=128.
__host__ __device__ constexpr uint32_t umma_idesc_m128_n128(bool bf16) {
  return (1u << 4) | ((bf16 ? 1u : 0u) << 7) | ((bf16 ? 1u : 0u) << 10) | (uint32_t(K2_NT >> 3) << 17) |
         (uint32_t(K2_BM >> 4) << 24);
}

// Rare path of the epilogue: put `key` into this thread's candidate list (k slots, stride K2_BM in shared
// memory, unsorted) by overwriting the current minimum, and return the new minimum = the thread's k-th best key
// (0 while fewer than k candidates are held).  Replace-min keeps the loads independent (no shifting chain);
// merge_partials_kernel does the final ordering.  *meta = held count | position of the minimum << 8.
static __device__ __noinline__ uint64_t k2_list_insert(uint64_t* mine, uint32_t* meta, int k, uint64_t key) {
  const uint32_t m = *meta;
  int count = int(m & 0xffu);
  if (count < k) {
    mine[size_t(count) * K2_BM] = key;
    ++count;
    if (count < k) {
      *meta = uint32_t(count);
      return 0ull;
    }
  } else {
    mine[size_t(m >> 8) * K2_BM] = key;
  }
  uint64_t mv = ~0ull;
  int mp = 0;
#pragma unroll 4
  for (int j = 0; j < k; ++j) {
    const uint64_t x = mine[size_t(j) * K2_BM];
    if (x < mv) {
      mv = x;
      mp = j;
    }
  }
  *meta = uint32_t(count) | (uint32_t(mp) << 8);
  return mv;
}

__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      :
      : "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
        "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]),
        "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]),
        "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// The epilogue warps of both K2 kernels (warps 2-5, thread = query of tile qt): read each accumulator back from tensor
// memory 32 columns at a time, filter, insert into the thread's candidate list, hand the accumulator back with
// release(acc); at the end write the list (or, in the probe pass, the best score) out.  acc_tmem = tensor-memory address
// of accumulator 0; accumulators are NACC x K2_NT columns from there.
template <bool DUMP, int NACC, typename Release>
__device__ __forceinline__ void k2_epilogue(const UmmaParams& p, int qt, int rs, int ntiles, uint64_t* lists,
                                            uint32_t* metas, uint32_t acc_tmem, uint32_t bar_tfull, Release release) {
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int k = p.k;
  const int quarter = warp & 3;              // TMEM lane quarter this warp may access
  const int ql = quarter * 32 + lane;        // query within the tile
  const int qglob = qt * K2_BM + ql;         // query within this launch
  const bool live = qglob < p.B;
  const bool warp_live = qt * K2_BM + quarter * 32 < p.B;   // any live query in this warp
  uint64_t* mine = lists + ql;               // my candidate list: mine[j * 128], j = 0 .. k-1 (unsorted)
  uint32_t* meta = metas + ql;
  for (int j = 0; j < k; ++j) mine[size_t(j) * K2_BM] = 0ull;
  *meta = 0u;
  // Rows reach a thread in ascending order, so an equal score can never displace a held one: the strict
  // compare `m > thr_f` is exact.  Padding queries never pass.
  // A proven lower bound of the final k-th score (from the probe pass) pre-loads the filter, so the scan does
  // not pay the warm-up in which every row beats an empty list.  `s >= floor` must pass: use the float just below.
  float thr_floor = -INFINITY;
  if (p.floor != nullptr && live) {
    const float f = p.floor[qglob];
    // the float just below f in the total order; below +-0 that is the largest negative subnormal, not -0.0
    // (which compares equal to 0 and would reject every row scoring exactly 0, e.g. for an all-zero query)
    if (f > -INFINITY) {
      const uint32_t o = f32_orderable(f);
      thr_floor = f32_from_orderable(o - (o == 0x80000000u ? 2u : 1u));
    }
  }
  float thr_f = live ? thr_floor : INFINITY;
  float best = -INFINITY;  // probe pass
  int acc = 0;
  uint32_t acc_phase = 0;
  for (int t = rs; t < ntiles; t += p.n_rslots) {
    const uint32_t row0 = p.row_begin + uint32_t(t) * K2_NT;
    const int nvalid = int(min(uint32_t(K2_NT), p.row_end - row0));
    mbar_wait(bar_tfull + acc * 8, acc_phase);
    tc_fence_after();
    if (warp_live) {
#pragma unroll 1
      for (int c = 0; c < K2_NT / 32; ++c) {
        uint32_t v[32];
        __syncwarp();
        tmem_ld_x32(acc_tmem + (uint32_t(quarter * 32) << 16) + uint32_t(acc * K2_NT + c * 32), v);
        tmem_wait_ld();
        if constexpr (DUMP) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const int col = c * 32 + j;
            if (col < nvalid && live)
              p.dump[int64_t(qglob) * p.dump_ld + int64_t(row0 - p.row_begin) + col] = __uint_as_float(v[j]);
          }
        } else {
          if (nvalid < K2_NT) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c * 32 + j >= nvalid) v[j] = 0xFF800000u;  // -inf: rows past the segment end
          }
          // two-level filter: max per group of 8 columns, then max of the 4 groups against my k-th best
          float gm[4];
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            float x = __uint_as_float(v[g * 8]);
#pragma unroll
            for (int j = 1; j < 8; ++j) x = fmaxf(x, __uint_as_float(v[g * 8 + j]));
            gm[g] = x;
          }
          const float m = fmaxf(fmaxf(gm[0], gm[1]), fmaxf(gm[2], gm[3]));
          if (p.probe_out != nullptr) {
            best = fmaxf(best, m);
          } else if (m > thr_f) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {
              if (gm[g] > thr_f) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                  const float s = __uint_as_float(v[g * 8 + j]);
                  if (s > thr_f) {
                    const uint64_t thr_key = k2_list_insert(mine, meta, k, make_key(s, row0 + uint32_t(c * 32 + g * 8 + j)));
                    thr_f = thr_key ? fmaxf(thr_floor, key_score(thr_key)) : thr_floor;
                  }
                }
              }
            }
          }
        }
      }
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) release(acc);
    if (++acc == NACC) {
      acc = 0;
      acc_phase ^= 1u;
    }
  }
  if constexpr (!DUMP) {
    if (p.probe_out != nullptr) {
      p.probe_out[size_t(qt * p.n_rslots + rs) * K2_BM + ql] = best;
    } else {
      uint64_t* dst = p.partial + (size_t(qt * p.n_rslots + rs) * K2_BM + ql) * k;
      for (int j = 0; j < k; ++j) dst[j] = mine[size_t(j) * K2_BM];
    }
  }
}

template <bool DUMP>
__global__ void __launch_bounds__(K2_THREADS, 1)
scan_umma_kernel(const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_x,
                 const UmmaParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  // Programmatic dependent launch: setup, tensor-memory allocation and the first index tiles run under the previous kernel
  // of the chain (prep / floor); only the warps that read what it wrote (queries, floors) or that write buffers it may
  // still read (partials, probe maxima) wait for it -- see the pdl_wait_prior_grid() calls below.
  pdl_launch_dependents();
  const int warp = threadIdx.x >> 5;
  const int ks = p.ks, nstages = p.nstages, k = p.k;

  const uint32_t q_s = smem_u32(smem);
  const uint32_t st_s = q_s + uint32_t(ks) * K2_SLICE;
  uint64_t* lists = reinterpret_cast<uint64_t*>(smem + size_t(ks + nstages) * K2_SLICE);  // [k][128]
  uint32_t* metas = reinterpret_cast<uint32_t*>(lists + size_t(k) * K2_BM);                     // [128]
  uint64_t* bars = reinterpret_cast<uint64_t*>(metas + K2_BM);
  const uint32_t bar_full = smem_u32(bars);                      // [K2_MAX_STAGES]
  const uint32_t bar_empty = bar_full + K2_MAX_STAGES * 8;       // [K2_MAX_STAGES]
  const uint32_t bar_tfull = bar_empty + K2_MAX_STAGES * 8;      // [K2_ACC]
  const uint32_t bar_tempty = bar_tfull + K2_ACC * 8;            // [K2_ACC]
  const uint32_t bar_q = bar_tempty + K2_ACC * 8;                // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * K2_MAX_STAGES + 2 * K2_ACC + 1);

  const int qt = blockIdx.x % p.n_qtiles;
  const int rs = blockIdx.x / p.n_qtiles;
  const uint32_t nrows = p.row_end - p.row_begin;
  const int ntiles_all = int((nrows + K2_NT - 1) / K2_NT);
  // probe pass: only the first probe_tiles tiles of this CTA's strided sequence
  const int ntiles = p.probe_out ? min(ntiles_all, rs + p.probe_tiles * p.n_rslots) : ntiles_all;

  if (threadIdx.x == 0) {
    if ((q_s & 1023u) != 0) __trap();  // SWIZZLE_128B operands need 1024-byte alignment
    for (int s = 0; s < K2_MAX_STAGES; ++s) {
      mbar_init(bar_full + s * 8, 1);
      mbar_init(bar_empty + s * 8, 1);
    }
    for (int a = 0; a < K2_ACC; ++a) {
      mbar_init(bar_tfull + a * 8, 1);
      mbar_init(bar_tempty + a * 8, 4);  // one arrival per epilogue warp
    }
    mbar_init(bar_q, 1);
    fence_mbar_init();
    tma_prefetch_desc(&tm_q);
    tma_prefetch_desc(&tm_x);
  }
  if (warp == 1) tmem_alloc_512(smem_u32(tmem_slot));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    // The whole warp runs the (warp-uniform) loop; one elected lane issues the copies.  Keeping control flow
    // uniform lets the compiler hold addresses / coordinates in uniform registers.
    const bool leader = elect_one();
    pdl_wait_prior_grid();   // the query tile was written by prep_queries_kernel
    if (leader) {
      mbar_arrive_expect_tx(bar_q, uint32_t(ks) * K2_SLICE);
      for (int s = 0; s < ks; ++s) tma_load_2d(q_s + s * K2_SLICE, &tm_q, bar_q, s * 64, qt * K2_BM);
    }
    int stage = 0;
    uint32_t phase = 0;
    for (int t = rs; t < ntiles; t += p.n_rslots) {
      const int32_t row0 = int32_t(p.row_begin + uint32_t(t) * K2_NT);
      for (int s = 0; s < ks; ++s) {
        mbar_wait(bar_empty + stage * 8, phase ^ 1u);
        if (leader) {
          mbar_arrive_expect_tx(bar_full + stage * 8, K2_SLICE);
          tma_load_2d(st_s + stage * K2_SLICE, &tm_x, bar_full + stage * 8, s * 64, row0);
        }
        __syncwarp();
        if (++stage == nstages) {
          stage = 0;
          phase ^= 1u;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    // Warp-uniform loop, one elected lane issues tcgen05.mma and the commits (same lane for both: a commit
    // tracks the MMAs of the thread that executes it).
    const bool leader = elect_one();
    const uint32_t idesc = p.idesc;
    mbar_wait(bar_q, 0);
    tc_fence_after();
    int stage = 0, acc = 0;
    uint32_t phase = 0, acc_phase = 0;
    for (int t = rs; t < ntiles; t += p.n_rslots) {
      mbar_wait(bar_tempty + acc * 8, acc_phase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + uint32_t(acc) * K2_NT;
      for (int s = 0; s < ks; ++s) {
        mbar_wait(bar_full + stage * 8, phase);
        tc_fence_after();
        const uint64_t b_desc = umma_smem_desc(st_s + stage * K2_SLICE);
        const uint64_t a_desc = umma_smem_desc(q_s + s * K2_SLICE);
        if (leader) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)  // 64-element slice = 4 x UMMA_K(16); +32 B per step inside the swizzle atom
            umma_f16(d_tmem, a_desc + uint64_t(kk * 2), b_desc + uint64_t(kk * 2), idesc, uint32_t((s | kk) != 0));
          umma_commit(bar_empty + stage * 8);
        }
        __syncwarp();
        if (++stage == nstages) {
          stage = 0;
          phase ^= 1u;
        }
      }
      if (leader) umma_commit(bar_tfull + acc * 8);
      __syncwarp();
      if (++acc == K2_ACC) {
        acc = 0;
        acc_phase ^= 1u;
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue: thread = query
    pdl_wait_prior_grid();     // floors come from the previous kernels; partials / probe maxima may still be read
    k2_epilogue<DUMP, K2_ACC>(p, qt, rs, ntiles, lists, metas, tmem_base, bar_tfull,
                              [&](int acc) { mbar_arrive(bar_tempty + acc * 8); });
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc_512(tmem_base);
}

// Per query: merge the RS per-CTA lists (sorted, k keys each).  One warp per query.
template <int KPL>
__global__ void merge_partials_kernel(const uint64_t* __restrict__ partial, int n_qtiles, int n_rslots, int B, int k,
                                      float* __restrict__ out_scores, int64_t* __restrict__ out_rows,
                                      int64_t row_base) {
  pdl_chain_prologue();
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= B) return;
  const int qt = q / K2_BM, ql = q % K2_BM;
  WarpTopK<KPL> m;
  m.clear();
  uint64_t thr = 0ull;
  // round-robin over the lists (entry j of every list before entry j+1), 8 loads in flight per lane
  thr = m.template merge_batched<8>(
      [&](int i) -> uint64_t {
        const int rs = i % n_rslots, j = i / n_rslots;
        return partial[(size_t(qt * n_rslots + rs) * K2_BM + ql) * k + j];
      },
      n_rslots * k, thr, k, lane);
#pragma unroll
  for (int j = 0; j < KPL; ++j) {
    const int pos = j * 32 + lane;
    if (pos < k) {
      const uint64_t key = m.key[j];
      out_scores[size_t(q) * k + pos] = key ? key_score(key) : -INFINITY;
      out_rows[size_t(q) * k + pos] = key ? int64_t(key_row(key)) + row_base : int64_t(-1);
    }
  }
}

// Probe reduction: per query, the k-th largest of the per-CTA best scores.  The RS values belong to RS distinct
// rows, so this is a lower bound of the query's final k-th best score (-inf when fewer than k CTAs probed).
template <int KPL>
__global__ void probe_floor_kernel(const float* __restrict__ probe, int n_qtiles, int n_rslots, int B, int k,
                                   float* __restrict__ floor) {
  pdl_chain_prologue();
  const int lane = threadIdx.x & 31;
  const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= B) return;
  const int qt = q / K2_BM, ql = q % K2_BM;
  WarpTopK<KPL> m;
  m.clear();
  uint64_t thr = 0ull;
  for (int i0 = 0; i0 < n_rslots; i0 += 32) {
    const int rs = i0 + lane;
    const bool valid = rs < n_rslots;
    const float v = valid ? probe[size_t(qt * n_rslots + rs) * K2_BM + ql] : -INFINITY;
    thr = m.offer_batch(make_key(v, uint32_t(rs)), valid && v > -INFINITY, thr, k, lane);
  }
  if (lane == 0) floor[q] = thr ? key_score(thr) : -INFINITY;
}

// fp32 queries -> L2-normalised bf16 (LanceDBStore._normalize, then narrowed for the tensor cores). Warp per query.
template <typename E>
__global__ void prep_queries_kernel(const float* __restrict__ q, E* __restrict__ out, int B, int dim,
                                    float* __restrict__ qerr = nullptr) {
  pdl_chain_prologue();
  const int lane = threadIdx.x & 31;
  const int qi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (qi >= B) return;
  const float* s = q + size_t(qi) * dim;
  float ss = 0.f;
  for (int i = lane; i < dim; i += 32) ss = fmaf(s[i], s[i], ss);
  ss = warp_allreduce_sum(ss);
  const float nrm = sqrtf(ss);
  float err2 = 0.f;
  for (int i = lane; i < dim; i += 32) {
    const float x = nrm > 0.f ? s[i] / nrm : s[i];
    float back;
    if constexpr (sizeof(E) == 2 && std::is_same<E, __half>::value) {
      const __half h = __float2half_rn(x);
      out[size_t(qi) * dim + i] = h;
      back = __half2float(h);
    } else {
      const __nv_bfloat16 h = __float2bfloat16_rn(x);
      out[size_t(qi) * dim + i] = h;
      back = __bfloat162float(h);
    }
    err2 = fmaf(x - back, x - back, err2);
  }
  // ||q_unit - q_16bit||_2: bounds how far the tensor-core score of ANY unit row can be from its fp32-query score
  // (Cauchy-Schwarz); used by the rescoring mode to prove its result exact
  if (qerr != nullptr) {
    err2 = warp_allreduce_sum(err2);
    if (lane == 0) qerr[qi] = sqrtf(err2);
  }
}
#endif  // __CUDACC__

// ------------------------------------------------------------------------------------------------ host side
struct UmmaIndexState {
  bool valid = false;
  const void* rows = nullptr;
  int64_t n_rows = 0;
  CUtensorMap map;
  // the query tile's map is cached too: a search re-encodes it only when the query copy moved or its shape changed
  bool q_valid = false;
  const void* q_ptr = nullptr;
  int q_rows = 0;
  CUtensorMap q_map;
};

typedef CUresult (*mmr_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                        CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                        CUtensorMapFloatOOBfill);

inline mmr_encode_tiled_fn umma_encode_fn() {
  static mmr_encode_tiled_fn fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<mmr_encode_tiled_fn>(sym);
  }
  return fn;
}

// [n_rows, dim] bf16 row-major -> boxes of [128 rows x 64 elements], 128-byte swizzle
inline bool umma_make_map(CUtensorMap* map, const void* base, int64_t n_rows, int dim, bool bf16 = true) {
  mmr_encode_tiled_fn fn = umma_encode_fn();
  if (!fn) return false;
  cuuint64_t gdim[2] = {cuuint64_t(dim), cuuint64_t(n_rows)};
  cuuint64_t gstr[1] = {cuuint64_t(dim) * 2};
  cuuint32_t box[2] = {64, 128};
  cuuint32_t estr[2] = {1, 1};
  return fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

inline size_t umma_align(size_t v) { return (v + 255) / 256 * 256; }

inline int umma_qtiles(int B) { return (B + K2_BM - 1) / K2_BM; }

inline size_t umma_workspace_bytes(int sm_count, int dim, int B, int k) {
  const int qtiles = std::min(umma_qtiles(B), sm_count);
  const int ctas = std::max(sm_count, qtiles);
  return umma_align(size_t(B) * dim * 2) + umma_align(size_t(ctas) * K2_BM * k * 8) +
         umma_align(size_t(ctas) * K2_BM * 4) + umma_align(size_t(B) * 4) + 256;
}

inline int& umma_last_launches() {  // kernels launched by the last umma_search on this thread
  static thread_local int n = 0;
  return n;
}
inline int umma_launches_per_search() { return umma_last_launches(); }

// smem plan: query tile + ring + lists + barriers
inline int umma_plan_stages(int dim, int k, size_t* smem_bytes) {
  const int ks = dim / 64;
  const size_t fixed = size_t(ks) * K2_SLICE + size_t(k) * K2_BM * 8 + K2_BM * 4 +
                       (2 * K2_MAX_STAGES + 2 * K2_ACC + 2) * 8 + 1024;
  int stages = int((size_t(K2_SMEM_LIMIT) - fixed) / K2_SLICE);
  stages = std::min(stages, K2_MAX_STAGES);
  if (smem_bytes) *smem_bytes = fixed + size_t(std::max(stages, 0)) * K2_SLICE;
  return stages;
}

// Which kernel family serves a batch that shares one row range.  The choice depends on the batch size and the
// storage type ONLY -- never on the number of rows -- so that a row-range shard of a table takes the same family
// (same query precision, same per-row arithmetic) as the whole table and sharded results stay bit-identical.
//   B <= 2  : K1 (fp32 queries, one launch, HBM-bound)      B >= 3, bf16/fp16 rows : K2 (16-bit queries on tcgen05)
inline bool umma_preferred(int dtype, int dim, int B, int k, int64_t nrows) {
  if ((dtype != MMR_BF16 && dtype != MMR_F16) || dim % 64 != 0 || B < 3) return false;
  if (nrows <= 0 || nrows >= (int64_t(1) << 31)) return false;
  return umma_plan_stages(dim, k, nullptr) >= 2;
}
}  // namespace mmr
