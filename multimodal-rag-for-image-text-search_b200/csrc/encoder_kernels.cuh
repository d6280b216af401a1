// Query encoders on the device (SURVEY 8f rank 2 / 3): the transformer kernels behind
//   embed_text_batch        (MiniLM-L6: BERT, 6 layers, hidden 384, mean pooling, L2 norm)   reference app/ml/embeddings.py:52-70
//   embed_query_for_images  (CLIP ViT-B/32 text tower: 12 pre-LN layers, hidden 512, causal, EOS pooling, projection, L2 norm)
//                                                                                              reference app/ml/embeddings.py:94-105
//   CrossEncoder.predict    (ms-marco-MiniLM-L-6: the same BERT + pooler + 1-logit classifier) reference app/ml/retrieve.py:132-155
// so that a query is born on the GPU and feeds mmr_search directly, and the one model of the ingest side
//   embed_images_batch      (CLIP ViT-B/32 vision tower: patchify + patch GEMM, class token, pre-LayerNorm, the same 12 pre-LN
//                            layers at hidden 768, not causal, class-token pooling, projection, L2 norm)
//                                                                                              reference app/ml/embeddings.py:73-91
// so that an image's index row is made by the same kernels as the query it is searched with.
//
// These models are small and latency-bound (a query is 8-40 tokens; 21 / 75 MB of bf16 weights stay in L2), so the
// kernels are shaped for short sequences and batch <= 128:
//   * every linear layer is ONE "swap-AB" tcgen05 GEMM: the WEIGHT tile is the 128-row M operand (features = TMEM lanes),
//     the tokens are the N operand (64 per tile), so a 16-token query still fills the tensor-core tile's M side and the
//     epilogue thread owns one output feature (bias / activation / residual without cross-lane traffic);
//     weights [N_out, K] bf16 are exactly nn.Linear's layout = K-major: TMA boxes with 128B swizzle, no transposes;
//   * attention is per (sequence, head) on CUDA cores in fp32 (S <= 512, head dim 32 / 64): K and V of the head live in
//     shared memory, one warp per query row;
//   * LayerNorm / embedding / pooling are warp-per-row fp32 kernels; the residual stream stays fp32, only GEMM inputs
//     are bf16.
// All kernels chain with programmatic dependent launch (pdl_chain_prologue) so the ~45 launches of a forward pass do not
// pay a launch gap each.
#pragma once
#include "scan_umma.cuh"

namespace mmr {

constexpr int ENC_THREADS = 192;
constexpr int ENC_BM = 128;   // output features per tile (UMMA M)
constexpr int ENC_W_SLICE = ENC_BM * 128;  // 16 KB: [128 features x 64 bf16]
constexpr int ENC_MAX_STAGES = 8;
// tokens per tile (UMMA N) is a template parameter NT in {64, 128, 256}: a single query (16 tokens) wants many small CTAs,
// a micro-batch of 128 queries or 64 rerank pairs (2k-8k tokens) wants fewer, larger ones (per-CTA setup amortised, weight
// tile re-read less often)

enum GemmEpilogue { EPI_BIAS_F32 = 0, EPI_BIAS_RES_F32 = 1, EPI_GELU_BF16 = 2, EPI_QUICKGELU_BF16 = 3 };

struct GemmParams {
  int32_t M, N, K;            // tokens, output features, input features
  int32_t nstages;
  const float* bias;          // [N]
  const float* residual;      // [M, N] fp32 (EPI_BIAS_RES_F32)
  float* out_f32;             // [M, N]
  __nv_bfloat16* out_bf16;    // [M, N]
  // LNX variant: the token operand is LN(ln_src) computed in the kernel (ln_src fp32 [M, K]); CTAs of feature tile 0 also
  // write the normalised rows to ln_out (fp32 [M, K], may be null, may NOT alias ln_src)
  const float* ln_src;
  const float* ln_g;
  const float* ln_b;
  float* ln_out;
  float ln_eps;
};

#ifdef __CUDACC__
__host__ __device__ constexpr uint32_t enc_idesc(int nt) {  // kind::f16, bf16 x bf16 -> f32, M = 128, N = nt, both K-major
  return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(nt >> 3) << 17) | (uint32_t(ENC_BM >> 4) << 24);
}
__device__ __forceinline__ void tmem_alloc_cols(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_cols(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// GELU(erf): erf by Abramowitz & Stegun 7.1.26 (|error| <= 1.5e-7, far below the bf16 rounding of the value it feeds) on the
// approximate reciprocal / exp2 units -- the FFN1 epilogue is issue-bound on its four warps.  Measured per FFN1 launch at 16384
// tokens (profiles/r02_encoder_summary.md): libm erff 74 us, this 0.97x of the whole pass; the same formula with IEEE
// reciprocal and exp2f() 101 us.  -DMMR_ENC_LIBM_ERF restores erff.
__device__ __forceinline__ float erf_as(float x) {
  const float ax = fabsf(x);
  float t, e;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fmaf(0.3275911f, ax, 1.0f)));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * ax * ax));
  return copysignf(fmaf(-p * t, e, 1.0f), x);
}
#ifdef MMR_ENC_LIBM_ERF
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
#else
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erf_as(x * 0.70710678118654752f)); }
#endif
__device__ __forceinline__ float quick_gelu(float x) { return x / (1.0f + __expf(-1.702f * x)); }

// out[t, f] = epilogue( sum_k X[t, k] * W[f, k] + bias[f] )      grid = (N / 128, ceil(M / NT))
// LNX = true: X = LayerNorm(ln_src) is computed HERE instead of by a layernorm_kernel launch in front (one dependent launch
// less per LayerNorm: at query sizes a forward pass is a chain of ~5 us launches, profiles/r02_encoder_summary.md).  The four
// epilogue warps (idle until the accumulator is ready) normalise the tile's tokens -- warp per token, bit for bit
// warp_layernorm's arithmetic -- and write the bf16 operand straight into shared memory in the layout TMA's SWIZZLE_128B would have
// produced (16-byte chunk c of row r at chunk c ^ (r & 7)); all K / 64 slices stay resident (K <= 512, NT = 64: <= 64 KB),
// the ring carries only weight tiles, and those start loading under the previous kernel (weights are not chain outputs).
template <int EPI, int NT, bool LNX = false>
__global__ void __launch_bounds__(ENC_THREADS, 1)
gemm_wt_kernel(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_x, const GemmParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  pdl_launch_dependents();   // barrier init / tensor-memory allocation run under the previous kernel of the forward pass;
                             // the producer (activations) and the epilogue (residual, outputs) wait for it below
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int nst = p.nstages;
  const int ks = p.K / 64;
  constexpr int ENC_NT = NT;
  constexpr int ENC_X_SLICE = NT * 128;                             // [NT tokens x 64 bf16]
  const uint32_t w_s = smem_u32(smem);                              // [nst][16 KB]
  const uint32_t x_s = w_s + uint32_t(nst) * ENC_W_SLICE;           // [nst][NT * 128 B]   (LNX: [K / 64][NT * 128 B])
  const int nx = LNX ? ks : nst;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + size_t(nst) * ENC_W_SLICE + size_t(nx) * ENC_X_SLICE);
  const uint32_t bar_full = smem_u32(bars);
  const uint32_t bar_empty = bar_full + ENC_MAX_STAGES * 8;
  const uint32_t bar_acc = bar_empty + ENC_MAX_STAGES * 8;
  const uint32_t bar_x = bar_acc + 8;                               // LNX: the normalised token operand is in shared memory
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * ENC_MAX_STAGES + 2);
  const int f0 = blockIdx.x * ENC_BM;
  const int t0 = blockIdx.y * ENC_NT;

  if (threadIdx.x == 0) {
    if ((w_s & 1023u) != 0) __trap();
    for (int s = 0; s < ENC_MAX_STAGES; ++s) {
      mbar_init(bar_full + s * 8, 1);
      mbar_init(bar_empty + s * 8, 1);
    }
    mbar_init(bar_acc, 1);
    mbar_init(bar_x, 128);
    fence_mbar_init();
    tma_prefetch_desc(&tm_w);
    if constexpr (!LNX) tma_prefetch_desc(&tm_x);
  }
  if (warp == 1) tmem_alloc_cols(smem_u32(tmem_slot), ENC_NT);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0;
    if constexpr (!LNX) pdl_wait_prior_grid();   // the activation tile is the previous kernel's output
    for (int s = 0; s < ks; ++s) {
      mbar_wait(bar_empty + stage * 8, phase ^ 1u);
      if (leader) {
        mbar_arrive_expect_tx(bar_full + stage * 8, LNX ? ENC_W_SLICE : ENC_W_SLICE + ENC_X_SLICE);
        tma_load_2d(w_s + stage * ENC_W_SLICE, &tm_w, bar_full + stage * 8, s * 64, f0);
        if constexpr (!LNX)
          tma_load_2d(x_s + stage * ENC_X_SLICE, &tm_x, bar_full + stage * 8, s * 64, t0);   // rows past M are zero-filled
      }
      __syncwarp();
      if (++stage == nst) {
        stage = 0;
        phase ^= 1u;
      }
    }
  } else if (warp == 1) {
    const bool leader = elect_one();
    const uint32_t idesc = enc_idesc(NT);
    int stage = 0;
    uint32_t phase = 0;
    if constexpr (LNX) mbar_wait(bar_x, 0);
    for (int s = 0; s < ks; ++s) {
      mbar_wait(bar_full + stage * 8, phase);
      tc_fence_after();
      const uint64_t a_desc = umma_smem_desc(w_s + stage * ENC_W_SLICE);
      const uint64_t b_desc = umma_smem_desc(x_s + (LNX ? s : stage) * ENC_X_SLICE);
      if (leader) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk)
          umma_f16(tmem_base, a_desc + uint64_t(kk * 2), b_desc + uint64_t(kk * 2), idesc, uint32_t((s | kk) != 0));
        umma_commit(bar_empty + stage * 8);
      }
      __syncwarp();
      if (++stage == nst) {
        stage = 0;
        phase ^= 1u;
      }
    }
    if (leader) umma_commit(bar_acc);
    __syncwarp();
  } else {
    // epilogue: thread = output feature (TMEM lane); 64 token columns
    const int quarter = warp & 3;
    const int f = f0 + quarter * 32 + lane;
    const float b = p.bias ? p.bias[f] : 0.f;
    float ln_gr[16], ln_br[16];
    if constexpr (LNX) {   // LayerNorm weights are not chain outputs: fetched under the previous kernel
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (i < (p.K >> 5)) {
          ln_gr[i] = p.ln_g[i * 32 + lane];
          ln_br[i] = p.ln_b[i * 32 + lane];
        }
    }
    pdl_wait_prior_grid();   // ln_src / residual / output buffers belong to the chain
    if constexpr (LNX) {
      // Warp per token with EXACTLY layernorm_kernel's arithmetic (lane l holds columns i * 32 + l, sums in the same order):
      // the folded and the separate path give bit-identical activations, so an embedding does not depend on whether its
      // pass was short enough to be folded.  Four tokens per warp per round with all their loads in flight together (one L2
      // latency per round, not per token).  Token rows past M are left as they are: an accumulator column depends on its own
      // token row only, and those columns are never stored.
      const int ni = p.K >> 5;
      const int nlive = min(NT, p.M - t0);
      const bool writer = blockIdx.x == 0 && p.ln_out != nullptr;
      for (int tb = warp - 2; tb < nlive; tb += 16) {
        float x[4][16];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            x[u][i] = 0.f;
            if (i < ni && tb + 4 * u < nlive) x[u][i] = __ldcg(p.ln_src + size_t(t0 + tb + 4 * u) * p.K + i * 32 + lane);
          }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int tt = tb + 4 * u;
          if (tt >= nlive) break;   // warp-uniform
          float sum = 0.f;
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (i < ni) sum += x[u][i];
          const float mean = warp_allreduce_sum(sum) / float(p.K);
          float var = 0.f;
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (i < ni) {
              const float d = x[u][i] - mean;
              var = fmaf(d, d, var);
            }
          const float rstd = rsqrtf(warp_allreduce_sum(var) / float(p.K) + p.ln_eps);
#pragma unroll
          for (int i = 0; i < 16; ++i)
            if (i < ni) {
              const int c = i * 32 + lane;
              const float y = (x[u][i] - mean) * rstd * ln_gr[i] + ln_br[i];
              if (writer) p.ln_out[size_t(t0 + tt) * p.K + c] = y;
              const int slice = c >> 6, cc = c & 63;
              const uint32_t dst = x_s + uint32_t(slice) * ENC_X_SLICE + uint32_t(tt) * 128u +
                                   (uint32_t((cc >> 3) ^ (tt & 7)) << 4) + uint32_t(cc & 7) * 2u;
              const __nv_bfloat16 yb = __float2bfloat16_rn(y);
              asm volatile("st.shared.b16 [%0], %1;" ::"r"(dst), "h"(*reinterpret_cast<const uint16_t*>(&yb)) : "memory");
            }
        }
      }
      fence_proxy_async();   // generic-proxy writes -> visible to the tensor core's async-proxy reads
      mbar_arrive(bar_x);
    }
    mbar_wait(bar_acc, 0);
    tc_fence_after();
#pragma unroll 1
    for (int c = 0; c < ENC_NT / 32; ++c) {
      uint32_t v[32];
      tmem_ld_x32(tmem_base + (uint32_t(quarter * 32) << 16) + uint32_t(c * 32), v);
      float res[32];
      if constexpr (EPI == EPI_BIAS_RES_F32) {
        // all residual loads are issued before the first store: `out` may alias `residual` (in-place residual stream), and
        // a load-store-load chain through possibly aliasing pointers serialises on global-memory latency
        // (36 us per GEMM in the first profile, profiles/r02_encoder_summary.md)
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const int t = t0 + c * 32 + j;
          res[j] = t < p.M ? __ldcg(p.residual + size_t(t) * p.N + f) : 0.f;
        }
      }
      tmem_wait_ld();
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        const int t = t0 + c * 32 + j;
        if (t < p.M) {
          float y = __uint_as_float(v[j]) + b;
          const size_t o = size_t(t) * p.N + f;   // consecutive lanes -> consecutive features: coalesced
          if constexpr (EPI == EPI_BIAS_F32) {
            p.out_f32[o] = y;
          } else if constexpr (EPI == EPI_BIAS_RES_F32) {
            p.out_f32[o] = y + res[j];
          } else if constexpr (EPI == EPI_GELU_BF16) {
            p.out_bf16[o] = __float2bfloat16_rn(gelu_erf(y));
          } else {
            p.out_bf16[o] = __float2bfloat16_rn(quick_gelu(y));
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc_cols(tmem_base, ENC_NT);
}

// ---------------------------------------------------------------------------------------------- row kernels (warp = token)
template <int H>
__device__ __forceinline__ void warp_layernorm(const float (&x)[H / 32], const float* __restrict__ g, const float* __restrict__ b,
                                               float eps, int lane, float (&y)[H / 32]) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < H / 32; ++i) s += x[i];
  const float mean = warp_allreduce_sum(s) / float(H);
  float v = 0.f;
#pragma unroll
  for (int i = 0; i < H / 32; ++i) {
    const float d = x[i] - mean;
    v = fmaf(d, d, v);
  }
  const float rstd = rsqrtf(warp_allreduce_sum(v) / float(H) + eps);
#pragma unroll
  for (int i = 0; i < H / 32; ++i) {
    const int c = i * 32 + lane;
    y[i] = (x[i] - mean) * rstd * g[c] + b[c];
  }
}

// BERT embeddings: LN(word[id] + pos[p] + type[tt]) -> fp32 residual stream + bf16 GEMM input.
// CLIP embeddings (ln_g == nullptr): tok[id] + pos[p] -> fp32 residual stream only.
template <int H>
__global__ void embed_kernel(const int32_t* __restrict__ ids, const int32_t* __restrict__ types, const float* __restrict__ word,
                             const float* __restrict__ pos, const float* __restrict__ type_emb, const float* __restrict__ ln_g,
                             const float* __restrict__ ln_b, float eps, int M, int S, float* __restrict__ x_f32,
                             __nv_bfloat16* __restrict__ x_bf16) {
  pdl_chain_prologue();
  const int lane = threadIdx.x & 31;
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= M) return;
  const int id = ids[t], p = t % S, tt = types ? types[t] : 0;
  float x[H / 32], y[H / 32];
#pragma unroll
  for (int i = 0; i < H / 32; ++i) {
    const int c = i * 32 + lane;
    x[i] = word[size_t(id) * H + c] + pos[size_t(p) * H + c] + (type_emb ? type_emb[size_t(tt) * H + c] : 0.f);
  }
  if (ln_g != nullptr) {
    warp_layernorm<H>(x, ln_g, ln_b, eps, lane, y);
  } else {
#pragma unroll
    for (int i = 0; i < H / 32; ++i) y[i] = x[i];
  }
#pragma unroll
  for (int i = 0; i < H / 32; ++i) {
    const int c = i * 32 + lane;
    x_f32[size_t(t) * H + c] = y[i];
    if (x_bf16) x_bf16[size_t(t) * H + c] = __float2bfloat16_rn(y[i]);
  }
}

// y = LN(x): out_f32 (may alias x, may be null) and / or out_bf16
template <int H>
__global__ void layernorm_kernel(const float* __restrict__ x, const float* __restrict__ g, const float* __restrict__ b, float eps,
                                 int M, float* __restrict__ out_f32, __nv_bfloat16* __restrict__ out_bf16) {
  pdl_chain_prologue();
  const int lane = threadIdx.x & 31;
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= M) return;
  float v[H / 32], y[H / 32];
#pragma unroll
  for (int i = 0; i < H / 32; ++i) v[i] = x[size_t(t) * H + i * 32 + lane];
  warp_layernorm<H>(v, g, b, eps, lane, y);
#pragma unroll
  for (int i = 0; i < H / 32; ++i) {
    const int c = i * 32 + lane;
    if (out_f32) out_f32[size_t(t) * H + c] = y[i];
    if (out_bf16) out_bf16[size_t(t) * H + c] = __float2bfloat16_rn(y[i]);
  }
}

// ---------------------------------------------------------------------------------------------- CLIP vision front end
// Patchify: pixels fp32 [B, C, S_img, S_img] (NCHW) -> the patch GEMM's token operand bf16 [B * NP, C * P * P], NP = (S_img / P)^2
// patches in row-major order (HF: conv output flattened over (h, w)), columns in (c, kh, kw) order = the flattened Conv2d
// weight [H, C, P, P].  Values are only rounded: out = bf16_rn(pixel).  One CTA per patch row; consecutive threads take
// consecutive columns, i.e. consecutive pixels of an image row (coalesced reads and writes).
__global__ void patchify_kernel(const float* __restrict__ pixels, int C, int S_img, int P, __nv_bfloat16* __restrict__ out) {
  pdl_chain_prologue();
  const int gw = S_img / P, np = gw * gw, cols = C * P * P;
  const int row = blockIdx.x, b = row / np, p = row % np;
  const int ph = p / gw, pw = p % gw;
  const float* img = pixels + size_t(b) * C * S_img * S_img;
  for (int col = threadIdx.x; col < cols; col += blockDim.x) {
    const int c = col / (P * P), r = col % (P * P), kh = r / P, kw = r % P;
    out[size_t(row) * cols + col] = __float2bfloat16_rn(img[(size_t(c) * S_img + ph * P + kh) * S_img + pw * P + kw]);
  }
}

// CLIP vision embeddings + pre-LayerNorm, warp per token: token 0 of an image = cls + pos[0], token 1 + p = patch_out[p] +
// pos[1 + p] (patch_out fp32 [B * (T - 1), H] = the patch GEMM's output), then LN(pre_ln_g, pre_ln_b) -> the fp32 residual
// stream (HF's pre_layrnorm output is the encoder's input hidden state).  T = tokens per image.
template <int H>
__global__ void vision_embed_kernel(const float* __restrict__ patch_out, const float* __restrict__ cls, const float* __restrict__ pos,
                                    const float* __restrict__ ln_g, const float* __restrict__ ln_b, float eps, int M, int T,
                                    float* __restrict__ x_f32) {
  pdl_chain_prologue();
  const int lane = threadIdx.x & 31;
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (t >= M) return;
  const int b = t / T, p = t % T;
  const float* src = p == 0 ? cls : patch_out + (size_t(b) * (T - 1) + p - 1) * H;
  float x[H / 32], y[H / 32];
#pragma unroll
  for (int i = 0; i < H / 32; ++i) {
    const int c = i * 32 + lane;
    x[i] = src[c] + pos[size_t(p) * H + c];
  }
  warp_layernorm<H>(x, ln_g, ln_b, eps, lane, y);
#pragma unroll
  for (int i = 0; i < H / 32; ++i) x_f32[size_t(t) * H + i * 32 + lane] = y[i];
}

// ---------------------------------------------------------------------------------------------- attention
// grid = (heads, B); one CTA = one head of one sequence; K (rows padded by 4 floats) and V of the head in shared memory
// (fp32).  A warp handles ATT_RQ query rows at a time: scores with lane = key (the K row is read once, as float4, for all
// ATT_RQ rows; the query rows are broadcast reads from shared memory; independent accumulators, no shuffles in the inner
// loop), softmax with warp reductions, P in shared memory, context with lane = output dim.
// mask[b, j] == 0 hides key j (padding); causal hides j > i (CLIP).
constexpr int ATT_NW = 8;   // warps per CTA
constexpr int ATT_RQ = 4;   // query rows per warp per pass

template <int DH>
inline size_t attention_smem_bytes(int S) {
  return (size_t(S) * (DH + 4) + size_t(S) * DH + size_t(ATT_NW) * ATT_RQ * DH + size_t(ATT_NW) * ATT_RQ * S) * 4;
}

template <int DH>
__global__ void __launch_bounds__(ATT_NW * 32) attention_kernel(const float* __restrict__ qkv, const int32_t* __restrict__ mask,
                                                               __nv_bfloat16* __restrict__ ctx, int S, int H, int causal) {
  extern __shared__ __align__(16) float att_smem[];
  pdl_chain_prologue();
  constexpr int KP = DH + 4;              // padded K row: float4 reads of different rows by a quarter warp hit distinct banks
  constexpr int DPL = DH / 32;            // output dims per lane
  const int h = blockIdx.x, b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* Ks = att_smem;                                   // [S][KP]
  float* Vs = Ks + size_t(S) * KP;                        // [S][DH]
  float* Qs = Vs + size_t(S) * DH + size_t(warp) * ATT_RQ * DH;                          // this warp's [RQ][DH]
  float* Ps = Vs + size_t(S) * DH + size_t(ATT_NW) * ATT_RQ * DH + size_t(warp) * ATT_RQ * S;   // this warp's [RQ][S]
  const size_t row0 = size_t(b) * S;
  const int ld = 3 * H;
  for (int i = threadIdx.x; i < S * (DH / 4); i += blockDim.x) {
    const int j = i / (DH / 4), d4 = i % (DH / 4);
    const float* src = qkv + (row0 + j) * ld + h * DH + d4 * 4;
    *reinterpret_cast<float4*>(Ks + j * KP + d4 * 4) = *reinterpret_cast<const float4*>(src + H);
    *reinterpret_cast<float4*>(Vs + j * DH + d4 * 4) = *reinterpret_cast<const float4*>(src + 2 * H);
  }
  __syncthreads();
  const float scale = rsqrtf(float(DH));
  for (int i0 = warp * ATT_RQ; i0 < S; i0 += ATT_NW * ATT_RQ) {
    // stage the (scaled) query rows of this pass
    for (int e = lane; e < ATT_RQ * DH; e += 32) {
      const int r = e / DH, d = e % DH;
      Qs[e] = (i0 + r < S) ? qkv[(row0 + i0 + r) * ld + h * DH + d] * scale : 0.f;
    }
    __syncwarp();
    const int jend = causal ? min(S, i0 + ATT_RQ) : S;
    float mx[ATT_RQ];
#pragma unroll
    for (int r = 0; r < ATT_RQ; ++r) mx[r] = -INFINITY;
    for (int j0 = 0; j0 < jend; j0 += 32) {
      const int j = j0 + lane;
      const float* kr = Ks + size_t(min(j, S - 1)) * KP;
      float sc[ATT_RQ];
#pragma unroll
      for (int r = 0; r < ATT_RQ; ++r) sc[r] = 0.f;
#pragma unroll
      for (int d4 = 0; d4 < DH / 4; ++d4) {
        const float4 k4 = *reinterpret_cast<const float4*>(kr + d4 * 4);
#pragma unroll
        for (int r = 0; r < ATT_RQ; ++r) {
          const float4 q4 = *reinterpret_cast<const float4*>(Qs + r * DH + d4 * 4);   // broadcast
          sc[r] = fmaf(q4.x, k4.x, fmaf(q4.y, k4.y, fmaf(q4.z, k4.z, fmaf(q4.w, k4.w, sc[r]))));
        }
      }
      const bool key_ok = j < S && (mask == nullptr || mask[row0 + min(j, S - 1)] != 0);
#pragma unroll
      for (int r = 0; r < ATT_RQ; ++r) {
        const bool ok = key_ok && j < jend && (!causal || j <= i0 + r);
        const float v = ok ? sc[r] : -INFINITY;
        if (j < S) Ps[r * S + j] = v;
        mx[r] = fmaxf(mx[r], v);
      }
    }
    float sum[ATT_RQ];
#pragma unroll
    for (int r = 0; r < ATT_RQ; ++r) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], o));
      sum[r] = 0.f;
    }
    __syncwarp();
    for (int j = lane; j < jend; j += 32) {
#pragma unroll
      for (int r = 0; r < ATT_RQ; ++r) {
        const float e = (mx[r] == -INFINITY) ? 0.f : __expf(Ps[r * S + j] - mx[r]);
        Ps[r * S + j] = e;
        sum[r] += e;
      }
    }
#pragma unroll
    for (int r = 0; r < ATT_RQ; ++r) sum[r] = warp_allreduce_sum(sum[r]);
    __syncwarp();
    float acc[ATT_RQ][DPL];
#pragma unroll
    for (int r = 0; r < ATT_RQ; ++r)
#pragma unroll
      for (int u = 0; u < DPL; ++u) acc[r][u] = 0.f;
    for (int j = 0; j < jend; ++j) {
      float vv[DPL];
#pragma unroll
      for (int u = 0; u < DPL; ++u) vv[u] = Vs[j * DH + u * 32 + lane];
#pragma unroll
      for (int r = 0; r < ATT_RQ; ++r) {
        const float pj = Ps[r * S + j];   // broadcast
#pragma unroll
        for (int u = 0; u < DPL; ++u) acc[r][u] = fmaf(pj, vv[u], acc[r][u]);
      }
    }
#pragma unroll
    for (int r = 0; r < ATT_RQ; ++r) {
      if (i0 + r < S) {
        const float inv = sum[r] > 0.f ? 1.f / sum[r] : 0.f;
#pragma unroll
        for (int u = 0; u < DPL; ++u)
          ctx[(row0 + i0 + r) * H + h * DH + u * 32 + lane] = __float2bfloat16_rn(acc[r][u] * inv);
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------- attention, long sequences
// Rerank passages are 128-512 tokens (reference index_build.py:14 splits at 512 tokens): there the fp32 kernel above is
// shared-memory-bound (five LDS per four FMAs in the P.V loop; 425 us per layer at 8 x 512, 75 % of the pass).  This one
// runs both contractions on the tensor cores, flash-attention style, with warp-level mma.sync m16n8k16 (bf16 in, fp32
// accumulate): the natural tile for head dim 32 / 64 -- a tcgen05 tile is 128 rows with the accumulator in tensor memory,
// and the online softmax between the two contractions would cross TMEM <-> registers twice per key block for a layer whose
// total work is 3 GFLOP.  grid = (heads, B, ceil(S / 128)); a CTA = 8 warps x 16 query rows; K and V [S][DH] of the
// head live in shared memory as bf16 (row pads make every ldmatrix conflict-free; V is transposed by ldmatrix.trans); scores never leave registers:
// per 64-key block S = Q K^T (fp32 accumulators), running max / sum, P packed to bf16 straight from the accumulator
// registers (the m16n8 C layout IS the m16n8k16 A layout), O += P V.  Q is scaled in fp32 before narrowing.
// Used for the cross-encoder (every sequence length: which kernel runs must not depend on what a pair is batched with; a
// pair's logit is independent of the padded length -- masked and zero-filled keys contribute exact zeros); the query
// encoders, whose embeddings are held to 1e-3 of fp32 torch, stay on the fp32 kernel.
constexpr int ATC_NW = 8;
constexpr int ATC_ROWS = ATC_NW * 16;   // query rows per CTA
constexpr int ATC_KB = 64;              // keys per online-softmax block
constexpr int ATC_MIN_S = 96;           // MMR_ENC_ATT_MMA=2 (measurement): every model from this sequence length on

template <int DH>
inline size_t attention_mma_smem_bytes(int S) {
  const int sp = (S + ATC_KB - 1) / ATC_KB * ATC_KB;
  return size_t(sp) * (DH + 8) * 2 * 2 + size_t(sp) * 4;   // K and V [sp][DH + 8] bf16, additive key mask
}

__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// four 8 x 8 b16 matrices; lane i supplies the address of row (i % 8) of matrix (i / 8).  Plain: thread T gets
// M[T / 4][2 (T % 4) .. +1]; .trans: M[2 (T % 4) .. +1][T / 4] -- exactly the m16n8k16 B fragments of a [key][dim] tile for
// Q K^T (plain: k = dim) and for P V (.trans: k = key).
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);   // .x (low half) = lo
  return *reinterpret_cast<const uint32_t*>(&v);
}

template <int DH>
__global__ void __launch_bounds__(ATC_NW * 32) attention_mma_kernel(const float* __restrict__ qkv, const int32_t* __restrict__ mask,
                                                                   __nv_bfloat16* __restrict__ ctx, int S, int H, int causal) {
  extern __shared__ __align__(16) uint8_t atc_smem[];
  pdl_chain_prologue();
  constexpr int KP = DH + 8;                      // K row pitch (bf16): 80 / 144 bytes -> the 8 rows of a fragment hit 8 bank groups
  const int sp = (S + ATC_KB - 1) / ATC_KB * ATC_KB;
  __nv_bfloat16* Ks = reinterpret_cast<__nv_bfloat16*>(atc_smem);                 // [sp][KP]
  __nv_bfloat16* Vs = Ks + size_t(sp) * KP;                                       // [sp][KP] (row-major: ldmatrix.trans transposes)
  float* madd = reinterpret_cast<float*>(Vs + size_t(sp) * KP);                   // [sp] 0 or -inf (padding keys, keys >= S)
  const int h = blockIdx.x, b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const size_t row0 = size_t(b) * S;
  const int ld = 3 * H;
  const int q_lo = blockIdx.z * ATC_ROWS;                                         // this CTA's query rows [q_lo, q_lo + 128)
  const int kend = causal ? min(sp, (min(q_lo + ATC_ROWS, S) + ATC_KB - 1) / ATC_KB * ATC_KB) : sp;   // keys this CTA can need

  // ---- stage K (row-major) and V (transposed) of this head as bf16, and the additive key mask ----
  // (four items per thread per round with all eight loads in flight before the first store: the loop is bound by the L2
  //  round trip, not by bytes -- 16 dependent round trips per CTA at S = 512 in the first version)
  for (int i0s = threadIdx.x; i0s < kend * (DH / 4); i0s += 4 * blockDim.x) {
    float4 k4[4], v4[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0s + u * blockDim.x;
      const int j = i / (DH / 4), d4 = (i % (DH / 4)) * 4;
      k4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      v4[u] = k4[u];
      if (i < kend * (DH / 4) && j < S) {
        const float* src = qkv + (row0 + j) * ld + h * DH + d4;
        k4[u] = __ldcg(reinterpret_cast<const float4*>(src + H));
        v4[u] = __ldcg(reinterpret_cast<const float4*>(src + 2 * H));
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0s + u * blockDim.x;
      if (i >= kend * (DH / 4)) break;
      const int j = i / (DH / 4), d4 = (i % (DH / 4)) * 4;
      uint2 kk;
      kk.x = pack_bf16x2(k4[u].x, k4[u].y);
      kk.y = pack_bf16x2(k4[u].z, k4[u].w);
      *reinterpret_cast<uint2*>(Ks + size_t(j) * KP + d4) = kk;
      uint2 vv;
      vv.x = pack_bf16x2(v4[u].x, v4[u].y);
      vv.y = pack_bf16x2(v4[u].z, v4[u].w);
      *reinterpret_cast<uint2*>(Vs + size_t(j) * KP + d4) = vv;
    }
  }
  for (int j = threadIdx.x; j < kend; j += blockDim.x)
    madd[j] = (j < S && (mask == nullptr || mask[row0 + j] != 0)) ? 0.f : -INFINITY;
  __syncthreads();

  const uint32_t ks_base = smem_u32(Ks), vs_base = smem_u32(Vs);
  const int i0 = q_lo + warp * 16;                // this warp's 16 query rows; thread owns rows i0 + g and i0 + g + 8
  if (i0 >= S) return;
  const int ra = i0 + g, rb = i0 + g + 8;
  // ---- Q fragments (A operand, row-major 16 x DH): scaled in fp32, narrowed to bf16 ----
  const float scale = rsqrtf(float(DH));
  uint32_t qa[DH / 16][4];
#pragma unroll
  for (int ks = 0; ks < DH / 16; ++ks) {
    const int c0 = ks * 16 + 2 * t;
    const float* pa = qkv + (row0 + min(ra, S - 1)) * ld + h * DH + c0;
    const float* pb = qkv + (row0 + min(rb, S - 1)) * ld + h * DH + c0;
    const float2 a_lo = *reinterpret_cast<const float2*>(pa), a_hi = *reinterpret_cast<const float2*>(pa + 8);
    const float2 b_lo = *reinterpret_cast<const float2*>(pb), b_hi = *reinterpret_cast<const float2*>(pb + 8);
    qa[ks][0] = pack_bf16x2(a_lo.x * scale, a_lo.y * scale);
    qa[ks][1] = pack_bf16x2(b_lo.x * scale, b_lo.y * scale);
    qa[ks][2] = pack_bf16x2(a_hi.x * scale, a_hi.y * scale);
    qa[ks][3] = pack_bf16x2(b_hi.x * scale, b_hi.y * scale);
  }
  float o[DH / 8][4];
#pragma unroll
  for (int dn = 0; dn < DH / 8; ++dn)
#pragma unroll
    for (int e = 0; e < 4; ++e) o[dn][e] = 0.f;
  float m_a = -INFINITY, m_b = -INFINITY, l_a = 0.f, l_b = 0.f;   // running max / (per-thread partial) sum of rows ra, rb

  const int wend = causal ? min(kend, (min(i0 + 16, S) + ATC_KB - 1) / ATC_KB * ATC_KB) : kend;
  for (int kb = 0; kb < wend; kb += ATC_KB) {
    // S block = Q K^T: 16 rows x 64 keys = 8 n-tiles
    float sc[ATC_KB / 8][4];
#pragma unroll
    for (int nt = 0; nt < ATC_KB / 8; ++nt) {
#pragma unroll
      for (int e = 0; e < 4; ++e) sc[nt][e] = 0.f;
      // lane i -> row (i % 8) of the n-tile's keys, dims (i / 8) * 8 .. +7 of a 32-dim half: one ldmatrix = two k-steps
      const uint32_t kaddr = ks_base + uint32_t((kb + nt * 8 + (lane & 7)) * KP + (lane >> 3) * 8) * 2u;
#pragma unroll
      for (int kh = 0; kh < DH / 32; ++kh) {
        uint32_t kf[4];
        ldmatrix_x4(kf, kaddr + kh * 64);
        mma_bf16_16816(sc[nt], qa[2 * kh], kf[0], kf[1]);
        mma_bf16_16816(sc[nt], qa[2 * kh + 1], kf[2], kf[3]);
      }
    }
    // masks + block max (thread holds keys kb + nt*8 + 2t, +1 of rows ra (e = 0, 1) and rb (e = 2, 3))
    float bm_a = -INFINITY, bm_b = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < ATC_KB / 8; ++nt) {
      const int j = kb + nt * 8 + 2 * t;
      const float2 ma = *reinterpret_cast<const float2*>(madd + j);
      sc[nt][0] += ma.x;
      sc[nt][1] += ma.y;
      sc[nt][2] += ma.x;
      sc[nt][3] += ma.y;
      if (causal) {
        if (j > ra) sc[nt][0] = -INFINITY;
        if (j + 1 > ra) sc[nt][1] = -INFINITY;
        if (j > rb) sc[nt][2] = -INFINITY;
        if (j + 1 > rb) sc[nt][3] = -INFINITY;
      }
      bm_a = fmaxf(bm_a, fmaxf(sc[nt][0], sc[nt][1]));
      bm_b = fmaxf(bm_b, fmaxf(sc[nt][2], sc[nt][3]));
    }
    bm_a = fmaxf(bm_a, __shfl_xor_sync(0xffffffffu, bm_a, 1));
    bm_a = fmaxf(bm_a, __shfl_xor_sync(0xffffffffu, bm_a, 2));
    bm_b = fmaxf(bm_b, __shfl_xor_sync(0xffffffffu, bm_b, 1));
    bm_b = fmaxf(bm_b, __shfl_xor_sync(0xffffffffu, bm_b, 2));
    const float mn_a = fmaxf(m_a, bm_a), mn_b = fmaxf(m_b, bm_b);
    const float ms_a = mn_a == -INFINITY ? 0.f : mn_a, ms_b = mn_b == -INFINITY ? 0.f : mn_b;   // all masked so far: p = 0
    const float f_a = __expf(m_a - ms_a), f_b = __expf(m_b - ms_b);                               // exp(-inf) = 0 on the first block
    m_a = mn_a;
    m_b = mn_b;
    l_a *= f_a;
    l_b *= f_b;
#pragma unroll
    for (int dn = 0; dn < DH / 8; ++dn) {
      o[dn][0] *= f_a;
      o[dn][1] *= f_a;
      o[dn][2] *= f_b;
      o[dn][3] *= f_b;
    }
#pragma unroll
    for (int nt = 0; nt < ATC_KB / 8; ++nt) {
      sc[nt][0] = __expf(sc[nt][0] - ms_a);
      sc[nt][1] = __expf(sc[nt][1] - ms_a);
      sc[nt][2] = __expf(sc[nt][2] - ms_b);
      sc[nt][3] = __expf(sc[nt][3] - ms_b);
      l_a += sc[nt][0] + sc[nt][1];
      l_b += sc[nt][2] + sc[nt][3];
    }
    // O += P V: four k-steps of 16 keys; the A fragment of k-step kk is n-tiles 2kk, 2kk+1 of the score block
#pragma unroll
    for (int kk = 0; kk < ATC_KB / 16; ++kk) {
      uint32_t pa[4];
      pa[0] = pack_bf16x2(sc[2 * kk][0], sc[2 * kk][1]);
      pa[1] = pack_bf16x2(sc[2 * kk][2], sc[2 * kk][3]);
      pa[2] = pack_bf16x2(sc[2 * kk + 1][0], sc[2 * kk + 1][1]);
      pa[3] = pack_bf16x2(sc[2 * kk + 1][2], sc[2 * kk + 1][3]);
      // lane i -> key kb + 16 kk + (i / 8 % 2) * 8 + i % 8, dims (dn + i / 16) * 8 .. +7: {b0, b1} of dn and of dn + 1
      const uint32_t vaddr = vs_base + uint32_t((kb + kk * 16 + ((lane >> 3) & 1) * 8 + (lane & 7)) * KP + (lane >> 4) * 8) * 2u;
#pragma unroll
      for (int dn = 0; dn < DH / 8; dn += 2) {
        uint32_t vf[4];
        ldmatrix_x4_trans(vf, vaddr + dn * 16);
        mma_bf16_16816(o[dn], pa, vf[0], vf[1]);
        mma_bf16_16816(o[dn + 1], pa, vf[2], vf[3]);
      }
    }
  }
  l_a += __shfl_xor_sync(0xffffffffu, l_a, 1);
  l_a += __shfl_xor_sync(0xffffffffu, l_a, 2);
  l_b += __shfl_xor_sync(0xffffffffu, l_b, 1);
  l_b += __shfl_xor_sync(0xffffffffu, l_b, 2);
  const float inv_a = l_a > 0.f ? 1.f / l_a : 0.f, inv_b = l_b > 0.f ? 1.f / l_b : 0.f;
#pragma unroll
  for (int dn = 0; dn < DH / 8; ++dn) {
    const int c = h * DH + dn * 8 + 2 * t;
    if (ra < S) *reinterpret_cast<uint32_t*>(ctx + (row0 + ra) * H + c) = pack_bf16x2(o[dn][0] * inv_a, o[dn][1] * inv_a);
    if (rb < S) *reinterpret_cast<uint32_t*>(ctx + (row0 + rb) * H + c) = pack_bf16x2(o[dn][2] * inv_b, o[dn][3] * inv_b);
  }
}

// ---------------------------------------------------------------------------------------------- heads (block = sequence)
__device__ __forceinline__ float block_sum(float v, float* red) {  // blockDim.x <= 1024, result broadcast
  v = warp_allreduce_sum(v);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = 0.f;
  for (int w = 0; w < int(blockDim.x >> 5); ++w) t += red[w];
  return t;
}

// sentence-transformers mean pooling over the attention mask, then L2 normalisation (Normalize module + the reference's
// own _normalize, app/ml/embeddings.py:46-49: a zero vector stays zero).  blockDim.x == H.
__global__ void mean_pool_norm_kernel(const float* __restrict__ x, const int32_t* __restrict__ mask, int S, int H,
                                      float* __restrict__ out) {
  __shared__ float red[32];
  pdl_chain_prologue();
  const int b = blockIdx.x, c = threadIdx.x;
  float s = 0.f, cnt = 0.f;
  for (int t = 0; t < S; ++t) {
    const float m = mask ? float(mask[size_t(b) * S + t] != 0) : 1.f;
    s = fmaf(m, x[(size_t(b) * S + t) * H + c], s);
    cnt += m;
  }
  const float e = s / fmaxf(cnt, 1e-9f);
  const float nrm = sqrtf(block_sum(e * e, red));
  out[size_t(b) * H + c] = nrm > 0.f ? e / nrm : e;
}

// CLIP head: hidden state at the pooled position -> final LayerNorm -> projection (no bias) -> L2 normalisation.
// blockDim.x == H >= projection dim P.  Text tower: the EOS position (eos_id == 2 reproduces the legacy argmax(input_ids)
// rule of HF's CLIP).  Vision tower (ids == nullptr): position 0, the class token.
__global__ void clip_head_kernel(const float* __restrict__ x, const int32_t* __restrict__ ids, int S, int H, int eos_id,
                                 const float* __restrict__ ln_g, const float* __restrict__ ln_b, float eps,
                                 const float* __restrict__ proj /* [P, H] */, int P, float* __restrict__ out) {
  extern __shared__ float head_smem[];   // [H] normalised hidden state
  __shared__ float red[32];
  __shared__ int s_pos;
  pdl_chain_prologue();
  const int b = blockIdx.x, c = threadIdx.x;
  if (c == 0) {
    int pos = 0;
    if (ids == nullptr) {
      // class token
    } else if (eos_id == 2) {
      int best = ids[size_t(b) * S];
      for (int t = 1; t < S; ++t)
        if (ids[size_t(b) * S + t] > best) {
          best = ids[size_t(b) * S + t];
          pos = t;
        }
    } else {
      for (int t = 0; t < S; ++t)
        if (ids[size_t(b) * S + t] == eos_id) {
          pos = t;
          break;
        }
    }
    s_pos = pos;
  }
  __syncthreads();
  const float v = x[(size_t(b) * S + s_pos) * H + c];
  const float mean = block_sum(v, red) / float(H);
  const float d = v - mean;
  const float rstd = rsqrtf(block_sum(d * d, red) / float(H) + eps);
  head_smem[c] = d * rstd * ln_g[c] + ln_b[c];
  __syncthreads();
  // projection: warp w computes outputs w, w + nwarps, ... with coalesced reads of the weight rows
  float* proj_out = head_smem + H;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int o0 = warp * 4; o0 < P; o0 += nwarps * 4) {   // 4 weight rows per warp in flight
    float a[4] = {0.f, 0.f, 0.f, 0.f};
    for (int i = lane; i < H; i += 32) {
      const float xv = head_smem[i];
#pragma unroll
      for (int u = 0; u < 4; ++u) a[u] = fmaf(proj[size_t(min(o0 + u, P - 1)) * H + i], xv, a[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float t = warp_allreduce_sum(a[u]);
      if (lane == 0 && o0 + u < P) proj_out[o0 + u] = t;
    }
  }
  __syncthreads();
  const float e = c < P ? proj_out[c] : 0.f;
  const float nrm = sqrtf(block_sum(e * e, red));
  if (c < P) out[size_t(b) * P + c] = nrm > 0.f ? e / nrm : e;
}

// Cross-encoder head (BertForSequenceClassification, one label): logit = w_c . tanh(W_p h_CLS + b_p) + b_c.  blockDim.x == H.
__global__ void cross_head_kernel(const float* __restrict__ x, int S, int H, const float* __restrict__ pool_w,
                                  const float* __restrict__ pool_b, const float* __restrict__ cls_w,
                                  const float* __restrict__ cls_b, float* __restrict__ out) {
  extern __shared__ float head_smem[];   // [H] CLS hidden state
  __shared__ float red[32];
  pdl_chain_prologue();
  const int b = blockIdx.x, c = threadIdx.x;
  head_smem[c] = x[(size_t(b) * S) * H + c];
  __syncthreads();
  float* pooled = head_smem + H;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int o0 = warp * 4; o0 < H; o0 += nwarps * 4) {   // 4 weight rows per warp in flight, coalesced reads
    float a[4] = {0.f, 0.f, 0.f, 0.f};
    for (int i = lane; i < H; i += 32) {
      const float xv = head_smem[i];
#pragma unroll
      for (int u = 0; u < 4; ++u) a[u] = fmaf(pool_w[size_t(min(o0 + u, H - 1)) * H + i], xv, a[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float t = warp_allreduce_sum(a[u]);
      if (lane == 0 && o0 + u < H) pooled[o0 + u] = tanhf(t + pool_b[o0 + u]);
    }
  }
  __syncthreads();
  const float logit = block_sum(pooled[c] * cls_w[c], red);
  if (c == 0) out[b] = logit + cls_b[0];
}

// fp32 -> bf16 weight conversion (set_weight)
__global__ void f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int64_t n) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    dst[i] = __float2bfloat16_rn(src[i]);
}
#endif  // __CUDACC__

}  // namespace mmr
