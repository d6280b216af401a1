// libmmr_b200.so -- device-side query encoders behind the C ABI (include/mmr_b200.h, "Query encoders").
// Host side: weight store, activation arena, the launch sequence of one forward pass.
#include <algorithm>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "abi_common.h"
#include "encoder_kernels.cuh"

using namespace mmr;
#define fail mmr_fail

namespace {

struct LayerW {
  __nv_bfloat16 *qkv_w = nullptr, *o_w = nullptr, *fc1_w = nullptr, *fc2_w = nullptr;   // [N_out, K] bf16
  float *qkv_b = nullptr, *o_b = nullptr, *fc1_b = nullptr, *fc2_b = nullptr;
  float *ln1_w = nullptr, *ln1_b = nullptr, *ln2_w = nullptr, *ln2_b = nullptr;
  CUtensorMap m_qkv, m_o, m_fc1, m_fc2;
};

bool make_map(CUtensorMap* map, const void* base, int64_t rows, int cols, int box_rows) {
  mmr_encode_tiled_fn fn = umma_encode_fn();
  if (!fn) return false;
  cuuint64_t gdim[2] = {cuuint64_t(cols), cuuint64_t(rows)};
  cuuint64_t gstr[1] = {cuuint64_t(cols) * 2};
  cuuint32_t box[2] = {64, cuuint32_t(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

struct mmr_encoder {
  int device = 0;
  mmr_encoder_config cfg{};     // vision: kind MMR_ENC_CLIP_VISION, max_positions = tokens per image, no vocabulary
  mmr_vision_config vcfg{};
  int patch_cols = 0;           // vision: C * P * P, the patch GEMM's K
  int out_dim = 0;
  std::mutex mu;
  std::vector<LayerW> layers;
  float *word = nullptr, *pos = nullptr, *type_emb = nullptr, *emb_ln_w = nullptr, *emb_ln_b = nullptr;
  float *final_ln_w = nullptr, *final_ln_b = nullptr, *proj_w = nullptr;                     // CLIP
  float *cls_emb = nullptr, *pre_ln_w = nullptr, *pre_ln_b = nullptr;                         // CLIP vision
  __nv_bfloat16* patch_w = nullptr;                                                           // [H, C * P * P]
  CUtensorMap m_patch_w;
  float *pool_w = nullptr, *pool_b = nullptr, *cls_w = nullptr, *cls_b = nullptr;            // cross-encoder
  std::vector<void*> owned;
  std::map<std::string, bool> seen;
  // activation arena for up to cap_tokens tokens
  int cap_tokens = 0, cap_seqs = 0;
  float *x = nullptr, *tmp = nullptr, *qkv = nullptr;
  __nv_bfloat16 *x16 = nullptr, *ctx16 = nullptr, *h16 = nullptr;
  int32_t *d_ids = nullptr, *d_mask = nullptr, *d_types = nullptr, *h_stage = nullptr;
  CUtensorMap m_x16, m_ctx16, m_h16;
  CUtensorMap m_patch;                     // vision: the patch matrix [B * NP, C * P * P] bf16, held in h16
  int maps_tokens = -1;
  int maps_narrow = -1;
  int nt_x = 64, nt_ctx = 64, nt_h = 64, nt_patch = 64;   // token tiles (= box rows) of the activation maps
};

static int dev_alloc(mmr_encoder* e, void** p, size_t bytes) {
  CUDA_TRY(cudaMalloc(p, std::max<size_t>(bytes, 16)));
  e->owned.push_back(*p);
  return MMR_OK;
}

// Device check and allocation of a validated config (cfg: text kinds; vc: also given for MMR_ENC_CLIP_VISION).
static int encoder_new(int device, const mmr_encoder_config* cfg, const mmr_vision_config* vc, mmr_encoder** out) {
  const int H = cfg->hidden, I = cfg->intermediate;
  int major = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) return fail(MMR_ERR_CUDA, "device %d is not sm_100: the encoders have no other backend", device);
  CUDA_TRY(cudaSetDevice(device));
  mmr_encoder* e = new mmr_encoder();
  e->device = device;
  e->cfg = *cfg;
  if (vc) {
    e->vcfg = *vc;
    e->patch_cols = vc->channels * vc->patch_size * vc->patch_size;
  }
  const bool clip = cfg->kind == MMR_ENC_CLIP_TEXT || cfg->kind == MMR_ENC_CLIP_VISION;
  e->out_dim = cfg->kind == MMR_ENC_CROSS ? 1 : (clip ? cfg->proj_dim : H);
  e->layers.resize(cfg->layers);
  int rc = MMR_OK;
  auto A = [&](void** p, size_t bytes) { if (rc == MMR_OK) rc = dev_alloc(e, p, bytes); };
  if (cfg->kind != MMR_ENC_CLIP_VISION) A((void**)&e->word, size_t(cfg->vocab_size) * H * 4);
  A((void**)&e->pos, size_t(cfg->max_positions) * H * 4);
  if (!clip) {
    A((void**)&e->type_emb, size_t(std::max(cfg->type_vocab, 1)) * H * 4);
    A((void**)&e->emb_ln_w, H * 4);
    A((void**)&e->emb_ln_b, H * 4);
  } else {
    A((void**)&e->final_ln_w, H * 4);
    A((void**)&e->final_ln_b, H * 4);
    A((void**)&e->proj_w, size_t(cfg->proj_dim) * H * 4);
  }
  if (cfg->kind == MMR_ENC_CLIP_VISION) {
    A((void**)&e->cls_emb, H * 4);
    A((void**)&e->pre_ln_w, H * 4);
    A((void**)&e->pre_ln_b, H * 4);
    A((void**)&e->patch_w, size_t(H) * e->patch_cols * 2);
    if (rc == MMR_OK && !make_map(&e->m_patch_w, e->patch_w, H, e->patch_cols, ENC_BM))
      rc = fail(MMR_ERR_CUDA, "cuTensorMapEncodeTiled failed for the patch embedding weight");
  }
  if (cfg->kind == MMR_ENC_CROSS) {
    A((void**)&e->pool_w, size_t(H) * H * 4);
    A((void**)&e->pool_b, H * 4);
    A((void**)&e->cls_w, H * 4);
    A((void**)&e->cls_b, 4);
  }
  for (auto& L : e->layers) {
    A((void**)&L.qkv_w, size_t(3 * H) * H * 2);
    A((void**)&L.o_w, size_t(H) * H * 2);
    A((void**)&L.fc1_w, size_t(I) * H * 2);
    A((void**)&L.fc2_w, size_t(H) * I * 2);
    A((void**)&L.qkv_b, 3 * H * 4);
    A((void**)&L.o_b, H * 4);
    A((void**)&L.fc1_b, I * 4);
    A((void**)&L.fc2_b, H * 4);
    A((void**)&L.ln1_w, H * 4);
    A((void**)&L.ln1_b, H * 4);
    A((void**)&L.ln2_w, H * 4);
    A((void**)&L.ln2_b, H * 4);
    if (rc == MMR_OK && (!make_map(&L.m_qkv, L.qkv_w, 3 * H, H, ENC_BM) || !make_map(&L.m_o, L.o_w, H, H, ENC_BM) ||
                         !make_map(&L.m_fc1, L.fc1_w, I, H, ENC_BM) || !make_map(&L.m_fc2, L.fc2_w, H, I, ENC_BM)))
      rc = fail(MMR_ERR_CUDA, "cuTensorMapEncodeTiled failed for an encoder weight");
  }
  if (rc != MMR_OK) {
    mmr_encoder_destroy(e);
    return rc;
  }
  *out = e;
  return MMR_OK;
}

extern "C" int mmr_encoder_create(int device, const mmr_encoder_config* cfg, mmr_encoder** out) {
  if (!out || !cfg) return fail(MMR_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (cfg->kind != MMR_ENC_MINILM && cfg->kind != MMR_ENC_CLIP_TEXT && cfg->kind != MMR_ENC_CROSS)
    return fail(MMR_ERR_INVALID, "unknown encoder kind %d", cfg->kind);
  const int H = cfg->hidden, I = cfg->intermediate;
  if ((H != 384 && H != 512) || H % cfg->heads != 0 || (H / cfg->heads != 32 && H / cfg->heads != 64))
    return fail(MMR_ERR_UNSUPPORTED, "hidden %d / heads %d: kernels are built for hidden 384 or 512 with head dim 32 or 64", H, cfg->heads);
  if (I % 128 != 0 || I % 64 != 0 || (3 * H) % 128 != 0) return fail(MMR_ERR_UNSUPPORTED, "intermediate size must be a multiple of 128");
  if (cfg->layers < 1 || cfg->vocab_size < 1 || cfg->max_positions < 1) return fail(MMR_ERR_INVALID, "bad config");
  return encoder_new(device, cfg, nullptr, out);
}

extern "C" int mmr_encoder_create_vision(int device, const mmr_vision_config* vc, mmr_encoder** out) {
  if (!out || !vc) return fail(MMR_ERR_INVALID, "NULL argument");
  *out = nullptr;
  const int H = vc->hidden;
  if (H != 768 || vc->heads < 1 || H % vc->heads != 0 || H / vc->heads != 64)
    return fail(MMR_ERR_UNSUPPORTED, "hidden %d / heads %d: the vision tower is built for hidden 768 with head dim 64", H, vc->heads);
  if (vc->layers < 1) return fail(MMR_ERR_INVALID, "layers = %d: must be >= 1", vc->layers);
  if (vc->channels < 1 || vc->patch_size < 1 || vc->image_size < 1)
    return fail(MMR_ERR_INVALID, "channels %d / image_size %d / patch_size %d: must be >= 1", vc->channels, vc->image_size, vc->patch_size);
  if (vc->image_size % vc->patch_size != 0)
    return fail(MMR_ERR_INVALID, "image_size %d is not a multiple of patch_size %d", vc->image_size, vc->patch_size);
  const int64_t cols = int64_t(vc->channels) * vc->patch_size * vc->patch_size;
  if (cols % 64 != 0 || cols > (1 << 20))
    return fail(MMR_ERR_UNSUPPORTED, "channels * patch_size^2 = %lld: the patch GEMM needs a multiple of 64 (at most 2^20)", (long long)cols);
  if (vc->intermediate < 128 || vc->intermediate % 128 != 0)
    return fail(MMR_ERR_UNSUPPORTED, "intermediate size %d must be a positive multiple of 128", vc->intermediate);
  const int64_t grid = vc->image_size / vc->patch_size, tokens = grid * grid + 1;
  if (tokens > 330)
    return fail(MMR_ERR_UNSUPPORTED, "%lld tokens per image (%lld patches + class token): the fp32 attention at head dim 64 takes 330 at most",
                (long long)tokens, (long long)(tokens - 1));
  if (vc->proj_dim < 1 || vc->proj_dim > H) return fail(MMR_ERR_INVALID, "proj_dim %d: must be in [1, hidden = %d]", vc->proj_dim, H);
  mmr_encoder_config cfg{};
  cfg.kind = MMR_ENC_CLIP_VISION;
  cfg.hidden = H;
  cfg.layers = vc->layers;
  cfg.heads = vc->heads;
  cfg.intermediate = vc->intermediate;
  cfg.max_positions = int32_t(tokens);
  cfg.proj_dim = vc->proj_dim;
  cfg.ln_eps = vc->ln_eps;
  return encoder_new(device, &cfg, vc, out);
}

extern "C" int mmr_encoder_destroy(mmr_encoder* e) {
  if (!e) return MMR_OK;
  cudaSetDevice(e->device);
  for (void* p : e->owned) cudaFree(p);
  if (e->h_stage) cudaFreeHost(e->h_stage);
  delete e;
  return MMR_OK;
}

extern "C" int mmr_encoder_out_dim(const mmr_encoder* e) { return e ? e->out_dim : 0; }

// name -> (destination, element count, is bf16 GEMM weight)
static bool weight_slot(mmr_encoder* e, const std::string& name, void** dst, int64_t* numel, bool* bf16) {
  const int H = e->cfg.hidden, I = e->cfg.intermediate;
  *bf16 = false;
  auto set = [&](void* p, int64_t n, bool b = false) { *dst = p; *numel = n; *bf16 = b; return p != nullptr; };
  if (name == "word_emb") return set(e->word, int64_t(e->cfg.vocab_size) * H);
  if (name == "pos_emb") return set(e->pos, int64_t(e->cfg.max_positions) * H);
  if (name == "type_emb") return set(e->type_emb, int64_t(std::max(e->cfg.type_vocab, 1)) * H);
  if (name == "emb_ln_w") return set(e->emb_ln_w, H);
  if (name == "emb_ln_b") return set(e->emb_ln_b, H);
  if (name == "final_ln_w") return set(e->final_ln_w, H);
  if (name == "final_ln_b") return set(e->final_ln_b, H);
  if (name == "proj_w") return set(e->proj_w, int64_t(e->cfg.proj_dim) * H);
  if (name == "patch_w") return set(e->patch_w, int64_t(H) * e->patch_cols, true);
  if (name == "cls_emb") return set(e->cls_emb, H);
  if (name == "pre_ln_w") return set(e->pre_ln_w, H);
  if (name == "pre_ln_b") return set(e->pre_ln_b, H);
  if (name == "pooler_w") return set(e->pool_w, int64_t(H) * H);
  if (name == "pooler_b") return set(e->pool_b, H);
  if (name == "cls_w") return set(e->cls_w, H);
  if (name == "cls_b") return set(e->cls_b, 1);
  int l = -1;
  char field[32] = {0};
  if (sscanf(name.c_str(), "L%d.%31s", &l, field) == 2 && l >= 0 && l < int(e->layers.size())) {
    LayerW& L = e->layers[l];
    const std::string f(field);
    if (f == "qkv_w") return set(L.qkv_w, int64_t(3 * H) * H, true);
    if (f == "o_w") return set(L.o_w, int64_t(H) * H, true);
    if (f == "fc1_w") return set(L.fc1_w, int64_t(I) * H, true);
    if (f == "fc2_w") return set(L.fc2_w, int64_t(H) * I, true);
    if (f == "qkv_b") return set(L.qkv_b, 3 * H);
    if (f == "o_b") return set(L.o_b, H);
    if (f == "fc1_b") return set(L.fc1_b, I);
    if (f == "fc2_b") return set(L.fc2_b, H);
    if (f == "ln1_w") return set(L.ln1_w, H);
    if (f == "ln1_b") return set(L.ln1_b, H);
    if (f == "ln2_w") return set(L.ln2_w, H);
    if (f == "ln2_b") return set(L.ln2_b, H);
  }
  return false;
}

extern "C" int mmr_encoder_set_weight(mmr_encoder* e, const char* name, const float* data_dev, int64_t numel, void* stream) {
  if (!e || !name || !data_dev) return fail(MMR_ERR_INVALID, "NULL argument");
  void* dst = nullptr;
  int64_t want = 0;
  bool bf16 = false;
  if (!weight_slot(e, name, &dst, &want, &bf16)) return fail(MMR_ERR_INVALID, "encoder has no weight named %s", name);
  if (numel != want) return fail(MMR_ERR_INVALID, "weight %s: %lld elements, expected %lld", name, (long long)numel, (long long)want);
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (bf16) {
    f32_to_bf16_kernel<<<std::min<int64_t>((numel + 255) / 256, 4096), 256, 0, st>>>(data_dev, static_cast<__nv_bfloat16*>(dst), numel);
    mmr_g_launches++;
    CUDA_TRY(cudaGetLastError());
  } else {
    CUDA_TRY(cudaMemcpyAsync(dst, data_dev, size_t(numel) * 4, cudaMemcpyDeviceToDevice, st));
  }
  e->seen[name] = true;
  return MMR_OK;
}

static int ensure_arena(mmr_encoder* e, int tokens, int seqs) {
  if (tokens <= e->cap_tokens && seqs <= e->cap_seqs) return MMR_OK;
  const int H = e->cfg.hidden, I = e->cfg.intermediate;
  const int cap = std::max(tokens, std::max(e->cap_tokens, 256));
  const int cs = std::max(seqs, std::max(e->cap_seqs, 8));
  // (old arena stays in `owned` until destroy: arenas only grow a few times)
  CUDA_TRY(cudaMalloc((void**)&e->x, size_t(cap) * H * 4));        e->owned.push_back(e->x);
  CUDA_TRY(cudaMalloc((void**)&e->tmp, size_t(cap) * H * 4));      e->owned.push_back(e->tmp);
  CUDA_TRY(cudaMalloc((void**)&e->qkv, size_t(cap) * 3 * H * 4));  e->owned.push_back(e->qkv);
  CUDA_TRY(cudaMalloc((void**)&e->x16, size_t(cap) * H * 2));      e->owned.push_back(e->x16);
  CUDA_TRY(cudaMalloc((void**)&e->ctx16, size_t(cap) * H * 2));    e->owned.push_back(e->ctx16);
  // h16 also holds a vision pass's patch matrix (B * NP < tokens rows of C * P * P), read before the first FFN1 writes h16
  CUDA_TRY(cudaMalloc((void**)&e->h16, size_t(cap) * std::max(I, e->patch_cols) * 2)); e->owned.push_back(e->h16);
  CUDA_TRY(cudaMalloc((void**)&e->d_ids, size_t(cap) * 3 * 4));    e->owned.push_back(e->d_ids);
  e->d_mask = e->d_ids + cap;
  e->d_types = e->d_ids + 2 * size_t(cap);
  if (e->h_stage) cudaFreeHost(e->h_stage);
  CUDA_TRY(cudaMallocHost((void**)&e->h_stage, size_t(cap) * 3 * 4));
  e->cap_tokens = cap;
  e->cap_seqs = cs;
  e->maps_tokens = -1;
  return MMR_OK;
}

static int enc_token_tile(int M) { return M <= 1024 ? 64 : (M <= 4096 ? 128 : 256); }
// Token tile of one GEMM: the M-based tile, halved while the grid (N / 128 feature tiles x token tiles) would leave SMs
// without their two CTAs -- the narrow GEMMs (out-proj and FFN2: N = hidden = 3-4 feature tiles) ran 96 CTAs on 148 SMs at
// 4096 tokens (profiles/r02_encoder_summary.md).  The tile never changes a result (accumulation runs along K only).
static int enc_token_tile_for(int M, int N) {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  int nt = enc_token_tile(M);
  if (options().enc_narrow_tiles == 0) return nt;
  // 128 -> 64 until every SM has its two CTAs; 256 -> 128 only when SMs would otherwise idle (at 16384 tokens the 256-token
  // tile with 192 CTAs beats 384 CTAs of 128: profiles/r02_encoder_summary.md)
  while (nt > 64 && int64_t(N / ENC_BM) * ((M + nt - 1) / nt) < (nt == 256 ? 1 : 2) * int64_t(sms)) nt >>= 1;
  return nt;
}

template <int EPI, int NT>
static int launch_gemm_nt(const CUtensorMap& mw, const CUtensorMap& mx, int M, int N, int K, const float* bias,
                          const float* residual, float* out_f32, __nv_bfloat16* out_bf16, cudaStream_t st) {
  static bool attr_done[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  GemmParams p{};
  p.M = M;
  p.N = N;
  p.K = K;
  const int stage_bytes = ENC_W_SLICE + NT * 128;
  p.nstages = std::max(2, std::min(std::min(ENC_MAX_STAGES, K / 64), (options().enc_gemm_smem_kb * 1024) / stage_bytes));
  p.bias = bias;
  p.residual = residual;
  p.out_f32 = out_f32;
  p.out_bf16 = out_bf16;
  const size_t smem = size_t(p.nstages) * stage_bytes + (2 * ENC_MAX_STAGES + 3) * 8 + 64;
  if (!attr_done[dev & 63]) {
    CUDA_TRY(cudaFuncSetAttribute(gemm_wt_kernel<EPI, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 210 * 1024));
    attr_done[dev & 63] = true;
  }
  CUDA_TRY(launch_pdl(gemm_wt_kernel<EPI, NT>, dim3(N / ENC_BM, (M + NT - 1) / NT), dim3(ENC_THREADS), smem, st, mw, mx, p));
  mmr_g_launches++;
  return MMR_OK;
}

template <int EPI>
static int launch_gemm(const CUtensorMap& mw, const CUtensorMap& mx, int nt, int M, int N, int K, const float* bias,
                       const float* residual, float* out_f32, __nv_bfloat16* out_bf16, cudaStream_t st) {
  switch (nt) {   // = the box rows of the activation map mx
    case 64: return launch_gemm_nt<EPI, 64>(mw, mx, M, N, K, bias, residual, out_f32, out_bf16, st);
    case 128: return launch_gemm_nt<EPI, 128>(mw, mx, M, N, K, bias, residual, out_f32, out_bf16, st);
    default: return launch_gemm_nt<EPI, 256>(mw, mx, M, N, K, bias, residual, out_f32, out_bf16, st);
  }
}

// The same GEMM with the LayerNorm in front of it folded in (gemm_wt_kernel<EPI, 64, true>): X = LN(ln_src), normalised rows
// also written to ln_out (fp32) when the residual stream needs them.  Token tile 64 only (the latency-bound regime).
template <int EPI>
static int launch_gemm_ln(const CUtensorMap& mw, const CUtensorMap& any_x_map, int M, int N, int K, const float* bias,
                          float* out_f32, __nv_bfloat16* out_bf16, const float* ln_src, const float* ln_g, const float* ln_b,
                          float ln_eps, float* ln_out, cudaStream_t st) {
  static bool attr_done[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  GemmParams p{};
  p.M = M;
  p.N = N;
  p.K = K;
  p.nstages = std::min(ENC_MAX_STAGES, K / 64);
  p.bias = bias;
  p.out_f32 = out_f32;
  p.out_bf16 = out_bf16;
  p.ln_src = ln_src;
  p.ln_g = ln_g;
  p.ln_b = ln_b;
  p.ln_out = ln_out;
  p.ln_eps = ln_eps;
  const size_t smem = size_t(p.nstages) * ENC_W_SLICE + size_t(K / 64) * (64 * 128) + (2 * ENC_MAX_STAGES + 3) * 8 + 64;
  if (!attr_done[dev & 63]) {
    CUDA_TRY(cudaFuncSetAttribute(gemm_wt_kernel<EPI, 64, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 210 * 1024));
    attr_done[dev & 63] = true;
  }
  CUDA_TRY(launch_pdl(gemm_wt_kernel<EPI, 64, true>, dim3(N / ENC_BM, (M + 63) / 64), dim3(ENC_THREADS), smem, st, mw, any_x_map, p));
  mmr_g_launches++;
  return MMR_OK;
}

// Shared memory of one attention launch, checked against the kernel's own limit (the opt-in size set below): the fp32
// kernel holds K and V of the head in fp32 (head dim 64: 330 tokens at most), the tensor-core kernel in bf16 (512 fit).
static int attention_smem(bool tensor_cores, int DH, int S, size_t* smem) {
  if (tensor_cores) {
    *smem = DH == 32 ? attention_mma_smem_bytes<32>(S) : attention_mma_smem_bytes<64>(S);
    if (*smem > 200 * 1024)
      return fail(MMR_ERR_UNSUPPORTED, "sequence length %d does not fit the tensor-core attention kernel (head dim %d)", S, DH);
  } else {
    *smem = DH == 32 ? attention_smem_bytes<32>(S) : attention_smem_bytes<64>(S);
    if (*smem > 220 * 1024)
      return fail(MMR_ERR_UNSUPPORTED, "sequence length %d does not fit the fp32 attention kernel (head dim %d: %d tokens at most)", S,
                  DH, DH == 32 ? 552 : 330);
  }
  return MMR_OK;
}

// One attention launch over qkv fp32 [B * S, 3H] -> ctx bf16 [B * S, H]: attention_mma_kernel (tensor_cores) or
// attention_kernel, head dim H / heads.  The forward pass and mmr_debug_enc_attention both launch through here.
static int launch_attention(bool tensor_cores, int B, int S, int H, int heads, int causal, const float* qkv, const int32_t* mask,
                            __nv_bfloat16* ctx, cudaStream_t st) {
  const int DH = H / heads;
  size_t smem = 0;
  const int rc = attention_smem(tensor_cores, DH, S, &smem);
  if (rc != MMR_OK) return rc;
  static bool att_attr[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (!att_attr[dev & 63]) {
    CUDA_TRY(cudaFuncSetAttribute(attention_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    CUDA_TRY(cudaFuncSetAttribute(attention_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    CUDA_TRY(cudaFuncSetAttribute(attention_mma_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    CUDA_TRY(cudaFuncSetAttribute(attention_mma_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    att_attr[dev & 63] = true;
  }
  const dim3 att_mma_grid(heads, B, (S + ATC_ROWS - 1) / ATC_ROWS);
  if (tensor_cores && DH == 32)
    CUDA_TRY(launch_pdl(attention_mma_kernel<32>, att_mma_grid, dim3(ATC_NW * 32), smem, st, qkv, mask, ctx, S, H, causal));
  else if (tensor_cores)
    CUDA_TRY(launch_pdl(attention_mma_kernel<64>, att_mma_grid, dim3(ATC_NW * 32), smem, st, qkv, mask, ctx, S, H, causal));
  else if (DH == 32)
    CUDA_TRY(launch_pdl(attention_kernel<32>, dim3(heads, B), dim3(ATT_NW * 32), smem, st, qkv, mask, ctx, S, H, causal));
  else
    CUDA_TRY(launch_pdl(attention_kernel<64>, dim3(heads, B), dim3(ATT_NW * 32), smem, st, qkv, mask, ctx, S, H, causal));
  mmr_g_launches++;
  return MMR_OK;
}

// Tensor maps of the activation buffers for a pass of M tokens (TMA zero-fills rows past M, so they depend on the live
// token count); patch_rows > 0 (vision) also maps the patch matrix.  Box rows of an activation map = the token tile of the
// GEMMs that read it: x16 feeds QKV (N = 3H) and FFN1 (N = I), ctx16 the out-projection and h16 FFN2 (both N = H), the patch
// matrix the patch GEMM (N = H).
static int ensure_maps(mmr_encoder* e, int M, int H, int patch_rows) {
  if (e->maps_tokens == M && e->maps_narrow == options().enc_narrow_tiles) return MMR_OK;
  const int I = e->cfg.intermediate;
  e->nt_x = enc_token_tile_for(M, std::min(3 * H, I));
  e->nt_ctx = enc_token_tile_for(M, H);
  e->nt_h = enc_token_tile_for(M, H);
  if (!make_map(&e->m_x16, e->x16, M, H, e->nt_x) || !make_map(&e->m_ctx16, e->ctx16, M, H, e->nt_ctx) ||
      !make_map(&e->m_h16, e->h16, M, I, e->nt_h))
    return fail(MMR_ERR_CUDA, "cuTensorMapEncodeTiled failed for the activations");
  if (patch_rows > 0) {
    e->nt_patch = enc_token_tile_for(patch_rows, H);
    if (!make_map(&e->m_patch, e->h16, patch_rows, e->patch_cols, e->nt_patch))
      return fail(MMR_ERR_CUDA, "cuTensorMapEncodeTiled failed for the patch matrix");
  }
  e->maps_tokens = M;
  e->maps_narrow = options().enc_narrow_tiles;
  return MMR_OK;
}

// Attention kernel of a model: the cross-encoder (rerank passages: 128-512 tokens) runs both attention contractions on the
// tensor cores, whatever the sequence length (kernel choice by model, never by batch shape); MMR_ENC_ATT_MMA=0: fp32 kernel
// everywhere, =2: every model from ATC_MIN_S tokens on (measurement)
static bool attention_on_tensor_cores(const mmr_encoder* e, int S) {
  const int att_opt = options().enc_att_mma;
  return att_opt == 2 ? S >= ATC_MIN_S : (att_opt == 1 && e->cfg.kind == MMR_ENC_CROSS);
}

// The pre-LN layer stack of both CLIP towers over the fp32 residual stream e->x [B * S, H]:
//   h = LN1(x); x = x + out_proj(attention(qkv(h))); h = LN2(x); x = x + fc2(quick_gelu(fc1(h)))
// Text: causal with the padding mask; vision: neither.  fuse_ln folds LN1 / LN2 into the QKV / FC1 GEMMs (H <= 512 only).
template <int H>
static int preln_layers(mmr_encoder* e, int B, int S, bool att_mma, int causal, const int32_t* mask, bool fuse_ln, cudaStream_t st) {
  const mmr_encoder_config& c = e->cfg;
  const int M = B * S, I = c.intermediate;
  const int wpb = 8;
  const dim3 rows_grid((M + wpb - 1) / wpb), rows_block(wpb * 32);
  for (LayerW& L : e->layers) {
    int rc;
    if (fuse_ln) {
      rc = launch_gemm_ln<EPI_BIAS_F32>(L.m_qkv, e->m_x16, M, 3 * H, H, L.qkv_b, e->qkv, nullptr, e->x, L.ln1_w, L.ln1_b, c.ln_eps,
                                        nullptr, st);
    } else {
      CUDA_TRY(launch_pdl(layernorm_kernel<H>, rows_grid, rows_block, 0, st, e->x, L.ln1_w, L.ln1_b, c.ln_eps, M, (float*)nullptr,
                          e->x16));
      mmr_g_launches++;
      rc = launch_gemm<EPI_BIAS_F32>(L.m_qkv, e->m_x16, e->nt_x, M, 3 * H, H, L.qkv_b, nullptr, e->qkv, nullptr, st);
    }
    if (rc != MMR_OK) return rc;
    rc = launch_attention(att_mma, B, S, H, c.heads, causal, e->qkv, mask, e->ctx16, st);
    if (rc != MMR_OK) return rc;
    rc = launch_gemm<EPI_BIAS_RES_F32>(L.m_o, e->m_ctx16, e->nt_ctx, M, H, H, L.o_b, e->x, e->x, nullptr, st);
    if (rc != MMR_OK) return rc;
    if (fuse_ln) {
      rc = launch_gemm_ln<EPI_QUICKGELU_BF16>(L.m_fc1, e->m_x16, M, I, H, L.fc1_b, nullptr, e->h16, e->x, L.ln2_w, L.ln2_b, c.ln_eps,
                                              nullptr, st);
    } else {
      CUDA_TRY(launch_pdl(layernorm_kernel<H>, rows_grid, rows_block, 0, st, e->x, L.ln2_w, L.ln2_b, c.ln_eps, M, (float*)nullptr,
                          e->x16));
      mmr_g_launches++;
      rc = launch_gemm<EPI_QUICKGELU_BF16>(L.m_fc1, e->m_x16, e->nt_x, M, I, H, L.fc1_b, nullptr, nullptr, e->h16, st);
    }
    if (rc != MMR_OK) return rc;
    rc = launch_gemm<EPI_BIAS_RES_F32>(L.m_fc2, e->m_h16, e->nt_h, M, H, I, L.fc2_b, e->x, e->x, nullptr, st);
    if (rc != MMR_OK) return rc;
  }
  return MMR_OK;
}

// The post-LN layer stack of BERT (MiniLM, cross-encoder): x = LN1(x + out_proj(attention(qkv(x))));
// x = LN2(x + fc2(gelu(fc1(x)))), with the padding mask.  fuse_ln folds LN1 into FC1 and LN2 into the next layer's QKV GEMM.
template <int H>
static int postln_layers(mmr_encoder* e, int B, int S, bool att_mma, bool fuse_ln, cudaStream_t st) {
  const mmr_encoder_config& c = e->cfg;
  const int M = B * S, I = c.intermediate;
  const int wpb = 8;
  const dim3 rows_grid((M + wpb - 1) / wpb), rows_block(wpb * 32);
  const LayerW* prev = nullptr;   // BERT: the layer whose closing LayerNorm (ln2 over e->tmp) is still pending
  for (LayerW& L : e->layers) {
    int rc;
    if (prev != nullptr) {   // BERT, fused: x = LN2_prev(tmp) computed by this layer's QKV GEMM
      rc = launch_gemm_ln<EPI_BIAS_F32>(L.m_qkv, e->m_x16, M, 3 * H, H, L.qkv_b, e->qkv, nullptr, e->tmp, prev->ln2_w, prev->ln2_b,
                                        c.ln_eps, e->x, st);
    } else {
      rc = launch_gemm<EPI_BIAS_F32>(L.m_qkv, e->m_x16, e->nt_x, M, 3 * H, H, L.qkv_b, nullptr, e->qkv, nullptr, st);
    }
    if (rc != MMR_OK) return rc;
    rc = launch_attention(att_mma, B, S, H, c.heads, 0, e->qkv, e->d_mask, e->ctx16, st);
    if (rc != MMR_OK) return rc;
    rc = launch_gemm<EPI_BIAS_RES_F32>(L.m_o, e->m_ctx16, e->nt_ctx, M, H, H, L.o_b, e->x, e->tmp, nullptr, st);
    if (rc != MMR_OK) return rc;
    if (fuse_ln) {
      rc = launch_gemm_ln<EPI_GELU_BF16>(L.m_fc1, e->m_x16, M, I, H, L.fc1_b, nullptr, e->h16, e->tmp, L.ln1_w, L.ln1_b, c.ln_eps,
                                         e->x, st);
    } else {
      CUDA_TRY(launch_pdl(layernorm_kernel<H>, rows_grid, rows_block, 0, st, e->tmp, L.ln1_w, L.ln1_b, c.ln_eps, M, e->x, e->x16));
      mmr_g_launches++;
      rc = launch_gemm<EPI_GELU_BF16>(L.m_fc1, e->m_x16, e->nt_x, M, I, H, L.fc1_b, nullptr, nullptr, e->h16, st);
    }
    if (rc != MMR_OK) return rc;
    rc = launch_gemm<EPI_BIAS_RES_F32>(L.m_fc2, e->m_h16, e->nt_h, M, H, I, L.fc2_b, e->x, e->tmp, nullptr, st);
    if (rc != MMR_OK) return rc;
    if (fuse_ln && &L != &e->layers.back()) {
      prev = &L;   // LN2 rides in the next layer's QKV GEMM
    } else {
      CUDA_TRY(launch_pdl(layernorm_kernel<H>, rows_grid, rows_block, 0, st, e->tmp, L.ln2_w, L.ln2_b, c.ln_eps, M, e->x, e->x16));
      mmr_g_launches++;
    }
  }
  return MMR_OK;
}

template <int H>
static int forward_t(mmr_encoder* e, int B, int S, float* out_dev, cudaStream_t st) {
  const mmr_encoder_config& c = e->cfg;
  const int M = B * S, DH = H / c.heads;
  const bool clip = c.kind == MMR_ENC_CLIP_TEXT;
  const int wpb = 8;
  const dim3 rows_grid((M + wpb - 1) / wpb), rows_block(wpb * 32);
  if (const int rc = ensure_maps(e, M, H, 0); rc != MMR_OK) return rc;
  const bool att_mma = attention_on_tensor_cores(e, S);
  size_t att_smem = 0;
  if (const int rc = attention_smem(att_mma, DH, S, &att_smem); rc != MMR_OK) return rc;   // before the first launch

  // embeddings
  if (clip)
    CUDA_TRY(launch_pdl(embed_kernel<H>, rows_grid, rows_block, 0, st, e->d_ids, (const int32_t*)nullptr, e->word, e->pos,
                        (const float*)nullptr, (const float*)nullptr, (const float*)nullptr, c.ln_eps, M, S, e->x,
                        (__nv_bfloat16*)nullptr));
  else
    CUDA_TRY(launch_pdl(embed_kernel<H>, rows_grid, rows_block, 0, st, e->d_ids, e->d_types, e->word, e->pos, e->type_emb,
                        e->emb_ln_w, e->emb_ln_b, c.ln_eps, M, S, e->x, e->x16));
  mmr_g_launches++;
  // LayerNorms in front of a GEMM can be folded into it (MMR_ENC_FUSE_LN=1: passes of <= 16 tokens, =2: whenever the token
  // tile is 64; bit-identical activations either way).  OFF by default -- measured (profiles/r02_encoder_summary.md): 44 -> 33 /
  // 86 -> 62 launches buy nothing (MiniLM 1 x 16: 0.229 -> 0.259 ms, from 128 tokens on clearly slower): a dependent launch
  // costs no more than the LayerNorm it carried, and every CTA of the GEMM repeats its token tile's LayerNorm.
  const int fuse_opt = options().enc_fuse_ln;
  const bool fuse_ln = fuse_opt == 2 ? enc_token_tile(M) == 64 : (fuse_opt == 1 && M <= 16);
  const int rc = clip ? preln_layers<H>(e, B, S, att_mma, 1, e->d_mask, fuse_ln, st) : postln_layers<H>(e, B, S, att_mma, fuse_ln, st);
  if (rc != MMR_OK) return rc;
  // head
  if (c.kind == MMR_ENC_MINILM)
    CUDA_TRY(launch_pdl(mean_pool_norm_kernel, dim3(B), dim3(H), 0, st, e->x, e->d_mask, S, H, out_dev));
  else if (clip)
    CUDA_TRY(launch_pdl(clip_head_kernel, dim3(B), dim3(H), size_t(H + c.proj_dim) * 4, st, e->x, e->d_ids, S, H, c.eos_token_id,
                        e->final_ln_w, e->final_ln_b, c.ln_eps, e->proj_w, c.proj_dim, out_dev));
  else
    CUDA_TRY(launch_pdl(cross_head_kernel, dim3(B), dim3(H), size_t(2 * H) * 4, st, e->x, S, H, e->pool_w, e->pool_b, e->cls_w,
                        e->cls_b, out_dev));
  mmr_g_launches++;
  return MMR_OK;
}

// ------------------------------------------------------------------------------------------------ CLIP vision tower
constexpr int VIS_H = 768;

// The vision front end for B images of C x S_img x S_img pixels, patch size P: patchify -> patch16 [B * NP, C P P] bf16
// (tensor map m_patch, token tile nt), patch GEMM (no bias) -> patch_out fp32 [B * NP, H], class token + positions +
// pre-LayerNorm -> x fp32 [B * (NP + 1), H].  The forward pass and mmr_debug_enc_patch_embed both launch through here.
static int launch_vision_front(int B, int C, int S_img, int P, const float* pixels, __nv_bfloat16* patch16, const CUtensorMap& m_patch_w,
                               const CUtensorMap& m_patch, int nt, float* patch_out, const float* cls, const float* pos,
                               const float* ln_g, const float* ln_b, float eps, float* x, cudaStream_t st) {
  const int np = (S_img / P) * (S_img / P), T = np + 1, M = B * T;
  CUDA_TRY(launch_pdl(patchify_kernel, dim3(B * np), dim3(256), 0, st, pixels, C, S_img, P, patch16));
  mmr_g_launches++;
  const int rc = launch_gemm<EPI_BIAS_F32>(m_patch_w, m_patch, nt, B * np, VIS_H, C * P * P, nullptr, nullptr, patch_out, nullptr, st);
  if (rc != MMR_OK) return rc;
  const int wpb = 8;
  CUDA_TRY(launch_pdl(vision_embed_kernel<VIS_H>, dim3((M + wpb - 1) / wpb), dim3(wpb * 32), 0, st, patch_out, cls, pos, ln_g, ln_b,
                      eps, M, T, x));
  mmr_g_launches++;
  return MMR_OK;
}

static int forward_vision(mmr_encoder* e, const float* pixels, int B, float* out_dev, cudaStream_t st) {
  const mmr_encoder_config& c = e->cfg;
  const mmr_vision_config& v = e->vcfg;
  const int T = c.max_positions, M = B * T;
  if (const int rc = ensure_maps(e, M, VIS_H, B * (T - 1)); rc != MMR_OK) return rc;
  const bool att_mma = attention_on_tensor_cores(e, T);
  size_t att_smem = 0;
  if (const int rc = attention_smem(att_mma, VIS_H / c.heads, T, &att_smem); rc != MMR_OK) return rc;   // before the first launch
  int rc = launch_vision_front(B, v.channels, v.image_size, v.patch_size, pixels, e->h16, e->m_patch_w, e->m_patch, e->nt_patch, e->tmp,
                               e->cls_emb, e->pos, e->pre_ln_w, e->pre_ln_b, c.ln_eps, e->x, st);
  if (rc != MMR_OK) return rc;
  // no mask, not causal; the LayerNorm-folded GEMM holds K <= 512 and is never used at hidden 768
  rc = preln_layers<VIS_H>(e, B, T, att_mma, 0, nullptr, false, st);
  if (rc != MMR_OK) return rc;
  CUDA_TRY(launch_pdl(clip_head_kernel, dim3(B), dim3(VIS_H), size_t(VIS_H + c.proj_dim) * 4, st, e->x, (const int32_t*)nullptr, T,
                      VIS_H, 0, e->final_ln_w, e->final_ln_b, c.ln_eps, e->proj_w, c.proj_dim, out_dev));
  mmr_g_launches++;
  return MMR_OK;
}

extern "C" int mmr_encoder_forward_pixels(mmr_encoder* e, const float* pixels_dev, int32_t B, float* out_dev, void* stream) {
  if (B < 1 || B > 65535) return fail(MMR_ERR_INVALID, "B = %d: must be in [1, 65535]", B);   // 65535: the attention grid's y
  if (!e || !pixels_dev || !out_dev) return fail(MMR_ERR_INVALID, "NULL argument");
  if (e->cfg.kind != MMR_ENC_CLIP_VISION)
    return fail(MMR_ERR_INVALID, "encoder kind %d takes token ids (mmr_encoder_forward), not pixels", e->cfg.kind);
  std::lock_guard<std::mutex> guard(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  const int rc = ensure_arena(e, B * e->cfg.max_positions, B);
  if (rc != MMR_OK) return rc;
  return forward_vision(e, pixels_dev, B, out_dev, static_cast<cudaStream_t>(stream));
}

extern "C" int mmr_encoder_forward(mmr_encoder* e, const int32_t* input_ids_host, const int32_t* attention_mask_host,
                                   const int32_t* token_type_host, int32_t B, int32_t S, float* out_dev, void* stream) {
  if (!e || !input_ids_host || !out_dev) return fail(MMR_ERR_INVALID, "NULL argument");
  if (e->cfg.kind == MMR_ENC_CLIP_VISION)
    return fail(MMR_ERR_INVALID, "a vision encoder takes pixels (mmr_encoder_forward_pixels), not token ids");
  if (B < 1 || S < 1) return fail(MMR_ERR_INVALID, "B and S must be >= 1");
  if (S > e->cfg.max_positions) return fail(MMR_ERR_INVALID, "sequence length %d > max_positions %d", S, e->cfg.max_positions);
  if (S > 512) return fail(MMR_ERR_UNSUPPORTED, "sequence length %d > 512", S);
  if (e->cfg.kind == MMR_ENC_CLIP_TEXT && e->cfg.proj_dim > e->cfg.hidden) return fail(MMR_ERR_UNSUPPORTED, "projection wider than hidden");
  std::lock_guard<std::mutex> guard(e->mu);
  CUDA_TRY(cudaSetDevice(e->device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int M = B * S;
  for (int i = 0; i < M; ++i)
    if (input_ids_host[i] < 0 || input_ids_host[i] >= e->cfg.vocab_size)
      return fail(MMR_ERR_INVALID, "token id %d out of range [0, %d)", input_ids_host[i], e->cfg.vocab_size);
  int rc = ensure_arena(e, M, B);
  if (rc != MMR_OK) return rc;
  // ids | mask | types ride in one pinned staging buffer, one H2D copy
  const size_t cap = size_t(e->cap_tokens);
  CUDA_TRY(cudaStreamSynchronize(st));  // the previous forward may still read the staging buffer's device copy
  memcpy(e->h_stage, input_ids_host, size_t(M) * 4);
  for (int i = 0; i < M; ++i) e->h_stage[cap + i] = attention_mask_host ? attention_mask_host[i] : 1;
  for (int i = 0; i < M; ++i) {
    const int t = token_type_host ? token_type_host[i] : 0;
    if (t < 0 || t >= std::max(e->cfg.type_vocab, 1)) return fail(MMR_ERR_INVALID, "token type %d out of range", t);
    e->h_stage[2 * cap + i] = t;
  }
  CUDA_TRY(cudaMemcpyAsync(e->d_ids, e->h_stage, cap * 3 * 4, cudaMemcpyHostToDevice, st));
  if (e->cfg.hidden == 384) return forward_t<384>(e, B, S, out_dev, st);
  return forward_t<512>(e, B, S, out_dev, st);
}

// ------------------------------------------------------------------------------------------------ validation hooks
// One launch of an encoder kernel on caller buffers, through the same launch code as the forward pass (tests compare each
// with a float64 reference).  Arguments are checked before any CUDA call.
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

template <int EPI>
static int debug_gemm_epi(int nt, bool fold_ln, int M, int N, int K, const void* x_dev, const float* ln_src_dev, const float* ln_g_dev,
                          const float* ln_b_dev, float ln_eps, float* ln_out_dev, const void* w_dev, const float* bias_dev,
                          const float* residual_dev, float* out_f32_dev, void* out_bf16_dev, cudaStream_t st) {
  CUtensorMap mw, mx;
  if (!make_map(&mw, w_dev, N, K, ENC_BM) || (!fold_ln && !make_map(&mx, x_dev, M, K, nt)))
    return fail(MMR_ERR_CUDA, "cuTensorMapEncodeTiled failed");
  __nv_bfloat16* o16 = static_cast<__nv_bfloat16*>(out_bf16_dev);
  if (fold_ln)   // the folded kernel never reads the activation map
    return launch_gemm_ln<EPI>(mw, mw, M, N, K, bias_dev, out_f32_dev, o16, ln_src_dev, ln_g_dev, ln_b_dev, ln_eps, ln_out_dev, st);
  return launch_gemm<EPI>(mw, mx, nt, M, N, K, bias_dev, residual_dev, out_f32_dev, o16, st);
}

extern "C" int mmr_debug_enc_gemm(int32_t epi, int32_t nt, int32_t fold_ln, int32_t M, int32_t N, int32_t K, const void* x_dev,
                                  const float* ln_src_dev, const float* ln_g_dev, const float* ln_b_dev, float ln_eps,
                                  float* ln_out_dev, const void* w_dev, const float* bias_dev, const float* residual_dev,
                                  float* out_f32_dev, void* out_bf16_dev, void* stream) {
  if (epi < EPI_BIAS_F32 || epi > EPI_QUICKGELU_BF16) return fail(MMR_ERR_INVALID, "unknown epilogue %d", epi);
  if (nt != 64 && nt != 128 && nt != 256) return fail(MMR_ERR_INVALID, "token tile %d: must be 64, 128 or 256", nt);
  if (fold_ln != 0 && fold_ln != 1) return fail(MMR_ERR_INVALID, "fold_ln must be 0 or 1");
  if (M < 1 || M > (1 << 22)) return fail(MMR_ERR_INVALID, "M = %d: must be in [1, 2^22]", M);
  if (N < ENC_BM || N % ENC_BM != 0 || N > 65535 * ENC_BM) return fail(MMR_ERR_INVALID, "N = %d: must be a positive multiple of 128", N);
  if (K < 64 || K % 64 != 0) return fail(MMR_ERR_INVALID, "K = %d: must be a positive multiple of 64", K);
  if (!w_dev || !aligned16(w_dev)) return fail(MMR_ERR_INVALID, "W must be a 16-byte aligned device pointer");
  if (fold_ln) {
    if (nt != 64) return fail(MMR_ERR_INVALID, "the LayerNorm-folded GEMM runs on the 64-token tile only (nt = %d)", nt);
    if (K != 384 && K != 512) return fail(MMR_ERR_INVALID, "the LayerNorm-folded GEMM needs K = 384 or 512 (K = %d)", K);
    if (epi == EPI_BIAS_RES_F32) return fail(MMR_ERR_INVALID, "the LayerNorm-folded GEMM has no residual epilogue");
    if (!ln_src_dev || !ln_g_dev || !ln_b_dev) return fail(MMR_ERR_INVALID, "fold_ln needs ln_src, ln_g and ln_b");
    if (ln_out_dev && static_cast<const void*>(ln_out_dev) == static_cast<const void*>(ln_src_dev))
      return fail(MMR_ERR_INVALID, "ln_out may not alias ln_src");
  } else if (!x_dev || !aligned16(x_dev)) {
    return fail(MMR_ERR_INVALID, "X must be a 16-byte aligned device pointer");
  }
  if ((epi == EPI_BIAS_F32 || epi == EPI_BIAS_RES_F32) && !out_f32_dev) return fail(MMR_ERR_INVALID, "epilogue %d needs out_f32", epi);
  if (epi == EPI_BIAS_RES_F32 && !residual_dev) return fail(MMR_ERR_INVALID, "the residual epilogue needs residual");
  if ((epi == EPI_GELU_BF16 || epi == EPI_QUICKGELU_BF16) && !out_bf16_dev) return fail(MMR_ERR_INVALID, "epilogue %d needs out_bf16", epi);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (epi) {
    case EPI_BIAS_F32:
      return debug_gemm_epi<EPI_BIAS_F32>(nt, fold_ln, M, N, K, x_dev, ln_src_dev, ln_g_dev, ln_b_dev, ln_eps, ln_out_dev, w_dev, bias_dev,
                                          residual_dev, out_f32_dev, out_bf16_dev, st);
    case EPI_BIAS_RES_F32:
      return debug_gemm_epi<EPI_BIAS_RES_F32>(nt, fold_ln, M, N, K, x_dev, ln_src_dev, ln_g_dev, ln_b_dev, ln_eps, ln_out_dev, w_dev,
                                              bias_dev, residual_dev, out_f32_dev, out_bf16_dev, st);
    case EPI_GELU_BF16:
      return debug_gemm_epi<EPI_GELU_BF16>(nt, fold_ln, M, N, K, x_dev, ln_src_dev, ln_g_dev, ln_b_dev, ln_eps, ln_out_dev, w_dev, bias_dev,
                                           residual_dev, out_f32_dev, out_bf16_dev, st);
    default:
      return debug_gemm_epi<EPI_QUICKGELU_BF16>(nt, fold_ln, M, N, K, x_dev, ln_src_dev, ln_g_dev, ln_b_dev, ln_eps, ln_out_dev, w_dev,
                                                bias_dev, residual_dev, out_f32_dev, out_bf16_dev, st);
  }
}

extern "C" int mmr_debug_enc_attention(int32_t tensor_cores, int32_t B, int32_t S, int32_t H, int32_t heads, int32_t causal,
                                       const float* qkv_dev, const int32_t* mask_dev, void* ctx_dev, void* stream) {
  if (tensor_cores != 0 && tensor_cores != 1) return fail(MMR_ERR_INVALID, "tensor_cores must be 0 or 1");
  if (causal != 0 && causal != 1) return fail(MMR_ERR_INVALID, "causal must be 0 or 1");
  if ((H != 384 && H != 512) || heads < 1 || H % heads != 0 || (H / heads != 32 && H / heads != 64))
    return fail(MMR_ERR_INVALID, "hidden %d / heads %d: hidden must be 384 or 512 with head dim 32 or 64", H, heads);
  if (B < 1 || B > 65535) return fail(MMR_ERR_INVALID, "B = %d: must be in [1, 65535]", B);
  if (S < 1 || S > 512) return fail(MMR_ERR_INVALID, "S = %d: must be in [1, 512]", S);
  if (!qkv_dev || !ctx_dev || !aligned16(qkv_dev) || !aligned16(ctx_dev))
    return fail(MMR_ERR_INVALID, "qkv and ctx must be 16-byte aligned device pointers");
  return launch_attention(tensor_cores != 0, B, S, H, heads, causal, qkv_dev, mask_dev, static_cast<__nv_bfloat16*>(ctx_dev),
                          static_cast<cudaStream_t>(stream));
}

extern "C" int mmr_debug_enc_layernorm(int32_t H, int32_t M, const float* x_dev, const float* g_dev, const float* b_dev, float eps,
                                       float* out_f32_dev, void* out_bf16_dev, void* stream) {
  if (H != 384 && H != 512) return fail(MMR_ERR_INVALID, "H = %d: must be 384 or 512", H);
  if (M < 1 || M > (1 << 22)) return fail(MMR_ERR_INVALID, "M = %d: must be in [1, 2^22]", M);
  if (!x_dev || !g_dev || !b_dev) return fail(MMR_ERR_INVALID, "NULL argument");
  if (!out_f32_dev && !out_bf16_dev) return fail(MMR_ERR_INVALID, "no output: out_f32 and out_bf16 are both NULL");
  const int wpb = 8;   // forward_t's rows_grid / rows_block
  const dim3 grid((M + wpb - 1) / wpb), block(wpb * 32);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  __nv_bfloat16* o16 = static_cast<__nv_bfloat16*>(out_bf16_dev);
  if (H == 384)
    CUDA_TRY(launch_pdl(layernorm_kernel<384>, grid, block, 0, st, x_dev, g_dev, b_dev, eps, M, out_f32_dev, o16));
  else
    CUDA_TRY(launch_pdl(layernorm_kernel<512>, grid, block, 0, st, x_dev, g_dev, b_dev, eps, M, out_f32_dev, o16));
  mmr_g_launches++;
  return MMR_OK;
}

extern "C" int mmr_debug_enc_patch_embed(int32_t H, int32_t C, int32_t image_size, int32_t patch, int32_t B, const float* pixels_dev,
                                         const void* patch_w_dev, const float* cls_dev, const float* pos_dev, const float* ln_g_dev,
                                         const float* ln_b_dev, float ln_eps, void* patch16_dev, float* patch_out_dev, float* x_dev,
                                         void* stream) {
  if (H != VIS_H) return fail(MMR_ERR_INVALID, "H = %d: the vision front end is built for hidden 768", H);
  if (C < 1 || patch < 1 || image_size < 1)
    return fail(MMR_ERR_INVALID, "C = %d, image_size = %d, patch = %d: must be >= 1", C, image_size, patch);
  if (image_size % patch != 0) return fail(MMR_ERR_INVALID, "image_size %d is not a multiple of patch %d", image_size, patch);
  const int64_t cols = int64_t(C) * patch * patch, grid = image_size / patch;
  if (cols % 64 != 0 || cols > (1 << 20)) return fail(MMR_ERR_INVALID, "C * patch^2 = %lld: must be a multiple of 64 (at most 2^20)", (long long)cols);
  if (B < 1 || B > 65535) return fail(MMR_ERR_INVALID, "B = %d: must be in [1, 65535]", B);
  if (int64_t(B) * (grid * grid + 1) > (1 << 22)) return fail(MMR_ERR_INVALID, "B x tokens per image must be <= 2^22");
  if (!pixels_dev || !cls_dev || !pos_dev || !ln_g_dev || !ln_b_dev || !patch_out_dev || !x_dev) return fail(MMR_ERR_INVALID, "NULL argument");
  if (!patch_w_dev || !patch16_dev || !aligned16(patch_w_dev) || !aligned16(patch16_dev))
    return fail(MMR_ERR_INVALID, "patch_w and patch16 must be 16-byte aligned device pointers");
  const int rows = B * int(grid * grid);
  const int nt = enc_token_tile_for(rows, H);   // the forward pass's tile for this patch count
  CUtensorMap mw, mx;
  if (!make_map(&mw, patch_w_dev, H, int(cols), ENC_BM) || !make_map(&mx, patch16_dev, rows, int(cols), nt))
    return fail(MMR_ERR_CUDA, "cuTensorMapEncodeTiled failed");
  return launch_vision_front(B, C, image_size, patch, pixels_dev, static_cast<__nv_bfloat16*>(patch16_dev), mw, mx, nt, patch_out_dev,
                             cls_dev, pos_dev, ln_g_dev, ln_b_dev, ln_eps, x_dev, static_cast<cudaStream_t>(stream));
}
