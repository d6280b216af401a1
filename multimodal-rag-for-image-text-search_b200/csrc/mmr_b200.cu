// libmmr_b200.so -- C ABI (include/mmr_b200.h) over the sm_100a scan kernels.
// Host side: argument checks, planning (which kernel, grid, workspace carve-up), launches.
#include "abi_common.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include "aux_kernels.cuh"
#include "common.cuh"
#include "scan_stream.cuh"
#include "scan_umma2.cuh"

using namespace mmr;

// ------------------------------------------------------------------------------------------------ errors
thread_local std::string mmr_g_err;
std::atomic<int64_t> mmr_g_launches{0};
static thread_local int g_last_kernel = 0;
static std::atomic<int64_t> g_rescore_reruns{0};
#define g_err mmr_g_err
#define g_launches mmr_g_launches
#define fail mmr_fail

int mmr_fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  mmr_g_err = buf;
  return code;
}

// ------------------------------------------------------------------------------------------------ index
struct mmr_index {
  int device = 0;
  int dim = 0;
  int dtype = MMR_BF16;
  int64_t n_rows = 0;
  const void* rows = nullptr;
  int64_t row_base = 0;
  std::vector<int64_t> seg;  // [n_segments + 1]
  int sm_count = 0;
  int query_precision = MMR_QP_AUTO;
  mutable uint8_t* h_flags = nullptr;   // pinned: per-query "proven exact" flags of the rescoring mode
  mutable int flags_cap = 0;
  // Host-buffer calls (mmr_search_host & co): one staging set per index, serialised by host_mu.
  //   h_q / d_q      pinned + device copy of the queries (only when they do not ride in the kernel parameters)
  //   h_box / d_box  MAPPED pinned mailbox: [flag u32 | pad to 64][scores f32 B*k | pad][rows i64 B*k]; the kernels write
  //                  results and the completion flag straight into it, the host spins on the flag
  std::mutex host_mu;
  float* h_q = nullptr;
  float* d_q = nullptr;
  uint8_t* h_box = nullptr;
  uint8_t* d_box = nullptr;
  uint32_t box_seq = 0;
  void* d_ws = nullptr;
  size_t ws_bytes = 0;
  int cap_b = 0, cap_k = 0;
  mutable UmmaIndexState umma;
  mutable Umma2IndexState umma2;
};

static int elem_bytes(int dtype) { return dtype == MMR_F32 ? 4 : 2; }

static int set_segments(mmr_index* ix, const int64_t* seg, int32_t nseg) {
  ix->seg.clear();
  if (seg == nullptr || nseg <= 0) {
    ix->seg = {0, ix->n_rows};
    return MMR_OK;
  }
  ix->seg.assign(seg, seg + nseg + 1);
  if (ix->seg.front() < 0 || ix->seg.back() > ix->n_rows) return fail(MMR_ERR_INVALID, "segment offsets out of range");
  for (int i = 0; i < nseg; ++i)
    if (ix->seg[i] > ix->seg[i + 1]) return fail(MMR_ERR_INVALID, "segment offsets must be ascending");
  return MMR_OK;
}

// ------------------------------------------------------------------------------------------------ options
static int* option_slot(const char* name) {
  Options& o = options();
  if (!name) return nullptr;
  if (!strcmp(name, "MMR_PDL")) return &o.pdl;
  if (!strcmp(name, "MMR_ENC_FUSE_LN")) return &o.enc_fuse_ln;
  if (!strcmp(name, "MMR_ENC_ATT_MMA")) return &o.enc_att_mma;
  if (!strcmp(name, "MMR_ENC_GEMM_SMEM_KB")) return &o.enc_gemm_smem_kb;
  if (!strcmp(name, "MMR_ENC_NARROW_TILES")) return &o.enc_narrow_tiles;
  if (!strcmp(name, "MMR_INLINE_QUERY")) return &o.inline_query;
  if (!strcmp(name, "MMR_MAILBOX")) return &o.mailbox;
  return nullptr;
}
static int parse_option(const char* v, int dflt) {
  if (!v || !v[0]) return dflt;
  return atoi(v);
}
static const char* kOptionNames[] = {"MMR_PDL", "MMR_INLINE_QUERY", "MMR_MAILBOX", "MMR_ENC_FUSE_LN", "MMR_ENC_ATT_MMA",
                                     "MMR_ENC_GEMM_SMEM_KB", "MMR_ENC_NARROW_TILES"};
namespace {
struct OptionsFromEnv {  // the environment is read once, when the library is loaded
  OptionsFromEnv() {
    for (const char* name : kOptionNames) {
      int* slot = option_slot(name);
      *slot = parse_option(getenv(name), *slot);
    }
  }
} g_options_from_env;
}  // namespace

extern "C" int mmr_set_option(const char* name, const char* value) {
  int* slot = option_slot(name);
  if (!slot) return fail(MMR_ERR_INVALID, "unknown option %s", name ? name : "(null)");
  Options defaults;
  Options& o = options();
  const int dflt = *(reinterpret_cast<int*>(&defaults) + (slot - reinterpret_cast<int*>(&o)));
  *slot = parse_option(value, dflt);
  return MMR_OK;
}
extern "C" int mmr_get_option(const char* name) {
  int* slot = option_slot(name);
  return slot ? *slot : -1;
}

extern "C" int mmr_abi_version(void) { return MMR_ABI_VERSION; }
extern "C" const char* mmr_last_error(void) { return g_err.c_str(); }
extern "C" int64_t mmr_launch_count(void) { return g_launches.load(); }
extern "C" int mmr_last_kernel(void) { return g_last_kernel; }
extern "C" int64_t mmr_rescore_reruns(void) { return g_rescore_reruns.load(); }

extern "C" int mmr_device_sm_count(int device, int* out_sms) {
  if (!out_sms) return fail(MMR_ERR_INVALID, "out_sms is NULL");
  CUDA_TRY(cudaDeviceGetAttribute(out_sms, cudaDevAttrMultiProcessorCount, device));
  return MMR_OK;
}

extern "C" int mmr_index_create(int device, int dim, int dtype, int64_t n_rows, const void* rows_dev,
                                const int64_t* seg_offsets_host, int32_t n_segments, int64_t row_base,
                                mmr_index** out) {
  if (!out) return fail(MMR_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (dtype != MMR_BF16 && dtype != MMR_F32 && dtype != MMR_F16) return fail(MMR_ERR_INVALID, "unknown dtype %d", dtype);
  if (dim <= 0 || n_rows < 0) return fail(MMR_ERR_INVALID, "bad shape [%lld, %d]", (long long)n_rows, dim);
  if (n_rows >= (int64_t(1) << 32)) return fail(MMR_ERR_UNSUPPORTED, "at most 2^32-1 rows per resident index");
  if (n_rows > 0 && rows_dev == nullptr) return fail(MMR_ERR_INVALID, "rows_dev is NULL");
  if ((reinterpret_cast<uintptr_t>(rows_dev) & 15) != 0) return fail(MMR_ERR_INVALID, "rows_dev must be 16-byte aligned");
  if (dim != 384 && dim != 512)
    return fail(MMR_ERR_UNSUPPORTED, "dim %d: kernels are built for 384 (MiniLM) and 512 (CLIP)", dim);
  int major = 0, minor = 0, sms = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  CUDA_TRY(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  if (major != 10) return fail(MMR_ERR_CUDA, "device %d is sm_%d%d; this library is sm_100a only", device, major, minor);
  mmr_index* ix = new mmr_index();
  ix->device = device;
  ix->dim = dim;
  ix->dtype = dtype;
  ix->n_rows = n_rows;
  ix->rows = rows_dev;
  ix->row_base = row_base;
  ix->sm_count = sms;
  int rc = set_segments(ix, seg_offsets_host, n_segments);
  if (rc != MMR_OK) {
    delete ix;
    return rc;
  }
  *out = ix;
  return MMR_OK;
}

extern "C" int mmr_index_update(mmr_index* ix, int64_t n_rows, const void* rows_dev, const int64_t* seg, int32_t nseg) {
  if (!ix) return fail(MMR_ERR_INVALID, "index is NULL");
  if (n_rows < 0 || n_rows >= (int64_t(1) << 32)) return fail(MMR_ERR_INVALID, "bad n_rows");
  if (n_rows > 0 && rows_dev == nullptr) return fail(MMR_ERR_INVALID, "rows_dev is NULL");
  if ((reinterpret_cast<uintptr_t>(rows_dev) & 15) != 0) return fail(MMR_ERR_INVALID, "rows_dev must be 16-byte aligned");
  ix->n_rows = n_rows;
  ix->rows = rows_dev;
  ix->umma.valid = false;
  ix->umma2.valid = false;
  return set_segments(ix, seg, nseg);
}

static void free_staging(mmr_index* ix) {
  if (ix->h_flags) cudaFreeHost(ix->h_flags);
  ix->h_flags = nullptr;
  ix->flags_cap = 0;
  if (ix->h_q) cudaFreeHost(ix->h_q);
  if (ix->h_box) cudaFreeHost(ix->h_box);
  if (ix->d_q) cudaFree(ix->d_q);
  if (ix->d_ws) cudaFree(ix->d_ws);
  ix->h_q = ix->d_q = nullptr;
  ix->h_box = ix->d_box = nullptr;
  ix->d_ws = nullptr;
  ix->cap_b = ix->cap_k = 0;
}

extern "C" int mmr_index_destroy(mmr_index* ix) {
  if (!ix) return MMR_OK;
  cudaSetDevice(ix->device);
  free_staging(ix);
  delete ix;
  return MMR_OK;
}

extern "C" int mmr_index_set_query_precision(mmr_index* ix, int mode) {
  if (!ix) return fail(MMR_ERR_INVALID, "index is NULL");
  if (mode != MMR_QP_AUTO && mode != MMR_QP_F32 && mode != MMR_QP_RESCORE)
    return fail(MMR_ERR_INVALID, "unknown query precision %d", mode);
  ix->query_precision = mode;
  return MMR_OK;
}

// ------------------------------------------------------------------------------------------------ loader
template <typename E>
static int launch_convert(const float* src, void* dst, int64_t n, int dim, int normalize, cudaStream_t st,
                          const int64_t* dst_row = nullptr) {
  if (n == 0) return MMR_OK;
  const int threads = 256;
  const int64_t blocks = std::min<int64_t>((n + 7) / 8, 148 * 16);
  convert_rows_kernel<E><<<(unsigned)blocks, threads, 0, st>>>(src, reinterpret_cast<E*>(dst), n, dim, normalize, dst_row);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return MMR_OK;
}

static int convert_dispatch(const float* src_dev, void* dst_dev, int dtype, int64_t n_rows, int dim, int normalize,
                            cudaStream_t st, const int64_t* dst_row_dev) {
  switch (dtype) {
    case MMR_BF16: return launch_convert<__nv_bfloat16>(src_dev, dst_dev, n_rows, dim, normalize, st, dst_row_dev);
    case MMR_F16: return launch_convert<__half>(src_dev, dst_dev, n_rows, dim, normalize, st, dst_row_dev);
    case MMR_F32: return launch_convert<float>(src_dev, dst_dev, n_rows, dim, normalize, st, dst_row_dev);
  }
  return fail(MMR_ERR_INVALID, "unknown dtype %d", dtype);
}

extern "C" int mmr_convert_rows_f32(const float* src_dev, void* dst_dev, int dtype, int64_t n_rows, int dim,
                                    int normalize, void* stream) {
  if (n_rows < 0 || dim <= 0) return fail(MMR_ERR_INVALID, "bad shape");
  if (n_rows > 0 && (!src_dev || !dst_dev)) return fail(MMR_ERR_INVALID, "NULL buffer");
  return convert_dispatch(src_dev, dst_dev, dtype, n_rows, dim, normalize, static_cast<cudaStream_t>(stream), nullptr);
}

// Pageable host memory -> pinned staging with a few threads (one memcpy thread tops out near 10 GB/s, well under the
// PCIe gen5 link), double-buffered against the H2D copy + convert kernel of the previous chunk.
static void parallel_memcpy(void* dst, const void* src, size_t bytes, int threads) {
  if (threads <= 1 || bytes < (size_t(4) << 20)) {
    memcpy(dst, src, bytes);
    return;
  }
  std::vector<std::thread> pool;
  const size_t per = (bytes / threads + 4095) / 4096 * 4096;
  for (int t = 0; t < threads; ++t) {
    const size_t o = size_t(t) * per;
    if (o >= bytes) break;
    const size_t len = std::min(per, bytes - o);
    pool.emplace_back([=]() { memcpy(static_cast<uint8_t*>(dst) + o, static_cast<const uint8_t*>(src) + o, len); });
  }
  for (auto& th : pool) th.join();
}

extern "C" int mmr_load_rows_f32_host_scatter(int device, const float* src_host, void* dst_dev, int dtype, int64_t n_rows,
                                              int dim, int normalize, const int64_t* dst_row_host, void* stream) {
  if (n_rows < 0 || dim <= 0) return fail(MMR_ERR_INVALID, "bad shape");
  if (n_rows == 0) return MMR_OK;
  if (!src_host || !dst_dev) return fail(MMR_ERR_INVALID, "NULL buffer");
  if (dtype != MMR_BF16 && dtype != MMR_F32 && dtype != MMR_F16) return fail(MMR_ERR_INVALID, "unknown dtype %d", dtype);
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t chunk_rows = std::max<int64_t>(1, (int64_t(64) << 20) / (int64_t(dim) * 4));  // 64 MiB chunks
  const size_t chunk_bytes = size_t(chunk_rows) * dim * 4;
  const size_t map_bytes = dst_row_host ? size_t(chunk_rows) * 8 : 0;
  uint8_t* h[2] = {nullptr, nullptr};
  uint8_t* d[2] = {nullptr, nullptr};
  cudaEvent_t done[2] = {nullptr, nullptr};
  int rc = MMR_OK;
  auto cleanup = [&]() {
    for (int i = 0; i < 2; ++i) {
      if (h[i]) cudaFreeHost(h[i]);
      if (d[i]) cudaFree(d[i]);
      if (done[i]) cudaEventDestroy(done[i]);
    }
  };
  for (int i = 0; i < 2; ++i) {
    if (cudaMallocHost(&h[i], chunk_bytes + map_bytes) != cudaSuccess ||
        cudaMalloc(&d[i], chunk_bytes + map_bytes) != cudaSuccess ||
        cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming) != cudaSuccess) {
      cleanup();
      return fail(MMR_ERR_CUDA, "staging allocation of %zu bytes failed", chunk_bytes + map_bytes);
    }
  }
  const int threads = int(std::min<unsigned>(8u, std::max(1u, std::thread::hardware_concurrency() / 2)));
  int slot = 0;
  for (int64_t r0 = 0; r0 < n_rows && rc == MMR_OK; r0 += chunk_rows, slot ^= 1) {
    const int64_t nr = std::min(chunk_rows, n_rows - r0);
    const size_t bytes = size_t(nr) * dim * 4;
    cudaEventSynchronize(done[slot]);  // staging slot free again
    parallel_memcpy(h[slot], src_host + r0 * dim, bytes, threads);
    if (dst_row_host) memcpy(h[slot] + chunk_bytes, dst_row_host + r0, size_t(nr) * 8);
    // one copy when the row map rides along (it sits right behind the chunk in both staging buffers)
    const size_t copy_bytes = dst_row_host ? chunk_bytes + size_t(nr) * 8 : bytes;
    if (cudaMemcpyAsync(d[slot], h[slot], copy_bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) {
      rc = fail(MMR_ERR_CUDA, "H2D copy failed");
      break;
    }
    const int64_t* map_dev = dst_row_host ? reinterpret_cast<const int64_t*>(d[slot] + chunk_bytes) : nullptr;
    const int eb = elem_bytes(dtype);
    void* dst = dst_row_host ? dst_dev : static_cast<void*>(static_cast<uint8_t*>(dst_dev) + size_t(r0) * dim * eb);
    rc = convert_dispatch(reinterpret_cast<const float*>(d[slot]), dst, dtype, nr, dim, normalize, st, map_dev);
    cudaEventRecord(done[slot], st);
  }
  cudaStreamSynchronize(st);
  cleanup();
  return rc;
}

extern "C" int mmr_load_rows_f32_host(int device, const float* src_host, void* dst_dev, int dtype, int64_t n_rows,
                                      int dim, int normalize, void* stream) {
  return mmr_load_rows_f32_host_scatter(device, src_host, dst_dev, dtype, n_rows, dim, normalize, nullptr, stream);
}

// Host-side helper of the columnar store: 64-bit hashes of n strings held Arrow-style (one byte buffer + n+1 int32
// offsets).  The store keeps (hash, row) sorted to find the rows an upsert replaces (delete-by-chunk_id,
// lancedb_store.py:91-92) without a Python dict over millions of ids.
extern "C" int mmr_hash_strings(const uint8_t* data, const int32_t* offsets, int64_t n, uint64_t* out) {
  if (n < 0 || (n > 0 && (!offsets || !out))) return fail(MMR_ERR_INVALID, "bad arguments");
  for (int64_t i = 0; i < n; ++i) {
    const uint8_t* p = data + offsets[i];
    const int32_t len = offsets[i + 1] - offsets[i];
    uint64_t h = 0xcbf29ce484222325ull ^ (uint64_t(uint32_t(len)) * 0x9E3779B97F4A7C15ull);
    int32_t j = 0;
    for (; j + 8 <= len; j += 8) {
      uint64_t w;
      memcpy(&w, p + j, 8);
      h = (h ^ w) * 0x100000001b3ull;
      h ^= h >> 29;
    }
    uint64_t tail = 0;
    if (j < len) memcpy(&tail, p + j, size_t(len - j));
    h = (h ^ tail) * 0x100000001b3ull;
    h ^= h >> 32;  // final avalanche (murmur3 fmix64)
    h *= 0xff51afd7ed558ccdull;
    h ^= h >> 33;
    h *= 0xc4ceb9fe1a85ec53ull;
    h ^= h >> 33;
    out[i] = h;
  }
  return MMR_OK;
}

// ------------------------------------------------------------------------------------------------ K1 launch
template <typename E, int D, int NQ, int KPL>
static int launch_stream_t(const StreamParams& p, int grid, cudaStream_t st) {
  using C = StreamCfg<E, D, NQ, KPL>;
  static bool attr_set[64] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 0 && dev < 64 && !attr_set[dev]) {
    CUDA_TRY(cudaFuncSetAttribute(scan_stream_kernel<E, D, NQ, KPL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  C::SMEM_BYTES));
    attr_set[dev] = true;
  }
  // MMR_PDL=1 (opt-in): launch with programmatic stream serialization so consecutive searches on one stream overlap
  // tail and head.  Contract: the queries of a search must not be produced by the kernel launched immediately before
  // it on the same stream (the scan starts before that kernel's memory is guaranteed visible).
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(C::THREADS);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = (p.items == nullptr && options().pdl) ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CUDA_TRY(cudaLaunchKernelEx(&cfg, scan_stream_kernel<E, D, NQ, KPL>, p));
  g_launches++;
  return MMR_OK;
}

template <typename E, int D>
static int launch_stream_ed(const StreamParams& p, int nq_pad, int kpl, int grid, cudaStream_t st) {
#define MMR_CASE(NQ_, KPL_) \
  if (nq_pad == NQ_ && kpl == KPL_) return launch_stream_t<E, D, NQ_, KPL_>(p, grid, st);
  MMR_CASE(1, 1) MMR_CASE(1, 2) MMR_CASE(2, 1) MMR_CASE(2, 2) MMR_CASE(4, 1) MMR_CASE(4, 2)
  if constexpr (sizeof(E) == 4) {  // fp32 rows stream half as many rows per byte: 8 queries per pass stay HBM-bound
    MMR_CASE(8, 1) MMR_CASE(8, 2)
  }
#undef MMR_CASE
  return fail(MMR_ERR_UNSUPPORTED, "no stream kernel for nq=%d kpl=%d", nq_pad, kpl);
}

static int launch_stream(const mmr_index* ix, const StreamParams& p, int nq_pad, int kpl, int grid, cudaStream_t st) {
  const int key = ix->dtype * 1000 + ix->dim;
  switch (key) {
    case MMR_BF16 * 1000 + 512: return launch_stream_ed<__nv_bfloat16, 512>(p, nq_pad, kpl, grid, st);
    case MMR_BF16 * 1000 + 384: return launch_stream_ed<__nv_bfloat16, 384>(p, nq_pad, kpl, grid, st);
    case MMR_F16 * 1000 + 512: return launch_stream_ed<__half, 512>(p, nq_pad, kpl, grid, st);
    case MMR_F16 * 1000 + 384: return launch_stream_ed<__half, 384>(p, nq_pad, kpl, grid, st);
    case MMR_F32 * 1000 + 512: return launch_stream_ed<float, 512>(p, nq_pad, kpl, grid, st);
    case MMR_F32 * 1000 + 384: return launch_stream_ed<float, 384>(p, nq_pad, kpl, grid, st);
  }
  return fail(MMR_ERR_UNSUPPORTED, "no stream kernel for dtype %d dim %d", ix->dtype, ix->dim);
}

// ------------------------------------------------------------------------------------------------ planning
// Workspace layout (bytes):
//   [0, 256)                          control block (two counters at +0: K1 arrival ticket / K6 claim + done)
//   [256, 256 + PART)                 partial top-k keys  (uniform: grid*8*k u64; varlen: n_items*K1_ITEM_NQ*k u64)
//   then (varlen only)                ScanItem[n_items], QuerySlot[B]
//   last                              the K2 slice (umma_workspace_bytes)
static constexpr size_t WS_CTRL = 256;
#ifndef MMR_VARLEN_ITEMS_PER_CTA
#define MMR_VARLEN_ITEMS_PER_CTA 8
#endif
static constexpr int VARLEN_ITEMS_PER_CTA = MMR_VARLEN_ITEMS_PER_CTA;   // varlen work items are per CTA (its eight warps interleave an item's chunks)
static constexpr int RANGES_PER_QUERY_BUDGET = 8;  // = B200Store's MAX_RANGES: a tenant is compacted before it owns more

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Upper bound of the varlen plan: ~VARLEN_ITEMS_PER_CTA pieces per CTA plus one (possibly short) piece per row range.
static int64_t varlen_item_cap(const mmr_index* ix, int64_t n_ranges) {
  return int64_t(ix->sm_count) * VARLEN_ITEMS_PER_CTA + n_ranges + 64;
}

// The tensor-core slice at the END of the workspace: K2's own buffers sized for the largest k (the rescoring mode runs K2
// with more candidates than the caller's k), then the rescoring buffers: candidate scores / rows [B, 64], ||q - q16|| [B],
// exact flags [B].
static size_t rescore_extra_bytes(int B) {
  return align_up(size_t(B) * MMR_MAX_K * 4, 256) + align_up(size_t(B) * MMR_MAX_K * 8, 256) + align_up(size_t(B) * 4, 256) +
         align_up(size_t(B), 256);
}
static size_t k2_slice_bytes(const mmr_index* ix, int B) {
  return umma_workspace_bytes(ix->sm_count, ix->dim, B, MMR_MAX_K) + rescore_extra_bytes(B);
}

static size_t workspace_bytes_for(const mmr_index* ix, int32_t B, int32_t k, int64_t n_ranges) {
  if (!ix || B <= 0 || k <= 0) return 0;
  const size_t kk = size_t(std::min<int32_t>(k, MMR_MAX_K));
  const size_t uniform = size_t(ix->sm_count) * 8 * kk * 8;
  const size_t items = size_t(varlen_item_cap(ix, n_ranges));
  const size_t varlen = align_up(items * K1_ITEM_NQ * kk * 8, 256) + align_up(items * sizeof(ScanItem), 256) +
                        align_up(size_t(B) * sizeof(QuerySlot), 256);
  size_t total = WS_CTRL + align_up(std::max(uniform, varlen), 256);
  total += k2_slice_bytes(ix, B);
  return total;
}

extern "C" size_t mmr_search_workspace_bytes(const mmr_index* ix, int32_t B, int32_t k) {
  return workspace_bytes_for(ix, B, k, int64_t(RANGES_PER_QUERY_BUDGET) * std::max(B, 0));
}
extern "C" size_t mmr_search_ranges_workspace_bytes(const mmr_index* ix, int32_t B, int32_t k, int64_t n_ranges) {
  return workspace_bytes_for(ix, B, k, std::max<int64_t>(n_ranges, 0));
}

struct ExchangeInfo {  // fused push by K1's last CTA (only when one launch covers all B queries)
  int n_peers = 0;
  uint32_t seq = 0;
  uint32_t wire_score_bytes = 0;
  uint64_t slot[MMR_MAX_PEERS] = {};
  uint64_t flag[MMR_MAX_PEERS] = {};
};

struct QuerySrc {   // where the fp32 queries are: device memory, or host memory to be carried in the kernel parameters
  const float* dev = nullptr;
  const float* host = nullptr;
};
struct Completion {  // optional mailbox flag (mapped host memory) released by the kernel that writes the final result
  uint32_t* flag_dev = nullptr;
  uint32_t seq = 0;
  bool armed = false;  // set by the launcher when the flag will really be written (single-launch paths only)
};

static int k1_group(const mmr_index* ix) { return ix->dtype == MMR_F32 ? 8 : 4; }  // queries per pass

static bool can_inline(const mmr_index* ix, int B) {
  return options().inline_query && B * ix->dim <= K1_INLINE_FLOATS && B <= 2;
}

static int search_uniform_stream(const mmr_index* ix, QuerySrc q, int B, int k, uint32_t r0, uint32_t r1,
                                 float* out_s, int64_t* out_r, uint8_t* ws, cudaStream_t st,
                                 const ExchangeInfo* xi = nullptr, Completion* done = nullptr) {
  const int kpl = k <= 32 ? 1 : 2;
  const int R = MMR_K1_ROWS;
  const int64_t nchunks = (int64_t(r1) - r0 + R - 1) / R;
  int grid = int(std::min<int64_t>(ix->sm_count, std::max<int64_t>(1, (nchunks + K1_NW - 1) / K1_NW)));
  const int group = k1_group(ix);
  if (q.dev == nullptr && !(q.host && can_inline(ix, B))) return fail(MMR_ERR_INVALID, "queries must be device-resident for this batch size");
  for (int q0 = 0; q0 < B; q0 += group) {
    const int nq = std::min(group, B - q0);
    const int nq_pad = nq <= 2 ? nq : (nq <= 4 ? 4 : 8);
    StreamParams p;
    memset(&p, 0, offsetof(StreamParams, qinline));
    p.rows = ix->rows;
    p.queries = q.dev;
    if (q.dev == nullptr) memcpy(p.qinline, q.host, size_t(B) * ix->dim * sizeof(float));
    p.q_first = q0;
    p.nq = nq;
    p.k = k;
    p.row_begin = r0;
    p.row_end = r1;
    p.partial = reinterpret_cast<uint64_t*>(ws + WS_CTRL);
    p.ticket = reinterpret_cast<unsigned int*>(ws);
    p.out_scores = out_s;
    p.out_rows = out_r;
    p.row_base = ix->row_base;
    if (B <= group) {  // one launch covers the batch: it may push to peers / ring the mailbox itself
      if (xi) {
        p.n_peers = xi->n_peers;
        p.seq = xi->seq;
        p.wire_score_bytes = xi->wire_score_bytes;
        for (int g = 0; g < xi->n_peers; ++g) {
          p.peer_slot[g] = xi->slot[g];
          p.peer_flag[g] = xi->flag[g];
        }
      }
      if (done && done->flag_dev && options().mailbox) {
        p.done_flag = done->flag_dev;
        p.done_seq = done->seq;
        done->armed = true;
      }
    }
    int rc = launch_stream(ix, p, nq_pad, kpl, grid, st);
    if (rc != MMR_OK) return rc;
  }
  g_last_kernel = 1;
  return MMR_OK;
}

// K6 -- the grouped varlen launch.  `ranges[b]` = the row ranges query b scans (a tenant is one base segment plus any
// appended delta segments).  Queries with identical range lists (= the same tenant) are grouped K1_ITEM_NQ at a time, and
// every work item is (one piece of one range, one query group): the rows of a tenant are read once per GROUP, not once
// per query (SURVEY 2.1 K6).  Scores are computed exactly as in the uniform K1 kernel (fp32 queries, same per-row
// arithmetic), so a request's result does not depend on what it was batched with.
typedef std::vector<std::pair<uint32_t, uint32_t>> RangeList;

static int search_varlen_stream(const mmr_index* ix, const float* q, const std::vector<RangeList>& ranges, int k,
                                float* out_s, int64_t* out_r, uint8_t* ws, size_t ws_bytes, cudaStream_t st) {
  const int B = int(ranges.size());
  const int kpl = k <= 32 ? 1 : 2;
  const int R = MMR_K1_ROWS;
  // 1. group the queries by range list (first-appearance order keeps the plan deterministic)
  std::map<RangeList, int> tenant_of;
  std::vector<std::vector<int>> members;
  std::vector<const RangeList*> tenant_ranges;
  for (int b = 0; b < B; ++b) {
    auto it = tenant_of.find(ranges[b]);
    if (it == tenant_of.end()) {
      it = tenant_of.emplace(ranges[b], int(members.size())).first;
      members.emplace_back();
      tenant_ranges.push_back(&it->first);
    }
    members[it->second].push_back(b);
  }
  // 2. size the pieces: about VARLEN_ITEMS_PER_CTA per CTA over everything this launch reads
  int64_t total_rows = 0, n_group_ranges = 0;
  for (size_t t = 0; t < members.size(); ++t) {
    const int64_t ngroups = (int64_t(members[t].size()) + K1_ITEM_NQ - 1) / K1_ITEM_NQ;
    for (auto& r : *tenant_ranges[t]) total_rows += (int64_t(r.second) - r.first) * ngroups;
    n_group_ranges += int64_t(tenant_ranges[t]->size()) * ngroups;
  }
  const int64_t target = int64_t(ix->sm_count) * VARLEN_ITEMS_PER_CTA;
  int64_t item_rows = std::max<int64_t>(64 * K1_NW, (total_rows + target - 1) / target);
  item_rows = (item_rows + R - 1) / R * R;
  // 3. emit items and per-query slots.  Three classes by group size -- 1 query (NQ = 1 instantiation: streams at the HBM
  //    roofline), 2 queries (NQ = 2), 3..4 queries (NQ = 4: four dot products per row byte, the slowest stream) -- so a batch
  //    that mostly hits distinct tenants does not pay the 4-query arithmetic on every row.
  constexpr int N_CLS = 3;
  static const int cls_nq[N_CLS] = {1, 2, K1_ITEM_NQ};
  std::vector<ScanItem> cls_items[N_CLS];
  std::vector<QuerySlot> slots(B);
  std::vector<int> slot_cls(B, 0);
  cls_items[0].reserve(size_t(std::min<int64_t>(target + n_group_ranges, 1 << 22)));
  for (size_t t = 0; t < members.size(); ++t) {
    const std::vector<int>& m = members[t];
    for (size_t g0 = 0; g0 < m.size(); g0 += K1_ITEM_NQ) {
      const int nq = int(std::min<size_t>(K1_ITEM_NQ, m.size() - g0));
      const int cls = nq == 1 ? 0 : nq == 2 ? 1 : 2;
      std::vector<ScanItem>& dst = cls_items[cls];
      const int item0 = int(dst.size());
      for (auto& r : *tenant_ranges[t]) {
        for (int64_t s = r.first; s < int64_t(r.second); s += item_rows) {
          ScanItem it;
          it.row_begin = uint32_t(s);
          it.row_end = uint32_t(std::min<int64_t>(s + item_rows, r.second));
          for (int j = 0; j < K1_ITEM_NQ; ++j) it.query[j] = m[g0 + std::min(j, nq - 1)];
          it.nq = nq;
          it.out = int(dst.size());   // list group inside its class; rebased below
          dst.push_back(it);
        }
      }
      for (int j = 0; j < nq; ++j) {
        slots[m[g0 + j]] = QuerySlot{item0, int(dst.size()) - item0, j, 0};
        slot_cls[m[g0 + j]] = cls;
      }
    }
  }
  int cls_first[N_CLS + 1] = {0};
  for (int c = 0; c < N_CLS; ++c) cls_first[c + 1] = cls_first[c] + int(cls_items[c].size());
  for (int b = 0; b < B; ++b) slots[b].item0 += cls_first[slot_cls[b]];
  // launch order inside a class: largest piece first (the kernel's CTAs claim items dynamically in this order, so the
  // launch ends on the smallest pieces); `out` keeps every item's lists where the query slots expect them
  auto by_size = [](const ScanItem& a, const ScanItem& b) { return a.row_end - a.row_begin > b.row_end - b.row_begin; };
  std::vector<ScanItem> items;
  items.reserve(size_t(cls_first[N_CLS]));
  for (int c = 0; c < N_CLS; ++c) {
    for (auto& it : cls_items[c]) it.out += cls_first[c];
    std::stable_sort(cls_items[c].begin(), cls_items[c].end(), by_size);
    items.insert(items.end(), cls_items[c].begin(), cls_items[c].end());
  }
  const int n_items = int(items.size());
  const size_t part_bytes = align_up(size_t(std::max(n_items, 1)) * K1_ITEM_NQ * k * 8, 256);
  const size_t item_bytes = align_up(size_t(std::max(n_items, 1)) * sizeof(ScanItem), 256);
  const size_t slot_bytes = align_up(size_t(B) * sizeof(QuerySlot), 256);
  const size_t k2_bytes = k2_slice_bytes(ix, B);
  if (WS_CTRL + part_bytes + item_bytes + slot_bytes + k2_bytes > ws_bytes)
    return fail(MMR_ERR_WORKSPACE,
                "workspace too small for %d work items over %lld row ranges: size it with "
                "mmr_search_ranges_workspace_bytes(index, B, k, n_ranges)", n_items, (long long)n_group_ranges);
  uint64_t* d_part = reinterpret_cast<uint64_t*>(ws + WS_CTRL);
  ScanItem* d_items = reinterpret_cast<ScanItem*>(ws + WS_CTRL + part_bytes);
  QuerySlot* d_slots = reinterpret_cast<QuerySlot*>(ws + WS_CTRL + part_bytes + item_bytes);
  // pageable sources: cudaMemcpyAsync stages them before returning, the vectors may die after this call
  if (n_items > 0) CUDA_TRY(cudaMemcpyAsync(d_items, items.data(), size_t(n_items) * sizeof(ScanItem), cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(d_slots, slots.data(), size_t(B) * sizeof(QuerySlot), cudaMemcpyHostToDevice, st));
  for (int cls = 0; cls < N_CLS; ++cls) {
    const int first = cls_first[cls];
    const int count = cls_first[cls + 1] - first;
    if (count <= 0) continue;
    const int nq_launch = cls_nq[cls];
    StreamParams p;
    memset(&p, 0, offsetof(StreamParams, qinline));
    p.rows = ix->rows;
    p.queries = q;
    p.nq = nq_launch;
    p.k = k;
    p.partial = d_part;   // indexed by ScanItem::out
    p.ticket = reinterpret_cast<unsigned int*>(ws);
    p.row_base = ix->row_base;
    p.items = d_items + first;
    p.n_items = count;
    p.item_nq = K1_ITEM_NQ;
    const int grid = int(std::min<int64_t>(ix->sm_count, count));
    int rc = launch_stream(ix, p, nq_launch, kpl, grid, st);
    if (rc != MMR_OK) return rc;
  }
  const int wpb = 4;
  if (kpl == 1)
    merge_items_kernel<1><<<(B + wpb - 1) / wpb, wpb * 32, 0, st>>>(d_part, d_slots, B, K1_ITEM_NQ, k, out_s, out_r, ix->row_base);
  else
    merge_items_kernel<2><<<(B + wpb - 1) / wpb, wpb * 32, 0, st>>>(d_part, d_slots, B, K1_ITEM_NQ, k, out_s, out_r, ix->row_base);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  g_last_kernel = 3;
  return MMR_OK;
}

template <typename E, int D>
static void launch_rescore_ed(const mmr_index* ix, const float* q, const float* cs, const int64_t* cr, const float* qerr, int B,
                              int kc, int k, float* out_s, int64_t* out_r, uint8_t* flags, cudaStream_t st) {
  if (k <= 32)
    rescore_kernel<E, D, 1><<<B, 256, 0, st>>>(ix->rows, q, cs, cr, qerr, kc, k, ix->row_base, out_s, out_r, flags);
  else
    rescore_kernel<E, D, 2><<<B, 256, 0, st>>>(ix->rows, q, cs, cr, qerr, kc, k, ix->row_base, out_s, out_r, flags);
}

// MMR_QP_RESCORE: the tensor cores nominate kc candidates per query, rescore_kernel re-scores them with the fp32 query in
// K1's arithmetic and proves the top-k exact; unproven queries (rare) are rerun on K1.  The result is bit-identical to
// searching every query alone -- at the price of one stream synchronisation inside the call (the flags are read on the host).
static int search_rescored(const mmr_index* ix, const float* q, int B, int k, uint32_t r0, uint32_t r1, float* out_s,
                           int64_t* out_r, uint8_t* ws, size_t ws_total, cudaStream_t st) {
  const int kc = k <= 16 ? 32 : MMR_MAX_K;
  uint8_t* slice = ws + ws_total - k2_slice_bytes(ix, B);
  uint8_t* extra = slice + umma_workspace_bytes(ix->sm_count, ix->dim, B, MMR_MAX_K);
  float* cand_s = reinterpret_cast<float*>(extra);
  int64_t* cand_r = reinterpret_cast<int64_t*>(extra + align_up(size_t(B) * MMR_MAX_K * 4, 256));
  float* qerr = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(cand_r) + align_up(size_t(B) * MMR_MAX_K * 8, 256));
  uint8_t* flags = reinterpret_cast<uint8_t*>(qerr) + align_up(size_t(B) * 4, 256);
  int rc = umma_search(ix->umma, ix->umma2, ix->rows, ix->n_rows, ix->dim, ix->dtype, ix->sm_count, q, B, kc, r0, r1,
                       ix->row_base, cand_s, cand_r, slice, st, g_err, nullptr, 0, qerr);
  if (rc != MMR_OK) return rc;
  g_launches += umma_launches_per_search();
  if (ix->dtype == MMR_BF16 && ix->dim == 512) launch_rescore_ed<__nv_bfloat16, 512>(ix, q, cand_s, cand_r, qerr, B, kc, k, out_s, out_r, flags, st);
  else if (ix->dtype == MMR_BF16) launch_rescore_ed<__nv_bfloat16, 384>(ix, q, cand_s, cand_r, qerr, B, kc, k, out_s, out_r, flags, st);
  else if (ix->dim == 512) launch_rescore_ed<__half, 512>(ix, q, cand_s, cand_r, qerr, B, kc, k, out_s, out_r, flags, st);
  else launch_rescore_ed<__half, 384>(ix, q, cand_s, cand_r, qerr, B, kc, k, out_s, out_r, flags, st);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  if (ix->flags_cap < B) {
    if (ix->h_flags) cudaFreeHost(ix->h_flags);
    ix->h_flags = nullptr;
    CUDA_TRY(cudaMallocHost(&ix->h_flags, size_t(std::max(B, 1024))));
    ix->flags_cap = std::max(B, 1024);
  }
  CUDA_TRY(cudaMemcpyAsync(ix->h_flags, flags, size_t(B), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  g_last_kernel = 2;
  int reruns = 0;
  for (int b = 0; b < B; ++b) {
    if (ix->h_flags[b]) continue;
    QuerySrc one;
    one.dev = q + size_t(b) * ix->dim;
    rc = search_uniform_stream(ix, one, 1, k, r0, r1, out_s + size_t(b) * k, out_r + size_t(b) * k, ws, st);
    if (rc != MMR_OK) return rc;
    ++reruns;
  }
  g_last_kernel = 2;
  g_rescore_reruns += reruns;
  return MMR_OK;
}

// One shared row range for the whole batch: K2 when allowed and preferred, else K1 passes.
static int search_uniform(const mmr_index* ix, QuerySrc q, int B, int k, uint32_t r0, uint32_t r1, float* out_s,
                          int64_t* out_r, uint8_t* ws, size_t ws_total, cudaStream_t st, const ExchangeInfo* xi = nullptr,
                          Completion* done = nullptr) {
  if (q.dev != nullptr && ix->query_precision != MMR_QP_F32 &&
      umma_preferred(ix->dtype, ix->dim, B, k, int64_t(r1) - r0)) {
    if (ix->query_precision == MMR_QP_RESCORE)
      return search_rescored(ix, q.dev, B, k, r0, r1, out_s, out_r, ws, ws_total, st);
    int rc = umma_search(ix->umma, ix->umma2, ix->rows, ix->n_rows, ix->dim, ix->dtype, ix->sm_count, q.dev, B, k, r0, r1,
                         ix->row_base, out_s, out_r, ws + ws_total - k2_slice_bytes(ix, B), st, g_err);
    if (rc == MMR_OK) {
      g_launches += umma_launches_per_search();
      g_last_kernel = 2;
    }
    return rc;
  }
  return search_uniform_stream(ix, q, B, k, r0, r1, out_s, out_r, ws, st, xi, done);
}

// true when a uniform batch of B queries would run on the tensor-core family
static bool uniform_takes_k2(const mmr_index* ix, int B, int k, int64_t nrows) {
  return ix->query_precision != MMR_QP_F32 && umma_preferred(ix->dtype, ix->dim, B, k, nrows);
}

static int check_search_args(const mmr_index* ix, int32_t B, int32_t k) {
  if (!ix) return fail(MMR_ERR_INVALID, "index is NULL");
  if (B <= 0) return fail(MMR_ERR_INVALID, "B must be >= 1");
  if (k < 1 || k > MMR_MAX_K) return fail(MMR_ERR_INVALID, "k must be in [1, %d]", MMR_MAX_K);
  return MMR_OK;
}

// segment ids -> one range per query; `uniform` = everybody scans the same range
static int ranges_from_segments(const mmr_index* ix, const int32_t* query_seg_host, int B, std::vector<RangeList>& out,
                                bool& uniform) {
  const int nseg = int(ix->seg.size()) - 1;
  out.assign(B, RangeList(1));
  uniform = true;
  for (int b = 0; b < B; ++b) {
    const int s = query_seg_host ? query_seg_host[b] : -1;
    if (s < -1 || s >= nseg) return fail(MMR_ERR_INVALID, "query %d: segment %d out of range [0, %d)", b, s, nseg);
    out[b][0] = s < 0 ? std::make_pair(uint32_t(0), uint32_t(ix->n_rows))
                      : std::make_pair(uint32_t(ix->seg[s]), uint32_t(ix->seg[s + 1]));
    if (out[b][0] != out[0][0]) uniform = false;
  }
  return MMR_OK;
}

extern "C" int mmr_search(const mmr_index* ix, const float* queries_dev, const int32_t* query_seg_host, int32_t B,
                          int32_t k, float* out_scores_dev, int64_t* out_rows_dev, void* workspace_dev,
                          size_t workspace_bytes, void* stream) {
  int rc = check_search_args(ix, B, k);
  if (rc != MMR_OK) return rc;
  if (!queries_dev || !out_scores_dev || !out_rows_dev || !workspace_dev) return fail(MMR_ERR_INVALID, "NULL buffer");
  const size_t need = workspace_bytes_for(ix, B, k, B);
  if (workspace_bytes < need) return fail(MMR_ERR_WORKSPACE, "workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
  std::vector<RangeList> ranges;
  bool uniform = true;
  rc = ranges_from_segments(ix, query_seg_host, B, ranges, uniform);
  if (rc != MMR_OK) return rc;
  QuerySrc q;
  q.dev = queries_dev;
  if (uniform)
    return search_uniform(ix, q, B, k, ranges[0][0].first, ranges[0][0].second, out_scores_dev, out_rows_dev, ws,
                          workspace_bytes, st);
  return search_varlen_stream(ix, queries_dev, ranges, k, out_scores_dev, out_rows_dev, ws, workspace_bytes, st);
}

// Explicit row ranges per query: query b scans ranges[range_off[b] .. range_off[b+1]) (pairs of [begin, end) row
// ordinals).  Used by stores that append delta segments between compactions.
static int parse_ranges(const mmr_index* ix, int B, const int32_t* range_off_host, const int64_t* ranges_host,
                        std::vector<RangeList>& per_query, bool& single_shared) {
  per_query.assign(B, RangeList());
  single_shared = true;
  for (int b = 0; b < B; ++b) {
    if (range_off_host[b + 1] < range_off_host[b]) return fail(MMR_ERR_INVALID, "range offsets must be ascending");
    for (int32_t r = range_off_host[b]; r < range_off_host[b + 1]; ++r) {
      const int64_t lo = ranges_host[2 * r], hi = ranges_host[2 * r + 1];
      if (lo < 0 || hi < lo || hi > ix->n_rows)
        return fail(MMR_ERR_INVALID, "query %d: bad row range [%lld, %lld)", b, (long long)lo, (long long)hi);
      if (hi > lo) per_query[b].push_back({uint32_t(lo), uint32_t(hi)});
    }
    // a row must not be offered twice to one query (the warp top-k assumes distinct keys): reject overlapping ranges
    RangeList sorted = per_query[b];
    std::sort(sorted.begin(), sorted.end());
    for (size_t i = 1; i < sorted.size(); ++i)
      if (sorted[i].first < sorted[i - 1].second)
        return fail(MMR_ERR_INVALID, "query %d: row ranges [%u, %u) and [%u, %u) overlap", b, sorted[i - 1].first,
                    sorted[i - 1].second, sorted[i].first, sorted[i].second);
    if (per_query[b].size() != 1 || per_query[b] != per_query[0]) single_shared = false;
  }
  return MMR_OK;
}

extern "C" int mmr_search_ranges(const mmr_index* ix, const float* queries_dev, int32_t B, int32_t k,
                                 const int32_t* range_off_host, const int64_t* ranges_host, float* out_scores_dev,
                                 int64_t* out_rows_dev, void* workspace_dev, size_t workspace_bytes, void* stream) {
  int rc = check_search_args(ix, B, k);
  if (rc != MMR_OK) return rc;
  if (!queries_dev || !range_off_host || !out_scores_dev || !out_rows_dev || !workspace_dev)
    return fail(MMR_ERR_INVALID, "NULL buffer");
  if (workspace_bytes < workspace_bytes_for(ix, B, k, 0)) return fail(MMR_ERR_WORKSPACE, "workspace too small");
  std::vector<RangeList> per_query;
  bool single_shared = true;
  rc = parse_ranges(ix, B, range_off_host, ranges_host, per_query, single_shared);
  if (rc != MMR_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* ws = static_cast<uint8_t*>(workspace_dev);
  QuerySrc q;
  q.dev = queries_dev;
  if (single_shared)  // everyone scans the same single range: the uniform kernels apply
    return search_uniform(ix, q, B, k, per_query[0][0].first, per_query[0][0].second, out_scores_dev, out_rows_dev, ws,
                          workspace_bytes, st);
  return search_varlen_stream(ix, queries_dev, per_query, k, out_scores_dev, out_rows_dev, ws, workspace_bytes, st);
}

// ------------------------------------------------------------------------------------------------ host-buffer calls
// Mailbox layout inside h_box / d_box (mapped pinned memory, same bytes seen by both sides):
static constexpr size_t BOX_HEADER = 64;
static size_t box_rows_off(int B, int k) { return BOX_HEADER + align_up(size_t(B) * k * 4, 16); }

static int ensure_staging(mmr_index* ix, int B, int k) {
  if (B <= ix->cap_b && k <= ix->cap_k) return MMR_OK;
  free_staging(ix);
  const int cb = std::max(B, 8), ck = std::max(k, 16);
  const size_t box_bytes = box_rows_off(cb, ck) + size_t(cb) * ck * 8;
  CUDA_TRY(cudaMallocHost(&ix->h_q, size_t(cb) * ix->dim * 4));
  CUDA_TRY(cudaMalloc(&ix->d_q, size_t(cb) * ix->dim * 4));
  CUDA_TRY(cudaHostAlloc(&ix->h_box, box_bytes, cudaHostAllocMapped));
  CUDA_TRY(cudaHostGetDevicePointer(reinterpret_cast<void**>(&ix->d_box), ix->h_box, 0));
  memset(ix->h_box, 0, box_bytes);
  ix->ws_bytes = workspace_bytes_for(ix, cb, ck, int64_t(RANGES_PER_QUERY_BUDGET) * cb);
  CUDA_TRY(cudaMalloc(&ix->d_ws, ix->ws_bytes));
  CUDA_TRY(cudaMemset(ix->d_ws, 0, ix->ws_bytes));
  ix->cap_b = cb;
  ix->cap_k = ck;
  return MMR_OK;
}

static inline void cpu_relax() {
#if defined(__x86_64__)
  _mm_pause();
#endif
}

// Wait for the mailbox flag to reach `seq`.  The kernel releases it at system scope right after its result stores, so
// the host sees the result a PCIe write later instead of after a stream synchronisation.  The stream is polled now and
// then so that a faulted kernel turns into an error instead of an endless spin.
static int wait_mailbox(mmr_index* ix, uint32_t seq, cudaStream_t st) {
  volatile uint32_t* flag = reinterpret_cast<volatile uint32_t*>(ix->h_box);
  for (uint64_t spins = 1;; ++spins) {
    if (*flag == seq) break;
    if ((spins & 4095) == 0) {
      cudaError_t e = cudaStreamQuery(st);
      if (e == cudaSuccess) {
        if (*flag == seq) break;
        return fail(MMR_ERR_CUDA, "search finished without ringing its mailbox");
      }
      if (e != cudaErrorNotReady) return fail(MMR_ERR_CUDA, "search failed: %s", cudaGetErrorString(e));
    }
    cpu_relax();
  }
  std::atomic_thread_fence(std::memory_order_acquire);
  return MMR_OK;
}

// Shared tail of the host-buffer calls: results are in the mailbox (written by the kernels through the mapped
// pointer); wait (flag or stream), then hand them to the caller.
static int finish_host_call(mmr_index* ix, const Completion& done, int B, int k, float* out_scores_host,
                            int64_t* out_rows_host, cudaStream_t st) {
  if (done.armed) {
    int rc = wait_mailbox(ix, done.seq, st);
    if (rc != MMR_OK) return rc;
  } else {
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  memcpy(out_scores_host, ix->h_box + BOX_HEADER, size_t(B) * k * 4);
  memcpy(out_rows_host, ix->h_box + box_rows_off(B, k), size_t(B) * k * 8);
  return MMR_OK;
}

extern "C" int mmr_search_host(mmr_index* ix, const float* queries_host, const int32_t* query_seg_host, int32_t B,
                               int32_t k, float* out_scores_host, int64_t* out_rows_host, void* stream) {
  int rc = check_search_args(ix, B, k);
  if (rc != MMR_OK) return rc;
  if (!queries_host || !out_scores_host || !out_rows_host) return fail(MMR_ERR_INVALID, "NULL buffer");
  std::lock_guard<std::mutex> guard(ix->host_mu);   // one staging set per index: concurrent callers take turns
  CUDA_TRY(cudaSetDevice(ix->device));
  rc = ensure_staging(ix, B, k);
  if (rc != MMR_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::vector<RangeList> ranges;
  bool uniform = true;
  rc = ranges_from_segments(ix, query_seg_host, B, ranges, uniform);
  if (rc != MMR_OK) return rc;
  float* box_s = reinterpret_cast<float*>(ix->d_box + BOX_HEADER);
  int64_t* box_r = reinterpret_cast<int64_t*>(ix->d_box + box_rows_off(B, k));
  Completion done;
  done.flag_dev = reinterpret_cast<uint32_t*>(ix->d_box);
  done.seq = ++ix->box_seq ? ix->box_seq : ++ix->box_seq;   // never 0
  const uint32_t r0 = ranges[0][0].first, r1 = ranges[0][0].second;
  if (uniform && can_inline(ix, B) && !uniform_takes_k2(ix, B, k, int64_t(r1) - r0)) {
    // the latency path of a single request: ONE launch carries the query in its parameters, the kernel's last CTA
    // writes the result and the flag into the mailbox -- no H2D copy, no D2H copy, no stream synchronisation
    QuerySrc q;
    q.host = queries_host;
    rc = search_uniform_stream(ix, q, B, k, r0, r1, box_s, box_r, static_cast<uint8_t*>(ix->d_ws), st, nullptr, &done);
  } else {
    memcpy(ix->h_q, queries_host, size_t(B) * ix->dim * 4);
    CUDA_TRY(cudaMemcpyAsync(ix->d_q, ix->h_q, size_t(B) * ix->dim * 4, cudaMemcpyHostToDevice, st));
    QuerySrc q;
    q.dev = ix->d_q;
    if (uniform)
      rc = search_uniform(ix, q, B, k, r0, r1, box_s, box_r, static_cast<uint8_t*>(ix->d_ws), ix->ws_bytes, st, nullptr, &done);
    else
      rc = search_varlen_stream(ix, ix->d_q, ranges, k, box_s, box_r, static_cast<uint8_t*>(ix->d_ws), ix->ws_bytes, st);
  }
  if (rc != MMR_OK) return rc;
  return finish_host_call(ix, done, B, k, out_scores_host, out_rows_host, st);
}

// ------------------------------------------------------------------------------------------------ fused exchange
static uint32_t xchg_score_bytes(int B, int k) { return uint32_t((size_t(B) * k * 4 + 7) / 8 * 8); }
static uint32_t xchg_wire_bytes(int B, int k) { return uint32_t((xchg_score_bytes(B, k) + size_t(B) * k * 8 + 15) / 16 * 16); }

extern "C" size_t mmr_exchange_buffer_bytes(int32_t G, int32_t B, int32_t k) {
  if (G <= 0 || G > MMR_XCHG_MAX_PEERS || B <= 0 || k <= 0) return 0;
  return size_t(MMR_XCHG_HEADER) + size_t(2) * G * xchg_wire_bytes(B, k);
}

extern "C" size_t mmr_search_exchange_workspace_bytes(const mmr_index* ix, int32_t B, int32_t k) {
  const size_t base = mmr_search_workspace_bytes(ix, B, k);
  return base ? base + align_up(xchg_wire_bytes(B, std::min<int32_t>(k, MMR_MAX_K)), 256) : 0;
}

// The exchange proper.  push_mask: which peers receive this rank's result (bit g); do_merge: whether this rank waits for
// all G slots and merges (every rank in the SPMD form; only the collecting device in the single-process form).
// Exactly one of {per_query ranges, uniform range} describes what is scanned.
static int exchange_impl(const mmr_index* ix, QuerySrc q, int B, int k, bool uniform, uint32_t r0, uint32_t r1,
                         const std::vector<RangeList>* per_query, const uint64_t* peer_bufs, int G, int rank, uint32_t seq,
                         uint32_t push_mask, bool do_merge, float* out_s, int64_t* out_r, uint8_t* ws, size_t base_ws,
                         cudaStream_t st, Completion* done) {
  const uint32_t score_bytes = xchg_score_bytes(B, k), wire_bytes = xchg_wire_bytes(B, k);
  const int parity = int(seq & 1u);
  uint8_t* wire = ws + base_ws;  // this rank's own result, [scores | rows]
  float* w_scores = reinterpret_cast<float*>(wire);
  int64_t* w_rows = reinterpret_cast<int64_t*>(wire + score_bytes);
  ExchangeInfo xi;
  xi.seq = seq;
  xi.wire_score_bytes = score_bytes;
  for (int g = 0; g < G; ++g) {
    if (!(push_mask >> g & 1u)) continue;
    xi.slot[xi.n_peers] = peer_bufs[g] + MMR_XCHG_HEADER + (size_t(parity) * G + rank) * wire_bytes;
    xi.flag[xi.n_peers] = peer_bufs[g] + (size_t(parity) * MMR_XCHG_MAX_PEERS + rank) * 4;
    ++xi.n_peers;
  }
  // 1. the shard-local scan
  bool pushed = false;
  const bool k2 = uniform && q.dev != nullptr && uniform_takes_k2(ix, B, k, int64_t(r1) - r0);
  if (uniform && !k2 && B <= k1_group(ix) && (q.dev != nullptr || can_inline(ix, B))) {
    // K1 computes and pushes in ONE kernel: its last CTA stores the result into the peers over NVLink
    int rc = search_uniform_stream(ix, q, B, k, r0, r1, w_scores, w_rows, ws, st, &xi);
    if (rc != MMR_OK) return rc;
    pushed = true;
  } else {
    if (q.dev == nullptr) return fail(MMR_ERR_INVALID, "this batch needs device-resident queries");
    int rc = uniform ? search_uniform(ix, q, B, k, r0, r1, w_scores, w_rows, ws, base_ws, st)
                     : search_varlen_stream(ix, q.dev, *per_query, k, w_scores, w_rows, ws, base_ws, st);
    if (rc != MMR_OK) return rc;
  }
  // 2. push (when the scan kernel did not do it itself)
  if (!pushed && xi.n_peers > 0) {
    PeerPtrs pp;
    for (int g = 0; g < MMR_XCHG_MAX_PEERS; ++g) {
      pp.slot[g] = g < xi.n_peers ? xi.slot[g] : 0;
      pp.flag[g] = g < xi.n_peers ? xi.flag[g] : 0;
    }
    push_wire_kernel<<<xi.n_peers, 256, 0, st>>>(wire, wire_bytes, pp, seq);
    g_launches++;
  }
  if (!do_merge) return MMR_OK;
  // 3. wait for every peer's slot, merge in place
  const uint8_t* local = reinterpret_cast<const uint8_t*>(peer_bufs[rank]);
  const int wpb = 4;
  const uint64_t timeout_ns = 5000000000ull;
  // With MMR_PDL=1 the wait+merge kernel is a programmatic dependent of the scan: it may become resident while the scan
  // still runs (it only spins on the flags, which the scan's last CTA releases at its very end) and the next search's
  // scan may in turn start behind it.  Otherwise plain stream order.
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((B + wpb - 1) / wpb);
  cfg.blockDim = dim3(wpb * 32);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = (pushed && options().pdl) ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  uint32_t* done_flag = nullptr;
  uint32_t done_seq = 0;
  if (done && done->flag_dev && cfg.gridDim.x == 1 && options().mailbox) {  // one block writes every result: it rings the mailbox
    done_flag = done->flag_dev;
    done_seq = done->seq;
    done->armed = true;
  }
  if (k <= 32)
    CUDA_TRY(cudaLaunchKernelEx(&cfg, merge_wait_kernel<1>, local, parity, seq, wire_bytes, score_bytes, int(G), int(B),
                                int(k), out_s, out_r, timeout_ns, done_flag, done_seq));
  else
    CUDA_TRY(cudaLaunchKernelEx(&cfg, merge_wait_kernel<2>, local, parity, seq, wire_bytes, score_bytes, int(G), int(B),
                                int(k), out_s, out_r, timeout_ns, done_flag, done_seq));
  g_launches++;
  return MMR_OK;
}

static int check_exchange_args(const mmr_index* ix, int B, int k, const uint64_t* peer_bufs_host, int G, int rank, uint32_t seq) {
  int rc = check_search_args(ix, B, k);
  if (rc != MMR_OK) return rc;
  if (!peer_bufs_host || G < 1 || G > MMR_XCHG_MAX_PEERS || rank < 0 || rank >= G)
    return fail(MMR_ERR_INVALID, "bad peer table (G=%d, rank=%d)", G, rank);
  if (seq == 0) return fail(MMR_ERR_INVALID, "seq must start at 1 and grow by 1 per search");
  return MMR_OK;
}

extern "C" int mmr_search_exchange(const mmr_index* ix, const float* queries_dev, const int32_t* query_seg_host,
                                   int32_t B, int32_t k, const uint64_t* peer_bufs_host, int32_t G, int32_t rank,
                                   uint32_t seq, float* out_scores_dev, int64_t* out_rows_dev, void* workspace_dev,
                                   size_t workspace_bytes, void* stream) {
  int rc = check_exchange_args(ix, B, k, peer_bufs_host, G, rank, seq);
  if (rc != MMR_OK) return rc;
  if (!queries_dev || !out_scores_dev || !out_rows_dev || !workspace_dev) return fail(MMR_ERR_INVALID, "NULL buffer");
  const size_t base_ws = mmr_search_workspace_bytes(ix, B, k);
  if (workspace_bytes < mmr_search_exchange_workspace_bytes(ix, B, k)) return fail(MMR_ERR_WORKSPACE, "workspace too small");
  std::vector<RangeList> ranges;
  bool uniform = true;
  rc = ranges_from_segments(ix, query_seg_host, B, ranges, uniform);
  if (rc != MMR_OK) return rc;
  QuerySrc q;
  q.dev = queries_dev;
  return exchange_impl(ix, q, B, k, uniform, ranges[0][0].first, ranges[0][0].second, &ranges, peer_bufs_host, G, rank, seq,
                       (G >= 32 ? 0xFFFFFFFFu : ((1u << G) - 1u)), true, out_scores_dev, out_rows_dev,
                       static_cast<uint8_t*>(workspace_dev), base_ws, static_cast<cudaStream_t>(stream), nullptr);
}

// The same exchange with HOST buffers (one process per GPU, e.g. under torchrun): for B <= 2 the query rides in the scan
// kernel's parameters, the wait+merge kernel writes the merged result and a completion flag into this index's mapped
// mailbox, and the host spins on the flag -- no copies, no stream synchronisation on the request path.
extern "C" int mmr_search_exchange_host(mmr_index* ix, const float* queries_host, const int32_t* query_seg_host, int32_t B,
                                        int32_t k, const uint64_t* peer_bufs_host, int32_t G, int32_t rank, uint32_t seq,
                                        float* out_scores_host, int64_t* out_rows_host, void* stream) {
  int rc = check_exchange_args(ix, B, k, peer_bufs_host, G, rank, seq);
  if (rc != MMR_OK) return rc;
  if (!queries_host || !out_scores_host || !out_rows_host) return fail(MMR_ERR_INVALID, "NULL buffer");
  std::lock_guard<std::mutex> guard(ix->host_mu);
  CUDA_TRY(cudaSetDevice(ix->device));
  rc = ensure_staging(ix, B, k);
  if (rc != MMR_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  std::vector<RangeList> ranges;
  bool uniform = true;
  rc = ranges_from_segments(ix, query_seg_host, B, ranges, uniform);
  if (rc != MMR_OK) return rc;
  // the exchange wire sits behind the search workspace: the staging workspace must hold both
  const size_t base_ws = workspace_bytes_for(ix, ix->cap_b, ix->cap_k, int64_t(RANGES_PER_QUERY_BUDGET) * ix->cap_b);
  const size_t need = base_ws + align_up(xchg_wire_bytes(ix->cap_b, ix->cap_k), 256);
  if (ix->ws_bytes < need) {
    if (ix->d_ws) cudaFree(ix->d_ws);
    ix->d_ws = nullptr;
    CUDA_TRY(cudaMalloc(&ix->d_ws, need));
    CUDA_TRY(cudaMemset(ix->d_ws, 0, need));
    ix->ws_bytes = need;
  }
  float* box_s = reinterpret_cast<float*>(ix->d_box + BOX_HEADER);
  int64_t* box_r = reinterpret_cast<int64_t*>(ix->d_box + box_rows_off(B, k));
  Completion done;
  done.flag_dev = reinterpret_cast<uint32_t*>(ix->d_box);
  done.seq = ++ix->box_seq ? ix->box_seq : ++ix->box_seq;
  QuerySrc q;
  const uint32_t r0 = ranges[0][0].first, r1 = ranges[0][0].second;
  if (uniform && can_inline(ix, B) && !uniform_takes_k2(ix, B, k, int64_t(r1) - r0)) {
    q.host = queries_host;
  } else {
    memcpy(ix->h_q, queries_host, size_t(B) * ix->dim * 4);
    CUDA_TRY(cudaMemcpyAsync(ix->d_q, ix->h_q, size_t(B) * ix->dim * 4, cudaMemcpyHostToDevice, st));
    q.dev = ix->d_q;
  }
  rc = exchange_impl(ix, q, B, k, uniform, r0, r1, &ranges, peer_bufs_host, G, rank, seq,
                     (G >= 32 ? 0xFFFFFFFFu : ((1u << G) - 1u)), true, box_s, box_r, static_cast<uint8_t*>(ix->d_ws),
                     base_ws, st, &done);
  if (rc != MMR_OK) return rc;
  return finish_host_call(ix, done, B, k, out_scores_host, out_rows_host, st);
}

// ------------------------------------------------------------------------------------------------ one process, G GPUs
// The reference has ONE store object in ONE process (app/ml/retrieve.py:21).  mmr_multi keeps that shape on a multi-GPU
// box: G row-range shards (one mmr_index per device, row_base = first global row), one launcher thread and one stream
// per device, and the same fused exchange as the SPMD form -- every shard's scan kernel stores its [B, k] result into the
// COLLECTOR device's exchange buffer over NVLink peer mappings, and the collector's wait+merge kernel writes the final
// result and a completion flag into a mapped host mailbox.  A request costs one kernel launch per device plus one merge
// launch; no copies, no stream synchronisation.
struct mmr_multi {
  int G = 0;
  std::vector<mmr_index*> shard;
  std::vector<cudaStream_t> stream;
  std::vector<uint8_t*> xbuf;
  std::vector<uint64_t> peer_ptrs;
  int cap_b = 0, cap_k = 0;
  uint32_t seq = 0;       // exchange sequence number (restarts with the exchange buffers)
  uint32_t mail_seq = 0;  // mailbox sequence number of the collector index (monotonic for the index's lifetime)
  std::mutex call_mu;  // one search at a time
  // job broadcast to the launcher threads
  std::vector<std::thread> workers;
  std::mutex mu;
  std::condition_variable cv;
  std::atomic<uint64_t> job_seq{0};
  std::atomic<int> pending{0};
  std::atomic<bool> stop{false};
  const float* q_host = nullptr;
  const std::vector<RangeList>* ranges = nullptr;  // global row ranges per query
  int B = 0, k = 0;
  std::vector<int> rc;
  std::vector<std::string> err;
};

static void multi_free_xbuf(mmr_multi* m) {
  for (int g = 0; g < m->G; ++g) {
    if (m->xbuf[g]) {
      cudaSetDevice(m->shard[g]->device);
      cudaFree(m->xbuf[g]);
      m->xbuf[g] = nullptr;
    }
  }
}

// runs on launcher thread g with device g current
static int multi_run_shard(mmr_multi* m, int g) {
  mmr_index* ix = m->shard[g];
  const int B = m->B, k = m->k;
  std::lock_guard<std::mutex> guard(ix->host_mu);
  int rc = ensure_staging(ix, std::max(B, m->cap_b), std::max(k, m->cap_k));
  if (rc != MMR_OK) return rc;
  const size_t base_ws = workspace_bytes_for(ix, ix->cap_b, ix->cap_k, int64_t(RANGES_PER_QUERY_BUDGET) * ix->cap_b);
  const size_t need = base_ws + align_up(xchg_wire_bytes(ix->cap_b, ix->cap_k), 256);
  if (ix->ws_bytes < need) {
    if (ix->d_ws) cudaFree(ix->d_ws);
    ix->d_ws = nullptr;
    CUDA_TRY(cudaMalloc(&ix->d_ws, need));
    CUDA_TRY(cudaMemset(ix->d_ws, 0, need));
    ix->ws_bytes = need;
  }
  // clip the global ranges to this shard
  const int64_t lo_g = ix->row_base, hi_g = ix->row_base + ix->n_rows;
  std::vector<RangeList> local(B);
  bool uniform = true;
  for (int b = 0; b < B; ++b) {
    for (auto& r : (*m->ranges)[b]) {
      const int64_t lo = std::max<int64_t>(r.first, lo_g), hi = std::min<int64_t>(r.second, hi_g);
      if (hi > lo) local[b].push_back({uint32_t(lo - lo_g), uint32_t(hi - lo_g)});
    }
    if (local[b].size() > 1 || local[b] != local[0]) uniform = false;
  }
  const uint32_t r0 = (uniform && !local[0].empty()) ? local[0][0].first : 0u;
  const uint32_t r1 = (uniform && !local[0].empty()) ? local[0][0].second : 0u;
  cudaStream_t st = m->stream[g];
  QuerySrc q;
  if (uniform && can_inline(ix, B) && !uniform_takes_k2(ix, B, k, int64_t(r1) - r0)) {
    q.host = m->q_host;
  } else {
    memcpy(ix->h_q, m->q_host, size_t(B) * ix->dim * 4);
    CUDA_TRY(cudaMemcpyAsync(ix->d_q, ix->h_q, size_t(B) * ix->dim * 4, cudaMemcpyHostToDevice, st));
    q.dev = ix->d_q;
  }
  Completion done;
  float* box_s = nullptr;
  int64_t* box_r = nullptr;
  if (g == 0) {  // the collector merges into its mailbox
    box_s = reinterpret_cast<float*>(ix->d_box + BOX_HEADER);
    box_r = reinterpret_cast<int64_t*>(ix->d_box + box_rows_off(B, k));
    done.flag_dev = reinterpret_cast<uint32_t*>(ix->d_box);
    done.seq = m->mail_seq;
  }
  rc = exchange_impl(ix, q, B, k, uniform, r0, r1, &local, m->peer_ptrs.data(), m->G, g, m->seq, 1u /* push to the collector */,
                     g == 0, box_s, box_r, static_cast<uint8_t*>(ix->d_ws), base_ws, st, g == 0 ? &done : nullptr);
  if (rc == MMR_OK && g == 0 && !done.armed) {
    // multi-block merge (B > 4): no flag from the kernel; ring the mailbox when the stream drains
    CUDA_TRY(cudaStreamSynchronize(st));
    *reinterpret_cast<volatile uint32_t*>(ix->h_box) = m->mail_seq;
  }
  return rc;
}

static void multi_worker(mmr_multi* m, int g) {
  cudaSetDevice(m->shard[g]->device);
  uint64_t seen = 0;
  for (;;) {
    // spin briefly (back-to-back requests find the launcher hot), then sleep on the condition variable
    int spins = 0;
    while (m->job_seq.load(std::memory_order_acquire) == seen && !m->stop.load(std::memory_order_relaxed)) {
      if (++spins < 20000) {
        cpu_relax();
      } else {
        std::unique_lock<std::mutex> lk(m->mu);
        m->cv.wait_for(lk, std::chrono::milliseconds(50), [&] {
          return m->job_seq.load(std::memory_order_acquire) != seen || m->stop.load(std::memory_order_relaxed);
        });
      }
    }
    if (m->stop.load(std::memory_order_relaxed)) return;
    seen = m->job_seq.load(std::memory_order_acquire);
    m->rc[g] = multi_run_shard(m, g);
    if (m->rc[g] != MMR_OK) m->err[g] = g_err;
    m->pending.fetch_sub(1, std::memory_order_acq_rel);
  }
}

extern "C" int mmr_multi_create(mmr_index** shards, int32_t G, mmr_multi** out) {
  if (!out) return fail(MMR_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (!shards || G < 1 || G > MMR_XCHG_MAX_PEERS) return fail(MMR_ERR_INVALID, "need 1..%d shards", MMR_XCHG_MAX_PEERS);
  for (int g = 0; g < G; ++g) {
    if (!shards[g]) return fail(MMR_ERR_INVALID, "shard %d is NULL", g);
    if (shards[g]->dim != shards[0]->dim || shards[g]->dtype != shards[0]->dtype)
      return fail(MMR_ERR_INVALID, "shards must share dim and dtype");
    for (int h = 0; h < g; ++h)
      if (shards[h]->device == shards[g]->device) return fail(MMR_ERR_INVALID, "one shard per device");
  }
  mmr_multi* m = new mmr_multi();
  m->G = G;
  m->shard.assign(shards, shards + G);
  m->stream.assign(G, nullptr);
  m->xbuf.assign(G, nullptr);
  m->peer_ptrs.assign(G, 0);
  m->rc.assign(G, MMR_OK);
  m->err.assign(G, std::string());
  const int collector = shards[0]->device;
  for (int g = 0; g < G; ++g) {
    const int dev = shards[g]->device;
    if (cudaSetDevice(dev) != cudaSuccess || cudaStreamCreateWithFlags(&m->stream[g], cudaStreamNonBlocking) != cudaSuccess) {
      delete m;
      return fail(MMR_ERR_CUDA, "cannot create a stream on device %d", dev);
    }
    if (dev != collector) {  // shard g's scan kernel stores into the collector's exchange buffer
      int can = 0;
      cudaDeviceCanAccessPeer(&can, dev, collector);
      if (!can) {
        delete m;
        return fail(MMR_ERR_CUDA, "device %d cannot access device %d (no NVLink / P2P)", dev, collector);
      }
      cudaError_t e = cudaDeviceEnablePeerAccess(collector, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
        delete m;
        return fail(MMR_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", dev, collector, cudaGetErrorString(e));
      }
      cudaGetLastError();
    }
  }
  for (int g = 0; g < G; ++g) m->workers.emplace_back(multi_worker, m, g);
  *out = m;
  return MMR_OK;
}

extern "C" int mmr_multi_destroy(mmr_multi* m) {
  if (!m) return MMR_OK;
  m->stop.store(true);
  {
    std::lock_guard<std::mutex> lk(m->mu);
    m->cv.notify_all();
  }
  for (auto& t : m->workers) t.join();
  multi_free_xbuf(m);
  for (int g = 0; g < m->G; ++g) {
    if (m->stream[g]) {
      cudaSetDevice(m->shard[g]->device);
      cudaStreamDestroy(m->stream[g]);
    }
  }
  delete m;
  return MMR_OK;
}

extern "C" int mmr_multi_search_host(mmr_multi* m, const float* queries_host, int32_t B, int32_t k,
                                     const int32_t* range_off_host, const int64_t* ranges_host, float* out_scores_host,
                                     int64_t* out_rows_host) {
  if (!m) return fail(MMR_ERR_INVALID, "multi handle is NULL");
  int rc = check_search_args(m->shard[0], B, k);
  if (rc != MMR_OK) return rc;
  if (!queries_host || !range_off_host || !out_scores_host || !out_rows_host) return fail(MMR_ERR_INVALID, "NULL buffer");
  std::lock_guard<std::mutex> call_guard(m->call_mu);
  // global ranges (validated against the global row count)
  int64_t total = 0;
  for (int g = 0; g < m->G; ++g) total = std::max<int64_t>(total, m->shard[g]->row_base + m->shard[g]->n_rows);
  std::vector<RangeList> per_query(B);
  for (int b = 0; b < B; ++b) {
    if (range_off_host[b + 1] < range_off_host[b]) return fail(MMR_ERR_INVALID, "range offsets must be ascending");
    for (int32_t r = range_off_host[b]; r < range_off_host[b + 1]; ++r) {
      const int64_t lo = ranges_host[2 * r], hi = ranges_host[2 * r + 1];
      if (lo < 0 || hi < lo || hi > total || hi >= (int64_t(1) << 32))
        return fail(MMR_ERR_INVALID, "query %d: bad row range [%lld, %lld)", b, (long long)lo, (long long)hi);
      if (hi > lo) per_query[b].push_back({uint32_t(lo), uint32_t(hi)});
    }
    RangeList sorted = per_query[b];
    std::sort(sorted.begin(), sorted.end());
    for (size_t i = 1; i < sorted.size(); ++i)
      if (sorted[i].first < sorted[i - 1].second) return fail(MMR_ERR_INVALID, "query %d: row ranges overlap", b);
  }
  // (re)size the exchange buffers: zeroed once, sequence numbers restart with them
  if (B > m->cap_b || k > m->cap_k) {
    for (int g = 0; g < m->G; ++g) CUDA_TRY((cudaSetDevice(m->shard[g]->device), cudaStreamSynchronize(m->stream[g])));
    multi_free_xbuf(m);
    const int cb = std::max(B, 8), ck = std::max(k, 16);
    const size_t bytes = mmr_exchange_buffer_bytes(m->G, cb, ck);
    for (int g = 0; g < m->G; ++g) {
      CUDA_TRY(cudaSetDevice(m->shard[g]->device));
      CUDA_TRY(cudaMalloc(&m->xbuf[g], bytes));
      CUDA_TRY(cudaMemset(m->xbuf[g], 0, bytes));
      CUDA_TRY(cudaDeviceSynchronize());
      m->peer_ptrs[g] = reinterpret_cast<uint64_t>(m->xbuf[g]);
    }
    m->cap_b = cb;
    m->cap_k = ck;
    m->seq = 0;
  }
  // NOTE the wire layout depends on (B, k): slots of different shapes never mix inside one sequence number
  m->seq += 1;
  {
    std::lock_guard<std::mutex> box_guard(m->shard[0]->host_mu);
    m->mail_seq = ++m->shard[0]->box_seq ? m->shard[0]->box_seq : ++m->shard[0]->box_seq;
  }
  m->q_host = queries_host;
  m->ranges = &per_query;
  m->B = B;
  m->k = k;
  m->pending.store(m->G, std::memory_order_release);
  {
    std::lock_guard<std::mutex> lk(m->mu);
    m->job_seq.fetch_add(1, std::memory_order_acq_rel);
  }
  m->cv.notify_all();
  while (m->pending.load(std::memory_order_acquire) != 0) cpu_relax();   // every launcher has issued its work
  for (int g = 0; g < m->G; ++g)
    if (m->rc[g] != MMR_OK) return fail(m->rc[g], "shard %d: %s", g, m->err[g].c_str());
  mmr_index* c = m->shard[0];
  CUDA_TRY(cudaSetDevice(c->device));
  rc = wait_mailbox(c, m->mail_seq, m->stream[0]);
  if (rc != MMR_OK) return rc;
  memcpy(out_scores_host, c->h_box + BOX_HEADER, size_t(B) * k * 4);
  memcpy(out_rows_host, c->h_box + box_rows_off(B, k), size_t(B) * k * 8);
  if (out_rows_host[0] == -2) return fail(MMR_ERR_CUDA, "exchange timed out: a shard never delivered its result");
  return MMR_OK;
}

// Debug / validation hook: raw K2 scores (tensor-core contraction only, no top-k) for rows [row_begin, row_end).
extern "C" int mmr_debug_umma_scores(const mmr_index* ix, const float* queries_dev, int32_t B, int64_t row_begin,
                                     int64_t row_end, float* out_scores_dev, int64_t out_ld, void* workspace_dev,
                                     size_t workspace_bytes, void* stream) {
  if (!ix || !queries_dev || !out_scores_dev || !workspace_dev) return fail(MMR_ERR_INVALID, "NULL argument");
  if (ix->dtype != MMR_BF16 && ix->dtype != MMR_F16) return fail(MMR_ERR_UNSUPPORTED, "K2 needs bf16 or fp16 rows");
  if (B <= 0 || row_begin < 0 || row_end > ix->n_rows || row_end <= row_begin || out_ld < row_end - row_begin)
    return fail(MMR_ERR_INVALID, "bad range");
  if (workspace_bytes < umma_workspace_bytes(ix->sm_count, ix->dim, B, MMR_MAX_K)) return fail(MMR_ERR_WORKSPACE, "workspace too small");
  int rc = umma_search(ix->umma, ix->umma2, ix->rows, ix->n_rows, ix->dim, ix->dtype, ix->sm_count, queries_dev, B, 10, uint32_t(row_begin),
                       uint32_t(row_end), 0, nullptr, nullptr, static_cast<uint8_t*>(workspace_dev),
                       static_cast<cudaStream_t>(stream), g_err, out_scores_dev, out_ld);
  if (rc == MMR_OK) g_launches += umma_launches_per_search();
  return rc;
}

// ------------------------------------------------------------------------------------------------ K4 / K5
extern "C" int mmr_merge_topk_strided(const float* scores_dev, const int64_t* rows_dev, int64_t score_shard_stride,
                                      int64_t row_shard_stride, int32_t G, int32_t B, int32_t k, float* out_scores_dev,
                                      int64_t* out_rows_dev, void* stream) {
  if (G <= 0 || B <= 0) return fail(MMR_ERR_INVALID, "G and B must be >= 1");
  if (k < 1 || k > MMR_MAX_K) return fail(MMR_ERR_INVALID, "k must be in [1, %d]", MMR_MAX_K);
  if (!scores_dev || !rows_dev || !out_scores_dev || !out_rows_dev) return fail(MMR_ERR_INVALID, "NULL buffer");
  if (score_shard_stride < int64_t(B) * k || row_shard_stride < int64_t(B) * k)
    return fail(MMR_ERR_INVALID, "shard stride smaller than B*k");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int wpb = 4;
  const int blocks = (B + wpb - 1) / wpb;
  if (k <= 32)
    merge_shards_kernel<1><<<blocks, wpb * 32, 0, st>>>(scores_dev, rows_dev, score_shard_stride, row_shard_stride, G, B,
                                                        k, out_scores_dev, out_rows_dev);
  else
    merge_shards_kernel<2><<<blocks, wpb * 32, 0, st>>>(scores_dev, rows_dev, score_shard_stride, row_shard_stride, G, B,
                                                        k, out_scores_dev, out_rows_dev);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return MMR_OK;
}

extern "C" int mmr_merge_topk(const float* scores_dev, const int64_t* rows_dev, int32_t G, int32_t B, int32_t k,
                              float* out_scores_dev, int64_t* out_rows_dev, void* stream) {
  return mmr_merge_topk_strided(scores_dev, rows_dev, int64_t(B) * k, int64_t(B) * k, G, B, k, out_scores_dev,
                                out_rows_dev, stream);
}

extern "C" int mmr_fuse(const float* text_scores_dev, const int64_t* text_rows_dev, int32_t kt,
                        const float* img_scores_dev, const int64_t* img_rows_dev, int32_t ki, int32_t B,
                        int32_t final_n, double tau, double* out_combined_dev, double* out_score_dev,
                        int64_t* out_rows_dev, int8_t* out_modality_dev, uint8_t* out_low_conf_dev, void* stream) {
  if (B <= 0) return fail(MMR_ERR_INVALID, "B must be >= 1");
  if (kt < 0 || kt > FUSE_MAXK || ki < 0 || ki > FUSE_MAXK) return fail(MMR_ERR_INVALID, "kt, ki must be in [0, %d]", FUSE_MAXK);
  if (final_n < 1) return fail(MMR_ERR_INVALID, "final_n must be >= 1");
  if ((kt > 0 && (!text_scores_dev || !text_rows_dev)) || (ki > 0 && (!img_scores_dev || !img_rows_dev)))
    return fail(MMR_ERR_INVALID, "NULL input buffer");
  if (!out_combined_dev || !out_score_dev || !out_rows_dev || !out_modality_dev || !out_low_conf_dev)
    return fail(MMR_ERR_INVALID, "NULL output buffer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int threads = 64;
  fuse_kernel<<<(B + threads - 1) / threads, threads, 0, st>>>(
      kt > 0 ? text_scores_dev : nullptr, kt > 0 ? text_rows_dev : nullptr, kt, ki > 0 ? img_scores_dev : nullptr,
      ki > 0 ? img_rows_dev : nullptr, ki, B, final_n, tau, out_combined_dev, out_score_dev, out_rows_dev,
      out_modality_dev, out_low_conf_dev);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return MMR_OK;
}

extern "C" int mmr_fuse_f64(const double* text_scores_dev, const int32_t* text_count_dev, const double* text_rerank_dev,
                            const int32_t* rerank_count_dev, const double* img_scores_dev, const int32_t* img_count_dev,
                            int32_t kt, int32_t ki, int32_t B, int32_t final_n, double tau, double* out_combined_dev,
                            int32_t* out_index_dev, uint8_t* out_low_conf_dev, void* stream) {
  if (B <= 0) return fail(MMR_ERR_INVALID, "B must be >= 1");
  if (kt < 0 || kt > FUSE_MAXK || ki < 0 || ki > FUSE_MAXK) return fail(MMR_ERR_INVALID, "kt, ki must be in [0, %d]", FUSE_MAXK);
  if (final_n < 1) return fail(MMR_ERR_INVALID, "final_n must be >= 1");
  if ((kt > 0 && (!text_scores_dev || !text_count_dev)) || (ki > 0 && (!img_scores_dev || !img_count_dev)))
    return fail(MMR_ERR_INVALID, "NULL input buffer");
  if (!out_combined_dev || !out_index_dev || !out_low_conf_dev) return fail(MMR_ERR_INVALID, "NULL output buffer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int threads = 32;
  fuse_full_kernel<<<(B + threads - 1) / threads, threads, 0, st>>>(
      kt > 0 ? text_scores_dev : nullptr, kt > 0 ? text_count_dev : nullptr, text_rerank_dev, rerank_count_dev,
      ki > 0 ? img_scores_dev : nullptr, ki > 0 ? img_count_dev : nullptr, kt, ki, B, final_n, tau, out_combined_dev,
      out_index_dev, out_low_conf_dev);
  g_launches++;
  CUDA_TRY(cudaGetLastError());
  return MMR_OK;
}
