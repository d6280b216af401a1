// CLIP image preprocessing on the device (mmr_image_preprocess): decoded 8-bit RGB images of any sizes -> pixel_values
// fp32 [B, 3, crop_h, crop_w], bit-identical to Pillow's `Image.resize(size, BICUBIC)` followed by HF's centre crop, rescale
// and normalise (CLIPImageProcessorPil).
//
// Pillow's 8-bit resample (libImaging/Resample.c): per axis, double-precision bicubic weights (a = -0.5) normalised to sum
// 1 and rounded to 22-bit fixed point; the horizontal pass runs first (only if the width changes) into a uint8 image, the
// vertical pass second (only if the height changes); each output is clip8((1 << 21) + sum pixel * k) with int32 sums.
// A skipped pass is the one-tap filter k = 1 << 22 here, which returns its input byte unchanged, so one code path serves
// every case.  Only the crop window's rows and columns are computed: each output depends on its own window only.
// Integer sums do not depend on their order, so the vertical pass accumulates input rows as they stream through.
//
// One CTA per (32 output columns, 16 output rows, image): it computes its columns' and rows' coefficients (a warp per
// output index, the weight sum in tap order on one lane), then streams the input rows its rows' windows cover in chunks:
// 16-byte loads of the row segments its columns' windows cover -> shared memory -> horizontal pass (uint8) -> vertical
// accumulation in registers.  The end maps each byte through the [3][256] rescale / normalise table, built on the host by
// HF's own functions, and stores coalesced NCHW rows.
#pragma once
#include <cstdint>

#include "common.cuh"

namespace mmr {

constexpr int PREP_THREADS = 256;
constexpr int PREP_WARPS = PREP_THREADS / 32;
constexpr int PREP_COLS = 32;              // output columns per CTA (= lanes: one coalesced 128-byte store per row)
constexpr int PREP_ROWS = 16;              // output rows per CTA
constexpr int PREP_OUT_PER_THREAD = 3 * PREP_ROWS * PREP_COLS / PREP_THREADS;
constexpr int PREP_MAX_CHUNK = 32;         // input rows per chunk
constexpr int PREP_RAW_BUDGET = 24 * 1024; // bytes of input row segments per chunk
constexpr int PREP_LAUNCH_IMAGES = 896;    // images per launch: their geometry rides in the kernel parameters

struct PrepImage {
  int64_t offset;                          // byte offset of the image (HWC RGB) in the source buffer, a multiple of 16
  int32_t h, w, out_h, out_w, top, left;   // input size, resized size, crop window origin in the resized image
};

// Kernel parameters (< 32764 bytes: no device copy of the geometry, nothing to keep alive after the launch).
struct PrepParams {
  float table[3][256];
  int32_t crop_h, crop_w;
  int32_t taps_x, taps_y;                  // coefficient row strides: the largest tap count over the launch's images
  int32_t seg_bytes, chunk_rows;           // shared row segment (multiple of 16) and rows per chunk
  PrepImage img[PREP_LAUNCH_IMAGES];
};

// Tap count of Pillow's bicubic filter for in_size -> out_size (ksize of precompute_coeffs), host and device.
__host__ __device__ inline int prep_taps(int in_size, int out_size) {
  if (in_size == out_size) return 1;       // the pass is skipped: identity tap
  const double scale = double(in_size) / double(out_size);
  const double fs = scale < 1.0 ? 1.0 : scale;
  return int(ceil(2.0 * fs)) * 2 + 1;
}

// Input columns (or rows) a run of n consecutive outputs can cover: (n - 1) * scale + 2 * support + 1 <= that + taps.
__host__ __device__ inline int prep_span(int in_size, int out_size, int n) {
  if (in_size == out_size) return n;
  return int(ceil(double(n - 1) * double(in_size) / double(out_size))) + prep_taps(in_size, out_size) + 2;
}

__device__ __forceinline__ double prep_bicubic(double x) {
  // ((a + 2) x - (a + 3)) x x + 1 for |x| < 1, (((x - 5) x + 8) x - 4) a for |x| < 2, a = -0.5; every operation rounded
  // on its own (no FMA contraction), as Pillow's compiled C rounds them
  x = fabs(x);
  if (x < 1.0) return __dadd_rn(__dmul_rn(__dmul_rn(__dadd_rn(__dmul_rn(1.5, x), -2.5), x), x), 1.0);
  if (x < 2.0) return __dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(__dmul_rn(__dadd_rn(x, -5.0), x), 8.0), x), -4.0), -0.5);
  return 0.0;
}

// Pillow's precompute_coeffs + normalize_coeffs_8bpc for output index xx of one axis, by one warp: first input index,
// tap count and 22-bit taps k[0, count).  wtmp: this warp's scratch of >= taps doubles.
__device__ void prep_axis_coeffs(int in_size, int out_size, int xx, double* wtmp, int32_t* k, int32_t* first, int32_t* count) {
  const int lane = threadIdx.x & 31;
  if (in_size == out_size) {
    if (lane == 0) {
      *first = xx;
      *count = 1;
      k[0] = 1 << 22;
    }
    return;
  }
  const double scale = __ddiv_rn(double(in_size), double(out_size));
  const double fs = scale < 1.0 ? 1.0 : scale;
  const double support = __dmul_rn(2.0, fs);
  const double center = __dmul_rn(__dadd_rn(double(xx), 0.5), scale);
  const double ss = __ddiv_rn(1.0, fs);
  const int xmin = max(int(__dadd_rn(__dsub_rn(center, support), 0.5)), 0);
  const int n = min(int(__dadd_rn(__dadd_rn(center, support), 0.5)), in_size) - xmin;
  for (int t = lane; t < n; t += 32) wtmp[t] = prep_bicubic(__dmul_rn(__dadd_rn(__dsub_rn(double(t + xmin), center), 0.5), ss));
  __syncwarp();
  double ww = 0.0;
  if (lane == 0)
    for (int t = 0; t < n; ++t) ww = __dadd_rn(ww, wtmp[t]);   // in tap order
  ww = __shfl_sync(0xffffffffu, ww, 0);
  for (int t = lane; t < n; t += 32) {
    const double w = ww != 0.0 ? __ddiv_rn(wtmp[t], ww) : wtmp[t];
    const double s = __dmul_rn(w, double(1 << 22));
    k[t] = w < 0.0 ? int(__dadd_rn(-0.5, s)) : int(__dadd_rn(s, 0.5));
  }
  if (lane == 0) {
    *first = xmin;
    *count = n;
  }
  __syncwarp();
}

__device__ __forceinline__ int32_t prep_clip8(int32_t acc) { return min(max(acc >> 22, 0), 255); }

__global__ void __launch_bounds__(PREP_THREADS) image_prep_kernel(const __grid_constant__ PrepParams p, const uint8_t* __restrict__ src,
                                                                  float* __restrict__ out) {
  extern __shared__ __align__(16) uint8_t prep_smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const PrepImage g = p.img[blockIdx.z];
  const int x0 = blockIdx.x * PREP_COLS, y0 = blockIdx.y * PREP_ROWS;
  const int ncols = min(PREP_COLS, p.crop_w - x0), nrows = min(PREP_ROWS, p.crop_h - y0);
  const int tmax = max(p.taps_x, p.taps_y);

  uint8_t* raw = prep_smem;                                                       // [chunk_rows][seg_bytes]
  float* table = reinterpret_cast<float*>(raw + size_t(p.chunk_rows) * p.seg_bytes);   // [3][256]
  double* wtmp = reinterpret_cast<double*>(table + 3 * 256);                       // [warps][tmax]
  int32_t* kx = reinterpret_cast<int32_t*>(wtmp + PREP_WARPS * tmax);             // [PREP_COLS][taps_x]
  int32_t* ky = kx + PREP_COLS * p.taps_x;                                        // [PREP_ROWS][taps_y]
  int32_t* xfirst = ky + PREP_ROWS * p.taps_y;
  int32_t* xcount = xfirst + PREP_COLS;
  int32_t* yfirst = xcount + PREP_COLS;
  int32_t* ycount = yfirst + PREP_ROWS;
  int32_t* rowshift = ycount + PREP_ROWS;                                         // [chunk_rows]: segment start - its 16-byte floor
  uint8_t* inter = reinterpret_cast<uint8_t*>(rowshift + PREP_MAX_CHUNK);         // [chunk_rows][PREP_COLS * 3]

  // the parameters alone decide the coefficients: compute them while the previous kernel drains
  pdl_launch_dependents();
  for (int i = tid; i < 3 * 256; i += PREP_THREADS) table[i] = (&p.table[0][0])[i];
  for (int i = warp; i < ncols + nrows; i += PREP_WARPS) {
    if (i < ncols)
      prep_axis_coeffs(g.w, g.out_w, g.left + x0 + i, wtmp + warp * tmax, kx + i * p.taps_x, xfirst + i, xcount + i);
    else
      prep_axis_coeffs(g.h, g.out_h, g.top + y0 + i - ncols, wtmp + warp * tmax, ky + (i - ncols) * p.taps_y, yfirst + i - ncols,
                       ycount + i - ncols);
  }
  __syncthreads();
  // window starts and ends are non-decreasing in the output index
  const int xlo = xfirst[0], xhi = xfirst[ncols - 1] + xcount[ncols - 1];
  const int ylo = yfirst[0], yhi = yfirst[nrows - 1] + ycount[nrows - 1];
  pdl_wait_prior_grid();

  const uint8_t* img = src + g.offset;
  int32_t acc[PREP_OUT_PER_THREAD];
#pragma unroll
  for (int q = 0; q < PREP_OUT_PER_THREAD; ++q) acc[q] = 1 << 21;
  const int n16 = p.seg_bytes / 16;
  for (int r0 = ylo; r0 < yhi; r0 += p.chunk_rows) {
    const int nr = min(p.chunk_rows, yhi - r0);
    // 1. row segments [xlo, xhi) of input rows r0 .. r0 + nr, from their 16-byte floor (the image is 16-byte aligned and
    //    padded to a multiple of 16, so no load leaves it)
    for (int i = tid; i < nr * n16; i += PREP_THREADS) {
      const int j = i / n16, v = i - j * n16;
      const int64_t start = (int64_t(r0 + j) * g.w + xlo) * 3, base = start & ~int64_t(15);
      const int64_t end = (int64_t(r0 + j) * g.w + xhi) * 3;
      if (v == 0) rowshift[j] = int32_t(start - base);
      if (base + 16 * v < end)
        *reinterpret_cast<uint4*>(raw + j * p.seg_bytes + 16 * v) = __ldg(reinterpret_cast<const uint4*>(img + base) + v);
    }
    __syncthreads();
    // 2. horizontal pass -> uint8 (row j, column i, channel c)
    for (int i = tid; i < nr * PREP_COLS * 3; i += PREP_THREADS) {
      const int j = i / (PREP_COLS * 3), xc = i - j * (PREP_COLS * 3), x = xc / 3, c = xc - 3 * x;
      if (x >= ncols) continue;
      const uint8_t* s = raw + j * p.seg_bytes + rowshift[j] + (xfirst[x] - xlo) * 3 + c;
      const int32_t* k = kx + x * p.taps_x;
      int32_t a = 1 << 21;
      for (int t = 0; t < xcount[x]; ++t) a += int32_t(s[3 * t]) * k[t];
      inter[j * (PREP_COLS * 3) + xc] = uint8_t(prep_clip8(a));
    }
    __syncthreads();
    // 3. vertical accumulation: output q of this thread is (channel, row) = (warp + 8 q) / 16, column = lane
#pragma unroll
    for (int q = 0; q < PREP_OUT_PER_THREAD; ++q) {
      const int cr = warp + PREP_WARPS * q, c = cr / PREP_ROWS, y = cr % PREP_ROWS;
      if (y >= nrows) continue;
      const int f = yfirst[y], lo = max(r0, f), hi = min(r0 + nr, f + ycount[y]);
      const int32_t* k = ky + y * p.taps_y;
      const uint8_t* s = inter + lane * 3 + c;
      for (int r = lo; r < hi; ++r) acc[q] += int32_t(s[(r - r0) * (PREP_COLS * 3)]) * k[r - f];
    }
    __syncthreads();
  }
  if (lane >= ncols) return;
#pragma unroll
  for (int q = 0; q < PREP_OUT_PER_THREAD; ++q) {
    const int cr = warp + PREP_WARPS * q, c = cr / PREP_ROWS, y = cr % PREP_ROWS;
    if (y >= nrows) continue;
    out[((size_t(blockIdx.z) * 3 + c) * p.crop_h + y0 + y) * p.crop_w + x0 + lane] = table[c * 256 + prep_clip8(acc[q])];
  }
}

// Dynamic shared memory of image_prep_kernel for a launch's layout (the carve-up at the top of the kernel).
inline size_t prep_smem_bytes(const PrepParams& p) {
  const int tmax = p.taps_x > p.taps_y ? p.taps_x : p.taps_y;
  return size_t(p.chunk_rows) * p.seg_bytes + 3 * 256 * 4 + size_t(PREP_WARPS) * tmax * 8 +
         size_t(PREP_COLS * p.taps_x + PREP_ROWS * p.taps_y + 2 * PREP_COLS + 2 * PREP_ROWS + PREP_MAX_CHUNK) * 4 +
         size_t(PREP_MAX_CHUNK) * PREP_COLS * 3;
}

}  // namespace mmr
