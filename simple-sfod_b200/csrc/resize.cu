// resize.cu -- weak augmentation of the input on the GPU (SURVEY.md 8f rank 3): detectron2's ResizeShortestEdge (uint8 path =
// PIL.Image.resize(BILINEAR)) followed by RandomFlip's np.flip, and the mapper's HWC -> CHW transpose, for a whole batch of
// differently sized images in one launch.
//
// Arithmetic contract: Pillow's 8-bit resampler (src/libImaging/Resample.c, PRECISION_BITS = 22), bit for bit.
//   horizontal pass, over the input rows the vertical taps use:  tmp[y][x] = clip8(2^21 + sum_k in[y][xmin_x + k] * kx[x][k])
//   vertical pass:                                                 out[y][x] = clip8(2^21 + sum_k tmp[ymin_y + k][x] * ky[y][k])
//   clip8(s) = s <= 0 ? 0 : s >= 255 << 22 ? 255 : s >> 22, int32 sums; the taps (host, ops.pil_resize_coeffs) are >= 0.
// Every byte of Pillow's temporary image depends only on its input row and the column taps, so a tile that recomputes the
// intermediate rows it needs reproduces that image exactly, and the result is bit-equal by construction.
//
// One CTA = one 32 x 64 output tile of one image, all three channels:
//   1. stage the input window the tile needs in shared memory: 16-byte loads of whole aligned row segments when a row (HWC)
//      or a channel row (CHW planes) is contiguous and the strides keep every segment at the same 16-byte phase, byte loads
//      otherwise;
//   2. horizontal pass into a uint8 (3, window rows, 64) intermediate: lane = output column, its taps in registers;
//   3. vertical pass: warp = output row (taps uniform across the warp), lane = output column; CHW bytes written to the mirrored
//      column when the flip flag is set.
// Taps past a column's xmax are zero, so the fixed KMAX-tap loops may read (and multiply by 0) bytes past the window: both
// shared buffers carry a tail pad for that.
#include "common.cuh"

namespace {

constexpr int kRTW = 64;        // output tile width (2 columns per lane)
constexpr int kRTH = 32;        // output tile height
constexpr int kRThreads = 256;
constexpr int kRWarps = kRThreads / 32;
constexpr int kRCols = kRTW / 32;
constexpr int kMaxKsize = 9;    // ksize = 2 * ceil(max(in / out, 1)) + 1: down-scale up to 4
constexpr int kWinPad = 64;     // >= 3 * kMaxKsize + 15: tail of the input window a zero tap may touch
constexpr int kRowPad = 1;      // extra intermediate rows past the last channel plane (times kMaxKsize below)

__device__ __forceinline__ unsigned char pil_clip8(int s) {
  return s <= 0 ? (unsigned char)0 : s >= (255 << 22) ? (unsigned char)255 : (unsigned char)(s >> 22);
}

// Largest window span (input pixels) a tile of `t` outputs needs along an axis whose ksize is <= kmax:
// xend - xmin <= (t - 1) * scale + 2 * support + 1 with scale <= support <= (kmax - 1) / 2.
__host__ __device__ constexpr int resize_span_max(int t, int kmax) { return (t + 1) * ((kmax - 1) / 2) + 2; }
// Bytes of one window row in shared memory: 3 * span for interleaved HWC, or three 16-byte-aligned lines for CHW planes,
// each including the 16-byte phase of the source.
__host__ __device__ constexpr int resize_row_cap(int span_max) { return 3 * ((span_max + 15 + 15) & ~15); }

template <int KMAX>
__global__ void __launch_bounds__(kRThreads) pil_resize_kernel(const sfod_resize_image *__restrict__ recs, const int *__restrict__ coeffs,
                                                              unsigned char *__restrict__ out, int max_out_h, int max_out_w) {
  extern __shared__ __align__(16) unsigned char rz_smem[];
  constexpr int kSpanX = resize_span_max(kRTW, KMAX), kSpanY = resize_span_max(kRTH, KMAX);
  constexpr int kRowCap = resize_row_cap(kSpanX);
  unsigned char *win = rz_smem;                                  // kSpanY rows of kRowCap bytes (+ kWinPad)
  unsigned char *mid = rz_smem + kSpanY * kRowCap + kWinPad;     // (3, kSpanY, kRTW) (+ KMAX rows)

  const sfod_resize_image r = recs[blockIdx.z];
  const int ox0 = blockIdx.x * kRTW, oy0 = blockIdx.y * kRTH;
  if (r.out_w > max_out_w || r.out_h > max_out_h || r.in_w <= 0 || r.in_h <= 0 || r.kx_size > KMAX || r.ky_size > KMAX ||
      r.kx_size <= 0 || r.ky_size <= 0)
    return;                                                      // malformed record: skipped (documented in the header)
  if (ox0 >= r.out_w || oy0 >= r.out_h) return;
  const int tw = min(kRTW, r.out_w - ox0), th = min(kRTH, r.out_h - oy0);
  const int *bx = coeffs + r.kx_offset, *kx = bx + 2 * r.out_w;  // (xmin, xmax) pairs, then taps
  const int *by = coeffs + r.ky_offset, *ky = by + 2 * r.out_h;
  const int ksx = r.kx_size, ksy = r.ky_size;
  const int wx0 = __ldg(bx + 2 * ox0), wx1 = __ldg(bx + 2 * (ox0 + tw - 1)) + __ldg(bx + 2 * (ox0 + tw - 1) + 1);
  const int wy0 = __ldg(by + 2 * oy0), wy1 = __ldg(by + 2 * (oy0 + th - 1)) + __ldg(by + 2 * (oy0 + th - 1) + 1);
  const int sx = wx1 - wx0, sy = wy1 - wy0;
  if (wx0 < 0 || wy0 < 0 || wx1 > r.in_w || wy1 > r.in_h || sx <= 0 || sy <= 0 || sx > kSpanX || sy > kSpanY) return;

  // ---- 1. input window -> shared memory
  const long long rs = r.stride_row, ps_g = r.stride_px, cs = r.stride_ch;
  const bool hwc = ps_g == 3 && cs == 1;
  const bool vec = (hwc || ps_g == 1) && (rs & 15) == 0 && (hwc || (cs & 15) == 0);
  int L, ps, pitch, phase;                                       // lines per window row, pixel step, line pitch, 16-byte phase
  if (vec) {
    L = hwc ? 1 : 3;
    ps = hwc ? 3 : 1;
    const uintptr_t a0 = reinterpret_cast<uintptr_t>(r.src + (long long)wy0 * rs + (long long)wx0 * ps);
    phase = (int)(a0 & 15);
    const int nchunk = (phase + sx * ps + 15) >> 4;
    pitch = nchunk * 16;
    const unsigned char *base = reinterpret_cast<const unsigned char *>(a0 - phase);
    // An aligned 16-byte block holding a byte of the row lies within the row's allocation: the over-read is harmless.
    for (int t = threadIdx.x; t < sy * L * nchunk; t += kRThreads) {
      const int line = t / nchunk, ch = t - line * nchunk;
      const int y = line / L, c = line - y * L;
      const uint4 v = __ldg(reinterpret_cast<const uint4 *>(base + (long long)y * rs + (long long)c * cs + ch * 16));
      *reinterpret_cast<uint4 *>(win + line * pitch + ch * 16) = v;
    }
  } else {                                                       // any strides: byte gather into interleaved rows
    L = 1;
    ps = 3;
    phase = 0;
    pitch = 3 * sx;
    for (int t = threadIdx.x; t < sy * 3 * sx; t += kRThreads) {
      const int y = t / (3 * sx), rem = t - y * 3 * sx;
      const int x = rem / 3, c = rem - x * 3;
      win[y * pitch + rem] = r.src[(long long)(wy0 + y) * rs + (long long)(wx0 + x) * ps_g + (long long)c * cs];
    }
  }
  __syncthreads();

  // ---- 2. horizontal pass (lane = output column, taps in registers) over every window row
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int xs[kRCols], tap[kRCols][KMAX];
#pragma unroll
  for (int j = 0; j < kRCols; ++j) {
    const int x = lane + 32 * j;
    const bool ok = x < tw;
    xs[j] = ok ? __ldg(bx + 2 * (ox0 + x)) - wx0 : 0;
#pragma unroll
    for (int k = 0; k < KMAX; ++k) tap[j][k] = (ok && k < ksx) ? __ldg(kx + (ox0 + x) * ksx + k) : 0;
  }
  for (int q = warp; q < 3 * sy; q += kRWarps) {
    const int c = q / sy, y = q - c * sy;
    const unsigned char *line = win + (y * L + (L == 3 ? c : 0)) * pitch + phase + (L == 1 ? c : 0);
    unsigned char *dst = mid + (c * kSpanY + y) * kRTW;
#pragma unroll
    for (int j = 0; j < kRCols; ++j) {
      const int x = lane + 32 * j;
      if (x >= tw) continue;
      int acc = 1 << 21;
#pragma unroll
      for (int k = 0; k < KMAX; ++k) acc += (int)line[ps * (xs[j] + k)] * tap[j][k];
      dst[x] = pil_clip8(acc);
    }
  }
  __syncthreads();

  // ---- 3. vertical pass (warp = output row, taps uniform across the warp) and the CHW store
  const long long plane = (long long)r.out_h * r.out_w;
  unsigned char *img = out + r.out_offset;
  for (int yy = warp; yy < th; yy += kRWarps) {
    const int oy = oy0 + yy;
    const int ys = __ldg(by + 2 * oy) - wy0;
    int tv[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) tv[k] = k < ksy ? __ldg(ky + oy * ksy + k) : 0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const unsigned char *col = mid + (c * kSpanY + ys) * kRTW;
      unsigned char *orow = img + c * plane + (long long)oy * r.out_w;
#pragma unroll
      for (int j = 0; j < kRCols; ++j) {
        const int x = lane + 32 * j;
        if (x >= tw) continue;
        int acc = 1 << 21;
#pragma unroll
        for (int k = 0; k < KMAX; ++k) acc += (int)col[k * kRTW + x] * tv[k];
        const int X = ox0 + x;
        orow[r.hflip ? r.out_w - 1 - X : X] = pil_clip8(acc);
      }
    }
  }
}

template <int KMAX>
size_t pil_resize_smem() {
  constexpr int kSpanX = resize_span_max(kRTW, KMAX), kSpanY = resize_span_max(kRTH, KMAX);
  return (size_t)kSpanY * resize_row_cap(kSpanX) + kWinPad + (size_t)(3 * kSpanY + kRowPad * KMAX) * kRTW;
}

template <int KMAX>
int launch_pil_resize(const sfod_resize_image *recs, int N, const int32_t *coeffs, uint8_t *out, int max_out_h, int max_out_w,
                      cudaStream_t st) {
  const size_t smem = pil_resize_smem<KMAX>();
  SFOD_CUDA_TRY(cudaFuncSetAttribute(pil_resize_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const dim3 grid((max_out_w + kRTW - 1) / kRTW, (max_out_h + kRTH - 1) / kRTH, N);
  pil_resize_kernel<KMAX><<<grid, kRThreads, smem, st>>>(recs, coeffs, out, max_out_h, max_out_w);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

}  // namespace

// =========================================================================== C ABI
SFOD_API int sfod_resize_pil(const sfod_resize_image *records_dev, int N, const int32_t *coeffs_dev, uint8_t *out, int max_out_h,
                             int max_out_w, int max_ksize, sfod_stream_t stream) {
  if (N < 0 || max_out_h <= 0 || max_out_w <= 0 || max_ksize <= 0) return SFOD_ERR_INVALID_ARG;
  if ((long long)max_out_h * max_out_w > 0x7FFFFFFFLL) return SFOD_ERR_INVALID_ARG;      // plane index must fit int32
  if (!records_dev || !coeffs_dev || !out) return SFOD_ERR_INVALID_ARG;
  if (max_ksize > kMaxKsize) return SFOD_ERR_UNSUPPORTED;
  if (N == 0) return SFOD_OK;
  if (N > 65535 || (max_out_h + kRTH - 1) / kRTH > 65535) return SFOD_ERR_UNSUPPORTED;   // grid limits
  const cudaStream_t st = sfod_cu(stream);
  if (max_ksize <= 3) return launch_pil_resize<3>(records_dev, N, coeffs_dev, out, max_out_h, max_out_w, st);
  if (max_ksize <= 5) return launch_pil_resize<5>(records_dev, N, coeffs_dev, out, max_out_h, max_out_w, st);
  if (max_ksize <= 7) return launch_pil_resize<7>(records_dev, N, coeffs_dev, out, max_out_h, max_out_w, st);
  return launch_pil_resize<9>(records_dev, N, coeffs_dev, out, max_out_h, max_out_w, st);
}
