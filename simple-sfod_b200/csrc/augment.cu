// augment.cu -- strong augmentation of the student's input on the GPU (SURVEY.md 8f rank 3).
// Replaces the CPU / PIL pipeline of reference daod/data/detection_utils.py:7-37 (applied per image in
// daod/data/mappers/two_crop_augmentation_mapper.py:141-157):
//     RandomApply([ColorJitter(0.4, 0.4, 0.4, 0.1)], p=0.8) -> RandomGrayscale(p=0.2) -> RandomApply([GaussianBlur((0.1, 2.0))], p=0.5)
//     -> ToTensor -> 3 x RandomErasing(value="random") -> ToPILImage
// on batches of uint8 CHW images that already live in HBM.  The random DECISIONS (which ops, in which order, which factors,
// sigma, rectangles) are drawn on the host exactly as torchvision draws them and handed over as small per-image parameter
// records; the kernels do the pixel work.
//
// Arithmetic contract (this TU is compiled with -fmad=false; every op is separately rounded):
//   * brightness / contrast / saturation / hue / grayscale follow Pillow's arithmetic (jitter_pixel): the reference's mapper hands
//     PIL images to the transforms, so torchvision's PIL path (ImageEnhance / Image.convert) is what the reference executes -- bit-exact;
//   * Gaussian blur: pil_blur_kernel reproduces Pillow's ImageFilter.GaussianBlur (three extended-box passes per axis in 8.24
//     fixed point) bit for bit -- the reference's filter;
//   * erasing writes byte(255 * v) (v ~ N(0, 1) from a counter-based generator, or a caller-provided noise tensor) into the
//     rectangles, which is what ToTensor -> erase(value="random") -> ToPILImage (`pic.mul(255).byte()`) leaves there.
#include "common.cuh"

namespace {

constexpr int kJThreads = 256;
constexpr int kOpBrightness = 0, kOpContrast = 1, kOpSaturation = 2, kOpHue = 3;

struct JitterRec {     // one per image; mirrors sfod_jitter_params
  int n_ops;           // 0..4 (0: ColorJitter not applied)
  int op[4];           // application order (torchvision: a random permutation of 0..3)
  float factor[4];     // blend alpha of op[k] (float32 of the Python float)
  int hue_shift[4];    // hue op: the shift byte uint8(int32(255 * hue)); ignored for the other ops
  int grayscale;       // RandomGrayscale hit: 3-channel gray AFTER the jitter
};

// ---- ColorJitter / RandomGrayscale in PILLOW's arithmetic: the reference hands PIL images to torchvision's transforms
// (daod/data/mappers/two_crop_augmentation_mapper.py:141-157), whose PIL path is ImageEnhance / Image.convert.  Restated from
// Pillow's libImaging (Blend.c, Convert.c) and torchvision/transforms/_functional_pil.py and pinned against the installed Pillow
// (oracle/pil_cpu.py, tests): bit-exact.
//   convert("L"):   L = (19595 R + 38470 G + 7471 B + 0x8000) >> 16
//   Image.blend(degenerate, image, alpha): (UINT8)(float)(deg + alpha * (img - deg)), clipped to [0, 255] when alpha is outside [0, 1]
//   Brightness: degenerate = 0;  Contrast: degenerate = int(mean(L) + 0.5);  Color (saturation): degenerate = L
//   adjust_hue: convert("HSV") (colorsys in float / double, see below), h += uint8(int32(255 hue)) mod 256, convert back
__device__ __forceinline__ unsigned char pil_L(unsigned char r, unsigned char g, unsigned char b) {
  return (unsigned char)((r * 19595u + g * 38470u + b * 7471u + 0x8000u) >> 16);
}
__device__ __forceinline__ unsigned char pil_blend(int deg, unsigned char img, float alpha) {
  const float t = __fadd_rn((float)deg, __fmul_rn(alpha, (float)((int)img - deg)));
  if (alpha >= 0.0f && alpha <= 1.0f) return (unsigned char)(int)t;
  return t <= 0.0f ? (unsigned char)0 : t >= 255.0f ? (unsigned char)255 : (unsigned char)(int)t;
}
__device__ __forceinline__ int clip8(int v) { return v < 0 ? 0 : v > 255 ? 255 : v; }
__device__ __forceinline__ void pil_hue_shift(unsigned char &R, unsigned char &G, unsigned char &B, int shift) {
  // rgb2hsv_row (Convert.c): float h, s, rc, gc, bc, cr; the literals 2.0 / 4.0 / 6.0 / 255.0 are doubles
  const int r = R, g = G, b = B;
  const int maxc = max(r, max(g, b)), minc = min(r, min(g, b));
  int uh = 0, us = 0;
  const int uv = maxc;
  if (minc != maxc) {
    const float cr = (float)(maxc - minc);
    const float s = __fdiv_rn(cr, (float)maxc);
    const float rc = __fdiv_rn((float)(maxc - r), cr), gc = __fdiv_rn((float)(maxc - g), cr), bc = __fdiv_rn((float)(maxc - b), cr);
    float h;
    if (r == maxc) h = __fsub_rn(bc, gc);
    else if (g == maxc) h = (float)(__dsub_rn(__dadd_rn(2.0, (double)rc), (double)bc));
    else h = (float)(__dsub_rn(__dadd_rn(4.0, (double)gc), (double)rc));
    const double hd = __dadd_rn(__ddiv_rn((double)h, 6.0), 1.0);
    h = (float)(hd - floor(hd));                                   // fmod(x, 1.0) for x in (0, 2): exact
    uh = clip8((int)__dmul_rn((double)h, 255.0));
    us = clip8((int)__dmul_rn((double)s, 255.0));
  }
  uh = (uh + shift) & 255;
  // hsv2rgb (Convert.c)
  if (us == 0) { R = G = B = (unsigned char)uv; return; }
  const double h6 = __ddiv_rn(__dmul_rn((double)(float)uh, 6.0), 255.0);
  const int i = (int)floor(h6);
  const float f = (float)__dsub_rn(h6, (double)(float)i);
  const float fs = (float)__ddiv_rn((double)(float)us, 255.0);
  const double v = (double)(float)uv;
  const int pp = clip8((int)round(__dmul_rn(v, __dsub_rn(1.0, (double)fs))));
  const int qq = clip8((int)round(__dmul_rn(v, __dsub_rn(1.0, __dmul_rn((double)fs, (double)f)))));
  const int tt = clip8((int)round(__dmul_rn(v, __dsub_rn(1.0, __dmul_rn((double)fs, __dsub_rn(1.0, (double)f))))));
  int ro, go, bo;
  switch (i % 6) {
    case 0: ro = uv; go = tt; bo = pp; break;
    case 1: ro = qq; go = uv; bo = pp; break;
    case 2: ro = pp; go = uv; bo = tt; break;
    case 3: ro = pp; go = qq; bo = uv; break;
    case 4: ro = tt; go = pp; bo = uv; break;
    default: ro = uv; go = pp; bo = qq; break;
  }
  R = (unsigned char)ro; G = (unsigned char)go; B = (unsigned char)bo;
}

// applies ops [0, upto) of the record to one pixel; `mean` = int(mean(L) + 0.5) of the image at the point where contrast is applied
__device__ __forceinline__ void jitter_pixel(const JitterRec &p, int upto, int mean, unsigned char &r, unsigned char &g, unsigned char &b) {
  for (int k = 0; k < upto; ++k) {
    const float f = p.factor[k];
    switch (p.op[k]) {
      case kOpBrightness: r = pil_blend(0, r, f); g = pil_blend(0, g, f); b = pil_blend(0, b, f); break;
      case kOpContrast: r = pil_blend(mean, r, f); g = pil_blend(mean, g, f); b = pil_blend(mean, b, f); break;
      case kOpSaturation: { const int l = pil_L(r, g, b); r = pil_blend(l, r, f); g = pil_blend(l, g, f); b = pil_blend(l, b, f); break; }
      default: pil_hue_shift(r, g, b, p.hue_shift[k]); break;
    }
  }
}

__device__ __forceinline__ int contrast_pos(const JitterRec &p) {
  for (int k = 0; k < p.n_ops; ++k) if (p.op[k] == kOpContrast) return k;
  return -1;
}

// pass A: sum of the gray levels of every image at the point where its contrast op applies (exact integer sum)
__global__ void __launch_bounds__(kJThreads) jitter_gray_sum_kernel(const unsigned char *__restrict__ img, const JitterRec *__restrict__ recs,
                                                                    int HW, unsigned long long *__restrict__ sums) {
  const int n = blockIdx.y;
  const JitterRec p = recs[n];
  const int cp = contrast_pos(p);
  if (cp < 0) return;
  const unsigned char *R = img + (size_t)n * 3 * HW, *G = R + HW, *B = G + HW;
  unsigned int local = 0;
  for (int i = blockIdx.x * kJThreads + threadIdx.x; i < HW; i += gridDim.x * kJThreads) {
    unsigned char r = R[i], g = G[i], b = B[i];
    jitter_pixel(p, cp, 0, r, g, b);
    local += pil_L(r, g, b);
  }
  local = __reduce_add_sync(0xFFFFFFFFu, local);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(sums + n, (unsigned long long)local);
}

// pass B: the whole op sequence (+ RandomGrayscale) per pixel
__global__ void __launch_bounds__(kJThreads) jitter_apply_kernel(const unsigned char *__restrict__ img, const JitterRec *__restrict__ recs,
                                                                 const unsigned long long *__restrict__ sums, int HW,
                                                                 unsigned char *__restrict__ out) {
  const int n = blockIdx.y;
  const JitterRec p = recs[n];
  // ImageStat mean = sum / count as a Python float, then int(mean + 0.5)
  const int mean = contrast_pos(p) >= 0 ? (int)((double)sums[n] / (double)HW + 0.5) : 0;
  const unsigned char *R = img + (size_t)n * 3 * HW, *G = R + HW, *B = G + HW;
  unsigned char *Ro = out + (size_t)n * 3 * HW, *Go = Ro + HW, *Bo = Go + HW;
  for (int i = blockIdx.x * kJThreads + threadIdx.x; i < HW; i += gridDim.x * kJThreads) {
    unsigned char r = R[i], g = G[i], b = B[i];
    jitter_pixel(p, p.n_ops, mean, r, g, b);
    if (p.grayscale) { const unsigned char l = pil_L(r, g, b); r = g = b = l; }
    Ro[i] = r; Go[i] = g; Bo[i] = b;
  }
}

// ---- PIL's ImageFilter.GaussianBlur, bit for bit.  The reference blurs with Pillow (reference daod/data/transforms/augmentations.py:18-21:
// x.filter(ImageFilter.GaussianBlur(radius=sigma))), which is NOT a Gaussian convolution: libImaging/BoxBlur.c approximates it with
// three passes of an "extended box blur" per axis (rows first, then columns), each pass in 8.24 fixed point and rounded to uint8:
//   out[x] = (ww * sum_{|d| <= r} in[c(x + d)] + fw * (in[c(x - r - 1)] + in[c(x + r + 1)]) + 2^23) >> 24,   c = clamp to the line,
// r = int(R), ww = uint32(2^24 / (2 R + 1)), fw = (2^24 - (2 r + 1) ww) / 2, R = the fractional box radius derived from sigma (host,
// ops.pil_blur_params).  All six passes run on one shared-memory tile: 32 x 32 outputs plus a halo of 3 (r + 1) pixels per side;
// every pass clamps in IMAGE coordinates, exactly as the line-by-line C code does, so borders are identical too.
constexpr int kPilMaxRadius = 9;   // box radius; sigma <= ~10
constexpr int kTile = 32;

__global__ void __launch_bounds__(256) pil_blur_kernel(const unsigned char *__restrict__ img, const int *__restrict__ radius,
                                                       const unsigned *__restrict__ wws, const unsigned *__restrict__ fws, int H, int W,
                                                       unsigned char *__restrict__ out) {
  extern __shared__ unsigned char pb_smem[];
  const int plane = blockIdx.z;          // n * 3 + c
  const int n = plane / 3;
  const int r = radius[n];
  const unsigned char *src = img + (size_t)plane * H * W;
  unsigned char *dst = out + (size_t)plane * H * W;
  const int x0 = blockIdx.x * kTile, y0 = blockIdx.y * kTile;
  if (r < 0) {                            // not blurred: copy
    for (int t = threadIdx.x; t < kTile * kTile; t += 256) {
      const int y = y0 + t / kTile, x = x0 + t % kTile;
      if (y < H && x < W) dst[(size_t)y * W + x] = src[(size_t)y * W + x];
    }
    return;
  }
  const unsigned ww = wws[n], fw = fws[n];
  const int h = 3 * (r + 1), TW = kTile + 2 * h;
  unsigned char *A = pb_smem, *B = pb_smem + TW * TW;
  const int ox = x0 - h, oy = y0 - h;     // image coordinates of tile cell (0, 0)
  for (int t = threadIdx.x; t < TW * TW; t += 256) {
    const int ty = t / TW, tx = t - ty * TW;
    const int y = min(max(oy + ty, 0), H - 1), x = min(max(ox + tx, 0), W - 1);
    A[t] = src[(size_t)y * W + x];
  }
  __syncthreads();
  // three horizontal passes over every row of the tile that lies inside the image
  for (int p = 1; p <= 3; ++p) {
    const int lo = p * (r + 1), wid = TW - 2 * lo;
    for (int t = threadIdx.x; t < TW * wid; t += 256) {
      const int ty = t / wid, tx = lo + (t - ty * wid);
      const int yi = oy + ty, xi = ox + tx;
      if (yi < 0 || yi >= H || xi < 0 || xi >= W) continue;
      const unsigned char *row = A + ty * TW;
      unsigned acc = 0;
      for (int d = -r; d <= r; ++d) acc += row[min(max(xi + d, 0), W - 1) - ox];
      const unsigned far = (unsigned)row[min(max(xi - r - 1, 0), W - 1) - ox] + (unsigned)row[min(max(xi + r + 1, 0), W - 1) - ox];
      B[ty * TW + tx] = (unsigned char)((acc * ww + far * fw + (1u << 23)) >> 24);
    }
    __syncthreads();
    unsigned char *tmp = A; A = B; B = tmp;
  }
  // three vertical passes over the output columns
  for (int p = 1; p <= 3; ++p) {
    const int lo = p * (r + 1), hgt = TW - 2 * lo;
    for (int t = threadIdx.x; t < hgt * kTile; t += 256) {
      const int ty = lo + t / kTile, tx = h + t % kTile;
      const int yi = oy + ty, xi = ox + tx;
      if (yi < 0 || yi >= H || xi >= W) continue;
      unsigned acc = 0;
      for (int d = -r; d <= r; ++d) acc += A[(min(max(yi + d, 0), H - 1) - oy) * TW + tx];
      const unsigned far = (unsigned)A[(min(max(yi - r - 1, 0), H - 1) - oy) * TW + tx] + (unsigned)A[(min(max(yi + r + 1, 0), H - 1) - oy) * TW + tx];
      B[ty * TW + tx] = (unsigned char)((acc * ww + far * fw + (1u << 23)) >> 24);
    }
    __syncthreads();
    unsigned char *tmp = A; A = B; B = tmp;
  }
  for (int t = threadIdx.x; t < kTile * kTile; t += 256) {
    const int ty = t / kTile, tx = t - ty * kTile;
    const int y = y0 + ty, x = x0 + tx;
    if (y < H && x < W) dst[(size_t)y * W + x] = A[(h + ty) * TW + h + tx];
  }
}

// ---- RandomErasing(value="random"): up to kMaxRects rectangles per image, applied in order
constexpr int kMaxRects = 4;
struct EraseRec { int n_rects; int rect[kMaxRects][4]; };   // (i, j, h, w) = top, left, height, width

__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// byte(255 * v): float -> int32 (truncation) -> low 8 bits, the value ToPILImage's `pic.mul(255).byte()` stores on x86
__device__ __forceinline__ unsigned char noise_byte(float v) { return (unsigned char)(__float2int_rz(__fmul_rn(v, 255.0f)) & 0xFF); }

__global__ void __launch_bounds__(256) erase_kernel(unsigned char *__restrict__ img, const EraseRec *__restrict__ recs,
                                                    const float *__restrict__ noise /* (N, kMaxRects, 3, H, W) or NULL */, int H, int W,
                                                    unsigned long long seed) {
  const int n = blockIdx.z / kMaxRects, k = blockIdx.z % kMaxRects;
  const EraseRec p = recs[n];
  if (k >= p.n_rects) return;
  const int i0 = p.rect[k][0], j0 = p.rect[k][1], h = p.rect[k][2], w = p.rect[k][3];
  // a later rectangle overwrites an earlier one: pixel ownership = the LAST rectangle that covers it
  const long long total = (long long)3 * h * w;
  for (long long t = (long long)blockIdx.x * 256 + threadIdx.x; t < total; t += (long long)gridDim.x * 256) {
    const int c = (int)(t / ((long long)h * w));
    const int rem = (int)(t - (long long)c * h * w);
    const int y = i0 + rem / w, x = j0 + rem % w;
    bool owned = true;
    for (int q = k + 1; q < p.n_rects; ++q)
      owned = owned && !(y >= p.rect[q][0] && y < p.rect[q][0] + p.rect[q][2] && x >= p.rect[q][1] && x < p.rect[q][1] + p.rect[q][3]);
    if (!owned) continue;
    float v;
    if (noise) {
      v = noise[((((size_t)n * kMaxRects + k) * 3 + c) * H + y) * W + x];
    } else {   // Box-Muller on two counter-based uniforms
      const unsigned long long key = mix64(seed + 0x9E3779B97F4A7C15ull * (((unsigned long long)(n * kMaxRects + k) << 40) | ((unsigned long long)c << 36) | (unsigned long long)(y * W + x)));
      const float u1 = ((float)(unsigned int)(key >> 40) + 1.0f) * (1.0f / 16777217.0f);   // (0, 1)
      const float u2 = (float)(unsigned int)((key >> 8) & 0xFFFFFFu) * (1.0f / 16777216.0f);
      v = sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
    }
    img[((size_t)n * 3 + c) * H * W + (size_t)y * W + x] = noise_byte(v);
  }
}

}  // namespace

// =========================================================================== C ABI
SFOD_API int sfod_color_jitter_pil(const uint8_t *images, int N, int H, int W, const sfod_jitter_params *params_dev, void *workspace,
                                   size_t workspace_bytes, uint8_t *out, sfod_stream_t stream) {
  static_assert(sizeof(sfod_jitter_params) == sizeof(JitterRec), "parameter record layout");
  if (N < 0 || H <= 0 || W <= 0) return SFOD_ERR_INVALID_ARG;
  if (N == 0) return SFOD_OK;
  if (!images || !params_dev || !out) return SFOD_ERR_INVALID_ARG;
  if (!workspace || workspace_bytes < (size_t)N * sizeof(unsigned long long)) return SFOD_ERR_WORKSPACE_TOO_SMALL;
  cudaStream_t st = sfod_cu(stream);
  unsigned long long *sums = static_cast<unsigned long long *>(workspace);
  SFOD_CUDA_TRY(cudaMemsetAsync(sums, 0, (size_t)N * sizeof(unsigned long long), st));
  const int HW = H * W;
  const unsigned gx = (unsigned)min(SFOD_NUM_SMS * 2, (HW + kJThreads - 1) / kJThreads);
  const JitterRec *recs = reinterpret_cast<const JitterRec *>(params_dev);
  jitter_gray_sum_kernel<<<dim3(gx, N), kJThreads, 0, st>>>(images, recs, HW, sums);
  SFOD_LAUNCH_CHECK();
  jitter_apply_kernel<<<dim3(gx, N), kJThreads, 0, st>>>(images, recs, sums, HW, out);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

SFOD_API int sfod_gaussian_blur_pil(const uint8_t *images, int N, int H, int W, const int32_t *radius_dev, const uint32_t *ww_dev,
                                    const uint32_t *fw_dev, int max_radius, uint8_t *out, sfod_stream_t stream) {
  if (N < 0 || H <= 0 || W <= 0 || max_radius < 0 || max_radius > kPilMaxRadius) return SFOD_ERR_INVALID_ARG;
  if (N == 0) return SFOD_OK;
  if (!images || !radius_dev || !ww_dev || !fw_dev || !out || images == out) return SFOD_ERR_INVALID_ARG;
  const int TW = kTile + 6 * (max_radius + 1);
  const size_t smem = 2 * (size_t)TW * TW;
  SFOD_CUDA_TRY(cudaFuncSetAttribute(pil_blur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((W + kTile - 1) / kTile, (H + kTile - 1) / kTile, N * 3);
  pil_blur_kernel<<<grid, 256, smem, sfod_cu(stream)>>>(images, radius_dev, ww_dev, fw_dev, H, W, out);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

SFOD_API int sfod_random_erase(uint8_t *images, int N, int H, int W, const sfod_erase_params *params_dev, const float *noise,
                               uint64_t seed, sfod_stream_t stream) {
  static_assert(sizeof(sfod_erase_params) == sizeof(EraseRec), "parameter record layout");
  if (N < 0 || H <= 0 || W <= 0) return SFOD_ERR_INVALID_ARG;
  if (N == 0) return SFOD_OK;
  if (!images || !params_dev) return SFOD_ERR_INVALID_ARG;
  dim3 grid(64, 1, N * kMaxRects);
  erase_kernel<<<grid, 256, 0, sfod_cu(stream)>>>(images, reinterpret_cast<const EraseRec *>(params_dev), noise, H, W,
                                                 (unsigned long long)seed);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}
