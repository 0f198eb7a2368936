// roi.cu -- ROIAlign (V1/V2) and ROIPool, forward and backward.
// Replaces torchvision.ops.roi_align / roi_pool as reached from d2 ROIPooler, constructed at reference
// daod/modeling/roi_heads/source_free_adaptive_teacher_roi_heads.py:42-47 and called at :117.
//
// Forward is write-bound: 100 352 B of output per VGG ROI against a 1.36 MB, L2-resident feature map
// (SURVEY.md 8d: 202.1 MB algorithmic for 2000 ROIs).  The fast kernel therefore
//   * reads a channels-last (NHWC) feature map so that one warp load covers 64 consecutive channels of
//     one pixel (fully coalesced), instead of torchvision's 4 scattered scalar taps per output element;
//   * exploits that bilinear sampling + bin averaging is separable: out = A . F . B^T per channel, with
//     A (PH x H) and B (PW x W) built once per ROI in shared memory -- each feature pixel of the ROI
//     region is loaded once per thread, not once per overlapping sample tap;
//   * stages the (256 channels x 49 bins) output tile in shared memory with a bank-conflict-free lane
//     permutation and writes it with ONE cp.async.bulk (TMA bulk) store of 50 176 contiguous bytes.
// The result differs from torchvision's per-sample summation order by a few ulp (<= 1e-5 relative,
// tested); `exact` selects a gather kernel that reproduces torchvision's order bit for bit.
#include "common.cuh"

namespace {

// --------------------------------------------------------------------------- layout transposes
// (N, C, HW) <-> (N, HW, C), 32x32 shared-memory tiles, coalesced on both sides.
__global__ void __launch_bounds__(256) transpose_kernel(const float *__restrict__ src, float *__restrict__ dst, int rows,
                                                        int cols) {
  // src: (batch, rows, cols) -> dst: (batch, cols, rows)
  __shared__ float tile[32][33];
  const size_t boff = (size_t)blockIdx.z * rows * cols;
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int i = ty; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + tx;
    if (r < rows && c < cols) tile[i][tx] = src[boff + (size_t)r * cols + c];
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + tx;
    if (r < rows && c < cols) dst[boff + (size_t)c * rows + r] = tile[tx][i];
  }
}

int launch_transpose(const float *src, float *dst, int batch, int rows, int cols, cudaStream_t st) {
  if (batch <= 0 || rows <= 0 || cols <= 0) return SFOD_OK;
  dim3 grid((cols + 31) / 32, (rows + 31) / 32, batch);
  transpose_kernel<<<grid, 256, 0, st>>>(src, dst, rows, cols);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

// --------------------------------------------------------------------------- ROI geometry (torchvision order)
struct RoiGeom {
  int n;                 // batch index
  float sh, sw, bh, bw;  // roi start (h, w), bin size
  int gh, gw;            // sampling grid
};

__device__ __forceinline__ RoiGeom roi_geometry(const float *__restrict__ roi, float scale, int aligned, int PH, int PW,
                                                int sampling_ratio) {
  RoiGeom g;
  g.n = (int)roi[0];
  const float offset = aligned ? 0.5f : 0.0f;
  const float rsw = __fsub_rn(__fmul_rn(roi[1], scale), offset);
  const float rsh = __fsub_rn(__fmul_rn(roi[2], scale), offset);
  const float rew = __fsub_rn(__fmul_rn(roi[3], scale), offset);
  const float reh = __fsub_rn(__fmul_rn(roi[4], scale), offset);
  float rw = __fsub_rn(rew, rsw), rh = __fsub_rn(reh, rsh);
  if (!aligned) { rw = fmaxf(rw, 1.0f); rh = fmaxf(rh, 1.0f); }
  g.bh = __fdiv_rn(rh, (float)PH);
  g.bw = __fdiv_rn(rw, (float)PW);
  g.gh = sampling_ratio > 0 ? sampling_ratio : (int)ceilf(__fdiv_rn(rh, (float)PH));
  g.gw = sampling_ratio > 0 ? sampling_ratio : (int)ceilf(__fdiv_rn(rw, (float)PW));
  g.sh = rsh; g.sw = rsw;
  return g;
}

// sample coordinate: start + p * bin + (i + .5) * bin / grid   (left-to-right, separately rounded)
__device__ __forceinline__ float sample_coord(float start, int p, float bin, int i, int grid) {
  return __fadd_rn(__fadd_rn(start, __fmul_rn((float)p, bin)), __fdiv_rn(__fmul_rn((float)i + 0.5f, bin), (float)grid));
}

// 1-D half of torchvision's bilinear_interpolate: returns false when the sample is outside [-1, size].
__device__ __forceinline__ bool bilinear_1d(float v, int size, int &lo, int &hi, float &l, float &h) {
  if (v < -1.0f || v > (float)size) return false;
  if (v <= 0.f) v = 0.f;
  lo = (int)v;
  if (lo >= size - 1) { hi = lo = size - 1; v = (float)lo; } else hi = lo + 1;
  l = __fsub_rn(v, (float)lo);
  h = __fsub_rn(1.0f, l);
  return true;
}

// --------------------------------------------------------------------------- exact forward (NCHW gather)
// One thread per output element; the summation order is torchvision's:
//   val += ((w1*v1 + w2*v2) + w3*v3) + w4*v4 over (iy, ix), then val / count.
__global__ void __launch_bounds__(256) roi_align_fwd_exact_kernel(const float *__restrict__ input, const float *__restrict__ rois,
                                                                  int N, int C, int H, int W, long long total, int PH, int PW,
                                                                  float scale, int sampling_ratio, int aligned,
                                                                  float *__restrict__ output) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int pw = (int)(idx % PW), ph = (int)((idx / PW) % PH);
  const int c = (int)((idx / ((long long)PW * PH)) % C);
  const long long r = idx / ((long long)PW * PH * C);
  const RoiGeom g = roi_geometry(rois + 5 * r, scale, aligned, PH, PW, sampling_ratio);
  float val = 0.f;
  if (g.n >= 0 && g.n < N) {
    const float *in = input + ((size_t)g.n * C + c) * H * W;
    for (int iy = 0; iy < g.gh; ++iy) {
      const float y = sample_coord(g.sh, ph, g.bh, iy, g.gh);
      int yl, yh; float ly, hy;
      const bool yok = bilinear_1d(y, H, yl, yh, ly, hy);
      for (int ix = 0; ix < g.gw; ++ix) {
        const float x = sample_coord(g.sw, pw, g.bw, ix, g.gw);
        int xl, xh; float lx, hx;
        if (!yok || !bilinear_1d(x, W, xl, xh, lx, hx)) continue;
        const float w1 = __fmul_rn(hy, hx), w2 = __fmul_rn(hy, lx), w3 = __fmul_rn(ly, hx), w4 = __fmul_rn(ly, lx);
        float t = __fadd_rn(__fmul_rn(w1, in[yl * W + xl]), __fmul_rn(w2, in[yl * W + xh]));
        t = __fadd_rn(t, __fmul_rn(w3, in[yh * W + xl]));
        t = __fadd_rn(t, __fmul_rn(w4, in[yh * W + xh]));
        val = __fadd_rn(val, t);
      }
    }
  }
  int cnt = g.gh * g.gw; if (cnt < 1) cnt = 1;
  output[idx] = __fdiv_rn(val, (float)cnt);
}

// generic backward (NCHW, one thread per output-gradient element, atomics), torchvision's formulation
__global__ void __launch_bounds__(256) roi_align_bwd_generic_kernel(const float *__restrict__ grad_out,
                                                                    const float *__restrict__ rois, int N, int C, int H, int W,
                                                                    long long total, int PH, int PW, float scale,
                                                                    int sampling_ratio, int aligned, float *__restrict__ grad_in) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int pw = (int)(idx % PW), ph = (int)((idx / PW) % PH);
  const int c = (int)((idx / ((long long)PW * PH)) % C);
  const long long r = idx / ((long long)PW * PH * C);
  const RoiGeom g = roi_geometry(rois + 5 * r, scale, aligned, PH, PW, sampling_ratio);
  if (g.n < 0 || g.n >= N) return;
  const float go = grad_out[idx];
  const float count = (float)(g.gh * g.gw);
  float *gi = grad_in + ((size_t)g.n * C + c) * H * W;
  for (int iy = 0; iy < g.gh; ++iy) {
    const float y = sample_coord(g.sh, ph, g.bh, iy, g.gh);
    int yl, yh; float ly, hy;
    if (!bilinear_1d(y, H, yl, yh, ly, hy)) continue;
    for (int ix = 0; ix < g.gw; ++ix) {
      const float x = sample_coord(g.sw, pw, g.bw, ix, g.gw);
      int xl, xh; float lx, hx;
      if (!bilinear_1d(x, W, xl, xh, lx, hx)) continue;
      atomicAdd(gi + yl * W + xl, __fdiv_rn(__fmul_rn(go, __fmul_rn(hy, hx)), count));
      atomicAdd(gi + yl * W + xh, __fdiv_rn(__fmul_rn(go, __fmul_rn(hy, lx)), count));
      atomicAdd(gi + yh * W + xl, __fdiv_rn(__fmul_rn(go, __fmul_rn(ly, hx)), count));
      atomicAdd(gi + yh * W + xh, __fdiv_rn(__fmul_rn(go, __fmul_rn(ly, lx)), count));
    }
  }
}

// --------------------------------------------------------------------------- separable fast path (7x7, NHWC)
// Bilinear sampling + bin averaging is separable: out = A . F . B^T per channel, A (7 x H) and B (7 x W) built once per
// ROI.  The kernels are bound by instruction issue and L2 latency, not by DRAM (the feature map is L2-resident and the
// 100 KB/ROI output is the only HBM traffic), so they are organised to minimise instructions and exposed latency:
//   * one work item = one ROI x 256 consecutive channels on a 128-thread CTA, 2 channels per thread (one LDG.64 per
//     pixel, a warp reads 256 contiguous bytes);
//   * forward: B is used in COMPACT form (each bin touches <= grid_w + 1 consecutive columns), its weights live in
//     registers, and the channel stride is a template constant so the 7 * NX pixel loads of a row are LDG.64 with
//     immediate offsets; backward and the wide-bin fallback use dense warp-uniform tables (2 LDS.128 per pixel);
//   * the 7 bin rows are produced in two passes (bins 0-3, then 4-6), which halves the accumulator registers
//     (28 pairs instead of 49) and lifts occupancy to 4 CTAs/SM; only rows shared by bins 3 and 4 are visited twice;
//   * the (256 x 49) output tile is staged in shared memory with a conflict-free lane permutation and leaves the SM
//     as ONE 50 176 B cp.async.bulk (TMA) store that drains while the next item is computed (persistent CTAs).
constexpr int kPH = 7, kPW = 7, kBins = kPH * kPW;
constexpr int kSepThreads = 128;           // 2 channels per thread
constexpr int kCT = 2 * kSepThreads;       // 256 channels per CTA
constexpr int kTileFloats = kCT * kBins;   // 12 544 floats = 50 176 B

struct SepSmem {
  float *tile;   // kTileFloats
  float *Ad;     // H * 8: Ad[y*8 + ph] = sum of y-weights of bin ph on row y, divided by grid_h
  float *Bd;     // W * 8
  int *lim;      // [0..3] ymin, ymax, xmin, xmax; [4..10] first row of bin ph; [11..17] last row of bin ph
                 // (the forward's table records add [18..26], see roi_sep_tables_kernel)
  float *Bc;     // forward only: compact column weights (see roi_sep_tables_kernel)
};
__host__ __device__ inline size_t sep_smem_bytes(int H, int W) {
  return (size_t)kTileFloats * 4 + (size_t)(H + W) * 8 * 4 + 32 * 4;
}
__device__ __forceinline__ SepSmem sep_carve(float *base, int H, int W) {
  SepSmem s;
  s.tile = base; s.Ad = base + kTileFloats; s.Bd = s.Ad + H * 8;
  s.lim = reinterpret_cast<int *>(s.Bd + W * 8);
  s.Bc = nullptr;
  return s;
}

// Build the dense separable weight tables of one ROI.  Called by all threads of the CTA.
__device__ __forceinline__ void sep_build_tables(const SepSmem &s, const RoiGeom &g, int H, int W) {
  const int tid = threadIdx.x;
  for (int i = tid; i < (H + W) * 8; i += blockDim.x) s.Ad[i] = 0.f;  // Ad and Bd are contiguous
  if (tid == 0) { s.lim[0] = H; s.lim[1] = -1; s.lim[2] = W; s.lim[3] = -1; }
  __syncthreads();
  if (tid < kPH) {
    const int ph = tid; int mn = H, mx = -1;
    const float inv = g.gh > 0 ? __fdiv_rn(1.0f, (float)g.gh) : 0.f;
    for (int iy = 0; iy < g.gh; ++iy) {
      int lo, hi; float l, h;
      if (!bilinear_1d(sample_coord(g.sh, ph, g.bh, iy, g.gh), H, lo, hi, l, h)) continue;
      s.Ad[lo * 8 + ph] += h * inv; s.Ad[hi * 8 + ph] += l * inv;
      mn = min(mn, lo); mx = max(mx, hi);
    }
    s.lim[4 + ph] = mn; s.lim[11 + ph] = mx;
    if (mx >= 0) { atomicMin(&s.lim[0], mn); atomicMax(&s.lim[1], mx); }
  } else if (tid >= 32 && tid < 32 + kPW) {
    const int pw = tid - 32; int mn = W, mx = -1;
    const float inv = g.gw > 0 ? __fdiv_rn(1.0f, (float)g.gw) : 0.f;
    for (int ix = 0; ix < g.gw; ++ix) {
      int lo, hi; float l, h;
      if (!bilinear_1d(sample_coord(g.sw, pw, g.bw, ix, g.gw), W, lo, hi, l, h)) continue;
      s.Bd[lo * 8 + pw] += h * inv; s.Bd[hi * 8 + pw] += l * inv;
      mn = min(mn, lo); mx = max(mx, hi);
    }
    if (mx >= 0) { atomicMin(&s.lim[2], mn); atomicMax(&s.lim[3], mx); }
  }
  __syncthreads();
}

// T[b] += B[x][b] * f for the two channels of this thread (weights are scalar, warp-uniform shared-memory broadcasts).
__device__ __forceinline__ void sep_row_fma(float2 (&T)[kPW], const float *__restrict__ bw, float2 f) {
  const float4 w0 = *reinterpret_cast<const float4 *>(bw), w1 = *reinterpret_cast<const float4 *>(bw + 4);
  T[0].x = fmaf(w0.x, f.x, T[0].x); T[0].y = fmaf(w0.x, f.y, T[0].y);
  T[1].x = fmaf(w0.y, f.x, T[1].x); T[1].y = fmaf(w0.y, f.y, T[1].y);
  T[2].x = fmaf(w0.z, f.x, T[2].x); T[2].y = fmaf(w0.z, f.y, T[2].y);
  T[3].x = fmaf(w0.w, f.x, T[3].x); T[3].y = fmaf(w0.w, f.y, T[3].y);
  T[4].x = fmaf(w1.x, f.x, T[4].x); T[4].y = fmaf(w1.x, f.y, T[4].y);
  T[5].x = fmaf(w1.y, f.x, T[5].x); T[5].y = fmaf(w1.y, f.y, T[5].y);
  T[6].x = fmaf(w1.z, f.x, T[6].x); T[6].y = fmaf(w1.z, f.y, T[6].y);
}

// Programmatic dependent launch: the table pre-kernel releases its dependents at once, the forward kernel is launched with
// programmatic stream serialization and blocks here until the pre-kernel's memory is visible -- launch latency and the
// prologue of the big kernel overlap the small one.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// ---- per-ROI table records (forward).  A small pre-kernel builds, for every ROI, the record the forward kernel needs:
//   ints  [0..31]  lim: [0..1] ymin, ymax; [2..3] xmin, xmax; [4..10] / [11..17] first / last row of bin ph;
//                       [18..24] first column of the compact window of bin pw; [25] window width of the ROI: 2, 3, 4, 6, 8
//                       (kNXMax + 1 = use the dense column tables); [26] image index (-1: invalid -> zero output); [27] ROI index
//   floats [32..87] Bc[pw*kNXMax + j]: weight of column lim[18+pw] + j for bin pw (the nonzero run of B's row pw)
//   floats [96..119] Bp[((pw>>1)*kNXPair + j)*2 + (pw&1)], pw < 6, j < kNXPair: the same weights with bins (0,1), (2,3), (4,5)
//                       interleaved -- the packed-fp32 slab forward loads a (bin 2i, bin 2i+1) weight pair with one 64-bit access
//   floats [128..128+8H) Ad[y*8 + ph], ph < 7; word y*8 + 7 holds (first bin fed by row y) | (number of such bins << 8)
// so that the persistent forward CTAs prefetch it with cp.async while they work on the previous ROI instead of spending
// ~20 % of their life in a latency-bound prologue (ROI load from DRAM, table build by 14 threads, two barriers).
constexpr int kNXMax = 8;                  // widest per-bin column window handled by the compact (sparse-in-x) forward
constexpr int kCostClasses = 16;           // ROI cost classes of the L2 forward's longest-processing-time-first order
constexpr int kNXPair = 4;                 // widest window the packed (slab) forward handles in compact form
constexpr int kRecPair = 96;               // first float of Bp
constexpr int kRecHead = 128;              // 32 ints + 7 x 8 compact weights + 3 x 4 weight pairs, padded
__host__ __device__ inline int sep_rec_floats(int H) { return kRecHead + 8 * H; }

__global__ void __launch_bounds__(128) roi_sep_tables_kernel(const float *__restrict__ rois, int R, int N, int H, int W, float scale,
                                                             int sampling_ratio, int aligned, float *__restrict__ recs,
                                                             int *__restrict__ bcnt, int *__restrict__ bucket) {
  extern __shared__ __align__(16) float tb_smem[];
  const int rec = sep_rec_floats(H);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 4 + warp;
  pdl_launch_dependents();   // the forward kernel may start its prologue; it waits (griddepcontrol.wait) before touching recs
  if (r >= R) return;
  float *my = tb_smem + (size_t)warp * rec;
  int *lim = reinterpret_cast<int *>(my);
  float *Bc = my + 32, *Ad = my + kRecHead;
  for (int i = lane; i < rec; i += 32) my[i] = 0.f;
  RoiGeom g = roi_geometry(rois + 5 * (size_t)r, scale, aligned, kPH, kPW, sampling_ratio);
  const bool valid = g.n >= 0 && g.n < N;
  if (!valid) { g.gh = 0; g.gw = 0; }
  __syncwarp();
  int ymn = H, ymx = -1, xmn = W, xmx = -1, nx = 0;
  if (lane < kPH) {
    const int ph = lane;
    const float inv = g.gh > 0 ? __fdiv_rn(1.0f, (float)g.gh) : 0.f;
    for (int iy = 0; iy < g.gh; ++iy) {
      int lo, hi; float l, h;
      if (!bilinear_1d(sample_coord(g.sh, ph, g.bh, iy, g.gh), H, lo, hi, l, h)) continue;
      Ad[lo * 8 + ph] += h * inv; Ad[hi * 8 + ph] += l * inv;
      ymn = min(ymn, lo); ymx = max(ymx, hi);
    }
    lim[4 + ph] = ymn; lim[11 + ph] = ymx;
  } else if (lane >= 8 && lane < 8 + kPW) {
    const int pw = lane - 8;
    for (int ix = 0; ix < g.gw; ++ix) {
      int lo, hi; float l, h;
      if (!bilinear_1d(sample_coord(g.sw, pw, g.bw, ix, g.gw), W, lo, hi, l, h)) continue;
      xmn = min(xmn, lo); xmx = max(xmx, hi);
    }
  }
  // window width of the ROI = widest bin, rounded up to a width the forward kernels are instantiated for
  const int bin_w = (lane >= 8 && lane < 8 + kPW && xmx >= 0) ? xmx - xmn + 1 : 0;
  const int wmax = __reduce_max_sync(0xFFFFFFFFu, bin_w);
  nx = wmax <= 2 ? 2 : wmax <= 3 ? 3 : wmax <= 4 ? 4 : wmax <= 6 ? 6 : wmax <= kNXMax ? kNXMax : kNXMax + 1;
  if (nx > W) nx = kNXMax + 1;   // map narrower than the window: dense tables
  if (lane >= 8 && lane < 8 + kPW) {
    const int pw = lane - 8;
    const float inv = g.gw > 0 ? __fdiv_rn(1.0f, (float)g.gw) : 0.f;
    // compact window [x0, x0 + nx) kept inside the row; it covers [xmn, xmx] because the bin is at most nx wide
    const int x0 = (xmx >= 0 && nx <= kNXMax) ? max(0, min(xmn, W - nx)) : 0;
    lim[18 + pw] = x0;
    if (nx <= kNXMax) {
      for (int ix = 0; ix < g.gw; ++ix) {   // same sample order as the dense table => identical sums
        int lo, hi; float l, h;
        if (!bilinear_1d(sample_coord(g.sw, pw, g.bw, ix, g.gw), W, lo, hi, l, h)) continue;
        Bc[pw * kNXMax + (lo - x0)] += h * inv; Bc[pw * kNXMax + (hi - x0)] += l * inv;
        if (pw < 6 && nx <= kNXPair) {   // same terms in the same order => identical sums
          float *Bp = my + kRecPair;
          Bp[(((pw >> 1) * kNXPair + (lo - x0)) << 1) + (pw & 1)] += h * inv; Bp[(((pw >> 1) * kNXPair + (hi - x0)) << 1) + (pw & 1)] += l * inv;
        }
      }
    }
  }
  ymn = __reduce_min_sync(0xFFFFFFFFu, ymn); ymx = __reduce_max_sync(0xFFFFFFFFu, ymx);
  xmn = __reduce_min_sync(0xFFFFFFFFu, xmn); xmx = __reduce_max_sync(0xFFFFFFFFu, xmx);
  if (lane == 0) {
    lim[0] = ymn; lim[1] = ymx; lim[2] = xmn; lim[3] = xmx; lim[25] = nx; lim[26] = valid ? g.n : -1; lim[27] = r;
    if (bucket) {   // cost class = log2 of the window area: the L2 forward pulls the most expensive ROIs first (LPT order)
      const int area = (ymx >= ymn && xmx >= xmn) ? (ymx - ymn + 1) * (xmx - xmn + 1) : 0;
      const int cls = area > 0 ? min(kCostClasses - 1, 32 - __clz(area)) : 0;
      bucket[(size_t)cls * R + atomicAdd(&bcnt[cls], 1)] = r;
    }
  }
  __syncwarp();
  for (int y = lane; y < H; y += 32) {   // bins fed by row y form a run [first, first + count): packed into the row's padding word
    int first = kPH, last = -1;
#pragma unroll
    for (int a = 0; a < kPH; ++a)
      if (Ad[y * 8 + a] != 0.f) { first = min(first, a); last = a; }
    Ad[y * 8 + 7] = __int_as_float(last >= 0 ? (first | ((last - first + 1) << 8)) : 0);
  }
  __syncwarp();
  float4 *dst = reinterpret_cast<float4 *>(recs + (size_t)r * rec);
  const float4 *src = reinterpret_cast<const float4 *>(my);
  for (int i = lane; i < rec / 4; i += 32) dst[i] = src[i];
}

// Dense column tables of one ROI for the rare wide-bin case (called by all threads of the CTA; CTA-uniform).
__device__ __forceinline__ void sep_build_x_dense(float *Bd, const RoiGeom &g, int W) {
  const int tid = threadIdx.x;
  for (int i = tid; i < W * 8; i += blockDim.x) Bd[i] = 0.f;
  __syncthreads();
  if (tid < kPW) {
    const int pw = tid;
    const float inv = g.gw > 0 ? __fdiv_rn(1.0f, (float)g.gw) : 0.f;
    for (int ix = 0; ix < g.gw; ++ix) {
      int lo, hi; float l, h;
      if (!bilinear_1d(sample_coord(g.sw, pw, g.bw, ix, g.gw), W, lo, hi, l, h)) continue;
      Bd[lo * 8 + pw] += h * inv; Bd[hi * 8 + pw] += l * inv;
    }
  }
  __syncthreads();
}

__device__ __forceinline__ void sep_tile_wait_free() {   // the previous ROI's bulk store has finished READING the tile
  if (threadIdx.x == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  __syncthreads();
}

// registers -> shared tile (flat [channel][49], the global layout).  Lanes 0-15 write their even channel while lanes
// 16-31 write their odd channel (and vice versa): word index (2*tid + j)*49 + k hits 32 distinct banks per instruction.
template <int PH0, int NPH, bool kFirst>
__device__ __forceinline__ void sep_store_acc(const float2 (&acc)[NPH][kPW], float *__restrict__ t0, float *__restrict__ t1, int half,
                                              bool active) {
  if (kFirst) sep_tile_wait_free();
  if (!active) return;
#pragma unroll
  for (int a = 0; a < NPH; ++a)
#pragma unroll
    for (int b = 0; b < kPW; ++b) {
      const float v0 = acc[a][b].x, v1 = acc[a][b].y;
      t0[(PH0 + a) * kPW + b] = half ? v1 : v0;
      t1[(PH0 + a) * kPW + b] = half ? v0 : v1;
    }
}

// One pass over the rows feeding bins [PH0, PH0 + NPH), dense column tables (2 LDS.128 of weights per pixel).
template <int PH0, int NPH, int kC>
__device__ __forceinline__ void sep_fwd_pass_dense(const SepSmem &s, const float2 *__restrict__ fbase2, int C, int W, int xmin, int xmax,
                                                   float *__restrict__ t0, float *__restrict__ t1, int half, bool active) {
  const int cs2 = (kC ? kC : C) >> 1;
  int y0 = s.lim[4 + PH0], y1 = s.lim[11 + PH0];
#pragma unroll
  for (int a = 1; a < NPH; ++a) { y0 = min(y0, s.lim[4 + PH0 + a]); y1 = max(y1, s.lim[11 + PH0 + a]); }
  float2 acc[NPH][kPW];
#pragma unroll
  for (int a = 0; a < NPH; ++a)
#pragma unroll
    for (int b = 0; b < kPW; ++b) acc[a][b] = make_float2(0.f, 0.f);
  for (int y = y0; y <= y1; ++y) {
    float2 T[kPW];
#pragma unroll
    for (int b = 0; b < kPW; ++b) T[b] = make_float2(0.f, 0.f);
    const float2 *prow = fbase2 + (size_t)y * W * cs2;
    for (int x = xmin; x <= xmax; ++x) sep_row_fma(T, s.Bd + x * 8, __ldg(prow + (size_t)x * cs2));
    const float4 av4 = *reinterpret_cast<const float4 *>(s.Ad + y * 8 + PH0);   // PH0 in {0, 4}: 16-byte aligned
    const float av[4] = {av4.x, av4.y, av4.z, av4.w};
#pragma unroll
    for (int a = 0; a < NPH; ++a) {
      if (av[a] != 0.f) {  // warp-uniform (broadcast shared-memory value)
#pragma unroll
        for (int b = 0; b < kPW; ++b) { acc[a][b].x = fmaf(av[a], T[b].x, acc[a][b].x); acc[a][b].y = fmaf(av[a], T[b].y, acc[a][b].y); }
      }
    }
  }
  sep_store_acc<PH0, NPH, PH0 == 0>(acc, t0, t1, half, active);
}

// The same pass with the column weights in compact form.  With the adaptive sampling grid every bin touches at most
// grid_w + 1 consecutive columns, so instead of 7 (mostly zero) weights per pixel of the ROI's bounding box a row costs
// 7 * NX pixel loads with ONE register-resident weight each: no weight traffic on the shared-memory crossbar and
// NX / (7 ns) of the FMAs.  Summation order per bin (ascending x) is that of the dense pass; the skipped terms are exact
// zeros.  NX = widest bin window of this ROI rounded up to a template instance; narrower bins carry zero weights.
template <int PH0, int NPH, int kC, int NX>
__device__ __forceinline__ void sep_fwd_pass_compact(const SepSmem &s, const float2 *__restrict__ fbase2, int C, int W,
                                                     float *__restrict__ t0, float *__restrict__ t1, int half, bool active) {
  const int cs2 = (kC ? kC : C) >> 1;
  int y0 = s.lim[4 + PH0], y1 = s.lim[11 + PH0];
#pragma unroll
  for (int a = 1; a < NPH; ++a) { y0 = min(y0, s.lim[4 + PH0 + a]); y1 = max(y1, s.lim[11 + PH0 + a]); }
  float bw[kPW][NX];
  int xo[kPW];
#pragma unroll
  for (int b = 0; b < kPW; ++b) {
    xo[b] = s.lim[18 + b] * cs2;
#pragma unroll
    for (int j = 0; j < NX; ++j) bw[b][j] = s.Bc[b * kNXMax + j];
  }
  float2 acc[NPH][kPW];
#pragma unroll
  for (int a = 0; a < NPH; ++a)
#pragma unroll
    for (int b = 0; b < kPW; ++b) acc[a][b] = make_float2(0.f, 0.f);
  // NX == 2 (the common case) is software-pipelined: the pixel loads of row y + 1 are issued before the accumulation of
  // row y, so each warp keeps a row of loads in flight while it (or its neighbours) issue FMAs; wider windows would spill
  constexpr bool kPipe = NX <= 2;
  float2 f[kPW][NX];
  if (kPipe) {
    const float2 *prow = fbase2 + (size_t)y0 * W * cs2;
#pragma unroll
    for (int b = 0; b < kPW; ++b)
#pragma unroll
      for (int j = 0; j < NX; ++j) f[b][j] = __ldg(prow + xo[b] + j * cs2);
  }
  for (int y = y0; y <= y1; ++y) {
    if (!kPipe) {
      const float2 *prow = fbase2 + (size_t)y * W * cs2;
#pragma unroll
      for (int b = 0; b < kPW; ++b)
#pragma unroll
        for (int j = 0; j < NX; ++j) f[b][j] = __ldg(prow + xo[b] + j * cs2);
    }
    float2 T[kPW];
#pragma unroll
    for (int b = 0; b < kPW; ++b) {
      T[b] = make_float2(bw[b][0] * f[b][0].x, bw[b][0] * f[b][0].y);
#pragma unroll
      for (int j = 1; j < NX; ++j) { T[b].x = fmaf(bw[b][j], f[b][j].x, T[b].x); T[b].y = fmaf(bw[b][j], f[b][j].y, T[b].y); }
    }
    if (kPipe && y < y1) {
      const float2 *prow = fbase2 + (size_t)(y + 1) * W * cs2;
#pragma unroll
      for (int b = 0; b < kPW; ++b)
#pragma unroll
        for (int j = 0; j < NX; ++j) f[b][j] = __ldg(prow + xo[b] + j * cs2);
    }
    const float4 av4 = *reinterpret_cast<const float4 *>(s.Ad + y * 8 + PH0);
    const float av[4] = {av4.x, av4.y, av4.z, av4.w};
#pragma unroll
    for (int a = 0; a < NPH; ++a) {
      if (av[a] != 0.f) {
#pragma unroll
        for (int b = 0; b < kPW; ++b) { acc[a][b].x = fmaf(av[a], T[b].x, acc[a][b].x); acc[a][b].y = fmaf(av[a], T[b].y, acc[a][b].y); }
      }
    }
  }
  sep_store_acc<PH0, NPH, PH0 == 0>(acc, t0, t1, half, active);
}

// Compact pass for wider windows (NX = 6 or 8, ROIs with a 5..7 sample grid per bin -- common on stride-16 maps): the
// weights are shared-memory broadcasts and a bin's NX pixels are loaded and folded one bin at a time; still NX / (7 ns)
// of the dense pass's FMAs and one LDS.32 instead of two LDS.128 per pixel load.
template <int PH0, int NPH, int kC, int NX>
__device__ __forceinline__ void sep_fwd_pass_compact_wide(const SepSmem &s, const float2 *__restrict__ fbase2, int C, int W,
                                                          float *__restrict__ t0, float *__restrict__ t1, int half, bool active) {
  const int cs2 = (kC ? kC : C) >> 1;
  int y0 = s.lim[4 + PH0], y1 = s.lim[11 + PH0];
#pragma unroll
  for (int a = 1; a < NPH; ++a) { y0 = min(y0, s.lim[4 + PH0 + a]); y1 = max(y1, s.lim[11 + PH0 + a]); }
  int xo[kPW];
#pragma unroll
  for (int b = 0; b < kPW; ++b) xo[b] = s.lim[18 + b] * cs2;
  float2 acc[NPH][kPW];
#pragma unroll
  for (int a = 0; a < NPH; ++a)
#pragma unroll
    for (int b = 0; b < kPW; ++b) acc[a][b] = make_float2(0.f, 0.f);
  for (int y = y0; y <= y1; ++y) {
    const float2 *prow = fbase2 + (size_t)y * W * cs2;
    float2 T[kPW];
#pragma unroll
    for (int b = 0; b < kPW; ++b) {
      float2 f[NX];
#pragma unroll
      for (int j = 0; j < NX; ++j) f[j] = __ldg(prow + xo[b] + j * cs2);
      const float *wb = s.Bc + b * kNXMax;
      T[b] = make_float2(wb[0] * f[0].x, wb[0] * f[0].y);
#pragma unroll
      for (int j = 1; j < NX; ++j) { T[b].x = fmaf(wb[j], f[j].x, T[b].x); T[b].y = fmaf(wb[j], f[j].y, T[b].y); }
    }
    const float4 av4 = *reinterpret_cast<const float4 *>(s.Ad + y * 8 + PH0);
    const float av[4] = {av4.x, av4.y, av4.z, av4.w};
#pragma unroll
    for (int a = 0; a < NPH; ++a) {
      if (av[a] != 0.f) {
#pragma unroll
        for (int b = 0; b < kPW; ++b) { acc[a][b].x = fmaf(av[a], T[b].x, acc[a][b].x); acc[a][b].y = fmaf(av[a], T[b].y, acc[a][b].y); }
      }
    }
  }
  sep_store_acc<PH0, NPH, PH0 == 0>(acc, t0, t1, half, active);
}

__host__ __device__ inline size_t sep_fwd_smem_bytes(int H, int W) {
  // output tile, two table records (current ROI / prefetched next ROI), dense column table of the fallback, work-item slots
  return (size_t)kTileFloats * 4 + 2 * (size_t)sep_rec_floats(H) * 4 + (size_t)W * 8 * 4 + 16;
}

// Persistent forward: CTAs pull (ROI, 256-channel slab) items from a global counter.  Per item and CTA: two barriers, no
// global-memory latency outside the row loops -- the table record of the NEXT item streams in through cp.async and the
// bulk store of the PREVIOUS item drains while the rows of the current one are accumulated.
template <int kC>
__global__ void __launch_bounds__(kSepThreads, 3) roi_align_fwd_sep_kernel(const float *__restrict__ feat /* NHWC */,
                                                                           const float *__restrict__ rois,
                                                                           const float *__restrict__ recs,
                                                                           unsigned *__restrict__ counter, const int *__restrict__ bcnt,
                                                                           const int *__restrict__ bucket, int N, int C, int H,
                                                                           int W, int R, float scale, int sampling_ratio,
                                                                           int aligned, float *__restrict__ output) {
  extern __shared__ __align__(128) float sep_smem[];
  const int rec = sep_rec_floats(H);
  float *tile = sep_smem, *tab = tile + kTileFloats, *Bd = tab + 2 * rec;
  int *s_item = reinterpret_cast<int *>(Bd + W * 8);
  const int tid = threadIdx.x;
  const int nslab = (C + kCT - 1) / kCT;
  const int nitems = R * nslab;
  int cur = blockIdx.x;
  if (cur >= nitems) return;
  unsigned long long l2_stream;   // the output stream must not evict the feature map from L2
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(l2_stream));
  // Items are pulled in order of DECREASING ROI cost (window area classes filled by the table kernel): with a few hundred
  // items per CTA and ROI costs spanning two orders of magnitude (2 x 2 ... 38 x 75 cells), arrival order leaves the tail of
  // the launch to whichever CTA drew a map-sized ROI last.
  __shared__ int s_pref[kCostClasses + 1];
  if (tid == 0 && bucket) {
    int acc = 0;
    for (int k = 0; k < kCostClasses; ++k) { s_pref[k] = acc; acc += bcnt[kCostClasses - 1 - k]; }
    s_pref[kCostClasses] = acc;
  }
  __syncthreads();
  auto roi_of = [&](int i) -> int {   // i-th ROI in decreasing-cost order (arrival order when no cost classes were built)
    if (!bucket) return i;
    int k = 0;
    while (k + 1 < kCostClasses && i >= s_pref[k + 1]) ++k;
    return bucket[(size_t)(kCostClasses - 1 - k) * R + (i - s_pref[k])];
  };
  auto fetch = [&](int item, int b) {
    const float4 *src = reinterpret_cast<const float4 *>(recs + (size_t)roi_of(item / nslab) * rec);
    const unsigned dst = (unsigned)__cvta_generic_to_shared(tab + b * rec);
    for (int i = tid; i < rec / 4; i += kSepThreads)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * i), "l"(src + i) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  fetch(cur, 0);
  if (tid == 0) s_item[1] = (int)(gridDim.x + atomicAdd(counter, 1u));
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  const int half = (tid >> 4) & 1;
  float *t0 = tile + (size_t)(2 * tid + half) * kBins;
  float *t1 = tile + (size_t)(2 * tid + 1 - half) * kBins;
  int buf = 0;
  for (;;) {
    const int nxt = s_item[buf ^ 1];
    if (nxt < nitems) fetch(nxt, buf ^ 1);
    int after = 0;
    if (tid == 0) after = (int)(gridDim.x + atomicAdd(counter, 1u));
    const int cbase = (cur % nslab) * kCT;
    SepSmem s;
    s.tile = tile; s.lim = reinterpret_cast<int *>(tab + buf * rec); s.Bc = tab + buf * rec + 32; s.Ad = tab + buf * rec + kRecHead;
    s.Bd = Bd;
    const int r = s.lim[27];   // the record carries its ROI index (items arrive in cost order, not in ROI order)
    const int n = s.lim[26];
    const bool empty = n < 0 || s.lim[1] < s.lim[0] || s.lim[3] < s.lim[2];
    const bool active = cbase + 2 * tid < C;
    const int c0 = active ? cbase + 2 * tid : cbase;   // idle lanes of a partial slab shadow a valid channel pair
    if (!empty) {
      const float2 *fbase2 = reinterpret_cast<const float2 *>(feat + (size_t)n * H * W * C + c0);
      const int nx = s.lim[25];   // CTA-uniform
      if (nx <= 2) {
        sep_fwd_pass_compact<0, 4, kC, 2>(s, fbase2, C, W, t0, t1, half, active);
        sep_fwd_pass_compact<4, 3, kC, 2>(s, fbase2, C, W, t0, t1, half, active);
      } else if (nx == 3) {
        sep_fwd_pass_compact<0, 4, kC, 3>(s, fbase2, C, W, t0, t1, half, active);
        sep_fwd_pass_compact<4, 3, kC, 3>(s, fbase2, C, W, t0, t1, half, active);
      } else if (nx == 4) {
        sep_fwd_pass_compact<0, 4, kC, 4>(s, fbase2, C, W, t0, t1, half, active);
        sep_fwd_pass_compact<4, 3, kC, 4>(s, fbase2, C, W, t0, t1, half, active);
      } else if (nx == 6) {
        sep_fwd_pass_compact_wide<0, 4, kC, 6>(s, fbase2, C, W, t0, t1, half, active);
        sep_fwd_pass_compact_wide<4, 3, kC, 6>(s, fbase2, C, W, t0, t1, half, active);
      } else if (nx == 8) {
        sep_fwd_pass_compact_wide<0, 4, kC, 8>(s, fbase2, C, W, t0, t1, half, active);
        sep_fwd_pass_compact_wide<4, 3, kC, 8>(s, fbase2, C, W, t0, t1, half, active);
      } else {   // wide bins (fixed sampling_ratio with bins wider than a pixel, or maps narrower than the window)
        const RoiGeom g = roi_geometry(rois + 5 * (size_t)r, scale, aligned, kPH, kPW, sampling_ratio);
        sep_build_x_dense(Bd, g, W);
        sep_fwd_pass_dense<0, 4, kC>(s, fbase2, C, W, s.lim[2], s.lim[3], t0, t1, half, active);
        sep_fwd_pass_dense<4, 3, kC>(s, fbase2, C, W, s.lim[2], s.lim[3], t0, t1, half, active);
      }
    } else {
      sep_tile_wait_free();
      if (active) {
#pragma unroll
        for (int k = 0; k < kBins; ++k) { t0[k] = 0.f; t1[k] = 0.f; }
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (tid == 0) s_item[buf] = after;
    __syncthreads();   // tile complete, next record landed, everybody is done with this record and this item slot
    if (tid == 0) {
      const int nch = min(kCT, C - cbase);
      const unsigned bytes = (unsigned)nch * kBins * 4u;
      float *dst = output + ((size_t)r * C + cbase) * kBins;
      const unsigned src = (unsigned)__cvta_generic_to_shared(tile);
      asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst), "r"(src), "r"(bytes), "l"(l2_stream) : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    cur = nxt; buf ^= 1;
    if (cur >= nitems) break;
  }
  if (tid == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---- slab-resident forward (the default when the map is small enough, e.g. VGG 18 x 37).
// The kernel above is bound by L2 latency: every pixel of every ROI is a ~500-cycle global load and the register file
// limits how many of them a warp keeps in flight.  Here the feature map of one image and 32 channels (H*W*128 B; 85 KB
// for 18 x 37) is made RESIDENT in shared memory and every ROI of that image is served from it: pixel reads become
// conflict-free 128 B LDS (lane = channel), the L2 sees each slab once per CTA instead of once per ROI, and a warp
// needs no memory-level parallelism at all.
//   * work = (32-channel slab, ROI) pairs, numbered slab-major and cut into one contiguous range per CTA (1 CTA/SM, 16
//     warps); a CTA loads the slab of each image that occurs in its range once, then its warps pull ROIs of that image
//     from a shared-memory ticket counter (ROIs may arrive in any image order; sorted input costs 1-2 slab loads per CTA);
//   * one warp = one ROI at a time, one channel per lane, all 49 accumulators in registers (single pass, no row is
//     visited twice), column weights compact and register-resident exactly as in the kernel above;
//   * the table record of the warp's NEXT ROI streams in through cp.async while the current one is accumulated, and
//     the warp's (32 x 49) result leaves as one 6 272 B bulk store that drains during the next ROI.
constexpr int kSlabCh = 32;
constexpr int kSlabStage = kSlabCh * kBins;            // 1 568 floats staged per warp
constexpr int kSlabMaxImages = 1024;                   // presence bitmap (32 words)
// Pixel stride of the resident slab in floats.  32: the source is channels-last, pixels are copied as they lie (16-byte
// cp.async).  33: the source is NCHW and is transposed ON THE WAY IN by 4-byte cp.async (lane = pixel of one channel plane,
// coalesced reads); the odd stride makes both the transposing writes (bank = px + c) and the compute reads (lane = channel)
// conflict-free, so the separate NCHW->NHWC transpose launch and its 8 B/element of traffic disappear.
constexpr int kPSNhwc = kSlabCh, kPSNchw = kSlabCh + 1;

__host__ __device__ inline size_t slab_floats(int H, int W, int ps) { return ((size_t)H * W * ps + 31) / 32 * 32; }
__host__ __device__ inline size_t slab_warp_floats(int H) { return (size_t)kSlabStage + 2 * (size_t)sep_rec_floats(H); }
__host__ __device__ inline size_t slab_smem_bytes(int H, int W, int warps, int ps) {
  return (slab_floats(H, W, ps) + (size_t)warps * slab_warp_floats(H)) * 4 + 40 * 4;
}

__device__ __forceinline__ void slab_stage_wait_free() {   // this warp's previous bulk store has finished reading its stage
  if ((threadIdx.x & 31) == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  __syncwarp();
}

// acc[a][:] += av[a] * T[:] for the run of bins a in [first, first + count) that row y feeds (first | count << 8 = info).
// A warp-uniform switch on the first bin and nested count tests: only the FMAs of bins that really use the row are
// issued (1-2 of the 7 for all but tiny ROIs), instead of 49 predicated ones.
// Packed-fp32 form of the accumulators (sm_100 fma.rn.f32x2): bins (0,1), (2,3), (4,5) of an output row travel as register
// pairs, bin 6 stays scalar -- 3 FFMA2 + 1 FFMA per fed bin row instead of 7 FFMA (the row weight is the FFMA2's broadcast
// `.F32` operand, no duplicate is materialised), and 3 FMUL2/FFMA2 + 1 scalar per column tap instead of 7; the column-weight
// pairs come from the record's interleaved copy (Bp) by 64-bit loads, the pixel pairs are adjacent LDS destinations: no MOV
// in the row loop (SASS: ~60 instead of ~75 instructions per row that feeds two bins).  Same products, same rounding, same
// summation order as the scalar form.  Measured (same box, ABAB): 8 images / 16 000 ROIs 324.6 -> 317 us from NCHW,
// 328.7 -> 314.2 us from channels-last; 1 image 64.5 -> 62.5-64.5 us.  The gain is a fraction of the instructions saved: an
// FFMA2 holds the FMA pipe for two cycles and the kernel waits on latency with four warps per scheduler.
struct SlabAcc {
  float2 p[kPH][3];
  float s[kPH];
};
template <int A0>
__device__ __forceinline__ void slab_acc_from_pk(SlabAcc &acc, const float (&av)[kPH], const float2 (&Tp)[3], float Ts, int count) {
  const float2 a2 = make_float2(av[A0], av[A0]);
#pragma unroll
  for (int i = 0; i < 3; ++i) acc.p[A0][i] = __ffma2_rn(a2, Tp[i], acc.p[A0][i]);
  acc.s[A0] = fmaf(av[A0], Ts, acc.s[A0]);
  if constexpr (A0 + 1 < kPH) {
    if (count > 1) slab_acc_from_pk<A0 + 1>(acc, av, Tp, Ts, count - 1);
  }
}
__device__ __forceinline__ void slab_accumulate_pk(SlabAcc &acc, const float (&av)[kPH], const float2 (&Tp)[3], float Ts, int info) {
  const int count = info >> 8;
  switch (info & 0xff) {
    case 0: slab_acc_from_pk<0>(acc, av, Tp, Ts, count); break;
    case 1: slab_acc_from_pk<1>(acc, av, Tp, Ts, count); break;
    case 2: slab_acc_from_pk<2>(acc, av, Tp, Ts, count); break;
    case 3: slab_acc_from_pk<3>(acc, av, Tp, Ts, count); break;
    case 4: slab_acc_from_pk<4>(acc, av, Tp, Ts, count); break;
    case 5: slab_acc_from_pk<5>(acc, av, Tp, Ts, count); break;
    default: slab_acc_from_pk<6>(acc, av, Tp, Ts, count); break;
  }
}

// rows of one ROI from the resident slab; S = slab + lane, compact column windows of width NX
template <int kImm>
__device__ __forceinline__ float slab_lds(unsigned addr) {   // ld.shared with an immediate byte offset
  float v;
  asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(addr), "n"(kImm));
  return v;
}

template <int NX, int kPS>
__device__ __forceinline__ void slab_rows_compact_pk(const float *__restrict__ S, int W, const int *__restrict__ lim,
                                                     const float *__restrict__ Bc, const float *__restrict__ Bp, const float *__restrict__ Ad,
                                                     SlabAcc &acc) {
  float2 bwp[3][NX];
  float bws[NX];
  unsigned pb[kPW];   // shared-window byte address of (row 0, first column of bin b, this lane's channel)
  const unsigned sbase = (unsigned)__cvta_generic_to_shared(S);
#pragma unroll
  for (int b = 0; b < kPW; ++b) pb[b] = sbase + (unsigned)lim[18 + b] * (kPS * 4);
#pragma unroll
  for (int j = 0; j < NX; ++j) {
#pragma unroll
    for (int i = 0; i < 3; ++i) bwp[i][j] = *reinterpret_cast<const float2 *>(Bp + ((i * kNXPair + j) << 1));   // (bin 2i, bin 2i+1)
    bws[j] = Bc[6 * kNXMax + j];
  }
  const int y0 = lim[0], y1 = lim[1];
  const unsigned rstride = (unsigned)W * (kPS * 4);
  // running addresses (row weights, the seven column windows): nothing in a row waits for an index multiplication
  const float *ad = Ad + y0 * 8;
#pragma unroll
  for (int b = 0; b < kPW; ++b) pb[b] += (unsigned)y0 * rstride;
  for (int y = y0; y <= y1; ++y, ad += 8) {
    const float4 a0 = *reinterpret_cast<const float4 *>(ad), a1 = *reinterpret_cast<const float4 *>(ad + 4);
    const float av[kPH] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z};
    const int info = __float_as_int(a1.w);
    unsigned pr[kPW];
#pragma unroll
    for (int b = 0; b < kPW; ++b) { pr[b] = pb[b]; pb[b] += rstride; }
    if (info == 0) continue;   // no bin uses this row
    float2 Tp[3];
    float Ts;
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      const unsigned p0 = pr[2 * i], p1 = pr[2 * i + 1];
      Tp[i] = __fmul2_rn(bwp[i][0], make_float2(slab_lds<0>(p0), slab_lds<0>(p1)));
      if (NX > 1) Tp[i] = __ffma2_rn(bwp[i][1 % NX], make_float2(slab_lds<kPS * 4>(p0), slab_lds<kPS * 4>(p1)), Tp[i]);
      if (NX > 2) Tp[i] = __ffma2_rn(bwp[i][2 % NX], make_float2(slab_lds<2 * kPS * 4>(p0), slab_lds<2 * kPS * 4>(p1)), Tp[i]);
      if (NX > 3) Tp[i] = __ffma2_rn(bwp[i][3 % NX], make_float2(slab_lds<3 * kPS * 4>(p0), slab_lds<3 * kPS * 4>(p1)), Tp[i]);
    }
    {
      const unsigned p = pr[6];
      Ts = bws[0] * slab_lds<0>(p);
      if (NX > 1) Ts = fmaf(bws[1 % NX], slab_lds<kPS * 4>(p), Ts);
      if (NX > 2) Ts = fmaf(bws[2 % NX], slab_lds<2 * kPS * 4>(p), Ts);
      if (NX > 3) Ts = fmaf(bws[3 % NX], slab_lds<3 * kPS * 4>(p), Ts);
    }
    slab_accumulate_pk(acc, av, Tp, Ts, info);
  }
}

// wide-bin fallback: dense column table Bd (W x 8, built by the warp in its own stage buffer)
template <int kPS>
__device__ __forceinline__ void slab_rows_dense(const float *__restrict__ S, int W, const int *__restrict__ lim,
                                                const float *__restrict__ Bd, const float *__restrict__ Ad, SlabAcc &acc) {
  const int y0 = lim[0], y1 = lim[1], x0 = lim[2], x1 = lim[3];
  for (int y = y0; y <= y1; ++y) {
    const float *row = S + y * W * kPS;
    float T[kPW];
#pragma unroll
    for (int b = 0; b < kPW; ++b) T[b] = 0.f;
    for (int x = x0; x <= x1; ++x) {
      const float f = row[x * kPS];
      const float4 w0 = *reinterpret_cast<const float4 *>(Bd + x * 8), w1 = *reinterpret_cast<const float4 *>(Bd + x * 8 + 4);
      T[0] = fmaf(w0.x, f, T[0]); T[1] = fmaf(w0.y, f, T[1]); T[2] = fmaf(w0.z, f, T[2]); T[3] = fmaf(w0.w, f, T[3]);
      T[4] = fmaf(w1.x, f, T[4]); T[5] = fmaf(w1.y, f, T[5]); T[6] = fmaf(w1.z, f, T[6]);
    }
    const float4 a0 = *reinterpret_cast<const float4 *>(Ad + y * 8), a1 = *reinterpret_cast<const float4 *>(Ad + y * 8 + 4);
    const float av[kPH] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z};
    if (__float_as_int(a1.w) != 0) {
      const float2 Tp[3] = {make_float2(T[0], T[1]), make_float2(T[2], T[3]), make_float2(T[4], T[5])};
      slab_accumulate_pk(acc, av, Tp, T[6], __float_as_int(a1.w));
    }
  }
}

template <int kWarps, int kPS>
__global__ void __launch_bounds__(kWarps * 32, 1) roi_align_fwd_slab_kernel(const float *__restrict__ feat /* kPS == 32: NHWC, 33: NCHW */,
                                                                            const float *__restrict__ rois,
                                                                            const float *__restrict__ recs, int N, int C, int H,
                                                                            int W, int R, float scale, int sampling_ratio,
                                                                            int aligned, float *__restrict__ output) {
  extern __shared__ __align__(128) float sep_smem[];
  const int rec = sep_rec_floats(H);
  const int HW = H * W;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float *slab = sep_smem;
  float *mine = slab + slab_floats(H, W, kPS) + (size_t)warp * slab_warp_floats(H);
  float *stage = mine, *recbuf = mine + kSlabStage;
  int *ctrl = reinterpret_cast<int *>(slab + slab_floats(H, W, kPS) + (size_t)kWarps * slab_warp_floats(H));
  int *s_ticket = ctrl, *s_invalid = ctrl + 1, *s_span = ctrl + 2;
  unsigned *s_present = reinterpret_cast<unsigned *>(ctrl + 8);   // kSlabMaxImages bits

  unsigned long long l2_stream;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(l2_stream));
  const int nslab = (C + kSlabCh - 1) / kSlabCh;
  const long long total = (long long)nslab * R;
  long long lo = total * blockIdx.x / gridDim.x;
  const long long hi = total * (blockIdx.x + 1) / gridDim.x;
  pdl_wait();   // the table records of the pre-kernel are visible from here on

  auto fetch_rec = [&](int r, int b) {   // warp-wide cp.async of one table record
    const float4 *src = reinterpret_cast<const float4 *>(recs + (size_t)r * rec);
    const unsigned dst = (unsigned)__cvta_generic_to_shared(recbuf + b * rec);
    for (int i = lane; i < rec / 4; i += 32)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * i), "l"(src + i) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  auto ticket = [&]() -> int {
    int t = 0;
    if (lane == 0) t = atomicAdd(s_ticket, 1);
    return __shfl_sync(0xFFFFFFFFu, t, 0);
  };

  while (lo < hi) {
    const int sl = (int)(lo / R), r_lo = (int)(lo - (long long)sl * R);
    const int r_hi = (int)min((long long)R, r_lo + (hi - lo));
    lo += r_hi - r_lo;
    const int cbase = sl * kSlabCh, nch = min(kSlabCh, C - cbase);
    // which images occur in [r_lo, r_hi)?
    if (tid < kSlabMaxImages / 32) s_present[tid] = 0u;
    if (tid == 0) *s_invalid = 0;
    __syncthreads();
    for (int r = r_lo + tid; r < r_hi; r += kWarps * 32) {
      const int img = reinterpret_cast<const int *>(recs + (size_t)r * rec)[26];
      if (img >= 0) atomicOr(&s_present[img >> 5], 1u << (img & 31)); else *s_invalid = 1;
    }
    __syncthreads();
    for (int n = -1; n < N; ++n) {   // n == -1: ROIs with an invalid image index (zero output, no slab needed)
      if (n < 0 ? (*s_invalid == 0) : !((s_present[n >> 5] >> (n & 31)) & 1u)) continue;   // CTA-uniform
      if (n >= 0) {
        const unsigned dst = (unsigned)__cvta_generic_to_shared(slab);
        if (kPS == kPSNhwc) {
          const float *src = feat + (size_t)n * HW * C + cbase;
          const int q4 = nch >> 2;   // 16-byte chunks per pixel
          for (int idx = tid; idx < HW * 8; idx += kWarps * 32) {
            const int px = idx >> 3, q = idx & 7;
            if (q < q4)
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * idx), "l"(src + (size_t)px * C + q * 4) : "memory");
          }
        } else {   // NCHW: one channel plane per warp pass, lanes over pixels; smem word px * 33 + c
          const float *src = feat + ((size_t)n * C + cbase) * HW;
          for (int c = warp; c < nch; c += kWarps) {
            const float *plane = src + (size_t)c * HW;
            for (int px = lane; px < HW; px += 32)
              asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * (unsigned)(px * kPS + c)), "l"(plane + px) : "memory");
          }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
      }
      // first / last ROI of this image inside the range (sorted input: the tickets then visit no foreign ROI)
      if (tid == 0) { s_span[0] = r_hi; s_span[1] = r_lo - 1; }
      __syncthreads();
      {
        int first = r_hi, last = r_lo - 1;
        for (int r = r_lo + tid; r < r_hi; r += kWarps * 32) {
          const int img = reinterpret_cast<const int *>(recs + (size_t)r * rec)[26];
          if (img == n || (n < 0 && img < 0)) { first = min(first, r); last = max(last, r); }
        }
        first = __reduce_min_sync(0xFFFFFFFFu, first); last = __reduce_max_sync(0xFFFFFFFFu, last);
        if (lane == 0 && last >= first) { atomicMin(&s_span[0], first); atomicMax(&s_span[1], last); }
      }
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncthreads();
      const int t_end = s_span[1] + 1;
      if (tid == 0) *s_ticket = s_span[0];
      __syncthreads();
      const float *S = slab + lane;
      int buf = 0;
      int t = ticket();
      if (t < t_end) fetch_rec(t, 0);
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      __syncwarp();
      while (t < t_end) {
        const int tn = ticket();
        if (tn < t_end) fetch_rec(tn, buf ^ 1);
        const float *rb = recbuf + buf * rec;
        const int *lim = reinterpret_cast<const int *>(rb);
        if (lim[26] == n || (n < 0 && lim[26] < 0)) {
          SlabAcc acc;
#pragma unroll
          for (int a = 0; a < kPH; ++a) {
#pragma unroll
            for (int i = 0; i < 3; ++i) acc.p[a][i] = make_float2(0.f, 0.f);
            acc.s[a] = 0.f;
          }
          const bool empty = n < 0 || lim[1] < lim[0] || lim[3] < lim[2];
          if (!empty) {
            const int nx = lim[25];
            if (nx <= 2) slab_rows_compact_pk<2, kPS>(S, W, lim, rb + 32, rb + kRecPair, rb + kRecHead, acc);
            else if (nx == 3) slab_rows_compact_pk<3, kPS>(S, W, lim, rb + 32, rb + kRecPair, rb + kRecHead, acc);
            else if (nx == 4) slab_rows_compact_pk<4, kPS>(S, W, lim, rb + 32, rb + kRecPair, rb + kRecHead, acc);
            else {   // wide bins: dense column table, built by this warp in its (drained) stage buffer
              slab_stage_wait_free();
              const RoiGeom g = roi_geometry(rois + 5 * (size_t)t, scale, aligned, kPH, kPW, sampling_ratio);
              for (int i = lane; i < W * 8; i += 32) stage[i] = 0.f;
              __syncwarp();
              if (lane < kPW) {
                const float inv = g.gw > 0 ? __fdiv_rn(1.0f, (float)g.gw) : 0.f;
                for (int ix = 0; ix < g.gw; ++ix) {
                  int xl, xh; float l, h;
                  if (!bilinear_1d(sample_coord(g.sw, lane, g.bw, ix, g.gw), W, xl, xh, l, h)) continue;
                  stage[xl * 8 + lane] += h * inv; stage[xh * 8 + lane] += l * inv;
                }
              }
              __syncwarp();
              slab_rows_dense<kPS>(S, W, lim, stage, rb + kRecHead, acc);
              __syncwarp();
            }
          }
          slab_stage_wait_free();
          if (lane < nch) {
#pragma unroll
            for (int a = 0; a < kPH; ++a) {   // stride 49: conflict-free
#pragma unroll
              for (int i = 0; i < 3; ++i) {
                stage[lane * kBins + a * kPW + 2 * i] = acc.p[a][i].x;
                stage[lane * kBins + a * kPW + 2 * i + 1] = acc.p[a][i].y;
              }
              stage[lane * kBins + a * kPW + 6] = acc.s[a];
            }
          }
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            float *dst = output + ((size_t)t * C + cbase) * kBins;
            const unsigned src = (unsigned)__cvta_generic_to_shared(stage);
            const unsigned bytes = (unsigned)nch * kBins * 4u;
            // the 1.6 GB output stream must not evict the feature map and the table records from L2
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst), "r"(src), "r"(bytes), "l"(l2_stream) : "memory");
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
        t = tn; buf ^= 1;
      }
      __syncthreads();   // every warp is done with this slab (and with the ticket counter)
    }
  }
  if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// Backward of the separable form: gF = A^T . gOut . B per channel pair, accumulated into an NHWC gradient with 8-byte
// vector reductions (red.global.add.v2.f32): one coalesced 256 B reduction per warp and pixel.  The reduction traffic at the
// L2 is the scarce resource, so every pixel row of the window receives exactly ONE reduction: the two register passes
// (bins 0-3, bins 3-6) PARTITION the rows instead of both visiting the rows that bins 3 and 4 share -- a row fed by any of
// the bins 4-6 ("B row") is written by the second pass, which carries bin 3 along (kSecond: go = bins 3..6); the first pass
// drops bin 3 on such rows and skips them unless one of the bins 0-2 feeds them too (ROIs smaller than a few cells).  With
// the ~5.5-row windows of the stride-32 map this removes a quarter of the reductions (7.5 -> 5.5 rows per ROI): 130 -> 121 us
// for 4 096 ROIs.  Measured and NOT kept (DESIGN.md section 7): a persistent variant with double-buffered tiles, records from
// the table pre-kernel and one channel per thread (170 us: the per-pixel weight loads are paid per thread, so halving the
// channels per thread doubles them); the same row partition in the L2 forward (R101-C4 211 -> 260 us: the fourth bin of the
// second pass costs 14 more accumulator registers and the kernel spills).
template <bool kSecond, int kC>
__device__ __forceinline__ void sep_bwd_pass(const SepSmem &s, float2 *__restrict__ gbase2, int C, int W, int xmin, int xmax,
                                             const float *__restrict__ t0, const float *__restrict__ t1, int half) {
  constexpr int PH0 = kSecond ? 3 : 0, NPH = 4;      // bins held in registers by this pass
  constexpr int R0 = kSecond ? 4 : 0, RN = kSecond ? 3 : 4;   // bins whose row ranges bound the pass
  const int cs2 = (kC ? kC : C) >> 1;
  int y0 = s.lim[4 + R0], y1 = s.lim[11 + R0];
#pragma unroll
  for (int a = 1; a < RN; ++a) { y0 = min(y0, s.lim[4 + R0 + a]); y1 = max(y1, s.lim[11 + R0 + a]); }
  float2 go[NPH][kPW];
#pragma unroll
  for (int a = 0; a < NPH; ++a)
#pragma unroll
    for (int b = 0; b < kPW; ++b) {
      const float u0 = t0[(PH0 + a) * kPW + b], u1 = t1[(PH0 + a) * kPW + b];
      go[a][b] = half ? make_float2(u1, u0) : make_float2(u0, u1);
    }
  for (int y = y0; y <= y1; ++y) {
    const float4 lo = *reinterpret_cast<const float4 *>(s.Ad + y * 8), hi = *reinterpret_cast<const float4 *>(s.Ad + y * 8 + 4);
    const bool b_row = hi.x != 0.f || hi.y != 0.f || hi.z != 0.f;   // fed by one of the bins 4-6: the second pass owns bin 3 here
    if (kSecond && !b_row) continue;
    const float av[4] = {kSecond ? lo.w : lo.x, kSecond ? hi.x : lo.y, kSecond ? hi.y : lo.z, kSecond ? hi.z : (b_row ? 0.f : lo.w)};
    float2 U[kPW];
#pragma unroll
    for (int b = 0; b < kPW; ++b) U[b] = make_float2(0.f, 0.f);
    bool any = false;
#pragma unroll
    for (int a = 0; a < NPH; ++a) {
      if (av[a] != 0.f) {
        any = true;
#pragma unroll
        for (int b = 0; b < kPW; ++b) { U[b].x = fmaf(av[a], go[a][b].x, U[b].x); U[b].y = fmaf(av[a], go[a][b].y, U[b].y); }
      }
    }
    if (!any) continue;
    float2 *grow = gbase2 + (size_t)y * W * cs2;
    for (int x = xmin; x <= xmax; ++x) {
      const float4 w0 = *reinterpret_cast<const float4 *>(s.Bd + x * 8), w1 = *reinterpret_cast<const float4 *>(s.Bd + x * 8 + 4);
      float2 v = make_float2(w0.x * U[0].x, w0.x * U[0].y);
      v.x = fmaf(w0.y, U[1].x, v.x); v.y = fmaf(w0.y, U[1].y, v.y);
      v.x = fmaf(w0.z, U[2].x, v.x); v.y = fmaf(w0.z, U[2].y, v.y);
      v.x = fmaf(w0.w, U[3].x, v.x); v.y = fmaf(w0.w, U[3].y, v.y);
      v.x = fmaf(w1.x, U[4].x, v.x); v.y = fmaf(w1.x, U[4].y, v.y);
      v.x = fmaf(w1.y, U[5].x, v.x); v.y = fmaf(w1.y, U[5].y, v.y);
      v.x = fmaf(w1.z, U[6].x, v.x); v.y = fmaf(w1.z, U[6].y, v.y);
      atomicAdd(grow + (size_t)x * cs2, v);   // result unused -> RED.E.ADD.F32x2
    }
  }
}

template <int kC>
__global__ void __launch_bounds__(kSepThreads, 4) roi_align_bwd_sep_kernel(const float *__restrict__ grad_out,
                                                                           const float *__restrict__ rois, int N, int C, int H,
                                                                           int W, float scale, int sampling_ratio, int aligned,
                                                                           float *__restrict__ grad_nhwc) {
  extern __shared__ __align__(128) float sep_smem[];
  const SepSmem s = sep_carve(sep_smem, H, W);
  const int r = blockIdx.x, cbase = blockIdx.y * kCT;
  const int tid = threadIdx.x;
  RoiGeom g = roi_geometry(rois + 5 * (size_t)r, scale, aligned, kPH, kPW, sampling_ratio);
  if (g.n < 0 || g.n >= N) return;
  const int nch = min(kCT, C - cbase);
  // asynchronous 128-bit staging of the contiguous (nch x 49) gradient tile: all ~25 copies of a thread are in flight at
  // once and land while the tables are built
  {
    const float4 *src = reinterpret_cast<const float4 *>(grad_out + ((size_t)r * C + cbase) * kBins);
    const unsigned dst = (unsigned)__cvta_generic_to_shared(s.tile);
    const int n4 = nch * kBins / 4;
    for (int i = tid; i < n4; i += kSepThreads)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * i), "l"(src + i) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  sep_build_tables(s, g, H, W);
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();   // publishes the tile
  const int ymin = s.lim[0], ymax = s.lim[1], xmin = s.lim[2], xmax = s.lim[3];
  const int c0 = cbase + 2 * tid;
  if (c0 >= C || ymax < ymin || xmax < xmin) return;
  const int half = (tid >> 4) & 1;
  const float *t0 = s.tile + (size_t)(2 * tid + half) * kBins;
  const float *t1 = s.tile + (size_t)(2 * tid + 1 - half) * kBins;
  float2 *gbase2 = reinterpret_cast<float2 *>(grad_nhwc + (size_t)g.n * H * W * C + c0);
  sep_bwd_pass<false, kC>(s, gbase2, C, W, xmin, xmax, t0, t1, half);
  sep_bwd_pass<true, kC>(s, gbase2, C, W, xmin, xmax, t0, t1, half);
}

// --------------------------------------------------------------------------- ROIPool
__global__ void __launch_bounds__(256) roi_pool_fwd_kernel(const float *__restrict__ input, const float *__restrict__ rois, int N,
                                                           int C, int H, int W, long long total, int PH, int PW, float scale,
                                                           float *__restrict__ output, int *__restrict__ argmax) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int pw = (int)(idx % PW), ph = (int)((idx / PW) % PH);
  const int c = (int)((idx / ((long long)PW * PH)) % C);
  const long long r = idx / ((long long)PW * PH * C);
  const float *roi = rois + 5 * r;
  const int b = (int)roi[0];
  const int rsw = (int)roundf(__fmul_rn(roi[1], scale)), rsh = (int)roundf(__fmul_rn(roi[2], scale));
  const int rew = (int)roundf(__fmul_rn(roi[3], scale)), reh = (int)roundf(__fmul_rn(roi[4], scale));
  const int rw = max(rew - rsw + 1, 1), rh = max(reh - rsh + 1, 1);
  const float bh = __fdiv_rn((float)rh, (float)PH), bw = __fdiv_rn((float)rw, (float)PW);
  int hs = (int)floorf(__fmul_rn((float)ph, bh)), ws = (int)floorf(__fmul_rn((float)pw, bw));
  int he = (int)ceilf(__fmul_rn((float)(ph + 1), bh)), we = (int)ceilf(__fmul_rn((float)(pw + 1), bw));
  hs = min(max(hs + rsh, 0), H); he = min(max(he + rsh, 0), H);
  ws = min(max(ws + rsw, 0), W); we = min(max(we + rsw, 0), W);
  const bool empty = (he <= hs) || (we <= ws);
  float maxval = empty ? 0.f : -FLT_MAX;
  int maxidx = -1;
  if (b >= 0 && b < N) {
    const float *in = input + ((size_t)b * C + c) * H * W;
    for (int h = hs; h < he; ++h)
      for (int w = ws; w < we; ++w) {
        const float v = in[h * W + w];
        if (v > maxval) { maxval = v; maxidx = h * W + w; }
      }
  } else if (!empty) maxval = 0.f;
  output[idx] = maxval;
  argmax[idx] = maxidx;
}

__global__ void __launch_bounds__(256) roi_pool_bwd_kernel(const float *__restrict__ grad_out, const float *__restrict__ rois,
                                                           const int *__restrict__ argmax, int N, int C, int H, int W,
                                                           long long total, int PH, int PW, float *__restrict__ grad_in) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int c = (int)((idx / ((long long)PW * PH)) % C);
  const long long r = idx / ((long long)PW * PH * C);
  const int b = (int)rois[5 * r];
  const int am = argmax[idx];
  if (am != -1 && b >= 0 && b < N) atomicAdd(grad_in + ((size_t)b * C + c) * H * W + am, grad_out[idx]);
}

bool sep_supported(int C, int H, int W, int PH, int PW) {
  // shared-memory budgets of the backward (dense tables), the persistent forward and the 4-ROI table pre-kernel
  return PH == kPH && PW == kPW && (C % 4) == 0 && sep_smem_bytes(H, W) <= 100 * 1024 && sep_fwd_smem_bytes(H, W) <= 100 * 1024 &&
         4 * (size_t)sep_rec_floats(H) * sizeof(float) <= 48 * 1024;
}

}  // namespace

// =========================================================================== C ABI
SFOD_API size_t sfod_roi_align_fwd_workspace_bytes(int N, int C, int H, int W, int R, int layout, int exact) {
  // exact kernel reads NCHW, separable kernel reads NHWC: a converted copy is needed when layouts differ; the separable
  // kernel also needs one table record per ROI and its work counter
  const bool need = exact ? (layout == SFOD_NHWC) : (layout == SFOD_NCHW);
  size_t bytes = need ? sfod_align_up((size_t)N * C * H * W * sizeof(float), 256) : 0;
  if (!exact) bytes += 256 + sfod_align_up((size_t)(R > 0 ? R : 0) * sep_rec_floats(H) * sizeof(float), 256) +
                       sfod_align_up((size_t)(R > 0 ? R : 0) * kCostClasses * sizeof(int), 256);
  // a channels-last call falls back to the exact kernel (which reads an NCHW copy) when the separable path does not support
  // the shape -- C % 4, the map size, or an output other than 7 x 7, which this query is not told
  if (!exact && layout == SFOD_NHWC) {
    const size_t nchw = sfod_align_up((size_t)N * C * H * W * sizeof(float), 256);
    if (bytes < nchw) bytes = nchw;
  }
  return bytes ? bytes : 256;
}

static int sep_fwd_grid(const void *kern, size_t smem, int items) {   // resident CTAs of the persistent forward
  int dev = 0, sms = 0, per_sm = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kSepThreads, smem) != cudaSuccess || per_sm < 1) return -1;
  const long long g = (long long)sms * per_sm;
  return (int)(g < items ? g : items);
}

SFOD_API int sfod_roi_align_fwd(const float *input, int layout, const float *rois, int N, int C, int H, int W, int R, int PH,
                                int PW, float spatial_scale, int sampling_ratio, int aligned, int exact, float *output,
                                void *workspace, size_t workspace_bytes, sfod_stream_t stream) {
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || R < 0 || PH <= 0 || PW <= 0) return SFOD_ERR_INVALID_ARG;
  if (layout != SFOD_NCHW && layout != SFOD_NHWC) return SFOD_ERR_INVALID_ARG;
  if (R == 0) return SFOD_OK;
  if (!input || !rois || !output) return SFOD_ERR_INVALID_ARG;
  cudaStream_t st = sfod_cu(stream);
  const bool fast = !exact && sep_supported(C, H, W, PH, PW) && sfod_aligned16(output);
  const size_t fbytes = (size_t)N * C * H * W * sizeof(float);
  if (fast) {
    unsigned char *ws = static_cast<unsigned char *>(workspace);
    const size_t rec_bytes = (size_t)sep_rec_floats(H) * sizeof(float);
    const size_t feat_ws = layout == SFOD_NCHW ? sfod_align_up(fbytes, 256) : 0;   // transposed copy (only some paths use it)
    const size_t rec_ws = sfod_align_up((size_t)R * rec_bytes, 256);
    if (!workspace || workspace_bytes < feat_ws + 256 + rec_ws + (size_t)R * kCostClasses * sizeof(int)) return SFOD_ERR_WORKSPACE_TOO_SMALL;
    if (!sfod_aligned16(ws + feat_ws) || !sfod_aligned16(input)) return SFOD_ERR_ALIGNMENT;
    unsigned *counter = reinterpret_cast<unsigned *>(ws + feat_ws);          // [0]: work counter; [16 .. 31]: cost-class counts
    int *bcnt = reinterpret_cast<int *>(ws + feat_ws) + 16;
    float *recs = reinterpret_cast<float *>(ws + feat_ws + 256);
    int *bucket = reinterpret_cast<int *>(ws + feat_ws + 256 + rec_ws);
    int sms = 0, cur_dev = 0, max_optin = 0;
    SFOD_CUDA_TRY(cudaGetDevice(&cur_dev));
    SFOD_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cur_dev));
    SFOD_CUDA_TRY(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, cur_dev));
    // Which forward?  (1) 32-channel slab resident in shared memory, read straight from the caller's layout; (2) per-ROI
    // loads from L2 for maps whose slab does not fit (R101-C4 res4: 38 x 75 x 32 x 4 B = 365 KB).  A 16-channel slab with two
    // half-warps per ROI (182 KB) was built and measured in round 2: parity-green but no faster than (2) -- 177 M warp
    // instructions at 43 % issue with 10 warps per SM (profiles/r2c_s16_ncu_summary.txt, DESIGN.md section 7); removed.
    const int ps = layout == SFOD_NCHW ? kPSNchw : kPSNhwc;
    const bool slab_ok = N <= kSlabMaxImages && (size_t)W * 8 <= (size_t)kSlabStage;
    const int slab_warps = !slab_ok ? 0 : slab_smem_bytes(H, W, 16, ps) <= (size_t)max_optin ? 16 : slab_smem_bytes(H, W, 8, ps) <= (size_t)max_optin ? 8 : 0;
    const float *feat = input;   // what the main kernel reads
    if (!slab_warps && layout == SFOD_NCHW) {   // path (2) reads channels-last
      int rc = launch_transpose(input, static_cast<float *>(workspace), N, C, H * W, st);
      if (rc) return rc;
      feat = static_cast<const float *>(workspace);
    }
    const bool l2_path = !slab_warps;
    // Cost-ordered items pay off when a CTA sees few of them (1 image: 18 items per CTA, 296 -> 211 us on R101-C4); with
    // hundreds per CTA the tail is small and arrival (image-major) order keeps one image's map hot in L2 (8 images: 1 494 us in
    // arrival order, 1 595 us in cost order).
    const long long l2_items = (long long)R * ((C + kCT - 1) / kCT);
    const bool lpt = l2_path && l2_items < 64LL * 3 * sms;
    if (l2_path) SFOD_CUDA_TRY(cudaMemsetAsync(counter, 0, 256, st));
    if (!lpt) { bcnt = nullptr; bucket = nullptr; }
    roi_sep_tables_kernel<<<(R + 3) / 4, 128, 4 * rec_bytes, st>>>(rois, R, N, H, W, spatial_scale, sampling_ratio, aligned, recs, bcnt, bucket);
    SFOD_LAUNCH_CHECK();
    if (slab_warps) {
      // launched with programmatic stream serialization: its prologue overlaps the table kernel (griddepcontrol.wait inside)
      cudaLaunchConfig_t cfg = {};
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
      attr[0].val.programmaticStreamSerializationAllowed = 1;
      cfg.gridDim = dim3(sms); cfg.stream = st; cfg.attrs = attr; cfg.numAttrs = 1;
#define SFOD_SLAB_LAUNCH(KERN, WARPS, SMEM)                                                                                  \
      do {                                                                                                                   \
        SFOD_CUDA_TRY(cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SMEM)));                 \
        cfg.blockDim = dim3((WARPS) * 32); cfg.dynamicSmemBytes = (SMEM);                                                    \
        SFOD_CUDA_TRY(cudaLaunchKernelEx(&cfg, KERN, feat, rois, (const float *)recs, N, C, H, W, R, spatial_scale,          \
                                         sampling_ratio, aligned, output));                                                  \
      } while (0)
      if (slab_warps == 16 && ps == kPSNchw) SFOD_SLAB_LAUNCH((roi_align_fwd_slab_kernel<16, kPSNchw>), 16, slab_smem_bytes(H, W, 16, ps));
      else if (slab_warps == 16) SFOD_SLAB_LAUNCH((roi_align_fwd_slab_kernel<16, kPSNhwc>), 16, slab_smem_bytes(H, W, 16, ps));
      else if (slab_warps == 8 && ps == kPSNchw) SFOD_SLAB_LAUNCH((roi_align_fwd_slab_kernel<8, kPSNchw>), 8, slab_smem_bytes(H, W, 8, ps));
      else SFOD_SLAB_LAUNCH((roi_align_fwd_slab_kernel<8, kPSNhwc>), 8, slab_smem_bytes(H, W, 8, ps));
#undef SFOD_SLAB_LAUNCH
      SFOD_LAUNCH_CHECK();
      return SFOD_OK;
    }
    const size_t smem = sep_fwd_smem_bytes(H, W);
    const int items = R * ((C + kCT - 1) / kCT);
#define SFOD_ROI_FWD(KC)                                                                                                     \
    do {                                                                                                                     \
      SFOD_CUDA_TRY(cudaFuncSetAttribute(roi_align_fwd_sep_kernel<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      const int grid = sep_fwd_grid(reinterpret_cast<const void *>(roi_align_fwd_sep_kernel<KC>), smem, items);             \
      if (grid < 1) return SFOD_ERR_UNSUPPORTED;                                                                                   \
      roi_align_fwd_sep_kernel<KC><<<grid, kSepThreads, smem, st>>>(feat, rois, recs, counter, bcnt, bucket, N, C, H, W, R, spatial_scale, \
                                                                    sampling_ratio, aligned, output);                        \
    } while (0)
    switch (C) {
      case 256: SFOD_ROI_FWD(256); break;
      case 512: SFOD_ROI_FWD(512); break;
      case 1024: SFOD_ROI_FWD(1024); break;
      case 2048: SFOD_ROI_FWD(2048); break;
      default: SFOD_ROI_FWD(0); break;
    }
#undef SFOD_ROI_FWD
    SFOD_LAUNCH_CHECK();
    return SFOD_OK;
  }
  const float *in = input;
  if (layout == SFOD_NHWC) {
    if (!workspace || workspace_bytes < fbytes) return SFOD_ERR_WORKSPACE_TOO_SMALL;
    int rc = launch_transpose(input, static_cast<float *>(workspace), N, H * W, C, st);
    if (rc) return rc;
    in = static_cast<const float *>(workspace);
  }
  const long long total = (long long)R * C * PH * PW;
  roi_align_fwd_exact_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(in, rois, N, C, H, W, total, PH, PW, spatial_scale,
                                                                             sampling_ratio, aligned, output);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

SFOD_API size_t sfod_roi_align_bwd_workspace_bytes(int N, int C, int H, int W, int layout) {
  return layout == SFOD_NCHW ? sfod_align_up((size_t)N * C * H * W * sizeof(float), 256) : 256;
}

SFOD_API int sfod_roi_align_bwd(const float *grad_out, const float *rois, int N, int C, int H, int W, int R, int PH, int PW,
                                float spatial_scale, int sampling_ratio, int aligned, float *grad_in, int layout,
                                void *workspace, size_t workspace_bytes, sfod_stream_t stream) {
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || R < 0 || PH <= 0 || PW <= 0 || !grad_in) return SFOD_ERR_INVALID_ARG;
  if (layout != SFOD_NCHW && layout != SFOD_NHWC) return SFOD_ERR_INVALID_ARG;
  cudaStream_t st = sfod_cu(stream);
  const size_t fbytes = (size_t)N * C * H * W * sizeof(float);
  if (R == 0) { SFOD_CUDA_TRY(cudaMemsetAsync(grad_in, 0, fbytes, st)); return SFOD_OK; }
  if (!grad_out || !rois) return SFOD_ERR_INVALID_ARG;
  const bool fast = sep_supported(C, H, W, PH, PW) && sfod_aligned16(grad_out) && sfod_aligned16(grad_in);
  if (fast) {
    float *acc = grad_in;
    if (layout == SFOD_NCHW) {
      if (!workspace || workspace_bytes < fbytes) return SFOD_ERR_WORKSPACE_TOO_SMALL;
      acc = static_cast<float *>(workspace);
    }
    SFOD_CUDA_TRY(cudaMemsetAsync(acc, 0, fbytes, st));
    const size_t smem = sep_smem_bytes(H, W);
    dim3 grid(R, (C + kCT - 1) / kCT);
#define SFOD_ROI_BWD(KC)                                                                                                     \
    do {                                                                                                                     \
      SFOD_CUDA_TRY(cudaFuncSetAttribute(roi_align_bwd_sep_kernel<KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
      roi_align_bwd_sep_kernel<KC><<<grid, kSepThreads, smem, st>>>(grad_out, rois, N, C, H, W, spatial_scale, sampling_ratio, aligned, acc); \
    } while (0)
    switch (C) {
      case 256: SFOD_ROI_BWD(256); break;
      case 512: SFOD_ROI_BWD(512); break;
      case 1024: SFOD_ROI_BWD(1024); break;
      case 2048: SFOD_ROI_BWD(2048); break;
      default: SFOD_ROI_BWD(0); break;
    }
#undef SFOD_ROI_BWD
    SFOD_LAUNCH_CHECK();
    if (layout == SFOD_NCHW) return launch_transpose(acc, grad_in, N, H * W, C, st);
    return SFOD_OK;
  }
  // generic: accumulate in NCHW
  float *acc = grad_in;
  if (layout == SFOD_NHWC) {
    if (!workspace || workspace_bytes < fbytes) return SFOD_ERR_WORKSPACE_TOO_SMALL;
    acc = static_cast<float *>(workspace);
  }
  SFOD_CUDA_TRY(cudaMemsetAsync(acc, 0, fbytes, st));
  const long long total = (long long)R * C * PH * PW;
  roi_align_bwd_generic_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(grad_out, rois, N, C, H, W, total, PH, PW,
                                                                               spatial_scale, sampling_ratio, aligned, acc);
  SFOD_LAUNCH_CHECK();
  if (layout == SFOD_NHWC) return launch_transpose(acc, grad_in, N, C, H * W, st);
  return SFOD_OK;
}

SFOD_API int sfod_roi_pool_fwd(const float *input, const float *rois, int N, int C, int H, int W, int R, int PH, int PW,
                               float spatial_scale, float *output, int32_t *argmax, sfod_stream_t stream) {
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || R < 0 || PH <= 0 || PW <= 0) return SFOD_ERR_INVALID_ARG;
  if (R == 0) return SFOD_OK;
  if (!input || !rois || !output || !argmax) return SFOD_ERR_INVALID_ARG;
  const long long total = (long long)R * C * PH * PW;
  roi_pool_fwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, sfod_cu(stream)>>>(input, rois, N, C, H, W, total, PH, PW,
                                                                                   spatial_scale, output, argmax);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

SFOD_API int sfod_roi_pool_bwd(const float *grad_out, const float *rois, const int32_t *argmax, int N, int C, int H, int W, int R,
                               int PH, int PW, float *grad_in, sfod_stream_t stream) {
  if (N <= 0 || C <= 0 || H <= 0 || W <= 0 || R < 0 || PH <= 0 || PW <= 0 || !grad_in) return SFOD_ERR_INVALID_ARG;
  cudaStream_t st = sfod_cu(stream);
  SFOD_CUDA_TRY(cudaMemsetAsync(grad_in, 0, (size_t)N * C * H * W * sizeof(float), st));
  if (R == 0) return SFOD_OK;
  if (!grad_out || !rois || !argmax) return SFOD_ERR_INVALID_ARG;
  const long long total = (long long)R * C * PH * PW;
  roi_pool_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(grad_out, rois, argmax, N, C, H, W, total, PH, PW, grad_in);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}
