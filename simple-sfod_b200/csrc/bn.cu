// bn.cu -- BatchNorm train-mode forward split for AdaBN statistic recomputation.
// Replaces the nn.BatchNorm2d train-mode forwards that reference daod/engine/trainers/base.py:274-299
// (test_refinement, after reset_bn_stats :318-323) and the no_grad teacher forward
// (source_free_adaptive_teacher.py:385-390) run only for their running-statistic side effect.
//
// HBM-bound: the statistics pass reads x once (4 B/element, SURVEY.md 8d: 777 MB per VGG image), the
// apply pass reads x and writes y (8 B/element).  Accuracy contract (1e-5 relative vs ATen's fp64
// accumulation): every thread accumulates at most 64 pivot-shifted elements in fp32, everything above
// that (warp, block, grid, and the E[x^2]-E[x]^2 combination) is fp64.
#include "common.cuh"
#include <cooperative_groups.h>
#include <string.h>

namespace {

constexpr int kThreads = 256;
constexpr int kChunk = 16384;  // elements of one (n, c) plane per CTA: 64 per thread
constexpr int kStatReplicas = 16;  // copies of the (sum, sum^2) totals the NHWC statistics kernel spreads its atomics over

__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}

// Adds the CTA's (count m, shifted sums about pivot K) to the unshifted fp64 channel totals.
__device__ __forceinline__ void flush_channel(double *stats, int c, double sd, double sd2, double m, double K) {
  // sum x = sd + m K ; sum x^2 = sd2 + 2 K sd + m K^2
  atomicAdd(stats + 2 * c, sd + m * K);
  atomicAdd(stats + 2 * c + 1, sd2 + 2.0 * K * sd + m * K * K);
}

// ---- NVLink peer-memory exchange of the statistics: inbox layout and the delivery step (described at the end of this file)
constexpr int kP2PMaxPayload = 4104;                   // 2 * 2048 + 1 doubles, rounded up to a multiple of 8
constexpr size_t kP2PHeaderBytes = 256;
constexpr int kP2PThreads = 1024;
constexpr long long kP2PSpinLimit = 6000000000ll;      // ~3 s of SM clocks: a missing peer must not hang the GPU

// One payload element on the wire: the two 32-bit halves of the double, each next to a copy of the exchange's 32-bit tag.
// An aligned 8-byte store is single-copy atomic, so each (half, tag) pair validates itself: the receiver needs neither a
// separate flag nor a fence between payload and flag -- one NVLink one-way latency per exchange (the "LL" idea of NCCL).
__device__ __forceinline__ uint4 *p2p_slot(char *inbox, int par, int src) {
  return reinterpret_cast<uint4 *>(inbox + kP2PHeaderBytes) + ((size_t)par * SFOD_P2P_MAX_RANKS + src) * kP2PMaxPayload;
}
__device__ __forceinline__ unsigned p2p_tag(unsigned long long epoch) { return (unsigned)(epoch & 0x7FFFFFFFull) | 0x80000000u; }   // never 0
__device__ __forceinline__ void p2p_store(uint4 *p, double v, unsigned tag) {
  const unsigned long long u = (unsigned long long)__double_as_longlong(v);
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"((unsigned)u), "r"(tag), "r"((unsigned)(u >> 32)), "r"(tag) : "memory");
}
__device__ __forceinline__ bool p2p_load(const uint4 *p, unsigned tag, double &v) {
  uint4 e;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(e.x), "=r"(e.y), "=r"(e.z), "=r"(e.w) : "l"(p) : "memory");
  v = __longlong_as_double((long long)(((unsigned long long)e.z << 32) | e.x));
  return e.y == tag && e.w == tag;
}

// Delivery step, called by all threads of one CTA: element i of `src` goes to slot [epoch & 1][rank] of every PEER's inbox.
__device__ __forceinline__ void p2p_push(const double *__restrict__ src, int n, const sfod_p2p_comm_t &comm, unsigned long long epoch) {
  const int par = (int)(epoch & 1ull);
  const unsigned tag = p2p_tag(epoch);
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = __ldcg(src + i);
    for (int p = 0; p < comm.world; ++p)
      if (p != comm.rank) p2p_store(p2p_slot(static_cast<char *>(comm.inbox[p]), par, comm.rank) + i, v, tag);
  }
}
constexpr unsigned long long kP2PPushed = ~0ull;   // value of the ticket word stats[2C + 1] once the statistics kernel has delivered the payload

template <bool kPush>
__global__ void __launch_bounds__(kThreads, kPush ? 8 : 1) bn_stats_nchw_kernel(const float *__restrict__ x, const float *__restrict__ pre_bias,
                                                                 int C, long long HW, double *__restrict__ stats, double local_count,
                                                                 sfod_p2p_comm_t comm) {
  __shared__ double red[2][kThreads / 32];
  const int plane = blockIdx.y;          // n * C + c
  if (local_count > 0.0 && blockIdx.x == 0 && plane == 0 && threadIdx.x == 0) stats[2 * C] = local_count;   // third part of the all-reduce payload
  const int c = plane % C;
  const long long start = (long long)blockIdx.x * kChunk;
  const long long len = min((long long)kChunk, HW - start);
  if (len <= 0 && !kPush) return;
  if (len > 0) {
  const float *p = x + (size_t)plane * HW + start;
  // The statistics are those of v = fl(x + pre_bias[c]) (the conv bias the reference adds before BatchNorm, fused here);
  // the pivot is expressed in x-space: (x + b) - (x0 + b) is evaluated as fl(fl(x + b) - K) with K = fl(x0 + b).
  const float pb = pre_bias ? pre_bias[c] : 0.f;
  const float K = x[(size_t)c * HW] + pb;     // pivot: first element of the channel in image 0
  float s = 0.f, s2 = 0.f;
  // peel to 16-byte alignment, then 128-bit loads
  const int mis = (int)((reinterpret_cast<uintptr_t>(p) >> 2) & 3);
  const int head = mis ? min((long long)(4 - mis), len) : 0;
  if (threadIdx.x < head) { const float d = (p[threadIdx.x] + pb) - K; s += d; s2 = fmaf(d, d, s2); }
  const float4 *p4 = reinterpret_cast<const float4 *>(p + head);
  const int n4 = (int)((len - head) >> 2);
#pragma unroll 4
  for (int i = threadIdx.x; i < n4; i += kThreads) {
    const float4 v = __ldg(p4 + i);
    const float d0 = (v.x + pb) - K, d1 = (v.y + pb) - K, d2 = (v.z + pb) - K, d3 = (v.w + pb) - K;
    s += (d0 + d1) + (d2 + d3);
    s2 = fmaf(d0, d0, s2); s2 = fmaf(d1, d1, s2); s2 = fmaf(d2, d2, s2); s2 = fmaf(d3, d3, s2);
  }
  const int tail0 = head + (n4 << 2);
  if (tail0 + (int)threadIdx.x < len) { const float d = (p[tail0 + threadIdx.x] + pb) - K; s += d; s2 = fmaf(d, d, s2); }
  double ds = warp_sum((double)s), ds2 = warp_sum((double)s2);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { red[0][warp] = ds; red[1][warp] = ds2; }
  __syncthreads();
  if (warp == 0) {
    ds = lane < kThreads / 32 ? red[0][lane] : 0.0;
    ds2 = lane < kThreads / 32 ? red[1][lane] : 0.0;
    ds = warp_sum(ds); ds2 = warp_sum(ds2);
    if (lane == 0) flush_channel(stats, c, ds, ds2, (double)len, (double)K);
  }
  }
  if constexpr (kPush) {
    // Multi-GPU: the CTA that finishes last (ticket word stats[2C + 1], zeroed with the totals) delivers the rank's 2C+1 payload
    // to every peer's inbox right here, so the NVLink latency overlaps the launch gap before the finalize kernel, which then
    // only polls for the peers' elements.
    __shared__ int s_last;
    unsigned long long *ticket = reinterpret_cast<unsigned long long *>(stats + 2 * C + 1);
    if (threadIdx.x == 0) {
      __threadfence();
      s_last = atomicAdd(ticket, 1ull) == (unsigned long long)gridDim.x * gridDim.y - 1ull;
    }
    __syncthreads();
    if (s_last) {
      __threadfence();
      const unsigned long long epoch = *reinterpret_cast<const unsigned long long *>(comm.inbox[comm.rank]) + 1ull;
      p2p_push(stats, 2 * C + 1, comm, epoch);
      if (threadIdx.x == 0) *ticket = kP2PPushed;
    }
  }
}

// NHWC: x viewed as (M = N*HW rows, C columns).  A CTA covers `cols` float4 column groups x `rowlanes`
// row lanes; each thread walks nrows (a multiple of 4, <= 64) rows with 128-bit loads (4 channels per load).
__global__ void __launch_bounds__(kThreads, 5) bn_stats_nhwc_kernel(const float *__restrict__ x, const float *__restrict__ pre_bias,
                                                                 long long M, int C, int cols, int rowlanes, int nrows,
                                                                 double *__restrict__ stats_replicas) {
  // fp64 atomics on one address are serialised by the L2 (~65 cycles each): with thousands of CTAs flushing 8 values per
  // column group into the same 2C totals that alone would cost as much as reading x.  CTAs therefore flush into one of
  // kStatReplicas copies (bn_fold_replicas_kernel adds them up afterwards).
  double *stats = stats_replicas + (size_t)(blockIdx.x % kStatReplicas) * 2 * C;
  extern __shared__ double sred[];  // rowlanes * cols * 9 doubles, then cols * 9 doubles, then cols * 4 floats
  const int G = C >> 2;
  const int col = threadIdx.x % cols, rl = threadIdx.x / cols;
  const int g = blockIdx.y * cols + col;
  const long long row0 = (long long)blockIdx.x * rowlanes * nrows;   // nrows <= 64 rows per thread
  const bool on = rl < rowlanes && g < G;
  float4 K = make_float4(0.f, 0.f, 0.f, 0.f);
  float4 s = K, s2 = K, pb = K;
  int cnt = 0;
  if (on) {
    if (pre_bias) pb = __ldg(reinterpret_cast<const float4 *>(pre_bias) + g);
    K = __ldg(reinterpret_cast<const float4 *>(x) + g);  // pivot: row 0
    K = make_float4(K.x + pb.x, K.y + pb.y, K.z + pb.z, K.w + pb.w);
    const float4 *p = reinterpret_cast<const float4 *>(x) + g;
    // batches of 4 rows: the four 128-bit loads are issued before any of them is consumed (bytes in flight, not
    // occupancy, decide the bandwidth of this kernel); rows beyond M load row M-1 and are masked out
    for (int i = 0; i < nrows; i += 4) {
      float4 v[4];
      bool ok[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const long long r = row0 + (long long)(i + j) * rowlanes + rl;
        ok[j] = r < M;
        v[j] = __ldg(p + (size_t)(ok[j] ? r : M - 1) * G);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float m = ok[j] ? 1.0f : 0.0f;
        const float d0 = m * ((v[j].x + pb.x) - K.x), d1 = m * ((v[j].y + pb.y) - K.y);
        const float d2 = m * ((v[j].z + pb.z) - K.z), d3 = m * ((v[j].w + pb.w) - K.w);
        s.x += d0; s.y += d1; s.z += d2; s.w += d3;
        s2.x = fmaf(d0, d0, s2.x); s2.y = fmaf(d1, d1, s2.y); s2.z = fmaf(d2, d2, s2.z); s2.w = fmaf(d3, d3, s2.w);
        cnt += ok[j] ? 1 : 0;
      }
    }
  }
  double *mine = sred + ((size_t)rl * cols + col) * 9;
  double *tot = sred + (size_t)rowlanes * cols * 9;              // [cols][9]
  float *piv = reinterpret_cast<float *>(tot + (size_t)cols * 9);   // [cols][4]
  if (rl < rowlanes) {
    mine[0] = s.x; mine[1] = s.y; mine[2] = s.z; mine[3] = s.w;
    mine[4] = s2.x; mine[5] = s2.y; mine[6] = s2.z; mine[7] = s2.w; mine[8] = (double)cnt;
    if (rl == 0) { piv[4 * col] = K.x; piv[4 * col + 1] = K.y; piv[4 * col + 2] = K.z; piv[4 * col + 3] = K.w; }
  }
  __syncthreads();
  for (int item = threadIdx.x; item < cols * 9; item += kThreads) {   // (column group, value) pairs in parallel
    double t = 0.0;
    for (int q = 0; q < rowlanes; ++q) t += sred[(size_t)q * cols * 9 + item];
    tot[item] = t;
  }
  __syncthreads();
  if (threadIdx.x < cols * 4) {   // one thread per channel of the CTA
    const int cl = threadIdx.x >> 2, kk = threadIdx.x & 3;
    const int gg = blockIdx.y * cols + cl;
    if (gg < G)
      flush_channel(stats, 4 * gg + kk, tot[cl * 9 + kk], tot[cl * 9 + 4 + kk], tot[cl * 9 + 8], (double)piv[4 * cl + kk]);
  }
}

__global__ void __launch_bounds__(128) bn_fold_replicas_kernel(const double *__restrict__ replicas, int C, double *__restrict__ stats,
                                                               double local_count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i == 0) stats[2 * C] = local_count;
  if (i >= 2 * C) return;
  double t = 0.0;
#pragma unroll
  for (int r = 0; r < kStatReplicas; ++r) t += replicas[(size_t)r * 2 * C + i];
  stats[i] = t;
}

// scalar fallback for NHWC with C % 4 != 0 (not used by any shipped config)
__global__ void __launch_bounds__(kThreads) bn_stats_nhwc_scalar_kernel(const float *__restrict__ x, const float *__restrict__ pre_bias,
                                                                        long long M, int C, double *__restrict__ stats) {
  const int c = blockIdx.x;
  const float pb = pre_bias ? pre_bias[c] : 0.f;
  double s = 0.0, s2 = 0.0;
  for (long long r = threadIdx.x; r < M; r += kThreads) { const double v = x[(size_t)r * C + c] + pb; s += v; s2 += v * v; }
  __shared__ double red[2][kThreads / 32];
  s = warp_sum(s); s2 = warp_sum(s2);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s; red[1][threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < kThreads / 32; ++w) { s += red[0][w]; s2 += red[1][w]; }
    stats[2 * c] += s; stats[2 * c + 1] += s2;
  }
}

// One channel: ATen batch_norm_cpu_update_stats arithmetic in fp64 on the channel's (sum x, sum x^2) and the element count n.
__device__ __forceinline__ void bn_finalize_channel(int c, double sum, double sumsq, double n, const float *__restrict__ weight,
                                                    const float *__restrict__ bias, float *__restrict__ running_mean,
                                                    float *__restrict__ running_var, double momentum, double eps,
                                                    float *__restrict__ scale, float *__restrict__ shift) {
  const double mean = sum / n;
  double var = sumsq / n - mean * mean;
  if (var < 0.0) var = 0.0;
  const double invstd = 1.0 / sqrt(var + eps);
  const float mean_f = (float)mean;
  if (running_mean) running_mean[c] = (float)(momentum * (double)mean_f + (1.0 - momentum) * (double)running_mean[c]);
  if (running_var) {
    const double unbiased = n > 1.0 ? var * n / (n - 1.0) : var;
    running_var[c] = (float)(momentum * unbiased + (1.0 - momentum) * (double)running_var[c]);
  }
  const double w = weight ? (double)weight[c] : 1.0, b = bias ? (double)bias[c] : 0.0;
  scale[c] = (float)(w * invstd);
  shift[c] = (float)(b - mean * w * invstd);
}

// One thread per channel.
__global__ void bn_finalize_kernel(const double *__restrict__ stats, int C, const float *__restrict__ weight,
                                   const float *__restrict__ bias, float *__restrict__ running_mean,
                                   float *__restrict__ running_var, long long *__restrict__ nbt, double momentum, double eps,
                                   float *__restrict__ scale, float *__restrict__ shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0 && nbt) *nbt += 1;
  if (c >= C) return;
  const double n = stats[2 * C];   // element count left by phase 1 (and summed over the ranks by an all-reduce): no host read between the phases
  bn_finalize_channel(c, stats[2 * c], stats[2 * c + 1], n, weight, bias, running_mean, running_var, momentum, eps, scale, shift);
}

template <bool kRelu>
__device__ __forceinline__ float bn1(float v, float pb, float sc, float sh) {
  const float y = fmaf(v + pb, sc, sh);   // fl(x + conv_bias) first, exactly the tensor the reference normalises
  return kRelu ? fmaxf(y, 0.f) : y;
}
// BatchNorm -> (+ residual) -> ReLU of a ResNet bottleneck's last convolution (detectron2 BottleneckBlock.forward:
// out = conv3(out) [conv + norm]; out += shortcut; out = relu_(out)): the normalised value is rounded to fp32 first,
// then the shortcut is added, as in the three separate passes it replaces (12 instead of 28 B/element).
template <bool kRelu>
__device__ __forceinline__ float bn1r(float v, float pb, float sc, float sh, float r) {
  const float y = __fadd_rn(fmaf(v + pb, sc, sh), r);
  return kRelu ? fmaxf(y, 0.f) : y;
}

template <bool kRelu, bool kRes>
__global__ void __launch_bounds__(kThreads) bn_apply_nchw_kernel(const float *__restrict__ x, const float *__restrict__ pre_bias,
                                                                 const float *__restrict__ res, float *__restrict__ y, int C, long long HW,
                                                                 const float *__restrict__ scale, const float *__restrict__ shift) {
  const int plane = blockIdx.y;
  const int c = plane % C;
  const long long start = (long long)blockIdx.x * kChunk;
  const long long len = min((long long)kChunk, HW - start);
  if (len <= 0) return;
  const float sc = scale[c], sh = shift[c], pb = pre_bias ? pre_bias[c] : 0.f;
  const float *p = x + (size_t)plane * HW + start;
  const float *r = kRes ? res + (size_t)plane * HW + start : nullptr;   // same 16-byte phase as x (checked by the host)
  float *q = y + (size_t)plane * HW + start;
  const int mis = (int)((reinterpret_cast<uintptr_t>(p) >> 2) & 3);
  const int head = mis ? min((long long)(4 - mis), len) : 0;
  if (threadIdx.x < head) q[threadIdx.x] = kRes ? bn1r<kRelu>(p[threadIdx.x], pb, sc, sh, r[threadIdx.x]) : bn1<kRelu>(p[threadIdx.x], pb, sc, sh);
  const float4 *p4 = reinterpret_cast<const float4 *>(p + head);
  const float4 *r4 = reinterpret_cast<const float4 *>(r + head);
  float4 *q4 = reinterpret_cast<float4 *>(q + head);
  const int n4 = (int)((len - head) >> 2);
#pragma unroll 4
  for (int i = threadIdx.x; i < n4; i += kThreads) {
    const float4 v = p4[i];
    if (kRes) {
      const float4 w = __ldg(r4 + i);
      q4[i] = make_float4(bn1r<kRelu>(v.x, pb, sc, sh, w.x), bn1r<kRelu>(v.y, pb, sc, sh, w.y), bn1r<kRelu>(v.z, pb, sc, sh, w.z), bn1r<kRelu>(v.w, pb, sc, sh, w.w));
    } else {
      q4[i] = make_float4(bn1<kRelu>(v.x, pb, sc, sh), bn1<kRelu>(v.y, pb, sc, sh), bn1<kRelu>(v.z, pb, sc, sh), bn1<kRelu>(v.w, pb, sc, sh));
    }
  }
  const int tail0 = head + (n4 << 2);
  if (tail0 + (int)threadIdx.x < len) {
    const int t = tail0 + threadIdx.x;
    q[t] = kRes ? bn1r<kRelu>(p[t], pb, sc, sh, r[t]) : bn1<kRelu>(p[t], pb, sc, sh);
  }
}

// Normalise (+ReLU) fused with the 2x2 / stride-2 max-pool that follows the last BN of every VGG stage
// (reference daod/modeling/meta_arch/vgg.py:10-24): reads x once (4 B/element), writes the pooled map (1 B/element).
// The affine map may have a negative scale, so it is applied per element BEFORE the max.
// kVec: W % 4 == 0 and 16-byte aligned planes -> one float4 per input row and thread, two outputs (float2 store).
constexpr int kPoolOutPerCta = 4096;  // pooled outputs per CTA
template <bool kRelu, bool kVec>
__global__ void __launch_bounds__(kThreads) bn_apply_pool_nchw_kernel(const float *__restrict__ x, const float *__restrict__ pre_bias,
                                                                      float *__restrict__ y, int C, int H, int W, int H2, int W2,
                                                                      const float *__restrict__ scale, const float *__restrict__ shift) {
  const int plane = blockIdx.y;
  const int c = plane % C;
  const float sc = scale[c], sh = shift[c], pb = pre_bias ? pre_bias[c] : 0.f;
  const float *p = x + (size_t)plane * H * W;
  float *q = y + (size_t)plane * H2 * W2;
  const int total = H2 * W2;
  const int o0 = blockIdx.x * kPoolOutPerCta;
  const int o1 = min(o0 + kPoolOutPerCta, total);
  if (kVec) {
    const int W2h = W2 >> 1;  // output pairs per row
    for (int i = (o0 >> 1) + threadIdx.x; i < (o1 >> 1); i += kThreads) {
      const int oy = i / W2h, oxp = i - oy * W2h;
      const float4 a = __ldg(reinterpret_cast<const float4 *>(p + (size_t)(2 * oy) * W) + oxp);
      const float4 b = __ldg(reinterpret_cast<const float4 *>(p + (size_t)(2 * oy + 1) * W) + oxp);
      float2 r;
      r.x = fmaxf(fmaxf(bn1<kRelu>(a.x, pb, sc, sh), bn1<kRelu>(a.y, pb, sc, sh)), fmaxf(bn1<kRelu>(b.x, pb, sc, sh), bn1<kRelu>(b.y, pb, sc, sh)));
      r.y = fmaxf(fmaxf(bn1<kRelu>(a.z, pb, sc, sh), bn1<kRelu>(a.w, pb, sc, sh)), fmaxf(bn1<kRelu>(b.z, pb, sc, sh), bn1<kRelu>(b.w, pb, sc, sh)));
      reinterpret_cast<float2 *>(q + (size_t)oy * W2)[oxp] = r;
    }
  } else {
    for (int o = o0 + threadIdx.x; o < o1; o += kThreads) {
      const int oy = o / W2, ox = o - oy * W2;
      const float *r0 = p + (size_t)(2 * oy) * W + 2 * ox;
      const float *r1 = r0 + W;
      const float v = fmaxf(fmaxf(bn1<kRelu>(__ldg(r0), pb, sc, sh), bn1<kRelu>(__ldg(r0 + 1), pb, sc, sh)),
                            fmaxf(bn1<kRelu>(__ldg(r1), pb, sc, sh), bn1<kRelu>(__ldg(r1 + 1), pb, sc, sh)));
      q[o] = v;
    }
  }
}

template <bool kRelu, bool kRes>
__global__ void __launch_bounds__(kThreads) bn_apply_nhwc_kernel(const float *__restrict__ x, const float *__restrict__ pre_bias,
                                                                 const float *__restrict__ res, float *__restrict__ y, long long total4, int G,
                                                                 const float *__restrict__ scale, const float *__restrict__ shift) {
  const float4 *x4 = reinterpret_cast<const float4 *>(x);
  const float4 *r4 = reinterpret_cast<const float4 *>(res);
  float4 *y4 = reinterpret_cast<float4 *>(y);
  const float4 *sc4 = reinterpret_cast<const float4 *>(scale), *sh4 = reinterpret_cast<const float4 *>(shift);
  const float4 *pb4 = reinterpret_cast<const float4 *>(pre_bias);
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < total4; i += (long long)gridDim.x * kThreads) {
    const int g = (int)(i % G);
    const float4 v = x4[i], sc = __ldg(sc4 + g), sh = __ldg(sh4 + g);
    const float4 pb = pre_bias ? __ldg(pb4 + g) : make_float4(0.f, 0.f, 0.f, 0.f);
    if (kRes) {
      const float4 w = __ldg(r4 + i);
      y4[i] = make_float4(bn1r<kRelu>(v.x, pb.x, sc.x, sh.x, w.x), bn1r<kRelu>(v.y, pb.y, sc.y, sh.y, w.y),
                          bn1r<kRelu>(v.z, pb.z, sc.z, sh.z, w.z), bn1r<kRelu>(v.w, pb.w, sc.w, sh.w, w.w));
    } else {
      y4[i] = make_float4(bn1<kRelu>(v.x, pb.x, sc.x, sh.x), bn1<kRelu>(v.y, pb.y, sc.y, sh.y), bn1<kRelu>(v.z, pb.z, sc.z, sh.z),
                          bn1<kRelu>(v.w, pb.w, sc.w, sh.w));
    }
  }
}

// NHWC normalise(+ReLU)+max-pool: one thread per (n, oy, ox, channel group of 4): four float4 loads, one float4 store.
template <bool kRelu>
__global__ void __launch_bounds__(kThreads) bn_apply_pool_nhwc_kernel(const float *__restrict__ x, const float *__restrict__ pre_bias,
                                                                      float *__restrict__ y, int N, int H, int W, int H2, int W2, int G,
                                                                      const float *__restrict__ scale, const float *__restrict__ shift) {
  const float4 *x4 = reinterpret_cast<const float4 *>(x);
  float4 *y4 = reinterpret_cast<float4 *>(y);
  const long long total = (long long)N * H2 * W2 * G;
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kThreads) {
    const int g = (int)(i % G);
    long long r = i / G;
    const int ox = (int)(r % W2); r /= W2;
    const int oy = (int)(r % H2);
    const int n = (int)(r / H2);
    const float4 sc = __ldg(reinterpret_cast<const float4 *>(scale) + g), sh = __ldg(reinterpret_cast<const float4 *>(shift) + g);
    const float4 pb = pre_bias ? __ldg(reinterpret_cast<const float4 *>(pre_bias) + g) : make_float4(0.f, 0.f, 0.f, 0.f);
    const size_t base = (((size_t)n * H + 2 * oy) * W + 2 * ox) * G + g;
    const float4 a = __ldg(x4 + base), b = __ldg(x4 + base + G), c = __ldg(x4 + base + (size_t)W * G), d = __ldg(x4 + base + (size_t)W * G + G);
    float4 o;
    o.x = fmaxf(fmaxf(bn1<kRelu>(a.x, pb.x, sc.x, sh.x), bn1<kRelu>(b.x, pb.x, sc.x, sh.x)), fmaxf(bn1<kRelu>(c.x, pb.x, sc.x, sh.x), bn1<kRelu>(d.x, pb.x, sc.x, sh.x)));
    o.y = fmaxf(fmaxf(bn1<kRelu>(a.y, pb.y, sc.y, sh.y), bn1<kRelu>(b.y, pb.y, sc.y, sh.y)), fmaxf(bn1<kRelu>(c.y, pb.y, sc.y, sh.y), bn1<kRelu>(d.y, pb.y, sc.y, sh.y)));
    o.z = fmaxf(fmaxf(bn1<kRelu>(a.z, pb.z, sc.z, sh.z), bn1<kRelu>(b.z, pb.z, sc.z, sh.z)), fmaxf(bn1<kRelu>(c.z, pb.z, sc.z, sh.z), bn1<kRelu>(d.z, pb.z, sc.z, sh.z)));
    o.w = fmaxf(fmaxf(bn1<kRelu>(a.w, pb.w, sc.w, sh.w), bn1<kRelu>(b.w, pb.w, sc.w, sh.w)), fmaxf(bn1<kRelu>(c.w, pb.w, sc.w, sh.w), bn1<kRelu>(d.w, pb.w, sc.w, sh.w)));
    y4[i] = o;
  }
}

template <bool kRelu>
__global__ void __launch_bounds__(kThreads) bn_apply_nhwc_scalar_kernel(const float *__restrict__ x, const float *__restrict__ pre_bias,
                                                                        const float *__restrict__ res, float *__restrict__ y, long long total, int C,
                                                                        const float *__restrict__ scale, const float *__restrict__ shift) {
  for (long long i = (long long)blockIdx.x * kThreads + threadIdx.x; i < total; i += (long long)gridDim.x * kThreads) {
    const int c = (int)(i % C);
    const float pb = pre_bias ? pre_bias[c] : 0.f;
    y[i] = res ? bn1r<kRelu>(x[i], pb, scale[c], shift[c], res[i]) : bn1<kRelu>(x[i], pb, scale[c], shift[c]);
  }
}


// ---- single-launch train-mode BatchNorm for activations that (mostly) fit the 126 MB L2: statistics -> grid barrier ->
// normalise (+residual)(+ReLU), one cooperative persistent kernel.  The unit of work is (chunk of <= 4096 elements of one (n, c)
// plane) x (one WARP): the late layers this kernel serves have small planes (38 x 75 = 2 850 elements on R101-C4 res4), so a
// CTA-wide pass per plane would spend its time in block barriers and in the latency of a handful of loads; eight independent
// warps per CTA keep eight chunks in flight.  Every warp owns a contiguous range of chunks; phase 1 accumulates the fp64 channel
// totals (<= 64 pivot-shifted fp32 terms per thread between fp64 folds, as in bn_stats_nchw_kernel), phase 2 walks the SAME
// chunks in reverse order, so the second read of x is served by L2 (most recently touched lines first): HBM sees ~4 B/element of
// reads + 4 B/element of writes instead of 12, and the layer is one launch instead of four (memset, statistics, finalize, apply).
constexpr int kFChunk = 4096;

template <bool kRelu, bool kRes>
__global__ void __launch_bounds__(kThreads, 2) bn_fused_nchw_kernel(const float *__restrict__ x, const float *__restrict__ pre_bias,
                                                                    const float *__restrict__ res, float *__restrict__ y, int NC, int C,
                                                                    long long HW, double *__restrict__ stats, double count,
                                                                    const float *__restrict__ weight, const float *__restrict__ bias,
                                                                    float *__restrict__ running_mean, float *__restrict__ running_var,
                                                                    long long *__restrict__ nbt, double momentum, double eps) {
  namespace cg = cooperative_groups;
  const int cpp = (int)((HW + kFChunk - 1) / kFChunk);            // chunks per plane
  const long long nchunks = (long long)NC * cpp;
  const int lane = threadIdx.x & 31;
  const long long wg = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5), nw = (long long)gridDim.x * (kThreads / 32);
  const long long q0 = nchunks * wg / nw, q1 = nchunks * (wg + 1) / nw;
  // ---------------- phase 1
  for (long long q = q0; q < q1; ++q) {
    const int plane = (int)(q / cpp), c = plane % C;
    const long long start = (q - (long long)plane * cpp) * kFChunk;
    const int len = (int)min((long long)kFChunk, HW - start);
    const float *p = x + (size_t)plane * HW + start;
    const float pb = pre_bias ? pre_bias[c] : 0.f;
    const float K = x[(size_t)c * HW] + pb;                       // pivot: first element of the channel in image 0
    const int mis = (int)((reinterpret_cast<uintptr_t>(p) >> 2) & 3);
    const int head = mis ? min(4 - mis, len) : 0;
    const float4 *p4 = reinterpret_cast<const float4 *>(p + head);
    const int n4 = (len - head) >> 2;
    const int tail0 = head + (n4 << 2);
    double ds = 0.0, ds2 = 0.0;
    {
      float s = 0.f, s2 = 0.f;
      if (lane < head) { const float d = (p[lane] + pb) - K; s += d; s2 = fmaf(d, d, s2); }
      if (tail0 + lane < len) { const float d = (p[tail0 + lane] + pb) - K; s += d; s2 = fmaf(d, d, s2); }
      ds += (double)s; ds2 += (double)s2;
    }
    for (int b = 0; b < n4; b += 32 * 16) {                      // 16 float4 (64 elements) per lane between fp64 folds
      float s = 0.f, s2 = 0.f;
      float4 v[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) { const int i = b + k * 32 + lane; v[k] = i < n4 ? p4[i] : make_float4(K - pb, K - pb, K - pb, K - pb); }
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        const float d0 = (v[k].x + pb) - K, d1 = (v[k].y + pb) - K, d2 = (v[k].z + pb) - K, d3 = (v[k].w + pb) - K;
        s += (d0 + d1) + (d2 + d3);
        s2 = fmaf(d0, d0, s2); s2 = fmaf(d1, d1, s2); s2 = fmaf(d2, d2, s2); s2 = fmaf(d3, d3, s2);
      }
      ds += (double)s; ds2 += (double)s2;
    }
    ds = warp_sum(ds); ds2 = warp_sum(ds2);
    if (lane == 0) flush_channel(stats, c, ds, ds2, (double)len, (double)K);
  }
  __threadfence();
  cg::this_grid().sync();
  // ---------------- phase 2: reverse order; the coefficients of up to 32 chunks are computed by the 32 lanes in parallel
  if (blockIdx.x == 0 && threadIdx.x == 0 && nbt) *nbt += 1;
  for (long long qq = q1; qq > q0; qq -= 32) {
    float sc_l = 0.f, sh_l = 0.f;
    {
      const long long myq = qq - 1 - lane;
      if (myq >= q0) {
        const int plane = (int)(myq / cpp), c = plane % C;
        const double mean = __ldcg(stats + 2 * c) / count;
        double var = __ldcg(stats + 2 * c + 1) / count - mean * mean;
        if (var < 0.0) var = 0.0;
        const double invstd = 1.0 / sqrt(var + eps);
        const double w = weight ? (double)weight[c] : 1.0, b = bias ? (double)bias[c] : 0.0;
        sc_l = (float)(w * invstd);
        sh_l = (float)(b - mean * w * invstd);
        if (plane < C && myq - (long long)plane * cpp == 0) {     // image 0, first chunk: owner of channel c's running statistics
          const float mean_f = (float)mean;
          if (running_mean) running_mean[c] = (float)(momentum * (double)mean_f + (1.0 - momentum) * (double)running_mean[c]);
          if (running_var) {
            const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
            running_var[c] = (float)(momentum * unbiased + (1.0 - momentum) * (double)running_var[c]);
          }
        }
      }
    }
    const int nq = (int)min((long long)32, qq - q0);
    for (int j = 0; j < nq; ++j) {
      const long long q = qq - 1 - j;
      const float sc = __shfl_sync(0xFFFFFFFFu, sc_l, j), sh = __shfl_sync(0xFFFFFFFFu, sh_l, j);
      const int plane = (int)(q / cpp), c = plane % C;
      const long long start = (q - (long long)plane * cpp) * kFChunk;
      const int len = (int)min((long long)kFChunk, HW - start);
      const float pb = pre_bias ? pre_bias[c] : 0.f;
      const float *p = x + (size_t)plane * HW + start;
      const float *r = kRes ? res + (size_t)plane * HW + start : nullptr;
      float *o = y + (size_t)plane * HW + start;
      const int mis = (int)((reinterpret_cast<uintptr_t>(p) >> 2) & 3);
      const int head = mis ? min(4 - mis, len) : 0;
      const float4 *p4 = reinterpret_cast<const float4 *>(p + head);
      const float4 *r4 = reinterpret_cast<const float4 *>(r + head);
      float4 *o4 = reinterpret_cast<float4 *>(o + head);
      const int n4 = (len - head) >> 2;
      const int tail0 = head + (n4 << 2);
      if (lane < head) o[lane] = kRes ? bn1r<kRelu>(p[lane], pb, sc, sh, r[lane]) : bn1<kRelu>(p[lane], pb, sc, sh);
      if (tail0 + lane < len) { const int t = tail0 + lane; o[t] = kRes ? bn1r<kRelu>(p[t], pb, sc, sh, r[t]) : bn1<kRelu>(p[t], pb, sc, sh); }
      for (int b = 0; b < n4; b += 32 * 8) {
        float4 v[8], w4[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int i = b + k * 32 + lane;
          if (i < n4) { v[k] = p4[i]; if (kRes) w4[k] = __ldg(r4 + i); }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const int i = b + k * 32 + lane;
          if (i < n4) {
            if (kRes) o4[i] = make_float4(bn1r<kRelu>(v[k].x, pb, sc, sh, w4[k].x), bn1r<kRelu>(v[k].y, pb, sc, sh, w4[k].y),
                                          bn1r<kRelu>(v[k].z, pb, sc, sh, w4[k].z), bn1r<kRelu>(v[k].w, pb, sc, sh, w4[k].w));
            else o4[i] = make_float4(bn1<kRelu>(v[k].x, pb, sc, sh), bn1<kRelu>(v[k].y, pb, sc, sh), bn1<kRelu>(v[k].z, pb, sc, sh),
                                     bn1<kRelu>(v[k].w, pb, sc, sh));
          }
        }
      }
    }
  }
}

}  // namespace

SFOD_API size_t sfod_bn_stats_bytes(int C) {
  return C > 0 ? sfod_align_up((size_t)C * (4 + 2 * kStatReplicas) * sizeof(double), 256) : 256;
}

static bool p2p_comm_ok(const sfod_p2p_comm_t *comm) {
  if (!comm || comm->world < 1 || comm->world > SFOD_P2P_MAX_RANKS || comm->rank < 0 || comm->rank >= comm->world) return false;
  for (int r = 0; r < comm->world; ++r)
    if (!comm->inbox[r]) return false;
  return true;
}

SFOD_API int sfod_bn_partial_stats(const float *x, const float *pre_bias, int layout, int N, int C, int64_t HW, double *stats_dev,
                                   const sfod_p2p_comm_t *comm, sfod_stream_t stream) {
  if (comm && !p2p_comm_ok(comm)) return SFOD_ERR_INVALID_ARG;
  if (comm && 2 * C + 1 > kP2PMaxPayload) return SFOD_ERR_UNSUPPORTED;
  if (!x || !stats_dev || N <= 0 || C <= 0 || HW <= 0) return SFOD_ERR_INVALID_ARG;
  if (layout != SFOD_NCHW && layout != SFOD_NHWC) return SFOD_ERR_INVALID_ARG;
  cudaStream_t st = sfod_cu(stream);
  SFOD_CUDA_TRY(cudaMemsetAsync(stats_dev, 0, ((size_t)C * 2 + 2) * sizeof(double), st));   // totals, count, ticket word
  if (layout == SFOD_NCHW) {
    const long long planes = (long long)N * C;
    const long long step = 65535 / C * (long long)C;  // grid.y limit; multiples of C keep channel = plane % C
    if (step == 0) return SFOD_ERR_UNSUPPORTED;
    const bool push = comm != nullptr && planes <= step;   // one launch covers the layer: its last CTA delivers the payload
    for (long long p0 = 0; p0 < planes; p0 += step) {
      const long long np = planes - p0 < step ? planes - p0 : step;
      dim3 grid((unsigned)((HW + kChunk - 1) / kChunk), (unsigned)np);
      const double cnt = p0 == 0 ? (double)N * (double)HW : 0.0;
      if (push) bn_stats_nchw_kernel<true><<<grid, kThreads, 0, st>>>(x + (size_t)p0 * HW, pre_bias, C, HW, stats_dev, cnt, *comm);
      else bn_stats_nchw_kernel<false><<<grid, kThreads, 0, st>>>(x + (size_t)p0 * HW, pre_bias, C, HW, stats_dev, cnt, sfod_p2p_comm_t{});
      SFOD_LAUNCH_CHECK();
    }
    return SFOD_OK;
  }
  const long long M = (long long)N * HW;
  if ((C & 3) || !sfod_aligned16(x) || (pre_bias && !sfod_aligned16(pre_bias))) {
    bn_stats_nhwc_scalar_kernel<<<C, kThreads, 0, st>>>(x, pre_bias, M, C, stats_dev);
    SFOD_LAUNCH_CHECK();
    const double cnt = (double)M;
    SFOD_CUDA_TRY(cudaMemcpyAsync(stats_dev + 2 * (size_t)C, &cnt, sizeof(double), cudaMemcpyHostToDevice, st));   // pageable 8 B: staged by the driver
    return SFOD_OK;
  }
  const int G = C >> 2;
  const int cols = G < 64 ? G : 64;
  const int rowlanes = kThreads / cols;
  const long long gy = (G + cols - 1) / cols;
  int nrows = 64;   // rows per thread: fewer for small maps so that the layer still fills the machine (>= 16 CTAs per SM)
  while (nrows > 8 && ((M + (long long)rowlanes * nrows - 1) / ((long long)rowlanes * nrows)) * gy < (long long)SFOD_NUM_SMS * 16) nrows >>= 1;
  dim3 grid((unsigned)((M + (long long)rowlanes * nrows - 1) / ((long long)rowlanes * nrows)), (unsigned)gy);
  const size_t smem = ((size_t)rowlanes * cols * 9 + (size_t)cols * 9) * sizeof(double) + (size_t)cols * 4 * sizeof(float);
  double *replicas = stats_dev + 4 * (size_t)C;
  SFOD_CUDA_TRY(cudaMemsetAsync(replicas, 0, (size_t)C * 2 * kStatReplicas * sizeof(double), st));   // totals were zeroed above
  bn_stats_nhwc_kernel<<<grid, kThreads, smem, st>>>(x, pre_bias, M, C, cols, rowlanes, nrows, replicas);
  SFOD_LAUNCH_CHECK();
  bn_fold_replicas_kernel<<<(2 * C + 127) / 128, 128, 0, st>>>(replicas, C, stats_dev, (double)N * (double)HW);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

namespace {
// normalise (+residual) (+ReLU) (+2x2 max-pool) with given per-channel scale / shift: the launches shared by the train-mode and
// the frozen-statistics entry points
int launch_bn_apply(const float *x, const float *pre_bias, const float *residual, float *y, int layout, int N, int C, int H, int W,
                    const float *scale, const float *shift, int fuse_relu, int fuse_maxpool2, cudaStream_t st) {
  const long long HW = (long long)H * W;
  if (fuse_maxpool2) {
    const int H2 = H / 2, W2 = W / 2;
    if (H2 == 0 || W2 == 0) return SFOD_OK;  // empty pooled map
    if (x == y) return SFOD_ERR_INVALID_ARG;  // the pooled output cannot alias the input
    if (layout == SFOD_NCHW) {
      const long long planes = (long long)N * C;
      const long long step = 65535 / C * (long long)C;
      if (step == 0) return SFOD_ERR_UNSUPPORTED;
      const bool vec = (W % 4 == 0) && (HW % 4 == 0) && sfod_aligned16(x) && ((reinterpret_cast<uintptr_t>(y) & 7u) == 0);
      for (long long p0 = 0; p0 < planes; p0 += step) {
        const long long np = planes - p0 < step ? planes - p0 : step;
        dim3 grid((unsigned)((H2 * W2 + kPoolOutPerCta - 1) / kPoolOutPerCta), (unsigned)np);
        const float *xp = x + (size_t)p0 * HW;
        float *yp = y + (size_t)p0 * H2 * W2;
        if (vec) {
          if (fuse_relu) bn_apply_pool_nchw_kernel<true, true><<<grid, kThreads, 0, st>>>(xp, pre_bias, yp, C, H, W, H2, W2, scale, shift);
          else bn_apply_pool_nchw_kernel<false, true><<<grid, kThreads, 0, st>>>(xp, pre_bias, yp, C, H, W, H2, W2, scale, shift);
        } else {
          if (fuse_relu) bn_apply_pool_nchw_kernel<true, false><<<grid, kThreads, 0, st>>>(xp, pre_bias, yp, C, H, W, H2, W2, scale, shift);
          else bn_apply_pool_nchw_kernel<false, false><<<grid, kThreads, 0, st>>>(xp, pre_bias, yp, C, H, W, H2, W2, scale, shift);
        }
        SFOD_LAUNCH_CHECK();
      }
      return SFOD_OK;
    }
    if ((C & 3) || !sfod_aligned16(x) || !sfod_aligned16(y) || (pre_bias && !sfod_aligned16(pre_bias))) return SFOD_ERR_UNSUPPORTED;
    const long long total = (long long)N * H2 * W2 * (C >> 2);
    const unsigned grid = (unsigned)min((long long)SFOD_NUM_SMS * 16, (total + kThreads - 1) / kThreads);
    if (fuse_relu) bn_apply_pool_nhwc_kernel<true><<<grid, kThreads, 0, st>>>(x, pre_bias, y, N, H, W, H2, W2, C >> 2, scale, shift);
    else bn_apply_pool_nhwc_kernel<false><<<grid, kThreads, 0, st>>>(x, pre_bias, y, N, H, W, H2, W2, C >> 2, scale, shift);
    SFOD_LAUNCH_CHECK();
    return SFOD_OK;
  }
  if (layout == SFOD_NCHW) {
    const long long planes = (long long)N * C;
    const long long step = 65535 / C * (long long)C;
    if (step == 0) return SFOD_ERR_UNSUPPORTED;
    for (long long p0 = 0; p0 < planes; p0 += step) {
      const long long np = planes - p0 < step ? planes - p0 : step;
      dim3 grid((unsigned)((HW + kChunk - 1) / kChunk), (unsigned)np);
      const float *xp = x + (size_t)p0 * HW, *rp = residual ? residual + (size_t)p0 * HW : nullptr;
      float *yp = y + (size_t)p0 * HW;
      if (residual) {
        if (fuse_relu) bn_apply_nchw_kernel<true, true><<<grid, kThreads, 0, st>>>(xp, pre_bias, rp, yp, C, HW, scale, shift);
        else bn_apply_nchw_kernel<false, true><<<grid, kThreads, 0, st>>>(xp, pre_bias, rp, yp, C, HW, scale, shift);
      } else {
        if (fuse_relu) bn_apply_nchw_kernel<true, false><<<grid, kThreads, 0, st>>>(xp, pre_bias, rp, yp, C, HW, scale, shift);
        else bn_apply_nchw_kernel<false, false><<<grid, kThreads, 0, st>>>(xp, pre_bias, rp, yp, C, HW, scale, shift);
      }
      SFOD_LAUNCH_CHECK();
    }
    return SFOD_OK;
  }
  const long long total = (long long)N * HW * C;
  if ((C & 3) || !sfod_aligned16(x) || !sfod_aligned16(y) || (pre_bias && !sfod_aligned16(pre_bias))) {
    const unsigned grid = (unsigned)min((long long)SFOD_NUM_SMS * 8, (total + kThreads - 1) / kThreads);
    if (fuse_relu) bn_apply_nhwc_scalar_kernel<true><<<grid, kThreads, 0, st>>>(x, pre_bias, residual, y, total, C, scale, shift);
    else bn_apply_nhwc_scalar_kernel<false><<<grid, kThreads, 0, st>>>(x, pre_bias, residual, y, total, C, scale, shift);
  } else {
    const long long total4 = total >> 2;
    const unsigned grid = (unsigned)min((long long)SFOD_NUM_SMS * 16, (total4 + kThreads - 1) / kThreads);
    if (residual) {
      if (fuse_relu) bn_apply_nhwc_kernel<true, true><<<grid, kThreads, 0, st>>>(x, pre_bias, residual, y, total4, C >> 2, scale, shift);
      else bn_apply_nhwc_kernel<false, true><<<grid, kThreads, 0, st>>>(x, pre_bias, residual, y, total4, C >> 2, scale, shift);
    } else {
      if (fuse_relu) bn_apply_nhwc_kernel<true, false><<<grid, kThreads, 0, st>>>(x, pre_bias, residual, y, total4, C >> 2, scale, shift);
      else bn_apply_nhwc_kernel<false, false><<<grid, kThreads, 0, st>>>(x, pre_bias, residual, y, total4, C >> 2, scale, shift);
    }
  }
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

// FrozenBatchNorm2d / eval-mode BatchNorm coefficients: y = x * scale + shift with scale = w / sqrt(running_var + eps),
// shift = b - running_mean * scale (detectron2 layers/batch_norm.py FrozenBatchNorm2d.forward, fp32 like the reference).
__global__ void bn_frozen_coeffs_kernel(int C, const float *__restrict__ weight, const float *__restrict__ bias,
                                        const float *__restrict__ running_mean, const float *__restrict__ running_var, float eps,
                                        float *__restrict__ scale, float *__restrict__ shift) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float w = weight ? weight[c] : 1.0f, b = bias ? bias[c] : 0.0f;
  const float sc = __fmul_rn(w, __frsqrt_rn(__fadd_rn(running_var[c], eps)));
  scale[c] = sc;
  shift[c] = __fsub_rn(b, __fmul_rn(running_mean[c], sc));
}
}  // namespace

SFOD_API size_t sfod_bn_frozen_scratch_bytes(int C) { return C > 0 ? sfod_align_up(2 * sfod_align_up((size_t)C, 4) * sizeof(float), 256) : 256; }

SFOD_API int sfod_bn_frozen_apply(const float *x, const float *residual, float *y, int layout, int N, int C, int H, int W,
                                  const float *weight, const float *bias, const float *running_mean, const float *running_var,
                                  double eps, int fuse_relu, void *scratch, sfod_stream_t stream) {
  if (!x || !y || !running_mean || !running_var || !scratch || N <= 0 || C <= 0 || H <= 0 || W <= 0) return SFOD_ERR_INVALID_ARG;
  if (layout != SFOD_NCHW && layout != SFOD_NHWC) return SFOD_ERR_INVALID_ARG;
  if (residual && ((reinterpret_cast<uintptr_t>(residual) ^ reinterpret_cast<uintptr_t>(x)) & 15u)) return SFOD_ERR_ALIGNMENT;
  cudaStream_t st = sfod_cu(stream);
  float *scale = static_cast<float *>(scratch);
  float *shift = scale + sfod_align_up((size_t)C, 4);
  bn_frozen_coeffs_kernel<<<(C + 127) / 128, 128, 0, st>>>(C, weight, bias, running_mean, running_var, (float)eps, scale, shift);
  SFOD_LAUNCH_CHECK();
  return launch_bn_apply(x, nullptr, residual, y, layout, N, C, H, W, scale, shift, fuse_relu, 0, st);
}

// Single-launch train-mode BatchNorm (statistics + running-stat update + normalise [+ residual] [+ ReLU]) for NCHW activations;
// see bn_fused_nchw_kernel.  Returns SFOD_ERR_UNSUPPORTED when the cooperative grid cannot be formed (the caller then uses the
// two-phase entry points, which is also the path for multi-GPU statistics and for the max-pool fusion).
SFOD_API int sfod_bn_train_fused(const float *x, const float *pre_bias, const float *residual, float *y, int N, int C, int H, int W,
                                 double *stats_dev, const float *weight, const float *bias, float *running_mean, float *running_var,
                                 int64_t *num_batches_tracked, double momentum, double eps, int fuse_relu, sfod_stream_t stream) {
  if (!x || !y || !stats_dev || N <= 0 || C <= 0 || H <= 0 || W <= 0) return SFOD_ERR_INVALID_ARG;
  if (residual && ((reinterpret_cast<uintptr_t>(residual) ^ reinterpret_cast<uintptr_t>(x)) & 15u)) return SFOD_ERR_ALIGNMENT;
  if (((reinterpret_cast<uintptr_t>(y) ^ reinterpret_cast<uintptr_t>(x)) & 15u)) return SFOD_ERR_ALIGNMENT;
  cudaStream_t st = sfod_cu(stream);
  const long long HW = (long long)H * W;
  const long long nchunks = (long long)N * C * ((HW + kFChunk - 1) / kFChunk);
  if ((long long)N * C > 0x7FFFFFFFll) return SFOD_ERR_UNSUPPORTED;
  int dev = 0, sms = 0, per_sm = 0, coop = 0;
  SFOD_CUDA_TRY(cudaGetDevice(&dev));
  SFOD_CUDA_TRY(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
  if (!coop) return SFOD_ERR_UNSUPPORTED;
  SFOD_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const void *kern = residual ? (fuse_relu ? (const void *)bn_fused_nchw_kernel<true, true> : (const void *)bn_fused_nchw_kernel<false, true>)
                              : (fuse_relu ? (const void *)bn_fused_nchw_kernel<true, false> : (const void *)bn_fused_nchw_kernel<false, false>);
  SFOD_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kThreads, 0));
  if (per_sm < 1) return SFOD_ERR_UNSUPPORTED;
  long long grid = (long long)sms * per_sm;
  const long long want = (nchunks + kThreads / 32 - 1) / (kThreads / 32);   // one chunk per warp at least
  if (grid > want) grid = want;
  SFOD_CUDA_TRY(cudaMemsetAsync(stats_dev, 0, (size_t)C * 2 * sizeof(double), st));
  int NC = N * C;
  double count = (double)N * (double)HW;
  long long hw = HW;
  long long *nbt = reinterpret_cast<long long *>(num_batches_tracked);
  void *args[] = {(void *)&x, (void *)&pre_bias, (void *)&residual, (void *)&y, (void *)&NC, (void *)&C, (void *)&hw, (void *)&stats_dev,
                  (void *)&count, (void *)&weight, (void *)&bias, (void *)&running_mean, (void *)&running_var, (void *)&nbt,
                  (void *)&momentum, (void *)&eps};
  SFOD_CUDA_TRY(cudaLaunchCooperativeKernel(kern, dim3((unsigned)grid), dim3(kThreads), args, 0, st));
  sfod_count_launch();
  return SFOD_OK;
}

// --------------------------------------------------------------------------------------------------------------------
// Multi-GPU statistics: one-shot all-reduce of the (sum x, sum x^2, count) payload over NVLink peer memory, fused into the
// finalize kernel (SURVEY.md 8e collective (2); reference daod/engine/trainers/base.py:270-337 run on several ranks).
//
// Every rank owns an INBOX (cudaMalloc'ed, exported with cudaIpcGetMemHandle and mapped by every peer):
//   [0]    uint64 counter  -- exchanges this rank has completed (the epoch of the next one is counter + 1; kept on the device so
//                             that a captured CUDA graph replays correctly)
//   [8]    uint32 timeouts -- exchanges abandoned because a peer's payload did not arrive (diagnostic; results are then invalid)
//   [256]  uint4 slot[2][8][kP2PMaxPayload]   slot[parity][src][i] = (lo32, tag, hi32, tag) of rank src's i-th payload double
// One exchange, executed by ONE CTA on every rank after its statistics pass: (1) store the local 2C+1 doubles into slot
// [epoch & 1][rank] of every PEER's inbox as 16-byte (value, tag) elements (NVLink P2P stores, coalesced; no fence, no flag:
// every 8-byte half carries the tag of this exchange); (2) every thread polls its element of each peer's slot in the own inbox
// until both tags match, and adds the contributions in rank order -- the same order on every rank, so all ranks obtain
// bit-identical totals; (3) the per-channel coefficients and running statistics are computed from the totals in the same kernel.
// 16 KB per rank and 512-channel layer cross NVLink once, with one one-way latency on the critical path; there is no separate
// collective launch and no host involvement.  Step (1) can also be taken by the statistics kernel itself (its last CTA, see
// bn_stats_nchw_kernel<true>), which hides the transfer behind the launch gap between the two phases.  Slot reuse is safe
// without a handshake: a rank that writes epoch e + 2 has completed exchange e + 1, for which every peer had delivered its
// epoch-(e+1) payload, which a peer does only after its own exchange e -- the last reader of the slot -- has finished
// (stream order); and a reader accepts an element only with the tag of its own epoch.
namespace {
__global__ void __launch_bounds__(kP2PThreads) bn_exchange_finalize_kernel(double *__restrict__ stats, int C, sfod_p2p_comm_t comm,
                                                                            const float *__restrict__ weight, const float *__restrict__ bias,
                                                                            float *__restrict__ running_mean, float *__restrict__ running_var,
                                                                            long long *__restrict__ nbt, double momentum, double eps,
                                                                            float *__restrict__ scale, float *__restrict__ shift) {
  __shared__ double tot[kP2PMaxPayload];
  __shared__ int s_timeout;
  char *mine = static_cast<char *>(comm.inbox[comm.rank]);
  unsigned long long *counter = reinterpret_cast<unsigned long long *>(mine);
  const unsigned long long epoch = *counter + 1ull;
  const int par = (int)(epoch & 1ull);
  const unsigned tag = p2p_tag(epoch);
  const int n = 2 * C + 1;
  if (threadIdx.x == 0) s_timeout = 0;
  // the statistics kernel's last CTA may already have delivered the payload (ticket word == kP2PPushed)
  const bool pushed = *reinterpret_cast<const unsigned long long *>(stats + 2 * C + 1) == kP2PPushed;   // CTA-uniform
  if (!pushed) p2p_push(stats, n, comm, epoch);
  __syncthreads();
  const long long t0 = clock64();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    double t = 0.0;
    for (int r = 0; r < comm.world; ++r) {   // rank order: the same sum on every rank
      double v;
      if (r == comm.rank) v = __ldcg(stats + i);   // own contribution straight from phase 1
      else {
        const uint4 *e = p2p_slot(mine, par, r) + i;
        while (!p2p_load(e, tag, v)) {
          if (clock64() - t0 > kP2PSpinLimit) { s_timeout = 1; v = 0.0; break; }
          __nanosleep(20);
        }
      }
      t += v;
    }
    tot[i] = t;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) stats[i] = tot[i];   // the totals of the concatenated batch, as the NCCL path leaves them
  const double cnt = tot[2 * C];
  for (int c = threadIdx.x; c < C; c += blockDim.x)
    bn_finalize_channel(c, tot[2 * c], tot[2 * c + 1], cnt, weight, bias, running_mean, running_var, momentum, eps, scale, shift);
  if (threadIdx.x == 0) {
    if (nbt) *nbt += 1;
    if (s_timeout) atomicAdd(reinterpret_cast<unsigned *>(mine + 8), 1u);
    *counter = epoch;
  }
}
}  // namespace

SFOD_API size_t sfod_p2p_inbox_bytes(void) {
  return kP2PHeaderBytes + 2 * (size_t)SFOD_P2P_MAX_RANKS * kP2PMaxPayload * sizeof(uint4);
}
SFOD_API int sfod_p2p_max_channels(void) { return (kP2PMaxPayload - 1) / 2; }

// With CUDA's lazy module loading the FIRST launch of a kernel may synchronise the context.  Ranks that share one process
// (and one GPU: tests) would deadlock if that happened while a peer's finalize kernel is already polling for this rank's
// payload, so every kernel a BatchNorm layer can launch is loaded up front.
static int p2p_preload_kernels() {
  const void *kernels[] = {
      (const void *)bn_stats_nchw_kernel<true>, (const void *)bn_stats_nchw_kernel<false>, (const void *)bn_stats_nhwc_kernel,
      (const void *)bn_fold_replicas_kernel, (const void *)bn_stats_nhwc_scalar_kernel, (const void *)bn_exchange_finalize_kernel,
      (const void *)bn_finalize_kernel,
      (const void *)bn_apply_nchw_kernel<true, true>, (const void *)bn_apply_nchw_kernel<true, false>,
      (const void *)bn_apply_nchw_kernel<false, true>, (const void *)bn_apply_nchw_kernel<false, false>,
      (const void *)bn_apply_pool_nchw_kernel<true, true>, (const void *)bn_apply_pool_nchw_kernel<true, false>,
      (const void *)bn_apply_pool_nchw_kernel<false, true>, (const void *)bn_apply_pool_nchw_kernel<false, false>,
      (const void *)bn_apply_nhwc_kernel<true, true>, (const void *)bn_apply_nhwc_kernel<true, false>,
      (const void *)bn_apply_nhwc_kernel<false, true>, (const void *)bn_apply_nhwc_kernel<false, false>,
      (const void *)bn_apply_pool_nhwc_kernel<true>, (const void *)bn_apply_pool_nhwc_kernel<false>,
      (const void *)bn_apply_nhwc_scalar_kernel<true>, (const void *)bn_apply_nhwc_scalar_kernel<false>};
  for (const void *k : kernels) {
    cudaFuncAttributes attr;
    SFOD_CUDA_TRY(cudaFuncGetAttributes(&attr, k));
  }
  return SFOD_OK;
}

SFOD_API int sfod_p2p_alloc(void **inbox, unsigned char *handle) {
  if (!inbox) return SFOD_ERR_INVALID_ARG;
  if (int rc = p2p_preload_kernels()) return rc;
  void *p = nullptr;
  SFOD_CUDA_TRY(cudaMalloc(&p, sfod_p2p_inbox_bytes()));
  cudaError_t e = cudaMemset(p, 0, sfod_p2p_inbox_bytes());
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess && handle) {
    static_assert(sizeof(cudaIpcMemHandle_t) == SFOD_P2P_HANDLE_BYTES, "IPC handle size");
    cudaIpcMemHandle_t h;
    e = cudaIpcGetMemHandle(&h, p);
    if (e == cudaSuccess) memcpy(handle, &h, sizeof(h));
  }
  if (e != cudaSuccess) { cudaFree(p); return SFOD_ERR_CUDA_BASE + (int)e; }
  *inbox = p;
  return SFOD_OK;
}
SFOD_API int sfod_p2p_open(const unsigned char *handle, void **peer_inbox) {
  if (!handle || !peer_inbox) return SFOD_ERR_INVALID_ARG;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  SFOD_CUDA_TRY(cudaIpcOpenMemHandle(peer_inbox, h, cudaIpcMemLazyEnablePeerAccess));
  return SFOD_OK;
}
SFOD_API int sfod_p2p_close(void *peer_inbox) {
  if (!peer_inbox) return SFOD_ERR_INVALID_ARG;
  SFOD_CUDA_TRY(cudaIpcCloseMemHandle(peer_inbox));
  return SFOD_OK;
}
SFOD_API int sfod_p2p_free(void *inbox) {
  if (!inbox) return SFOD_ERR_INVALID_ARG;
  SFOD_CUDA_TRY(cudaFree(inbox));
  return SFOD_OK;
}
SFOD_API int sfod_p2p_status(const sfod_p2p_comm_t *comm, uint64_t *exchanges, uint32_t *timeouts) {
  if (!comm || comm->world < 1 || comm->world > SFOD_P2P_MAX_RANKS || comm->rank < 0 || comm->rank >= comm->world) return SFOD_ERR_INVALID_ARG;
  unsigned long long head[2] = {0, 0};
  SFOD_CUDA_TRY(cudaMemcpy(head, comm->inbox[comm->rank], sizeof(head), cudaMemcpyDeviceToHost));   // synchronises with the stream's work
  if (exchanges) *exchanges = head[0];
  if (timeouts) *timeouts = (uint32_t)(head[1] & 0xFFFFFFFFull);
  return SFOD_OK;
}

// stats_dev layout: [0, 2C) (sum x, sum x^2); [2C] element count (written by phase 1; with [0, 2C) it forms the 2C+1
// all-reduce payload); [2C + 1] ticket word of the statistics kernel's payload delivery; [2C + 2, ...) float scale / shift
// scratch of phase 2; [4C, ...) replica totals of the NHWC pass.
SFOD_API int sfod_bn_finalize_apply(const float *x, const float *pre_bias, const float *residual, float *y, int layout, int N, int C,
                                    int H, int W, double *stats_dev, const sfod_p2p_comm_t *comm, const float *weight, const float *bias,
                                    float *running_mean, float *running_var, int64_t *num_batches_tracked, double momentum, double eps,
                                    int fuse_relu, int fuse_maxpool2, sfod_stream_t stream) {
  if (!stats_dev || N <= 0 || C <= 0 || H <= 0 || W <= 0) return SFOD_ERR_INVALID_ARG;
  if (comm && !p2p_comm_ok(comm)) return SFOD_ERR_INVALID_ARG;
  if (comm && 2 * C + 1 > kP2PMaxPayload) return SFOD_ERR_UNSUPPORTED;
  if (layout != SFOD_NCHW && layout != SFOD_NHWC) return SFOD_ERR_INVALID_ARG;
  if (residual && fuse_maxpool2) return SFOD_ERR_INVALID_ARG;
  if (residual && x && ((reinterpret_cast<uintptr_t>(residual) ^ reinterpret_cast<uintptr_t>(x)) & 15u)) return SFOD_ERR_ALIGNMENT;
  cudaStream_t st = sfod_cu(stream);
  float *scale = reinterpret_cast<float *>(stats_dev + 2 * (size_t)C + 2);
  float *shift = scale + sfod_align_up((size_t)C, 4);
  long long *nbt = reinterpret_cast<long long *>(num_batches_tracked);
  if (comm)   // one CTA: the exchange is a single block that polls for every peer's payload
    bn_exchange_finalize_kernel<<<1, kP2PThreads, 0, st>>>(stats_dev, C, *comm, weight, bias, running_mean, running_var, nbt, momentum,
                                                           eps, scale, shift);
  else
    bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(stats_dev, C, weight, bias, running_mean, running_var, nbt, momentum, eps, scale,
                                                        shift);
  SFOD_LAUNCH_CHECK();
  if (!x || !y) return SFOD_OK;  // statistics-only mode (AdaBN does not need the normalised output of the last layer)
  return launch_bn_apply(x, pre_bias, residual, y, layout, N, C, H, W, scale, shift, fuse_relu, fuse_maxpool2, st);
}
