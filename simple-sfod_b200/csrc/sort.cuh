// sort.cuh -- segmented ascending sort of 64-bit keys (hand-written bitonic network).
//
// Used for: per-image top-k / full descending sort of RPN objectness logits (d2
// find_top_rpn_proposals step 1, reached from reference rpn.py:54-56), the stable score order
// torchvision's nms starts from, and the (class, score) order of Fast R-CNN candidates
// (reference roi_heads/fast_rcnn.py:122-133).  Ties are made impossible by packing the element
// index into the low key bits, which yields exactly the "value descending, index ascending"
// order of a stable sort.
//
// Layout: S segments of P keys each (P a power of two >= 512), contiguous: keys[s*P + i].
// A thread owns kE = 8 consecutive keys in registers; compare-exchange distance j is served
//   j < 8         : in registers (static indices),
//   8 <= j < 256  : warp shuffles (partner lane = lane ^ (j/8)),
//   j >= 256      : one swizzled shared-memory exchange per stage (conflict-free 64-bit banks),
//   j >= keys/CTA : distributed-shared-memory exchange between the CTAs of a thread-block cluster (a 16 384-key tile is
//                   spread over 8 CTAs = 8 SMs x 4 warps instead of 32 warps queueing on one SM),
//   j >= tile     : global-memory exchange kernel (only when P > 16384, e.g. 34 200 R101 anchors).
// The kernels have internal linkage: every translation unit that sorts (detect.cu, evaluate.cu) holds its own copy.
#pragma once
#include "common.cuh"

namespace bsort {

constexpr int kE = 8;              // keys per thread (8: half the serial work per thread of 16, one more shuffle stage)
constexpr int kMaxTile = 16384;    // keys per cluster tile (8 CTAs x 256 threads x 8 keys)
constexpr int kClusterMinKeys = 2048; // a tile is spread over tile / 2048 (<= 8) CTAs of a cluster
constexpr unsigned long long kSentinel = 0xFFFFFFFFFFFFFFFFull;

__device__ __forceinline__ void cex(unsigned long long &a, unsigned long long &b, bool asc) {
  const bool sw = (a > b) == asc;
  const unsigned long long lo = sw ? b : a, hi = sw ? a : b;
  a = lo; b = hi;
}

// In-register stages j = JMAX, JMAX/2, ..., 1 for merge size k.  `asc_thread` is the direction when
// k >= 16 (uniform over the thread's 16 keys); for k < 16 the direction depends on the register index.
template <int K>
__device__ __forceinline__ void reg_stages_small_k(unsigned long long (&a)[kE]) {
  // k < 16: direction = ((r & K) == 0)
#pragma unroll
  for (int j = K / 2; j >= 1; j >>= 1) {
#pragma unroll
    for (int r = 0; r < kE; ++r)
      if ((r & j) == 0) cex(a[r], a[r | j], (r & K) == 0);
  }
}
__device__ __forceinline__ void reg_stages(unsigned long long (&a)[kE], int jstart, bool asc) {
  // jstart in {kE/2, ..., 1}: run j = jstart..1
#pragma unroll
  for (int j = kE / 2; j >= 1; j >>= 1) {
    if (j <= jstart) {
#pragma unroll
      for (int r = 0; r < kE; ++r)
        if ((r & j) == 0) cex(a[r], a[r | j], asc);
    }
  }
}

__device__ __forceinline__ unsigned long long shfl_xor_u64(unsigned long long v, int lane_mask) {
  unsigned lo = (unsigned)v, hi = (unsigned)(v >> 32);
  lo = __shfl_xor_sync(0xFFFFFFFFu, lo, lane_mask);
  hi = __shfl_xor_sync(0xFFFFFFFFu, hi, lane_mask);
  return ((unsigned long long)hi << 32) | lo;
}

__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ const unsigned long long *cluster_peer(const unsigned long long *p, unsigned rank) {
  unsigned long long out;
  asm volatile("mapa.u64 %0, %1, %2;" : "=l"(out) : "l"(reinterpret_cast<unsigned long long>(p)), "r"(rank));
  return reinterpret_cast<const unsigned long long *>(out);
}

// Runs the bitonic stages for merge sizes k = k_lo .. k_hi (powers of two, k_lo >= 2) restricted to
// compare distances j < tile, on a tile of `tile` keys owned by a cluster of `cl` CTAs (ctile = tile / cl = 16 * blockDim.x
// keys per CTA, this CTA being number `rank`).  `gbase` is the global index (within the segment) of THIS CTA's first key:
// it defines directions.  smem: ctile keys.
__device__ __forceinline__ void block_bitonic(unsigned long long (&a)[kE], unsigned long long *smem, int tile, int ctile,
                                              int rank, long long gbase, int k_lo, int k_hi) {
  const int t = threadIdx.x;
  const long long g0 = gbase + (long long)t * kE;  // global index of a[0]
  for (long long k = k_lo; k <= k_hi; k <<= 1) {
    if (k < kE) {
      if (k == 2) reg_stages_small_k<2>(a);
      else if (k == 4) reg_stages_small_k<4>(a);
      else reg_stages_small_k<(kE > 8 ? 8 : 4)>(a);   // only reached when kE == 16
      continue;
    }
    const bool asc = (g0 & k) == 0;
    long long j = k >> 1;
    if (j >= tile) j = tile >> 1;
    // cluster stages: the partner key lives at the same position of CTA rank ^ (j / ctile)
    for (; j >= ctile; j >>= 1) {
      const int rj = (int)(j / ctile);
      const int sw = t & (kE - 1);
      __syncthreads();      // own threads are done with the shared-memory stage before
#pragma unroll
      for (int r = 0; r < kE; ++r) smem[t * kE + (r ^ sw)] = a[r];
      cluster_sync_all();   // all tiles of the cluster are published
      const unsigned long long *peer = cluster_peer(smem, (unsigned)(rank ^ rj));
      const bool take_min = (((rank & rj) == 0) == asc);
#pragma unroll
      for (int r = 0; r < kE; ++r) {
        const unsigned long long o = peer[t * kE + (r ^ sw)];
        a[r] = take_min ? (a[r] < o ? a[r] : o) : (a[r] > o ? a[r] : o);
      }
      cluster_sync_all();   // every peer has read this CTA's tile before anything overwrites it
    }
    // shared-memory stages
    for (; j >= 32 * kE; j >>= 1) {
      const int tj = (int)(j / kE);
      const int sw = t & (kE - 1);
      __syncthreads();
#pragma unroll
      for (int r = 0; r < kE; ++r) smem[t * kE + (r ^ sw)] = a[r];
      __syncthreads();
      const int p = t ^ tj;
      const bool lower = (t & tj) == 0;
#pragma unroll
      for (int r = 0; r < kE; ++r) {
        const unsigned long long o = smem[p * kE + (r ^ sw)];
        const bool take_min = (lower == asc);
        a[r] = take_min ? (a[r] < o ? a[r] : o) : (a[r] > o ? a[r] : o);
      }
    }
    // warp-shuffle stages
    for (; j >= kE; j >>= 1) {
      const int lj = (int)(j / kE);
      const bool lower = (t & lj) == 0;
      const bool take_min = (lower == asc);
#pragma unroll
      for (int r = 0; r < kE; ++r) {
        const unsigned long long o = shfl_xor_u64(a[r], lj);
        a[r] = take_min ? (a[r] < o ? a[r] : o) : (a[r] > o ? a[r] : o);
      }
    }
    // in-register stages j = kE/2..1
    reg_stages(a, kE / 2, asc);
  }
}

// Tile kernel: grid (cl * P / tile, S) launched as clusters of cl CTAs along x; block tile/cl/16 threads; dynamic smem
// tile/cl*8 bytes.
static __global__ void __launch_bounds__(kClusterMinKeys / kE) bitonic_tile_kernel(unsigned long long *keys, int P, int tile, int cl, int k_lo, int k_hi) {
  extern __shared__ unsigned long long sort_smem[];
  const int ctile = tile / cl, rank = (int)(blockIdx.x % (unsigned)cl);
  unsigned long long *seg = keys + (size_t)blockIdx.y * P + (size_t)blockIdx.x * ctile;
  unsigned long long a[kE];
  const int t = threadIdx.x;
  // 128-bit loads of the thread's 16 consecutive keys
  const ulonglong2 *src = reinterpret_cast<const ulonglong2 *>(seg + t * kE);
#pragma unroll
  for (int r = 0; r < kE / 2; ++r) { ulonglong2 v = src[r]; a[2 * r] = v.x; a[2 * r + 1] = v.y; }
  block_bitonic(a, sort_smem, tile, ctile, rank, (long long)blockIdx.x * ctile, k_lo, k_hi);
  ulonglong2 *dst = reinterpret_cast<ulonglong2 *>(seg + t * kE);
#pragma unroll
  for (int r = 0; r < kE / 2; ++r) dst[r] = make_ulonglong2(a[2 * r], a[2 * r + 1]);
}

// Global exchange for one stage (k, j) with j >= tile: grid (P/2/256, S), block 256.
static __global__ void __launch_bounds__(256) bitonic_global_kernel(unsigned long long *keys, int P, long long k, long long j) {
  unsigned long long *seg = keys + (size_t)blockIdx.y * P;
  const long long tt = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tt >= P / 2) return;
  const long long i = ((tt & ~(j - 1)) << 1) | (tt & (j - 1));
  const long long p = i | j;
  unsigned long long x = seg[i], y = seg[p];
  const bool asc = (i & k) == 0;
  if ((x > y) == asc) { seg[i] = y; seg[p] = x; }
}

static inline int next_pow2(long long n, int min_p = 512) {
  long long p = min_p;
  while (p < n) p <<= 1;
  return (int)p;
}

// Host driver: sort S segments of P keys each, ascending.
static inline int segmented_sort(unsigned long long *keys, int S, int P, cudaStream_t stream) {
  if (S <= 0) return SFOD_OK;
  if (P < 512 || (P & (P - 1))) return SFOD_ERR_INVALID_ARG;
  const int tile = P < kMaxTile ? P : kMaxTile;
  int cl = tile / kClusterMinKeys;   // keys per CTA >= 2048 (4 warps); portable cluster sizes only
  if (cl > 8) cl = 8;
  if (cl < 1) cl = 1;
  const int ctile = tile / cl;
  const size_t smem = (size_t)ctile * sizeof(unsigned long long);
  if (smem > 48 * 1024)
    SFOD_CUDA_TRY(cudaFuncSetAttribute(bitonic_tile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxTile * 8));
  dim3 grid(cl * (P / tile), S);
  auto launch_tile = [&](int k_lo, int k_hi) -> int {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = dim3(ctile / kE, 1, 1); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cl; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    SFOD_CUDA_TRY(cudaLaunchKernelEx(&cfg, bitonic_tile_kernel, keys, P, tile, cl, k_lo, k_hi));
    sfod_count_launch();
    return SFOD_OK;
  };
  int rc = launch_tile(2, tile);
  if (rc) return rc;
  for (long long k = (long long)tile * 2; k <= P; k <<= 1) {
    for (long long j = k >> 1; j >= tile; j >>= 1) {
      dim3 g2((unsigned)((P / 2 + 255) / 256), S);
      bitonic_global_kernel<<<g2, 256, 0, stream>>>(keys, P, k, j);
      SFOD_LAUNCH_CHECK();
    }
    rc = launch_tile((int)k, (int)k);
    if (rc) return rc;
  }
  return SFOD_OK;
}

}  // namespace bsort
