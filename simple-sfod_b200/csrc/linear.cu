// linear.cu -- fp32 fully connected layer y = act(x W^T + b) on the tcgen05 tensor cores with 3xTF32 arithmetic.
//
// Each operand v is split into hi = v truncated to TF32 and lo = tf32_rna(v - hi) (v - hi is exact in fp32), and the product is
// accumulated as lo*hi + hi*lo + hi*hi: three kind::tf32 MMAs whose operands carry at most 11 significant bits, so the result
// does not depend on how the MMA unit treats the low bits of an fp32 container.  |lo| < 2^-10 |v|; the dropped lo*lo term is
// < 2^-20 and the rounding of lo < 2^-21 relative per product (2^-22 on average).
//
// The tensor cores' fp32 accumulation does not round to nearest, so a single accumulator over K = 25088 would drift.  The
// MMAs therefore accumulate CHUNK k-blocks at a time into one of two TMEM buffers, and the epilogue warps add each finished
// chunk into fp32 registers (round to nearest) while the MMAs fill the other buffer.
//
// Per CTA one 128x128 output tile.  Warp 0: TMA producer (mbarrier ring of STAGES stages of hi/lo tiles of x and W, 128-byte
// swizzle).  Warp 1: TMEM allocator and single-thread MMA issuer.  Warps 2-5: chunk drains, then bias, activation and store.
#include "common.cuh"

#include <cuda.h>
#include <cudaTypedefs.h>

namespace {

constexpr int BM = 128, BN = 128;
constexpr int BK = 32;                        // fp32 elements per k-block: 128 bytes, one SWIZZLE_128B row
constexpr int UMMA_K = 8;                     // K of one kind::tf32 MMA
constexpr int STAGES = 3;
constexpr int TILE_BYTES = BM * BK * 4;       // 16 KB (BM == BN: the A and B tiles have the same size)
constexpr int STAGE_BYTES = 4 * TILE_BYTES;   // x_hi, x_lo, W_hi, W_lo
constexpr int CHUNK = 8;                      // k-blocks per TMEM accumulation chunk
constexpr int TMEM_COLS = 2 * BN;             // two fp32 accumulator buffers of BN columns
constexpr int THREADS = 192;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 128;   // + alignment slack + barriers and the TMEM address
static_assert(BM == BN, "A and B tiles share TILE_BYTES");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t *b, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t *b, uint32_t parity) {
  const uint32_t a = smem_u32(b);
  uint32_t done = 0;
  while (!done) {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                 : "=r"(done) : "r"(a), "r"(parity) : "memory");
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t *b) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void tma_load(const CUtensorMap *map, void *dst, int c0, int c1, uint64_t *bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
               ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// Shared-memory matrix descriptor: K-major, 128-byte swizzle, 8-row core-matrix groups 1024 bytes apart (SBO), version 1.
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
  return static_cast<uint64_t>((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (static_cast<uint64_t>(1024 >> 4) << 32) |
         (1ull << 46) | (2ull << 61);
}

// Instruction descriptor of kind::tf32: fp32 accumulator, tf32 A and B, both K-major, M = BM, N = BN.
constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(BN >> 3) << 17) |
                            (static_cast<uint32_t>(BM >> 4) << 24);

__device__ __forceinline__ void mma_tf32(uint32_t d, uint64_t a, uint64_t b, uint32_t accumulate) {
  asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
               "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}"
               ::"r"(d), "l"(a), "l"(b), "r"(kIdesc), "r"(accumulate));
}
// Arrives on `bar` once every MMA this thread issued so far has completed.
__device__ __forceinline__ void mma_commit(uint64_t *bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 consecutive fp32 columns of this thread's TMEM lane.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
               "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                 "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                 "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ float tf32_rna(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}

// hi = v truncated to TF32 (low 13 mantissa bits cleared), lo = tf32_rna(v - hi): both carry v's sign.
// Inf must come out of the three products as it comes out of v*w.  With a partner of the same sign in all three terms,
// Inf*lo + Inf*hi cannot become Inf - Inf (round-to-nearest hi would give lo the opposite sign half of the time), and a nonzero v
// whose lo would be 0 (v has <= 11 significant bits, or is infinite) gets lo = +-2^-126, the smallest normal, so that Inf * lo is
// not Inf * 0 = NaN.  That lo adds |partner| * 2^-126, far below the fp32 resolution of the product for any |v|, |w| > 2^-50.
// NaN becomes the NaN with every mantissa bit set: truncating a NaN whose payload sits in the low bits would make it Inf.
__device__ __forceinline__ void split_tf32(float v, float &hi, float &lo) {
  if (isnan(v)) { hi = __uint_as_float(0x7FFFFFFFu); lo = 0.f; return; }
  hi = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
  lo = isinf(v) ? 0.f : tf32_rna(__fsub_rn(v, hi));
  if (lo == 0.f && v != 0.f) lo = copysignf(1.17549435e-38f, v);
}

__global__ void __launch_bounds__(256) split_tf32_kernel(const float4 *__restrict__ in, float4 *__restrict__ hi,
                                                         float4 *__restrict__ lo, int64_t n4) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    const float4 v = in[i];
    float4 h, l;
    split_tf32(v.x, h.x, l.x);
    split_tf32(v.y, h.y, l.y);
    split_tf32(v.z, h.z, l.z);
    split_tf32(v.w, h.w, l.w);
    hi[i] = h;
    lo[i] = l;
  }
}

__global__ void __launch_bounds__(THREADS, 1)
linear_3xtf32_kernel(const __grid_constant__ CUtensorMap x_hi, const __grid_constant__ CUtensorMap x_lo,
                     const __grid_constant__ CUtensorMap w_hi, const __grid_constant__ CUtensorMap w_lo,
                     const float *__restrict__ bias, float *__restrict__ y, int M, int N, int K, int relu) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~static_cast<uintptr_t>(1023));
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + STAGES * STAGE_BYTES);   // stage landed (TMA transaction bytes)
  uint64_t *empty = full + STAGES;                                              // stage consumed (MMA commit)
  uint64_t *acc_full = empty + STAGES;                                          // TMEM chunk finished (MMA commit)
  uint64_t *acc_empty = acc_full + 2;                                           // TMEM chunk drained (128 epilogue threads)
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_empty + 2);

  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int n0 = blockIdx.x * BN, m0 = blockIdx.y * BM;
  const int nk = (K + BK - 1) / BK;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "n"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int kb = 0; kb < nk; ++kb) {
        const int s = kb % STAGES;
        mbar_wait(&empty[s], ((kb / STAGES) & 1) ^ 1);
        uint8_t *st = smem + s * STAGE_BYTES;
        mbar_expect_tx(&full[s], STAGE_BYTES);
        const int k0 = kb * BK;
        tma_load(&x_hi, st, k0, m0, &full[s]);
        tma_load(&x_lo, st + TILE_BYTES, k0, m0, &full[s]);
        tma_load(&w_hi, st + 2 * TILE_BYTES, k0, n0, &full[s]);
        tma_load(&w_lo, st + 3 * TILE_BYTES, k0, n0, &full[s]);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      for (int kb = 0; kb < nk; ++kb) {
        const int c = kb / CHUNK, buf = c & 1;
        const bool chunk_start = kb % CHUNK == 0;
        const uint32_t d = tmem + buf * BN;
        if (chunk_start) {
          mbar_wait(&acc_empty[buf], ((c >> 1) & 1) ^ 1);
          tc_fence_after();
        }
        const int s = kb % STAGES;
        mbar_wait(&full[s], (kb / STAGES) & 1);
        tc_fence_after();
        const uint32_t a_hi = smem_u32(smem + s * STAGE_BYTES), a_lo = a_hi + TILE_BYTES;
        const uint32_t b_hi = a_hi + 2 * TILE_BYTES, b_lo = a_hi + 3 * TILE_BYTES;
#pragma unroll
        for (int j = 0; j < BK / UMMA_K; ++j) {
          const uint32_t off = j * UMMA_K * 4;   // bytes along K inside the 128-byte swizzle row
          mma_tf32(d, smem_desc(a_lo + off), smem_desc(b_hi + off), !(chunk_start && j == 0));
          mma_tf32(d, smem_desc(a_hi + off), smem_desc(b_lo + off), 1);
          mma_tf32(d, smem_desc(a_hi + off), smem_desc(b_hi + off), 1);
        }
        mma_commit(&empty[s]);
        if (kb % CHUNK == CHUNK - 1 || kb == nk - 1) mma_commit(&acc_full[buf]);
      }
    }
  } else {
    const int q = warp & 3;   // a warp reads the TMEM lanes 32 * (warp % 4) ..
    float acc[BN];
#pragma unroll
    for (int i = 0; i < BN; ++i) acc[i] = 0.f;
    const int nchunks = (nk + CHUNK - 1) / CHUNK;
    for (int c = 0; c < nchunks; ++c) {
      const int buf = c & 1;
      mbar_wait(&acc_full[buf], (c >> 1) & 1);
      tc_fence_after();
      const uint32_t taddr = tmem + (static_cast<uint32_t>(q * 32) << 16) + buf * BN;
#pragma unroll
      for (int h = 0; h < BN / 32; ++h) {
        uint32_t r[32];
        tmem_ld32(taddr + h * 32, r);
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[h * 32 + i] = __fadd_rn(acc[h * 32 + i], __uint_as_float(r[i]));
      }
      tc_fence_before();
      mbar_arrive(&acc_empty[buf]);
    }
    const int row = m0 + q * 32 + lane;
    if (row < M) {
      float *out = y + static_cast<int64_t>(row) * N + n0;
#pragma unroll
      for (int c4 = 0; c4 < BN; c4 += 4) {
        if (n0 + c4 < N) {   // N % 16 == 0: a group of four columns is either inside or outside
          float v[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            v[i] = bias != nullptr ? __fadd_rn(acc[c4 + i], __ldg(bias + n0 + c4 + i)) : acc[c4 + i];
            if (relu && v[i] < 0.f) v[i] = 0.f;   // NaN stays NaN, as torch.relu
          }
          *reinterpret_cast<float4 *>(out + c4) = make_float4(v[0], v[1], v[2], v[3]);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS));
  }
}

struct SplitPlanes { float *w_hi, *w_lo, *x_hi, *x_lo; };

template <typename Ws> SplitPlanes carve(Ws &ws, int64_t M, int64_t N, int64_t K) {
  SplitPlanes p;
  p.w_hi = ws.template take<float>(N * K);
  p.w_lo = ws.template take<float>(N * K);
  p.x_hi = ws.template take<float>(M * K);
  p.x_lo = ws.template take<float>(M * K);
  return p;
}

// K-major (rows, K) fp32 plane, boxes of BK x 128 with the 128-byte swizzle the MMA descriptors expect.
int encode_plane(PFN_cuTensorMapEncodeTiled_v12000 encode, CUtensorMap *map, const float *base, int64_t rows, int64_t K) {
  const cuuint64_t dims[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(rows)};
  const cuuint64_t strides[1] = {static_cast<cuuint64_t>(K) * 4};
  const cuuint32_t box[2] = {BK, 128};
  const cuuint32_t elem[2] = {1, 1};
  CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(base), dims, strides, box, elem,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);   // rows and columns outside the plane read as zero
  return r == CUDA_SUCCESS ? SFOD_OK : SFOD_ERR_UNSUPPORTED;
}

int launch_split(const float *in, float *hi, float *lo, int64_t n, cudaStream_t st) {
  const int64_t n4 = n / 4;
  const int blocks = static_cast<int>(n4 / 256 + 1 < SFOD_NUM_SMS * 16 ? n4 / 256 + 1 : SFOD_NUM_SMS * 16);
  split_tf32_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4 *>(in), reinterpret_cast<float4 *>(hi),
                                            reinterpret_cast<float4 *>(lo), n4);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

}  // namespace

SFOD_API size_t sfod_linear_3xtf32_workspace_bytes(int64_t M, int N, int K) {
  if (M < 0 || N < 0 || K < 0) return 0;
  SfodWsSize ws;
  carve(ws, M, N, K);
  return ws.off;
}

SFOD_API int sfod_linear_3xtf32(const float *x, int64_t M, int K, const float *w, int N, const float *bias, int act, float *y,
                                void *workspace, size_t workspace_bytes, sfod_stream_t stream) {
  if (x == nullptr || w == nullptr || y == nullptr || M < 0 || K <= 0 || N <= 0 || (act != 0 && act != 1))
    return SFOD_ERR_INVALID_ARG;
  if (K % 4 != 0 || N % 16 != 0 || (M + BM - 1) / BM > 65535) return SFOD_ERR_UNSUPPORTED;
  if (!sfod_aligned16(x) || !sfod_aligned16(w) || !sfod_aligned16(y) || !sfod_aligned16(workspace)) return SFOD_ERR_ALIGNMENT;
  if (M == 0) return SFOD_OK;
  SfodWs ws(workspace, workspace_bytes);
  const SplitPlanes p = carve(ws, M, N, K);
  if (!ws.ok) return SFOD_ERR_WORKSPACE_TOO_SMALL;

  void *fn = nullptr;
  cudaDriverEntryPointQueryResult q;
  SFOD_CUDA_TRY(cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &fn, 12000, cudaEnableDefault, &q));
  if (fn == nullptr || q != cudaDriverEntryPointSuccess) return SFOD_ERR_UNSUPPORTED;
  const auto encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  CUtensorMap maps[4];
  int rc;
  if ((rc = encode_plane(encode, &maps[0], p.x_hi, M, K)) != SFOD_OK) return rc;
  if ((rc = encode_plane(encode, &maps[1], p.x_lo, M, K)) != SFOD_OK) return rc;
  if ((rc = encode_plane(encode, &maps[2], p.w_hi, N, K)) != SFOD_OK) return rc;
  if ((rc = encode_plane(encode, &maps[3], p.w_lo, N, K)) != SFOD_OK) return rc;
  SFOD_CUDA_TRY(cudaFuncSetAttribute(linear_3xtf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));

  const cudaStream_t st = sfod_cu(stream);
  // W is split on every call: its values can change in place (the teacher's EMA writes through raw pointers).
  if ((rc = launch_split(w, p.w_hi, p.w_lo, static_cast<int64_t>(N) * K, st)) != SFOD_OK) return rc;
  if ((rc = launch_split(x, p.x_hi, p.x_lo, M * K, st)) != SFOD_OK) return rc;
  // blockIdx.x walks N fastest: the CTAs resident at one time share few row blocks of x and stream the same K slices of W.
  const dim3 grid((N + BN - 1) / BN, static_cast<unsigned>((M + BM - 1) / BM));
  linear_3xtf32_kernel<<<grid, THREADS, SMEM_BYTES, st>>>(maps[0], maps[1], maps[2], maps[3], bias, y, static_cast<int>(M), N, K,
                                                          act);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}
