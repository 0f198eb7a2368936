// detect.cu -- C-ABI entry points for proposal selection, NMS, Fast R-CNN post-processing and the
// pseudo-label filter.  Compiled with -fmad=false: every fp32 operation that feeds an integer decision
// (sort order, IoU > thr, score > thr) is separately rounded, in the reference's operation order.
#include "common.cuh"
#include "sort.cuh"
#include "nms.cuh"
#include "rpn.cuh"
#include "frcnn.cuh"
#include "match.cuh"
#include "sample.cuh"

// ===================================================================== generic torchvision-style NMS
namespace {

__global__ void __launch_bounds__(256) nms_make_keys_kernel(const float *__restrict__ scores, long long n, int P,
                                                            unsigned long long *__restrict__ keys) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P) return;
  keys[i] = i < n ? (((unsigned long long)(~sfod_score_key(scores[i])) << 32) | (unsigned)i) : bsort::kSentinel;
}

__global__ void __launch_bounds__(256) nms_max_coord_kernel(const float *__restrict__ boxes, long long n4,
                                                            unsigned *__restrict__ maxkey) {
  unsigned best = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    const unsigned k = sfod_score_key(boxes[i]);
    best = k > best ? k : best;
  }
  for (int o = 16; o > 0; o >>= 1) { const unsigned v = __shfl_xor_sync(0xFFFFFFFFu, best, o); best = v > best ? v : best; }
  if ((threadIdx.x & 31) == 0) atomicMax(maxkey, best);
}

__global__ void __launch_bounds__(256) nms_gather_kernel(const unsigned long long *__restrict__ keys, long long n,
                                                         const float4 *__restrict__ boxes, const long long *__restrict__ idxs,
                                                         int use_trick, const unsigned *__restrict__ maxkey,
                                                         float4 *__restrict__ sboxes, int *__restrict__ scls,
                                                         nmsk::Seg *__restrict__ seg) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j == 0) { seg->start = 0; seg->len = (int)n; }
  if (j >= n) return;
  const unsigned i = (unsigned)(keys[j] & 0xFFFFFFFFull);
  float4 b = boxes[i];
  if (idxs) {
    const long long c = idxs[i];
    if (use_trick) {
      const float off = __fmul_rn((float)c, __fadd_rn(sfod_key_score(*maxkey), 1.0f));
      b = make_float4(__fadd_rn(b.x, off), __fadd_rn(b.y, off), __fadd_rn(b.z, off), __fadd_rn(b.w, off));
    }
    scls[j] = (int)c;
  }
  sboxes[j] = b;
}

__global__ void __launch_bounds__(256) nms_emit_kernel(const unsigned long long *__restrict__ keys,
                                                       const int *__restrict__ keep_rank, const int *__restrict__ keep_count,
                                                       long long n, long long *__restrict__ keep_out,
                                                       long long *__restrict__ num_keep) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int cnt = *keep_count;
  if (q == 0) *num_keep = cnt;
  if (q >= n) return;
  keep_out[q] = q < cnt ? (long long)(keys[keep_rank[q]] & 0xFFFFFFFFull) : -1;
}

struct NmsBuf {
  unsigned long long *keys; float4 *sboxes; int *scls; nmsk::Seg *seg; unsigned long long *mask; int *keep_rank;
  int *keep_count; unsigned *maxkey; int P; int wstride;
};
template <typename WS> void nms_carve(WS &ws, long long n, NmsBuf &b) {
  b.P = bsort::next_pow2(n);
  b.wstride = (int)((n + 63) / 64);
  b.keys = ws.template take<unsigned long long>((size_t)b.P);
  b.sboxes = ws.template take<float4>((size_t)n);
  b.scls = ws.template take<int>((size_t)n);
  b.seg = ws.template take<nmsk::Seg>(1);
  b.mask = ws.template take<unsigned long long>((size_t)n * b.wstride);
  b.keep_rank = ws.template take<int>((size_t)n);
  b.keep_count = ws.template take<int>(1);
  b.maxkey = ws.template take<unsigned>(1);
}

}  // namespace

SFOD_API size_t sfod_nms_workspace_bytes(int64_t n) {
  if (n <= 0) return 256;
  SfodWsSize ws; NmsBuf b; nms_carve(ws, n, b);
  return ws.off;
}

SFOD_API int sfod_nms(const float *boxes, const float *scores, const int64_t *idxs, int64_t n, double iou_threshold,
                      int64_t coord_trick_max_n, int64_t *keep_out, int64_t *num_keep_dev, void *workspace,
                      size_t workspace_bytes, sfod_stream_t stream) {
  if (n < 0 || !num_keep_dev) return SFOD_ERR_INVALID_ARG;
  cudaStream_t st = sfod_cu(stream);
  if (n == 0) { SFOD_CUDA_TRY(cudaMemsetAsync(num_keep_dev, 0, sizeof(int64_t), st)); return SFOD_OK; }
  if (!boxes || !scores || !keep_out) return SFOD_ERR_INVALID_ARG;
  if (!sfod_aligned16(boxes)) return SFOD_ERR_ALIGNMENT;
  if (n > (1ll << 30)) return SFOD_ERR_UNSUPPORTED;
  SfodWs ws(workspace, workspace_bytes); NmsBuf b; nms_carve(ws, n, b);
  if (!ws.ok) return SFOD_ERR_WORKSPACE_TOO_SMALL;
  const int use_trick = (idxs != nullptr && n <= coord_trick_max_n) ? 1 : 0;
  nms_make_keys_kernel<<<(b.P + 255) / 256, 256, 0, st>>>(scores, n, b.P, b.keys);
  SFOD_LAUNCH_CHECK();
  int rc = bsort::segmented_sort(b.keys, 1, b.P, st);
  if (rc) return rc;
  if (use_trick) {
    SFOD_CUDA_TRY(cudaMemsetAsync(b.maxkey, 0, sizeof(unsigned), st));
    nms_max_coord_kernel<<<64, 256, 0, st>>>(boxes, n * 4, b.maxkey);
    SFOD_LAUNCH_CHECK();
  }
  nms_gather_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(b.keys, n, reinterpret_cast<const float4 *>(boxes),
                                                                 reinterpret_cast<const long long *>(idxs), use_trick,
                                                                 b.maxkey, b.sboxes, b.scls, b.seg);
  SFOD_LAUNCH_CHECK();
  const int *cls = (idxs && !use_trick) ? b.scls : nullptr;
  rc = nmsk::run_segmented(b.sboxes, cls, b.seg, 1, (int)n, (int)n, b.wstride, iou_threshold, (int)n, (int)n, b.mask,
                           b.keep_rank, b.keep_count, st);
  if (rc) return rc;
  nms_emit_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(b.keys, b.keep_rank, b.keep_count, n,
                                                               reinterpret_cast<long long *>(keep_out),
                                                               reinterpret_cast<long long *>(num_keep_dev));
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

// ===================================================================== RPN proposal selection
SFOD_API size_t sfod_rpn_select_workspace_bytes(const sfod_rpn_params *p) {
  if (!p || p->N <= 0 || p->HWA <= 0) return 256;
  SfodWsSize ws; rpnk::Plan pl; rpnk::carve(ws, p, pl, nullptr);
  return ws.off;
}

SFOD_API int sfod_rpn_select(const sfod_rpn_params *p, const float *logits, const float *deltas, const float *anchors,
                             const int32_t *image_hw_dev, float *out_boxes, float *out_logits, int64_t *out_src_index,
                             int32_t *out_count_dev, int32_t *invalid_count_dev, void *workspace, size_t workspace_bytes,
                             sfod_stream_t stream) {
  if (!p || !logits || !deltas || !image_hw_dev || !out_boxes || !out_logits || !out_src_index || !out_count_dev ||
      !invalid_count_dev)
    return SFOD_ERR_INVALID_ARG;
  if (p->N <= 0 || p->HWA <= 0 || p->pre_nms_topk <= 0 || p->post_nms_topk <= 0) return SFOD_ERR_INVALID_ARG;
  if (!anchors && (p->A <= 0 || p->A > 64 || p->Hf <= 0 || p->Wf <= 0 || p->Hf * p->Wf * p->A != p->HWA))
    return SFOD_ERR_INVALID_ARG;
  const bool native = p->head_layout == 1;
  if (p->head_layout != 0 && p->head_layout != 1) return SFOD_ERR_INVALID_ARG;
  if (native && (p->A <= 0 || p->Hf <= 0 || p->Wf <= 0 || (long long)p->Hf * p->Wf * p->A != p->HWA)) return SFOD_ERR_INVALID_ARG;
  if ((!native && !sfod_aligned16(deltas)) || !sfod_aligned16(out_boxes) || (anchors && !sfod_aligned16(anchors))) return SFOD_ERR_ALIGNMENT;
  cudaStream_t st = sfod_cu(stream);
  SfodWs ws(workspace, workspace_bytes); rpnk::Plan pl; rpnk::Buffers b;
  rpnk::carve(ws, p, pl, &b);
  if (!ws.ok) return SFOD_ERR_WORKSPACE_TOO_SMALL;
  const int N = p->N;
  {
    dim3 grid((pl.P + 255) / 256, N);
    if (native) rpnk::rpn_make_keys_kernel<true><<<grid, 256, 0, st>>>(logits, p->HWA, pl.P, p->A, p->Hf * p->Wf, b.keys);
    else rpnk::rpn_make_keys_kernel<false><<<grid, 256, 0, st>>>(logits, p->HWA, pl.P, 1, p->HWA, b.keys);
    SFOD_LAUNCH_CHECK();
  }
  int rc = bsort::segmented_sort(b.keys, N, pl.P, st);
  if (rc) return rc;
  rpnk::CellAnchors cell;
  for (int i = 0; i < 64 * 4; ++i) cell.v[i] = p->cell_anchors[i];
  auto decode = native ? rpnk::rpn_decode_compact_kernel<true> : rpnk::rpn_decode_compact_kernel<false>;
  decode<<<N, rpnk::kDecodeThreads, 0, st>>>(
      b.keys, pl.P, logits, deltas, reinterpret_cast<const float4 *>(anchors), cell,
      p->HWA, p->A, p->Wf, p->Hf * p->Wf, p->stride, p->anchor_offset, p->weights[0], p->weights[1], p->weights[2], p->weights[3],
      p->scale_clamp, pl.topk, p->min_box_size, image_hw_dev, b.sboxes, b.sscores, b.ssrc, b.segs, invalid_count_dev);
  SFOD_LAUNCH_CHECK();
  rc = nmsk::run_segmented(b.sboxes, nullptr, b.segs, N, pl.topk, pl.topk, pl.wstride, p->nms_thresh, p->post_nms_topk,
                           p->post_nms_topk, b.mask, b.keep_rank, b.keep_count, st);
  if (rc) return rc;
  {
    dim3 grid((p->post_nms_topk + 255) / 256, N);
    rpnk::rpn_gather_kernel<<<grid, 256, 0, st>>>(b.sboxes, b.sscores, b.ssrc, b.keep_rank, b.keep_count, pl.topk,
                                                      p->post_nms_topk, reinterpret_cast<float4 *>(out_boxes), out_logits,
                                                      reinterpret_cast<long long *>(out_src_index), out_count_dev);
    SFOD_LAUNCH_CHECK();
  }
  return SFOD_OK;
}

// ===================================================================== Fast R-CNN post-processing
SFOD_API size_t sfod_frcnn_postprocess_workspace_bytes(const sfod_frcnn_params *p) {
  if (!p || p->N <= 0 || p->K <= 0 || p->max_rows_per_image <= 0 || p->topk <= 0) return 256;
  SfodWsSize ws; frk::Plan pl; frk::carve(ws, p, pl, nullptr);
  return ws.off;
}

SFOD_API int sfod_frcnn_postprocess(const sfod_frcnn_params *p, const float *cls_logits, const float *deltas,
                                    const float *proposals, const int32_t *row_offsets_dev, const int32_t *image_hw_dev,
                                    float *det_boxes, float *det_scores, int64_t *det_classes, int64_t *det_rows,
                                    int32_t *det_count_dev, int32_t *pseudo_count_dev, float *probs_out, float *boxes_out,
                                    void *workspace, size_t workspace_bytes, sfod_stream_t stream) {
  if (!p || !cls_logits || !deltas || !proposals || !row_offsets_dev || !image_hw_dev || !det_boxes || !det_scores ||
      !det_classes || !det_rows || !det_count_dev || !pseudo_count_dev)
    return SFOD_ERR_INVALID_ARG;
  if (p->N <= 0 || p->R < 0 || p->K <= 0 || p->max_rows_per_image <= 0 || p->topk <= 0) return SFOD_ERR_INVALID_ARG;
  if (p->rows_stride < 0 || (p->rows_stride > 0 && (p->rows_stride > p->max_rows_per_image || (long long)p->rows_stride * p->N != p->R)))
    return SFOD_ERR_INVALID_ARG;
  if (p->K > frk::kMaxK) return SFOD_ERR_UNSUPPORTED;
  if ((long long)p->max_rows_per_image * p->K >= (1ll << 24)) return SFOD_ERR_UNSUPPORTED;
  if (!sfod_aligned16(deltas) || !sfod_aligned16(proposals) || !sfod_aligned16(det_boxes) ||
      (boxes_out && !sfod_aligned16(boxes_out)))
    return SFOD_ERR_ALIGNMENT;
  cudaStream_t st = sfod_cu(stream);
  SfodWs ws(workspace, workspace_bytes); frk::Plan pl; frk::Buffers b;
  frk::carve(ws, p, pl, &b);
  if (!ws.ok) return SFOD_ERR_WORKSPACE_TOO_SMALL;
  if (pl.P > (1 << 20) || pl.P2 > bsort::kMaxTile * 64) return SFOD_ERR_UNSUPPORTED;
  const int N = p->N, K = p->K;
  SFOD_CUDA_TRY(cudaMemsetAsync(b.keys, 0xFF, (size_t)N * pl.P * sizeof(unsigned long long), st));
  SFOD_CUDA_TRY(cudaMemsetAsync(b.maxc, 0, (size_t)N * sizeof(int), st));
  if (p->R > 0) {
    frk::frcnn_decode_keys_kernel<<<(p->R + 127) / 128, 128, 0, st>>>(
        cls_logits, deltas, reinterpret_cast<const float4 *>(proposals), row_offsets_dev, image_hw_dev, N, p->R, K,
        p->class_agnostic, p->rows_stride, pl.Rmax, pl.P, p->weights[0], p->weights[1], p->weights[2], p->weights[3], p->scale_clamp,
        p->score_thresh, b.cand_boxes, b.keys, b.maxc, probs_out, boxes_out);
    SFOD_LAUNCH_CHECK();
  }
  int rc = bsort::segmented_sort(b.keys, N, pl.P, st);
  if (rc) return rc;
  frk::frcnn_segments_kernel<<<N, 128, (K + 1) * sizeof(int), st>>>(b.keys, pl.P, K, b.segs, b.cand_count);
  SFOD_LAUNCH_CHECK();
  {
    dim3 grid((pl.P + 255) / 256, N);
    frk::frcnn_gather_sorted_kernel<<<grid, 256, 0, st>>>(b.keys, pl.P, K, pl.Rmax, b.cand_boxes, b.cand_count, b.maxc,
                                                                 p->coord_trick_max_n, b.sboxes);
    SFOD_LAUNCH_CHECK();
  }
  rc = nmsk::run_segmented(b.sboxes, nullptr, b.segs, N * K, pl.Rmax, pl.Rmax, pl.wstride, p->nms_thresh, p->topk, p->topk,
                           b.mask, b.keep_rank, b.keep_count, st);
  if (rc) return rc;
  frk::frcnn_merge_keys_kernel<<<N, 256, 0, st>>>(b.keys, pl.P, K, b.segs, b.keep_rank, b.keep_count, p->topk, pl.P2,
                                                         b.keys2, b.total_kept);
  SFOD_LAUNCH_CHECK();
  rc = bsort::segmented_sort(b.keys2, N, pl.P2, st);
  if (rc) return rc;
  frk::frcnn_emit_kernel<<<N, 128, 0, st>>>(b.keys2, pl.P2, K, pl.Rmax, b.cand_boxes, b.total_kept, p->topk,
                                                   p->pseudo_thresh, reinterpret_cast<float4 *>(det_boxes), det_scores,
                                                   reinterpret_cast<long long *>(det_classes),
                                                   reinterpret_cast<long long *>(det_rows), det_count_dev, pseudo_count_dev);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

// ===================================================================== stand-alone box decode / softmax / filter
namespace {

__global__ void __launch_bounds__(256) apply_deltas_kernel(const float4 *__restrict__ deltas, const float4 *__restrict__ boxes,
                                                           long long R, int k, float wx, float wy, float ww, float wh,
                                                           float scale_clamp, float4 *__restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R * k) return;
  out[i] = sfod_decode_box(boxes[i / k], deltas[i], wx, wy, ww, wh, scale_clamp);
}

__global__ void __launch_bounds__(128) softmax_kernel(const float *__restrict__ x, long long R, int K1, float *__restrict__ out) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= R) return;
  const float *xr = x + r * K1; float *o = out + r * K1;
  float m = xr[0];
  for (int k = 1; k < K1; ++k) { const float v = xr[k]; if (v > m || v != v) m = v; }
  float s = 0.f;
  for (int k = 0; k < K1; ++k) s = __fadd_rn(s, sfod_exp_cr(__fsub_rn(xr[k], m)));
  for (int k = 0; k < K1; ++k) o[k] = __fdiv_rn(sfod_exp_cr(__fsub_rn(xr[k], m)), s);
}

constexpr int kSelThreads = 256;
__global__ void __launch_bounds__(kSelThreads) threshold_select_kernel(const float *__restrict__ values,
                                                                       const int *__restrict__ counts, int stride, float thres,
                                                                       long long *__restrict__ out_index,
                                                                       int *__restrict__ out_count) {
  __shared__ int warp_tot[kSelThreads / 32];
  __shared__ int running;
  const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = min(counts[s], stride);
  if (tid == 0) running = 0;
  __syncthreads();
  for (int base = 0; base < n; base += kSelThreads) {
    const int j = base + tid;
    const bool keep = j < n && values[(size_t)s * stride + j] > thres;
    const unsigned bal = __ballot_sync(0xFFFFFFFFu, keep);
    if (lane == 0) warp_tot[warp] = __popc(bal);
    __syncthreads();
    int off = running;
    for (int w = 0; w < warp; ++w) off += warp_tot[w];
    if (keep) out_index[(size_t)s * stride + off + __popc(bal & ((1u << lane) - 1u))] = j;
    __syncthreads();
    if (tid == 0) { int tot = 0; for (int w = 0; w < kSelThreads / 32; ++w) tot += warp_tot[w]; running += tot; }
    __syncthreads();
  }
  if (tid == 0) out_count[s] = running;
}


// Per-class confidence filter of the adaptive-threshold pseudo-labelling variant (reference
// daod/modeling/adaptive_thresh/adaptive_confidence.py:21-33 used by adaptive_threshold_bbox /
// prediction_threshold_bbox, daod/engine/trainers/source_free_adaptive_teacher.py:185-254): keep entry j of segment s iff
// values[s][j] >= class_thresh[classes[s][j]]  (note >=, the reference's `confidence >= threshold * ...`).
__global__ void __launch_bounds__(kSelThreads) class_threshold_select_kernel(const float *__restrict__ values,
                                                                             const long long *__restrict__ classes,
                                                                             const int *__restrict__ counts, int stride, int K,
                                                                             const float *__restrict__ class_thresh,
                                                                             long long *__restrict__ out_index,
                                                                             int *__restrict__ out_count) {
  __shared__ int warp_tot[kSelThreads / 32];
  __shared__ int running;
  const int s = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n = min(counts[s], stride);
  if (tid == 0) running = 0;
  __syncthreads();
  for (int base = 0; base < n; base += kSelThreads) {
    const int j = base + tid;
    bool keep = false;
    if (j < n) {
      const long long c = classes[(size_t)s * stride + j];
      keep = c >= 0 && c < K && values[(size_t)s * stride + j] >= class_thresh[c];
    }
    const unsigned bal = __ballot_sync(0xFFFFFFFFu, keep);
    if (lane == 0) warp_tot[warp] = __popc(bal);
    __syncthreads();
    int off = running;
    for (int w = 0; w < warp; ++w) off += warp_tot[w];
    if (keep) out_index[(size_t)s * stride + off + __popc(bal & ((1u << lane) - 1u))] = j;
    __syncthreads();
    if (tid == 0) { int tot = 0; for (int w = 0; w < kSelThreads / 32; ++w) tot += warp_tot[w]; running += tot; }
    __syncthreads();
  }
  if (tid == 0) out_count[s] = running;
}

// count_label_prediction (reference source_free_adaptive_teacher.py:282-296): per-class number of entries with
// value > thres over ALL segments (one launch for the batch instead of a bincount per image); hist (K) int64, zeroed here.
__global__ void __launch_bounds__(256) class_histogram_kernel(const float *__restrict__ values, const long long *__restrict__ classes,
                                                              const int *__restrict__ counts, int S, int stride, int K, float thres,
                                                              unsigned long long *__restrict__ hist) {
  extern __shared__ unsigned int sh_hist[];
  for (int k = threadIdx.x; k < K; k += blockDim.x) sh_hist[k] = 0;
  __syncthreads();
  for (int s = blockIdx.x; s < S; s += gridDim.x) {
    const int n = min(counts[s], stride);
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
      const long long c = classes[(size_t)s * stride + j];
      if (c >= 0 && c < K && values[(size_t)s * stride + j] > thres) atomicAdd(&sh_hist[c], 1u);
    }
  }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x) if (sh_hist[k]) atomicAdd(&hist[k], (unsigned long long)sh_hist[k]);
}

}  // namespace

SFOD_API int sfod_apply_deltas(const float *deltas, const float *boxes, int64_t R, int k, const float *weights4_host,
                               float scale_clamp, float *out, sfod_stream_t stream) {
  if (R < 0 || k <= 0 || !weights4_host) return SFOD_ERR_INVALID_ARG;
  if (R == 0) return SFOD_OK;
  if (!deltas || !boxes || !out) return SFOD_ERR_INVALID_ARG;
  if (!sfod_aligned16(deltas) || !sfod_aligned16(boxes) || !sfod_aligned16(out)) return SFOD_ERR_ALIGNMENT;
  const long long tot = R * k;
  apply_deltas_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, sfod_cu(stream)>>>(
      reinterpret_cast<const float4 *>(deltas), reinterpret_cast<const float4 *>(boxes), R, k, weights4_host[0],
      weights4_host[1], weights4_host[2], weights4_host[3], scale_clamp, reinterpret_cast<float4 *>(out));
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

SFOD_API int sfod_softmax_lastdim(const float *x, int64_t R, int K1, float *out, sfod_stream_t stream) {
  if (R < 0 || K1 <= 0) return SFOD_ERR_INVALID_ARG;
  if (R == 0) return SFOD_OK;
  if (!x || !out) return SFOD_ERR_INVALID_ARG;
  softmax_kernel<<<(unsigned)((R + 127) / 128), 128, 0, sfod_cu(stream)>>>(x, R, K1, out);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

SFOD_API int sfod_threshold_select(const float *values, const int32_t *counts_dev, int S, int stride, float thres,
                                   int64_t *out_index, int32_t *out_count_dev, sfod_stream_t stream) {
  if (S < 0 || stride < 0) return SFOD_ERR_INVALID_ARG;
  if (S == 0) return SFOD_OK;
  if (!values || !counts_dev || !out_index || !out_count_dev) return SFOD_ERR_INVALID_ARG;
  threshold_select_kernel<<<S, kSelThreads, 0, sfod_cu(stream)>>>(values, counts_dev, stride, thres,
                                                                 reinterpret_cast<long long *>(out_index), out_count_dev);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

static unsigned long long g_sfod_launches = 0;
void sfod_count_launch() { __atomic_fetch_add(&g_sfod_launches, 1ull, __ATOMIC_RELAXED); }
SFOD_API uint64_t sfod_debug_launch_count(void) { return __atomic_load_n(&g_sfod_launches, __ATOMIC_RELAXED); }

SFOD_API int sfod_class_threshold_select(const float *values, const int64_t *classes, const int32_t *counts_dev, int S, int stride,
                                         int K, const float *class_thresh_dev, int64_t *out_index, int32_t *out_count_dev,
                                         sfod_stream_t stream) {
  if (S < 0 || stride < 0 || K <= 0) return SFOD_ERR_INVALID_ARG;
  if (S == 0) return SFOD_OK;
  if (!values || !classes || !counts_dev || !class_thresh_dev || !out_index || !out_count_dev) return SFOD_ERR_INVALID_ARG;
  class_threshold_select_kernel<<<S, kSelThreads, 0, sfod_cu(stream)>>>(values, reinterpret_cast<const long long *>(classes),
                                                                       counts_dev, stride, K, class_thresh_dev,
                                                                       reinterpret_cast<long long *>(out_index), out_count_dev);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

SFOD_API int sfod_class_histogram(const float *values, const int64_t *classes, const int32_t *counts_dev, int S, int stride, int K,
                                  float thres, int64_t *hist_dev, sfod_stream_t stream) {
  if (S < 0 || stride < 0 || K <= 0 || K > 8192 || !hist_dev) return SFOD_ERR_INVALID_ARG;
  cudaStream_t st = sfod_cu(stream);
  SFOD_CUDA_TRY(cudaMemsetAsync(hist_dev, 0, (size_t)K * sizeof(int64_t), st));
  if (S == 0) return SFOD_OK;
  if (!values || !classes || !counts_dev) return SFOD_ERR_INVALID_ARG;
  const int grid = S < SFOD_NUM_SMS ? S : SFOD_NUM_SMS;
  class_histogram_kernel<<<grid, 256, (size_t)K * sizeof(unsigned int), st>>>(values, reinterpret_cast<const long long *>(classes),
                                                                             counts_dev, S, stride, K, thres,
                                                                             reinterpret_cast<unsigned long long *>(hist_dev));
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}

SFOD_API int sfod_abi_version(void) { return 3; }

SFOD_API size_t sfod_abi_sizeof(int which) {
  switch (which) {
    case 0: return sizeof(sfod_ema_tensor);
    case 1: return sizeof(sfod_rpn_params);
    case 2: return sizeof(sfod_frcnn_params);
    case 3: return sizeof(sfod_p2p_comm);
    case 4: return sizeof(sfod_jitter_params);
    case 5: return sizeof(sfod_erase_params);
    case 6: return sizeof(sfod_resize_image);
    case 7: return sizeof(sfod_coco_eval_params);
    default: return 0;
  }
}

SFOD_API const char *sfod_status_string(int status) {
  switch (status) {
    case SFOD_OK: return "ok";
    case SFOD_ERR_INVALID_ARG: return "invalid argument";
    case SFOD_ERR_WORKSPACE_TOO_SMALL: return "workspace too small";
    case SFOD_ERR_UNSUPPORTED: return "unsupported configuration";
    case SFOD_ERR_ALIGNMENT: return "pointer not 16-byte aligned";
    default: return status >= SFOD_ERR_CUDA_BASE ? cudaGetErrorString((cudaError_t)(status - SFOD_ERR_CUDA_BASE)) : "unknown";
  }
}

// ===================================================================== fused pairwise_iou + Matcher
SFOD_API size_t sfod_iou_match_workspace_bytes(int M) { return sfod_align_up((size_t)(M > 0 ? M : 1) * sizeof(int), 256); }

SFOD_API int sfod_iou_match(const float *gt_boxes, const float *boxes, int M, int N, const float *thresholds, const int *labels,
                            int num_thresholds, int allow_low_quality, int64_t *matches, int8_t *match_labels, float *matched_vals,
                            void *workspace, size_t workspace_bytes, sfod_stream_t stream) {
  if (M < 0 || N < 0 || num_thresholds < 0 || num_thresholds > matchk::kMaxThresholds || !labels) return SFOD_ERR_INVALID_ARG;
  if (num_thresholds > 0 && !thresholds) return SFOD_ERR_INVALID_ARG;
  if (N == 0) return SFOD_OK;
  if (!boxes || !matches || !match_labels || (M > 0 && !gt_boxes)) return SFOD_ERR_INVALID_ARG;
  if (!sfod_aligned16(boxes) || (M > 0 && !sfod_aligned16(gt_boxes))) return SFOD_ERR_ALIGNMENT;
  for (int q = 1; q < num_thresholds; ++q)
    if (thresholds[q] < thresholds[q - 1]) return SFOD_ERR_INVALID_ARG;
  cudaStream_t st = sfod_cu(stream);
  matchk::Thresholds th;
  th.count = num_thresholds;
  for (int q = 0; q < matchk::kMaxThresholds; ++q) th.t[q] = q < num_thresholds ? thresholds[q] : 0.f;
  for (int q = 0; q <= matchk::kMaxThresholds; ++q) th.label[q] = q <= num_thresholds ? labels[q] : 0;
  const bool lowq = allow_low_quality && M > 0;
  int *gt_max = nullptr;
  if (lowq) {
    if (!workspace || workspace_bytes < (size_t)M * sizeof(int)) return SFOD_ERR_WORKSPACE_TOO_SMALL;
    gt_max = static_cast<int *>(workspace);
    SFOD_CUDA_TRY(cudaMemsetAsync(gt_max, 0, (size_t)M * sizeof(int), st));
  }
  const unsigned grid = (unsigned)((N + matchk::kThreads - 1) / matchk::kThreads);
  matchk::match_kernel<<<grid, matchk::kThreads, 0, st>>>(reinterpret_cast<const float4 *>(gt_boxes), reinterpret_cast<const float4 *>(boxes),
                                                          M, N, th, reinterpret_cast<long long *>(matches),
                                                          reinterpret_cast<signed char *>(match_labels), matched_vals, gt_max);
  SFOD_LAUNCH_CHECK();
  if (lowq) {
    matchk::low_quality_kernel<<<grid, matchk::kThreads, 0, st>>>(reinterpret_cast<const float4 *>(gt_boxes),
                                                                  reinterpret_cast<const float4 *>(boxes), M, N, gt_max,
                                                                  reinterpret_cast<signed char *>(match_labels));
    SFOD_LAUNCH_CHECK();
  }
  return SFOD_OK;
}

// ===================================================================== batched subsample_labels
SFOD_API int sfod_subsample_labels(const int64_t *labels, const int32_t *offsets, int num_segments, int num_samples, int max_positive,
                                   int64_t bg_label, uint64_t seed, int64_t *sampled, int32_t *counts, sfod_stream_t stream) {
  if (num_segments < 0 || num_samples <= 0 || max_positive < 0 || max_positive > num_samples) return SFOD_ERR_INVALID_ARG;
  // selection buffer: the negatives start at num_pos and are padded to a power of two: num_pos + 2 (num_samples - num_pos) <= 2 num_samples
  if (2 * num_samples > samplek::kMaxSamples) return SFOD_ERR_UNSUPPORTED;
  if (num_segments == 0) return SFOD_OK;
  if (!labels || !offsets || !sampled || !counts) return SFOD_ERR_INVALID_ARG;
  // `offsets` is a HOST array: it travels in the kernel parameters, <= 255 segments per launch (the hash key uses the
  // segment index within the call, so a split call keeps keys distinct through the seed)
  for (int s0 = 0; s0 < num_segments; s0 += samplek::kMaxSegments) {
    const int ns = num_segments - s0 < samplek::kMaxSegments ? num_segments - s0 : samplek::kMaxSegments;
    samplek::Offsets off;
    for (int i = 0; i <= ns; ++i) off.v[i] = offsets[s0 + i];
    samplek::subsample_kernel<<<ns, samplek::kThreads, 0, sfod_cu(stream)>>>(
        reinterpret_cast<const long long *>(labels), off, num_samples, max_positive, (long long)bg_label,
        (unsigned long long)seed + 0x632BE59BD9B4E019ull * (unsigned long long)(s0 / samplek::kMaxSegments),
        reinterpret_cast<long long *>(sampled) + (size_t)s0 * num_samples, counts + 2 * (size_t)s0);
    SFOD_LAUNCH_CHECK();
  }
  return SFOD_OK;
}
