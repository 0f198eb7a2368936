// evaluate.cu -- COCO box AP on the device, bit-equal to pycocotools' COCOeval (iouType "bbox"): evaluate() + accumulate().
//
// Replaces the evaluation the reference runs through detectron2's COCOEvaluator (reference daod/evaluation/, called from
// test_refinement, daod/engine/trainers/base.py:300, from the --eval-only runs of train_net*.py and from EvalHook).  Every
// output of COCOeval.evaluate / accumulate is a count, a comparison or one IEEE fp64 division, so the result is exact:
//
//   1. coco_eval_match_kernel, one CTA per (image, category):
//      stable descending score order of the image's detections (NaN last, as np.argsort(-score, kind="mergesort")), the
//      first maxDets[-1] of the category; bbIou (maskApi.c) in fp64 in its operation order; COCOeval.evaluateImg's greedy
//      matching for every (area range, IoU threshold) pair, one lane each.  Per detection and area range one word: bit t =
//      true positive at threshold t, bit 16 + t = false positive (neither = ignored); plus the rank within the category and
//      one 64-bit sort key; per (category, area range) the number of non-ignored gt (npig, atomics: exact).
//   2. One ascending sort (sort.cuh) of the keys (category << 56) | (~score_key << 24) | (image * P + rank in the image): per
//      category the score-descending order of accumulate's np.argsort(-dtScores, kind="mergesort") over the detections
//      concatenated in image order.  The order does not depend on the area range, and the maxDet-truncated lists are
//      sub-sequences of it (rank < maxDet), so one sort serves every (category, area range, maxDet).
//   3. coco_eval_accumulate_kernel, one CTA per (category, area range, maxDet, threshold): cumulative tp / fp (integers),
//      rc = tp / npig, pr = tp / (fp + tp + 2^-52), the precision envelope (suffix maximum), np.searchsorted(rc, recThrs,
//      "left") and the -1 / 0 conventions of accumulate().  The scan runs backwards over the sorted keys so that the suffix
//      maximum and the cumulative sums come out of one pass.
#include "common.cuh"
#include "sort.cuh"

namespace {

constexpr int kMatchThreads = 128;
constexpr int kAccThreads = 256;
constexpr int kMaxDetsCap = 128;        // maxDets[-1] <= 128: ranks fit a byte
constexpr int kMaxSlots = 1024;         // detections per image row
constexpr int kMaxGtPerImage = 1024;
constexpr int kIouTableCap = 4096;      // doubles: the D x G IoU table when it fits, otherwise recomputed (same arithmetic)

struct EvalArgs {
  sfod_coco_eval_params p;
  const int64_t *gt_off;       // (I + 1), device copy of the caller's host offsets
  const double *gt_box;        // (n_gt, 4) XYWH
  const double *gt_area;
  const uint8_t *gt_crowd;
  const int64_t *gt_id;
  const int64_t *gt_cat;
  const float *dt_box;         // (I, P, 4) XYWH
  const float *dt_score;       // (I, P)
  const int64_t *dt_cls;       // (I, P)
  const int32_t *dt_count;     // (I)
  int32_t *npig;               // (K, A)
  unsigned long long *keys;    // (Psort)
  uint32_t *flags;             // (I * P, A)
  uint8_t *rank;               // (I * P)
  double *precision, *scores, *recall;
  int gmax, tab_cap, trunc;   // trunc = maxDets[-1]
};

// fp32 score -> 32-bit key, larger = earlier in a descending sort; NaN is 0 (numpy sorts NaN last).
__device__ __forceinline__ uint32_t eval_key(float s) { return s != s ? 0u : sfod_score_key(s); }
__device__ __forceinline__ double key_to_score(uint32_t k) { return k == 0u ? (double)__int_as_float(0x7fc00000) : (double)sfod_key_score(k); }

// maskApi.c::bbIou for one pair (the loop body, with its operation order).
__device__ __forceinline__ double bb_iou(const double *d, double da, const double *g, double ga, bool crowd) {
  const double w = __dsub_rn(fmin(__dadd_rn(d[2], d[0]), __dadd_rn(g[2], g[0])), fmax(d[0], g[0]));
  if (w <= 0) return 0.0;
  const double h = __dsub_rn(fmin(__dadd_rn(d[3], d[1]), __dadd_rn(g[3], g[1])), fmax(d[1], g[1]));
  if (h <= 0) return 0.0;
  const double i = __dmul_rn(w, h);
  const double u = crowd ? da : __dsub_rn(__dadd_rn(da, ga), i);
  return __ddiv_rn(i, u);
}

struct MatchSmem {   // byte offsets into the dynamic shared memory
  size_t skey, scls, dbox, darea, dpos, flagw, gbox, garea, gid, gcrowd, gig, gord, gtm, tab, total;
};

__host__ __device__ inline MatchSmem match_smem_layout(int P, int gmax, int tab_cap, int AT) {
  MatchSmem s;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 15) / 16 * 16; return r; };
  const int gw = (gmax + 31) / 32;
  s.tab = take((size_t)tab_cap * 8);
  s.dbox = take((size_t)kMaxDetsCap * 4 * 8);
  s.darea = take((size_t)kMaxDetsCap * 8);
  s.gbox = take((size_t)gmax * 4 * 8);
  s.garea = take((size_t)gmax * 8);
  s.gid = take((size_t)gmax * 8);
  s.skey = take((size_t)P * 4);
  s.scls = take((size_t)P * 4);
  s.dpos = take((size_t)kMaxDetsCap * 4);
  s.flagw = take((size_t)kMaxDetsCap * SFOD_COCO_MAX_AREA_RNGS * 4);
  s.gtm = take((size_t)AT * gw * 4);
  s.gord = take((size_t)SFOD_COCO_MAX_AREA_RNGS * gmax * 2);
  s.gcrowd = take((size_t)gmax);
  s.gig = take((size_t)gmax);
  s.total = o;
  return s;
}

__global__ void __launch_bounds__(kMatchThreads) coco_eval_match_kernel(const EvalArgs args) {
  extern __shared__ __align__(16) unsigned char smem[];
  const sfod_coco_eval_params &p = args.p;
  const int img = blockIdx.x, k = blockIdx.y, tid = threadIdx.x;
  const int P = p.dt_stride, A = p.n_area_rngs, T = p.n_iou_thrs;
  const int trunc = args.trunc;
  const MatchSmem L = match_smem_layout(P, args.gmax, args.tab_cap, A * T);
  uint32_t *skey = reinterpret_cast<uint32_t *>(smem + L.skey);
  int32_t *scls = reinterpret_cast<int32_t *>(smem + L.scls);
  double *dbox = reinterpret_cast<double *>(smem + L.dbox);
  double *darea = reinterpret_cast<double *>(smem + L.darea);
  int32_t *dpos = reinterpret_cast<int32_t *>(smem + L.dpos);
  uint32_t *flagw = reinterpret_cast<uint32_t *>(smem + L.flagw);
  double *gbox = reinterpret_cast<double *>(smem + L.gbox);
  double *garea = reinterpret_cast<double *>(smem + L.garea);
  int64_t *gid = reinterpret_cast<int64_t *>(smem + L.gid);
  uint8_t *gcrowd = smem + L.gcrowd;
  uint8_t *gig = smem + L.gig;       // bit a: ignored in area range a
  uint16_t *gord = reinterpret_cast<uint16_t *>(smem + L.gord);
  uint32_t *gtm = reinterpret_cast<uint32_t *>(smem + L.gtm);
  double *tab = reinterpret_cast<double *>(smem + L.tab);
  __shared__ int s_nk, s_G;
  __shared__ int s_wsum[kMatchThreads / 32];
  __shared__ double s_iou[SFOD_COCO_MAX_IOU_THRS], s_area[SFOD_COCO_MAX_AREA_RNGS][2];
  if (tid < T) s_iou[tid] = p.iou_thrs[tid];
  if (tid < A) { s_area[tid][0] = p.area_rng[tid][0]; s_area[tid][1] = p.area_rng[tid][1]; }

  // ---- detections of the image: score keys and classes
  int n = args.dt_count[img];
  n = n < 0 ? 0 : (n > P ? P : n);
  const size_t row = (size_t)img * P;
  if (tid == 0) { s_nk = 0; s_G = 0; }
  for (int j = tid; j < n; j += kMatchThreads) {
    skey[j] = eval_key(args.dt_score[row + j]);
    const int64_t c = args.dt_cls[row + j];
    scls[j] = (c >= 0 && c < p.n_categories) ? (int)c : -1;
  }
  __syncthreads();
  // rank in the image's stable descending order, and in the category's; the first `trunc` of the category are kept
  for (int j = tid; j < n; j += kMatchThreads) {
    if (scls[j] != k) continue;
    const uint32_t kj = skey[j];
    int r_all = 0, r_cat = 0;
    for (int q = 0; q < n; ++q) {
      const uint32_t kq = skey[q];
      const bool before = kq > kj || (kq == kj && q < j);
      r_all += before;
      r_cat += before && scls[q] == k;
    }
    atomicAdd(&s_nk, 1);
    if (r_cat < trunc) {
      const float4 b = reinterpret_cast<const float4 *>(args.dt_box)[row + j];
      double *db = dbox + 4 * r_cat;
      db[0] = (double)b.x; db[1] = (double)b.y; db[2] = (double)b.z; db[3] = (double)b.w;
      darea[r_cat] = __dmul_rn((double)b.z, (double)b.w);       // loadRes: area = w * h (exact for fp32 w, h)
      dpos[r_cat] = r_all;
      const unsigned long long pos = (unsigned long long)(row + r_all);
      args.keys[pos] = ((unsigned long long)k << 56) | ((unsigned long long)(~kj) << 24) | pos;
      args.rank[pos] = (uint8_t)r_cat;
    }
  }
  // ---- ground truth of (image, category), in annotation order
  const int64_t g0 = args.gt_off[img], g1 = args.gt_off[img + 1];
  const int lane = tid & 31, warp = tid >> 5;
  for (int64_t base = g0; base < g1; base += kMatchThreads) {
    const int64_t gi = base + tid;
    const bool mine = gi < g1 && args.gt_cat[gi] == k;
    const unsigned bal = __ballot_sync(0xFFFFFFFFu, mine);
    if (lane == 0) s_wsum[warp] = __popc(bal);
    __syncthreads();
    int off = s_G;
    for (int w = 0; w < warp; ++w) off += s_wsum[w];
    off += __popc(bal & ((1u << lane) - 1u));
    if (mine) {
      const double *src = args.gt_box + 4 * gi;
      double *gb = gbox + 4 * off;
      gb[0] = src[0]; gb[1] = src[1]; gb[2] = src[2]; gb[3] = src[3];
      const double area = args.gt_area[gi];
      const bool crowd = args.gt_crowd[gi] != 0;
      garea[off] = area;
      gid[off] = args.gt_id[gi];
      gcrowd[off] = crowd;
      uint8_t ig = 0;
      for (int a = 0; a < A; ++a)
        if (crowd || area < s_area[a][0] || area > s_area[a][1]) ig |= (uint8_t)(1u << a);
      gig[off] = ig;
    }
    __syncthreads();
    if (tid == 0) { int s = 0; for (int w = 0; w < kMatchThreads / 32; ++w) s += s_wsum[w]; s_G += s; }
    __syncthreads();
  }
  __syncthreads();
  const int G = s_G;
  const int D = s_nk < trunc ? s_nk : trunc;
  if (D == 0 && G == 0) return;            // evaluateImg returns None
  // npig and the per-area gt order (stable sort by _ignore: the non-ignored first)
  if (tid < A) {
    const int a = tid;
    int c = 0;
    for (int g = 0; g < G; ++g)
      if (!((gig[g] >> a) & 1)) gord[a * args.gmax + c++] = (uint16_t)g;
    if (c) atomicAdd(&args.npig[k * A + a], c);
    for (int g = 0; g < G; ++g)
      if ((gig[g] >> a) & 1) gord[a * args.gmax + c++] = (uint16_t)g;
  }
  const bool use_tab = D * G <= args.tab_cap;
  if (use_tab)
    for (int idx = tid; idx < D * G; idx += kMatchThreads) {
      const int d = idx / G, g = idx - d * G;
      const double *gb = gbox + 4 * g;
      tab[idx] = bb_iou(dbox + 4 * d, darea[d], gb, __dmul_rn(gb[2], gb[3]), gcrowd[g]);
    }
  const int gw = (args.gmax + 31) / 32;
  for (int idx = tid; idx < A * T * gw; idx += kMatchThreads) gtm[idx] = 0u;
  for (int idx = tid; idx < D * A; idx += kMatchThreads) flagw[idx] = 0u;
  __syncthreads();
  // ---- evaluateImg: one lane per (area range, threshold)
  if (tid < A * T) {
    const int a = tid / T, t = tid - a * T;
    uint32_t *mbits = gtm + tid * gw;
    const uint16_t *ord = gord + a * args.gmax;
    const double thr = s_iou[t], cap = 1 - 1e-10;
    const double t0 = cap < thr ? cap : thr;      // min([t, 1 - 1e-10])
    const double lo = s_area[a][0], hi = s_area[a][1];
    for (int d = 0; d < D; ++d) {
      double iou = t0;
      int m = -1;
      bool m_ig = false;
      for (int x = 0; x < G; ++x) {
        const int g = ord[x];
        if (((mbits[g >> 5] >> (g & 31)) & 1u) && !gcrowd[g]) continue;
        const bool g_ig = (gig[g] >> a) & 1;
        if (m > -1 && !m_ig && g_ig) break;
        double v;
        if (use_tab) v = tab[d * G + g];
        else { const double *gb = gbox + 4 * g; v = bb_iou(dbox + 4 * d, darea[d], gb, __dmul_rn(gb[2], gb[3]), gcrowd[g]); }
        if (v < iou) continue;
        iou = v; m = g; m_ig = g_ig;
      }
      bool ig = false, matched_id = false;
      if (m > -1) {
        mbits[m >> 5] |= 1u << (m & 31);
        ig = m_ig;
        matched_id = gid[m] != 0;                 // dtMatches holds the gt id: id 0 reads as "unmatched"
      }
      if (!matched_id && (darea[d] < lo || darea[d] > hi)) ig = true;
      const uint32_t bits = ig ? 0u : (matched_id ? (1u << t) : (1u << (16 + t)));
      if (bits) atomicOr(&flagw[d * A + a], bits);
    }
  }
  __syncthreads();
  for (int idx = tid; idx < D * A; idx += kMatchThreads) {
    const int d = idx / A, a = idx - d * A;
    args.flags[(row + dpos[d]) * A + a] = flagw[idx];
  }
}

// ---- block scans over kAccThreads threads (inclusive, in thread order)
template <typename V, typename Op>
__device__ __forceinline__ V block_inclusive_scan(V v, V *sh, Op op) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const V u = __shfl_up_sync(0xFFFFFFFFu, v, o);
    if (lane >= o) v = op(v, u);
  }
  if (lane == 31) sh[warp] = v;
  __syncthreads();
  V pre = V();
  bool has = false;
  for (int w = 0; w < warp; ++w) { pre = has ? op(pre, sh[w]) : sh[w]; has = true; }
  __syncthreads();
  return has ? op(pre, v) : v;
}

struct AddI { __device__ int operator()(int a, int b) const { return a + b; } };
struct MaxD { __device__ double operator()(double a, double b) const { return a > b ? a : b; } };

__device__ __forceinline__ unsigned long long lower_bound_keys(const unsigned long long *keys, long long n, unsigned long long v) {
  long long lo = 0, hi = n;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (keys[mid] < v) lo = mid + 1; else hi = mid;
  }
  return (unsigned long long)lo;
}

__global__ void __launch_bounds__(kAccThreads) coco_eval_accumulate_kernel(const EvalArgs args, long long n_keys) {
  const sfod_coco_eval_params &p = args.p;
  const int K = p.n_categories, A = p.n_area_rngs, M = p.n_max_dets, R = p.n_rec_thrs;
  const int m = blockIdx.x % M, a = (blockIdx.x / M) % A, k = blockIdx.x / (M * A), t = blockIdx.y;
  const int tid = threadIdx.x;
  __shared__ double q[SFOD_COCO_MAX_REC_THRS], ss[SFOD_COCO_MAX_REC_THRS], s_rec[SFOD_COCO_MAX_REC_THRS];
  __shared__ long long s_lo, s_hi;
  __shared__ int s_tot[3];
  __shared__ int sh_i[kAccThreads / 32];
  __shared__ double sh_d[kAccThreads / 32];
  auto cell = [&](int r) { return ((((size_t)t * R + r) * K + k) * A + a) * M + m; };
  const int npig = args.npig[k * A + a];
  if (npig == 0) {                                 // no non-ignored gt: COCOeval leaves -1
    for (int r = tid; r < R; r += kAccThreads) { args.precision[cell(r)] = -1.0; args.scores[cell(r)] = -1.0; }
    if (tid == 0) args.recall[(((size_t)t * K + k) * A + a) * M + m] = -1.0;
    return;
  }
  if (tid == 0) {
    s_lo = (long long)lower_bound_keys(args.keys, n_keys, (unsigned long long)k << 56);
    s_hi = (long long)lower_bound_keys(args.keys, n_keys, (unsigned long long)(k + 1) << 56);
    s_tot[0] = s_tot[1] = s_tot[2] = 0;
  }
  for (int r = tid; r < R; r += kAccThreads) { q[r] = 0.0; ss[r] = 0.0; s_rec[r] = p.rec_thrs[r]; }
  __syncthreads();
  const long long lo = s_lo, hi = s_hi;
  const int max_det = m == 0 ? p.max_dets[0] : m == 1 ? p.max_dets[1] : m == 2 ? p.max_dets[2] : p.max_dets[3];
  const uint32_t tp_bit = 1u << t, fp_bit = 1u << (16 + t);
  const unsigned long long pos_mask = (1ull << 24) - 1;
  // totals of the maxDet-truncated list
  int c_tp = 0, c_fp = 0, c_inc = 0;
  for (long long e = lo + tid; e < hi; e += kAccThreads) {
    const unsigned long long pos = args.keys[e] & pos_mask;
    if (args.rank[pos] >= max_det) continue;
    const uint32_t f = args.flags[pos * A + a];
    c_inc += 1; c_tp += (f & tp_bit) != 0; c_fp += (f & fp_bit) != 0;
  }
  if (c_inc) atomicAdd(&s_tot[2], c_inc);
  if (c_tp) atomicAdd(&s_tot[0], c_tp);
  if (c_fp) atomicAdd(&s_tot[1], c_fp);
  __syncthreads();
  const int TP = s_tot[0], FP = s_tot[1], NINC = s_tot[2];
  const double npig_d = (double)npig, eps = 2.220446049250313e-16;    // np.spacing(1)
  // backwards over the sorted list: thread 0 takes the last element of each chunk
  int carry_tp = 0, carry_fp = 0, carry_inc = 0;
  double carry_max = 0.0;
  for (long long end = hi; end > lo; end -= kAccThreads) {
    const long long e = end - 1 - tid;
    int inc = 0, tpf = 0, fpf = 0;
    uint32_t skey = 0;
    if (e >= lo) {
      const unsigned long long key = args.keys[e], pos = key & pos_mask;
      if (args.rank[pos] < max_det) {
        const uint32_t f = args.flags[pos * A + a];
        inc = 1; tpf = (f & tp_bit) != 0; fpf = (f & fp_bit) != 0;
        skey = ~(uint32_t)(key >> 24);
      }
    }
    const int s_tp = block_inclusive_scan(tpf, sh_i, AddI());
    const int s_fp = block_inclusive_scan(fpf, sh_i, AddI());
    const int s_inc = block_inclusive_scan(inc, sh_i, AddI());
    const int tp_cum = TP - (carry_tp + s_tp) + tpf;          // cumulative sums up to and including this element
    const int fp_cum = FP - (carry_fp + s_fp) + fpf;
    const int inc_before = NINC - (carry_inc + s_inc);
    const double tpd = (double)tp_cum, fpd = (double)fp_cum;
    const double pr = inc ? __ddiv_rn(tpd, __dadd_rn(__dadd_rn(fpd, tpd), eps)) : 0.0;
    double env = block_inclusive_scan(pr, sh_d, MaxD());
    env = env > carry_max ? env : carry_max;                  // precision envelope: max over this and every later element
    if (inc && (tpf || inc_before == 0)) {                    // recall steps here: searchsorted(rc, recThrs, "left") lands on it
      const double rc = __ddiv_rn(tpd, npig_d);
      const double rc_prev = __ddiv_rn((double)(tp_cum - tpf), npig_d);
      const double score = key_to_score(skey);
      for (int r = 0; r < R; ++r) {
        const double x = s_rec[r];
        if ((inc_before == 0 || rc_prev < x) && !(rc < x)) { q[r] = env; ss[r] = score; }
      }
    }
    // carries for the next (earlier) chunk: the last thread holds the chunk totals
    __shared__ int s_c[3];
    __shared__ double s_cm;
    if (tid == kAccThreads - 1) { s_c[0] = s_tp; s_c[1] = s_fp; s_c[2] = s_inc; s_cm = env; }
    __syncthreads();
    carry_tp += s_c[0]; carry_fp += s_c[1]; carry_inc += s_c[2]; carry_max = s_cm;
    __syncthreads();
  }
  __syncthreads();
  for (int r = tid; r < R; r += kAccThreads) { args.precision[cell(r)] = q[r]; args.scores[cell(r)] = ss[r]; }
  if (tid == 0) args.recall[(((size_t)t * K + k) * A + a) * M + m] = NINC ? __ddiv_rn((double)TP, npig_d) : 0.0;
}

struct EvalWs {
  int64_t *gt_off; int32_t *npig; unsigned long long *keys; uint32_t *flags; uint8_t *rank;
  int psort;
};

template <typename W>
static EvalWs carve(W &ws, const sfod_coco_eval_params *p) {
  EvalWs e;
  const long long slots = (long long)p->n_images * p->dt_stride;
  e.psort = bsort::next_pow2(slots < 1 ? 1 : slots);
  e.gt_off = ws.template take<int64_t>((size_t)p->n_images + 1);
  e.npig = ws.template take<int32_t>((size_t)p->n_categories * p->n_area_rngs);
  e.keys = ws.template take<unsigned long long>((size_t)e.psort);
  e.flags = ws.template take<uint32_t>((size_t)(slots < 1 ? 1 : slots) * p->n_area_rngs);
  e.rank = ws.template take<uint8_t>((size_t)(slots < 1 ? 1 : slots));
  return e;
}

static int check_params(const sfod_coco_eval_params *p) {
  if (!p) return SFOD_ERR_INVALID_ARG;
  if (p->n_images < 0 || p->n_categories < 1 || p->dt_stride < 1 || p->n_iou_thrs < 1 || p->n_rec_thrs < 1 ||
      p->n_area_rngs < 1 || p->n_max_dets < 1)
    return SFOD_ERR_INVALID_ARG;
  for (int m = 0; m < p->n_max_dets && m < SFOD_COCO_MAX_MAX_DETS; ++m)
    if (p->max_dets[m] < 1) return SFOD_ERR_INVALID_ARG;
  if (p->n_categories > SFOD_COCO_MAX_CATEGORIES || p->dt_stride > kMaxSlots || p->n_iou_thrs > SFOD_COCO_MAX_IOU_THRS ||
      p->n_rec_thrs > SFOD_COCO_MAX_REC_THRS || p->n_area_rngs > SFOD_COCO_MAX_AREA_RNGS || p->n_max_dets > SFOD_COCO_MAX_MAX_DETS)
    return SFOD_ERR_UNSUPPORTED;
  for (int m = 0; m < p->n_max_dets; ++m)
    if (p->max_dets[m] > kMaxDetsCap) return SFOD_ERR_UNSUPPORTED;
  if ((long long)p->n_images * p->dt_stride >= (1ll << 24))
    return SFOD_ERR_UNSUPPORTED;   // image * P + rank must fit the 24 low bits of a sort key
  return SFOD_OK;
}

}  // namespace

SFOD_API size_t sfod_coco_eval_workspace_bytes(const sfod_coco_eval_params *p) {
  if (check_params(p) != SFOD_OK) return 0;
  SfodWsSize ws;
  carve(ws, p);
  return ws.off;
}

SFOD_API int sfod_coco_eval(const sfod_coco_eval_params *p, const int64_t *gt_offsets, const double *gt_boxes,
                            const double *gt_area, const uint8_t *gt_iscrowd, const int64_t *gt_ids, const int64_t *gt_categories,
                            const float *dt_boxes, const float *dt_scores, const int64_t *dt_classes, const int32_t *dt_counts,
                            double *precision, double *scores, double *recall, void *workspace, size_t workspace_bytes,
                            sfod_stream_t stream) {
  int rc = check_params(p);
  if (rc) return rc;
  if (!gt_offsets || !precision || !scores || !recall) return SFOD_ERR_INVALID_ARG;
  const int I = p->n_images;
  if (I > 0 && (!dt_boxes || !dt_scores || !dt_classes || !dt_counts)) return SFOD_ERR_INVALID_ARG;
  if (gt_offsets[0] != 0) return SFOD_ERR_INVALID_ARG;
  int gmax = 0;
  for (int i = 0; i < I; ++i) {
    const int64_t g = gt_offsets[i + 1] - gt_offsets[i];
    if (g < 0) return SFOD_ERR_INVALID_ARG;          // gt not sorted by image
    if (g > kMaxGtPerImage) return SFOD_ERR_UNSUPPORTED;
    if (g > gmax) gmax = (int)g;
  }
  const int64_t n_gt = gt_offsets[I];
  if (n_gt > 2147483647ll) return SFOD_ERR_UNSUPPORTED;
  if (n_gt > 0 && (!gt_boxes || !gt_area || !gt_iscrowd || !gt_ids || !gt_categories)) return SFOD_ERR_INVALID_ARG;
  if (!sfod_aligned16(dt_boxes)) return SFOD_ERR_ALIGNMENT;
  SfodWs ws(workspace, workspace_bytes);
  const EvalWs e = carve(ws, p);
  if (!ws.ok) return SFOD_ERR_WORKSPACE_TOO_SMALL;

  const int A = p->n_area_rngs, T = p->n_iou_thrs;
  const int trunc = p->max_dets[p->n_max_dets - 1];
  const int dmax = trunc < p->dt_stride ? trunc : p->dt_stride;
  const int gm = gmax < 1 ? 1 : gmax;
  int tab_cap = dmax * gm;
  if (tab_cap > kIouTableCap) tab_cap = kIouTableCap;
  const MatchSmem L = match_smem_layout(p->dt_stride, gm, tab_cap, A * T);

  EvalArgs args;
  args.p = *p;
  args.gt_off = e.gt_off; args.gt_box = gt_boxes; args.gt_area = gt_area; args.gt_crowd = gt_iscrowd; args.gt_id = gt_ids;
  args.gt_cat = gt_categories;
  args.dt_box = dt_boxes; args.dt_score = dt_scores; args.dt_cls = dt_classes; args.dt_count = dt_counts;
  args.npig = e.npig; args.keys = e.keys; args.flags = e.flags; args.rank = e.rank;
  args.precision = precision; args.scores = scores; args.recall = recall;
  args.gmax = gm; args.tab_cap = tab_cap; args.trunc = trunc;

  cudaStream_t s = sfod_cu(stream);
  SFOD_CUDA_TRY(cudaMemcpyAsync(e.gt_off, gt_offsets, sizeof(int64_t) * ((size_t)I + 1), cudaMemcpyHostToDevice, s));
  SFOD_CUDA_TRY(cudaMemsetAsync(e.npig, 0, sizeof(int32_t) * (size_t)p->n_categories * A, s));
  SFOD_CUDA_TRY(cudaMemsetAsync(e.keys, 0xFF, sizeof(unsigned long long) * (size_t)e.psort, s));
  if (I > 0) {
    if (L.total > 48 * 1024)
      SFOD_CUDA_TRY(cudaFuncSetAttribute(coco_eval_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));
    coco_eval_match_kernel<<<dim3(I, p->n_categories), kMatchThreads, L.total, s>>>(args);
    SFOD_LAUNCH_CHECK();
    rc = bsort::segmented_sort(e.keys, 1, e.psort, s);
    if (rc) return rc;
  }
  coco_eval_accumulate_kernel<<<dim3(p->n_categories * A * p->n_max_dets, T), kAccThreads, 0, s>>>(args, e.psort);
  SFOD_LAUNCH_CHECK();
  return SFOD_OK;
}
