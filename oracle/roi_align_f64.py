"""Float64 reference of ROIAlign with the CUDA kernels' fp32 geometry (test infrastructure).

Every ROIAlign kernel of csrc/roi.cu computes the same geometry in fp32, with separately rounded operations in torchvision's
CPU order (roi_geometry, sample_coord, bilinear_1d): the ROI start and bin size, the sampling grid, each sample coordinate,
the in/out decision at [-1, size], the clamp, lo / hi and the 1-D weights l, h.  Those decisions are discontinuous -- a sample
one ulp outside [-1, size] is dropped, the adaptive grid ceil(roi_h / 7) jumps where roi_h / 7 is an integer -- so the
reference reproduces them bit for bit in numpy float32 (each numpy float32 operation is one correctly rounded IEEE
operation) and only the accumulation is done in float64.

Bilinear sampling followed by the bin average is a linear operator S per image, rows (ROI, bin), columns (y, x):

    S[(r, ph, pw), (y, x)] = A[r, ph, y] * B[r, pw, x] / count_r,
    A[r, ph, y] = sum over the samples iy of bin ph of h_y (at row lo) and l_y (at row hi),   count_r = max(gh * gw, 1)

(B likewise along x).  The fp32 factors are exact in float64, so S carries only float64 rounding.  Then

    forward  = S . X,   error scale S . |X|       backward = S^T . G,  error scale S^T . |G|

(the weights are non-negative).  Two term counts go with every output element: ``nnz``, the non-zeros of its row (forward)
or column (backward) of S, i.e. the (pixel, bin) products a kernel that merges the samples into weight tables sums; and
``terms``, the same count before the samples are merged (one per sample corner with a non-zero weight), i.e. what a kernel
that visits sample by sample sums.  S is built per image and per chunk of ROIs, so 1 000 R101 ROIs with 1 024 channels need
a few hundred MB of host memory at most.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp

F32 = np.float32
DENSE = 9   # window class of the dense column tables (kNXMax + 1 in roi.cu)


def _np(t) -> np.ndarray:
    return t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)


def geometry(rois, scale, aligned, PH, PW, sampling_ratio):
    """roi_geometry (roi.cu): per ROI the image index, the fp32 start / bin size and the sampling grid (gh, gw)."""
    r = np.asarray(_np(rois), dtype=F32).reshape(-1, 5)
    s, off = F32(scale), F32(0.5 if aligned else 0.0)
    rsw, rsh, rew, reh = (r[:, k] * s - off for k in (1, 2, 3, 4))
    rw, rh = rew - rsw, reh - rsh
    if not aligned:
        rw, rh = np.maximum(rw, F32(1.0)), np.maximum(rh, F32(1.0))
    bh, bw = rh / F32(PH), rw / F32(PW)
    if sampling_ratio > 0:
        gh = np.full(len(r), sampling_ratio, np.int64); gw = gh.copy()
    else:
        gh, gw = np.ceil(bh).astype(np.int64), np.ceil(bw).astype(np.int64)
    return dict(n=r[:, 0].astype(np.int64), sh=rsh, sw=rsw, bh=bh, bw=bw, gh=gh, gw=gw)


def axis_samples(start, binsz, grid, P, size):
    """sample_coord + bilinear_1d along one axis for every (ROI, bin p, sample i): arrays of shape (R, P, G).

    Returns the fp32 coordinate v, the in-range mask (i < grid and -1 <= v <= size), lo, hi and the fp32 weights l, h."""
    G = max(int(grid.max(initial=0)), 1)
    p = np.arange(P, dtype=F32)[None, :, None]
    i = np.arange(G, dtype=F32)[None, None, :]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        v = (start[:, None, None] + p * binsz[:, None, None]) + ((i + F32(0.5)) * binsz[:, None, None]) / grid.astype(F32)[:, None, None]
    ok = (np.arange(G)[None, None, :] < grid[:, None, None]) & (v >= F32(-1.0)) & (v <= F32(size))
    vc = np.where(ok, np.where(v <= 0, F32(0.0), v), F32(0.0)).astype(F32)
    lo = vc.astype(np.int64)
    top = lo >= size - 1
    lo = np.where(top, size - 1, lo)
    hi = np.where(top, lo, lo + 1)
    vc = np.where(top, lo.astype(F32), vc)
    l = (vc - lo.astype(F32)).astype(F32)
    h = (F32(1.0) - l).astype(F32)
    return dict(v=v, ok=ok, lo=lo, hi=hi, l=l, h=h)


def _axis_operator(ax, size):
    """Merged 1-D weights (sum of h at lo and l at hi, float64) and the per-entry count of non-zero sample terms."""
    R, P, G = ax["ok"].shape
    A = np.zeros((R, P, size)); T = np.zeros((R, P, size), np.int64)
    rr, pp, _ = np.nonzero(ax["ok"])
    okm = ax["ok"]
    for idx, wt in ((ax["lo"][okm], ax["h"][okm]), (ax["hi"][okm], ax["l"][okm])):
        nz = wt != 0
        np.add.at(A, (rr[nz], pp[nz], idx[nz]), wt[nz].astype(np.float64))
        np.add.at(T, (rr[nz], pp[nz], idx[nz]), 1)
    return A, T


def window_class(ax, W):
    """roi_sep_tables_kernel (roi.cu:296-300): the widest per-bin column window of the ROI, rounded up to 2, 3, 4, 6, 8,
    or DENSE (wider than 8, or wider than the map)."""
    ok = ax["ok"]
    xmn = np.where(ok, ax["lo"], W).min(axis=2)
    xmx = np.where(ok, ax["hi"], -1).max(axis=2)
    wmax = np.where(xmx >= 0, xmx - xmn + 1, 0).max(axis=1)
    nx = np.select([wmax <= 2, wmax <= 3, wmax <= 4, wmax <= 6, wmax <= 8], [2, 3, 4, 6, 8], DENSE)
    return np.where(nx > W, DENSE, nx)


class RoiAlignF64:
    """The reference for one call: ``RoiAlignF64(rois, N, H, W, scale, aligned, sampling_ratio, PH, PW)``."""

    def __init__(self, rois, N, H, W, scale, aligned, sampling_ratio, PH=7, PW=7):
        self.N, self.H, self.W, self.PH, self.PW = N, H, W, PH, PW
        self.g = geometry(rois, scale, aligned, PH, PW, sampling_ratio)
        self.R = len(self.g["n"])
        self.valid = (self.g["n"] >= 0) & (self.g["n"] < N)
        self.count = np.maximum(self.g["gh"] * self.g["gw"], 1).astype(np.float64)
        self.ay = axis_samples(self.g["sh"], self.g["bh"], self.g["gh"], PH, H)
        self.ax = axis_samples(self.g["sw"], self.g["bw"], self.g["gw"], PW, W)
        self.nx = window_class(self.ax, W)

    # ------------------------------------------------------------------ the operator
    def operator(self, idx):
        """S (float64) and the matching term counts for the ROIs ``idx`` (all of one image): CSR matrices of shape
        (len(idx) * PH * PW, H * W); rows (ROI, ph, pw), columns y * W + x.  Also the per-row nnz / terms, (len, PH, PW)."""
        idx = np.asarray(idx, np.int64)
        PH, PW, H, W = self.PH, self.PW, self.H, self.W
        sub = lambda ax: {k: v[idx] for k, v in ax.items()}
        A, TA = _axis_operator(sub(self.ay), H)
        B, TB = _axis_operator(sub(self.ax), W)
        A[~self.valid[idx]] = 0.0; TA[~self.valid[idx]] = 0
        ry, py, yy = np.nonzero(A)                 # ordered by ROI
        rx, px, xx = np.nonzero(B)
        cx = np.bincount(rx, minlength=len(idx))
        xs = np.concatenate([[0], np.cumsum(cx)])[:-1]
        rep = cx[ry]                               # every (ph, y) entry pairs with every (pw, x) entry of its ROI
        ey = np.repeat(np.arange(len(ry)), rep)
        k = np.arange(len(ey)) - np.repeat(np.concatenate([[0], np.cumsum(rep)])[:-1], rep)
        ex = xs[ry[ey]] + k
        r = ry[ey]
        rows = (r * PH + py[ey]) * PW + px[ex]
        cols = yy[ey] * W + xx[ex]
        vals = A[r, py[ey], yy[ey]] * B[r, px[ex], xx[ex]] / self.count[idx][r]
        terms = TA[r, py[ey], yy[ey]] * TB[r, px[ex], xx[ex]]
        shape = (len(idx) * PH * PW, H * W)
        S = sp.csr_matrix((vals, (rows, cols)), shape=shape)
        T = sp.csr_matrix((terms.astype(np.float64), (rows, cols)), shape=shape)
        ny = (A != 0).sum(2); nxc = (B != 0).sum(2)
        ty = TA.sum(2); tx = TB.sum(2)
        nnz = ny[:, :, None] * nxc[:, None, :]
        tr = ty[:, :, None] * tx[:, None, :]
        return S, T, nnz, tr

    def _groups(self, idx, chunk):
        idx = np.asarray(idx, np.int64)
        n = np.where(self.valid[idx], self.g["n"][idx], -1)
        for img in np.unique(n):
            sel = idx[n == img]
            for s in range(0, len(sel), chunk):
                yield int(img), sel[s:s + chunk]

    # ------------------------------------------------------------------ forward / backward
    def forward(self, x, idx=None, chunk=128):
        """Yields (rows, ref, scale, nnz, terms) per chunk of the ROIs ``idx`` (default: all), each of shape
        (len(rows), C, PH, PW): ref = S . X and scale = S . |X| in float64.  Invalid image indices give zero rows."""
        x = _np(x)
        C = x.shape[1]
        idx = np.arange(self.R) if idx is None else np.asarray(idx, np.int64)
        cache = {}
        for img, rows in self._groups(idx, chunk):
            shp = (len(rows), self.PH, self.PW, C)
            if img < 0:
                z = np.zeros(shp).transpose(0, 3, 1, 2)
                zi = np.zeros((len(rows), C, self.PH, self.PW), np.int64)
                yield rows, z, z, zi, zi
                continue
            if img not in cache:
                cache.clear()
                xi = x[img].reshape(C, -1).T.astype(np.float64)
                cache[img] = np.ascontiguousarray(np.hstack([xi, np.abs(xi)]))
            S, _, nnz, terms = self.operator(rows)
            both = S @ cache[img]
            ref = both[:, :C].reshape(shp).transpose(0, 3, 1, 2)
            scale = both[:, C:].reshape(shp).transpose(0, 3, 1, 2)
            yield rows, ref, scale, np.broadcast_to(nnz[:, None], ref.shape), np.broadcast_to(terms[:, None], ref.shape)

    def backward(self, g, chunk=128):
        """(grad, scale, nnz, terms), each (N, C, H, W): grad = S^T . G and scale = S^T . |G| in float64; nnz / terms are
        the contributions each pixel receives (column counts of S before / after merging the samples)."""
        g = _np(g)
        C = g.shape[1]
        N, H, W, PH, PW = self.N, self.H, self.W, self.PH, self.PW
        out = np.zeros((N, H * W, 2 * C)); nnz = np.zeros((N, H * W)); terms = np.zeros((N, H * W))
        for img, rows in self._groups(np.arange(self.R), chunk):
            if img < 0:
                continue
            S, T, _, _ = self.operator(rows)
            gi = g[rows].transpose(0, 2, 3, 1).reshape(-1, C).astype(np.float64)
            out[img] += S.T @ np.hstack([gi, np.abs(gi)])
            nnz[img] += np.asarray((S != 0).sum(axis=0)).ravel()
            terms[img] += np.asarray(T.sum(axis=0)).ravel()
        to = lambda a: a.reshape(N, H, W, C).transpose(0, 3, 1, 2)
        cnt = lambda a: np.broadcast_to(a.reshape(N, 1, H, W), (N, C, H, W))
        return to(out[:, :, :C]), to(out[:, :, C:]), cnt(nnz), cnt(terms)

    # ------------------------------------------------------------------ the same fp32 terms in torchvision's order
    def _corner_terms(self):
        ay, ax = self.ay, self.ax
        ok = ay["ok"][:, :, None, :, None] & ax["ok"][:, None, :, None, :] & self.valid[:, None, None, None, None]
        w = lambda a, b: (ay[a][:, :, None, :, None] * ax[b][:, None, :, None, :]).astype(F32)
        ylo, yhi = ay["lo"][:, :, None, :, None], ay["hi"][:, :, None, :, None]
        xlo, xhi = ax["lo"][:, None, :, None, :], ax["hi"][:, None, :, None, :]
        corners = [(w("h", "h"), ylo, xlo), (w("h", "l"), ylo, xhi), (w("l", "h"), yhi, xlo), (w("l", "l"), yhi, xhi)]
        return ok, corners

    def fp32_forward(self, x):
        """torchvision's CPU forward in fp32 from these factors: val += ((w1 v1 + w2 v2) + w3 v3) + w4 v4 over (iy, ix),
        then val / count.  (R, C, PH, PW) float32."""
        x = np.asarray(_np(x), F32)
        ok, corners = self._corner_terms()
        n = np.clip(self.g["n"], 0, self.N - 1)[:, None, None, None, None]
        R, PH, PW, Gy, Gx = ok.shape
        val = np.zeros((R, PH, PW, x.shape[1]), F32)
        for iy in range(Gy):
            for ix in range(Gx):
                t = None
                for w, yi, xi in corners:
                    wv = np.broadcast_to(w, ok.shape)[..., iy, ix][..., None]
                    px = x[np.broadcast_to(n, ok.shape)[..., iy, ix], :, np.broadcast_to(yi, ok.shape)[..., iy, ix],
                           np.broadcast_to(xi, ok.shape)[..., iy, ix]]
                    p = (wv * px).astype(F32)
                    t = p if t is None else (t + p).astype(F32)
                val = np.where(ok[..., iy, ix][..., None], (val + t).astype(F32), val)
        return (val / self.count.astype(F32)[:, None, None, None]).astype(F32).transpose(0, 3, 1, 2)

    def fp32_backward(self, g):
        """torchvision's CPU backward in fp32: ROIs, channels, bins and samples in order, g_k = (go * w_k) / count added to
        the four corners one after another.  (N, C, H, W) float32."""
        g = np.asarray(_np(g), F32)
        out = np.zeros((self.N, g.shape[1], self.H, self.W), F32)
        ok, corners = self._corner_terms()
        cnt = self.count.astype(F32)
        for r in np.nonzero(self.valid)[0]:
            n = self.g["n"][r]
            for ph in range(self.PH):
                for pw in range(self.PW):
                    go = g[r, :, ph, pw]
                    for iy, ix in zip(*np.nonzero(ok[r, ph, pw])):
                        for w, yi, xi in corners:
                            wv = np.broadcast_to(w, ok.shape)[r, ph, pw, iy, ix]
                            y = np.broadcast_to(yi, ok.shape)[r, ph, pw, iy, ix]
                            xx = np.broadcast_to(xi, ok.shape)[r, ph, pw, iy, ix]
                            out[n, :, y, xx] = (out[n, :, y, xx] + ((go * wv).astype(F32) / cnt[r]).astype(F32)).astype(F32)
        return out


# ---------------------------------------------------------------------------------------------------- ROI sets
def _ulp_neighbours(x, K):
    """The 2K + 1 float32 values x - K ulps ... x + K ulps (monotone through zero)."""
    b = int(np.array(x, F32).view(np.int32))
    key = b if b >= 0 else -(b & 0x7FFFFFFF)
    keys = key + np.arange(-K, K + 1, dtype=np.int64)
    bits = np.where(keys >= 0, keys, (-keys) | 0x80000000).astype(np.uint32)
    return bits.view(F32)


def _pick_around(values, target):
    """Indices of the candidates whose value equals ``target`` and of the nearest ones strictly below and above it."""
    out = []
    eq = np.nonzero(values == target)[0]
    if len(eq):
        out.append(eq[len(eq) // 2])
    for side in (values < target, values > target):
        c = np.nonzero(side)[0]
        if len(c):
            out.append(c[np.argmin(np.abs(values[c].astype(np.float64) - float(target)))])
    return out


def _edge_boxes(axis, size, other, scale, aligned, sr, K=96):
    """Boxes (feature frame of the other axis = ``other``) whose first sample (targets -1, 0 and interior integers, varying the
    near edge) or last sample (targets size - 1 and size, varying the far edge) lands exactly on the target in fp32, and on the
    nearest representable positions on either side of it."""
    s, off = float(scale), 0.5 if aligned else 0.0
    out = []
    ints = sorted({1, size // 2, max(size - 2, 1)} - {0, size - 1, size}) if size > 2 else []
    for t in [-1.0, 0.0, float(size - 1), float(size)] + [float(k) for k in ints]:
        upper = t >= size - 1
        for hgt in (0.7, 3.3, 0.45 * size + 1.9):
            bh = hgt / 7.0
            g = sr if sr > 0 else max(int(np.ceil(bh)), 1)
            first = 0.5 * bh / g if not upper else 6.0 * bh + (g - 0.5) * bh / g
            lo_f = t - first
            near, far = F32((lo_f + off) / s), F32((lo_f + hgt + off) / s)
            cands = _ulp_neighbours(far if upper else near, K)
            lo_c = np.full(len(cands), near, F32) if upper else cands
            hi_c = cands if upper else np.full(len(cands), far, F32)
            o1, o2 = other
            if axis == 0:
                boxes = np.stack([np.full_like(lo_c, o1), lo_c, np.full_like(lo_c, o2), hi_c], 1)
            else:
                boxes = np.stack([lo_c, np.full_like(lo_c, o1), hi_c, np.full_like(lo_c, o2)], 1)
            geo = geometry(np.hstack([np.zeros((len(boxes), 1), F32), boxes]), scale, aligned, 7, 7, sr)
            st, bn, gr = (geo["sh"], geo["bh"], geo["gh"]) if axis == 0 else (geo["sw"], geo["bw"], geo["gw"])
            v = axis_samples(st, bn, gr, 7, size)["v"]
            vals = v[np.arange(len(v)), 6, np.maximum(gr - 1, 0)] if upper else v[:, 0, 0]
            out += [boxes[i] for i in _pick_around(vals.astype(F32), F32(t))]
    return out


def _grid_boxes(axis, other, scale, aligned, sr, rng, K=96):
    """Boxes whose extent / 7 is exactly 1, 2, 3 feature pixels in fp32 (the adaptive grid count ceil(roi / 7) jumps there),
    and the nearest extents on either side."""
    s, off = float(scale), 0.5 if aligned else 0.0
    out = []
    for k in (1, 2, 3):
        lo = F32((rng.uniform(0, 4) + off) / s)
        cands = _ulp_neighbours(F32(float(lo) + 7 * k / s), K)
        lo_c = np.full(len(cands), lo, F32)
        o1, o2 = other
        if axis == 0:
            boxes = np.stack([np.full_like(lo_c, o1), lo_c, np.full_like(lo_c, o2), cands], 1)
        else:
            boxes = np.stack([lo_c, np.full_like(lo_c, o1), cands, np.full_like(lo_c, o2)], 1)
        geo = geometry(np.hstack([np.zeros((len(boxes), 1), F32), boxes]), scale, aligned, 7, 7, sr)
        out += [boxes[i] for i in _pick_around(geo["bh" if axis == 0 else "bw"], F32(k))]
    return out


def roi_set(H, W, scale, aligned, sampling_ratio, seed, sweep=300, wide=300):
    """The ROI set of the path tests, as (R, 4) float32 boxes in image coordinates (x1, y1, x2, y2):

    * a log-uniform sweep of widths and heights from 0.1 feature pixel to 1.2x the map, centres over the map and its border;
    * wide boxes (7 to 250 feature pixels across: bins of 1 to 36 pixels), so that every compact column window and the
      dense tables occur on every map;
    * edge boxes: a sample exactly on -1, 0, size - 1, size and on interior integers, and on the nearest fp32 positions on
      either side (the in/out decision and the clamp of bilinear_1d), along y and along x;
    * boxes whose extent / 7 is exactly 1, 2 or 3 and one step either side (the adaptive grid count);
    * zero and negative extents, and boxes entirely outside the map."""
    rng = np.random.default_rng(seed)
    s = float(scale)

    def rand_boxes(n, wlo, whi, hlo, hhi, spread):
        w = np.exp(rng.uniform(np.log(wlo), np.log(whi), n)); h = np.exp(rng.uniform(np.log(hlo), np.log(hhi), n))
        cx = W / 2 + rng.uniform(-spread, spread, n) * W; cy = H / 2 + rng.uniform(-spread, spread, n) * H
        return np.stack([cx - w / 2, cy - h / 2, cx + w / 2, cy + h / 2], 1) / s

    parts = [rand_boxes(sweep, 0.1, 1.2 * W, 0.1, 1.2 * H, 0.6), rand_boxes(wide, 7.0, 250.0, 0.3, 1.2 * H, 0.3)]
    special = []
    for axis, size, osize in ((0, H, W), (1, W, H)):
        for _ in range(2):
            o = rng.uniform(-0.5, osize / 2); other = (F32(o / s), F32((o + rng.uniform(0.5, osize / 2)) / s))
            special += _edge_boxes(axis, size, other, scale, aligned, sampling_ratio)
        special += _grid_boxes(axis, other, scale, aligned, sampling_ratio, rng)
    parts.append(np.array(special, np.float64).reshape(-1, 4))
    c = np.array([W / 3, H / 3]) / s
    d = rng.uniform(0.5, 3.0, (4, 2)) / s
    parts.append(np.array([[*c, *c], [*(c + d[0]), *(c + d[0])],                              # zero extent
                           [*(c + d[1]), *c], [c[0], c[1] + d[2, 1], c[0] + d[2, 0], c[1]],  # negative extents
                           [*(c + d[3]), c[0], c[1] + d[3, 1]], [c[0] + d[3, 0], c[1], c[0], c[1] + d[3, 1]]]))
    out = np.array([[-40, -30, -5, -2], [W + 3, 0, W + 50, H], [0, H + 2.5, W, H + 9], [-9, -9, -1.5, H + 1],
                    [W + 1.25, -4, W + 2, -1.25], [-3, H + 1.01, W + 4, H + 30]], np.float64) / s
    parts.append(out)                                                                           # entirely outside the map
    return np.concatenate(parts).astype(F32)
