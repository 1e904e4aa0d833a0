"""A plain float64 restatement of cv::SIFT::create(2500, 3, 0.04, 5, 1.2)->detectAndCompute (OpenCV 4.x
sift.simd.hpp), numpy / scipy only, no cv2.

Each stage is a function of the previous stage's output, so a test can feed it the GPU kernel's own previous stage
(csrc/sift.cu, read back by vstab_b200.k_sift_stages) and check one kernel at a time:

    base_image(u8)                      2x INTER_LINEAR upsample (exact), blur to sigma 1.2
    blur64(img, taps)                   separable Gaussian, BORDER_REFLECT_101 (repeated for tiny octaves)
    next_octave_base(g3)                nearest 2x decimation of Gaussian 3
    extrema(gauss)                      DoG 3x3x3 extrema, |v| > floor(0.5 * 0.04 / 3 * 255), 5 px border
    refine(gauss, cand)                 adjustLocalExtrema: <= 5 steps, contrast test, edge test
    orientations(gauss, refined)        calcOrientationHist: 36 bins, [1 4 6 4 1] / 16, peaks >= 0.8 max
    select(kps, rows, size_ratio)       removeDuplicatedSorted, retainBest(2500) with ties, octave -1 rescale, size filter
    descriptors(gauss, kps)             calcSIFTDescriptor: 4x4x8 trilinear, normalise, clip 0.2, normalise, x512

Everything is float64 except what OpenCV's definition fixes in float32: the Gaussian taps (getGaussianKernel(CV_32F)),
the initial sigma (computed in float by createInitialImage) and the DoG, which OpenCV stores as float32 images.
Keypoints are structured arrays of KP_DTYPE; `octave` is cv::KeyPoint::octave's packed word."""
import math

import numpy as np
from scipy import ndimage

N_LAYERS = 3
N_GAUSS = N_LAYERS + 3
BORDER = 5                      # SIFT_IMG_BORDER
CONTRAST_THR = 0.04
EDGE_THR = 5.0
SIGMA = 1.2
N_FEATURES = 2500
MAX_INTERP_STEPS = 5
ORI_BINS = 36
ORI_RADIUS = 4.5                # SIFT_ORI_RADIUS = 3 * SIFT_ORI_SIG_FCTR
ORI_SIG_FCTR = 1.5
ORI_PEAK_RATIO = 0.8
DESCR_WIDTH = 4
DESCR_BINS = 8
DESCR_SCL_FCTR = 3.0
DESCR_MAG_THR = 0.2
INT_DESCR_FCTR = 512.0
FLT_EPSILON = float(np.finfo(np.float32).eps)
DOG_THRESHOLD = math.floor(0.5 * CONTRAST_THR / N_LAYERS * 255)      # cvFloor, = 1

KP_DTYPE = np.dtype([("x", "<f4"), ("y", "<f4"), ("size", "<f4"), ("angle", "<f4"), ("response", "<f4"), ("octave", "<i4")])


def cv_round(v):
    """cvRound: round half to even (lrint)."""
    return np.rint(v).astype(np.int64)


# ------------------------------------------------------------------ Gaussian kernels
def kernel_size(sigma):
    """GaussianBlur(Size(), sigma) on a float image: cvRound(sigma * 4 * 2 + 1) | 1."""
    return int(np.rint(sigma * 8 + 1)) | 1


def gaussian_taps(sigma):
    """getGaussianKernel(ksize, sigma, CV_32F) (its bit-exact construction: exp(-x^2 / 2 sigma^2), the sum of the two
    halves plus the centre, each tap times 1 / sum), as float32 taps held in float64."""
    n = kernel_size(sigma)
    half = (n - 1) // 2
    x = np.arange(-half, 0, dtype=np.float64)
    side = np.exp(x * x * (-0.5 / (sigma * sigma)))
    s = side.sum() * 2.0 + 1.0
    k = np.concatenate([side, [1.0], side[::-1]]) * (1.0 / s)
    return k.astype(np.float32).astype(np.float64)


def sigmas():
    """The blur of the base image (createInitialImage computes it in float) and the five incremental sigmas of an
    octave (buildGaussianPyramid, double)."""
    s = np.float32(SIGMA)
    init = float(np.sqrt(np.maximum(s * s - np.float32(0.5 * 0.5 * 4), np.float32(0.01))))
    k = 2.0 ** (1.0 / N_LAYERS)
    inc = []
    for i in range(1, N_GAUSS):
        prev = k ** (i - 1) * SIGMA
        tot = prev * k
        inc.append(math.sqrt(tot * tot - prev * prev))
    return init, inc


def all_taps():
    """[taps of the base blur, taps of Gaussian 1 .. 5]."""
    init, inc = sigmas()
    return [gaussian_taps(init)] + [gaussian_taps(s) for s in inc]


# ------------------------------------------------------------------ blur, base image, octaves
def reflect101(idx, n):
    """borderInterpolate(BORDER_REFLECT_101), reflected as often as needed (kernels wider than the image)."""
    idx = np.asarray(idx, np.int64).copy()
    if n == 1:
        return np.zeros_like(idx)
    while True:
        lo, hi = idx < 0, idx >= n
        if not (lo.any() or hi.any()):
            return idx
        idx[lo] = -idx[lo]
        idx[hi] = 2 * n - 2 - idx[hi]


def blur64(img, taps, rows=None):
    """Separable blur in float64 with BORDER_REFLECT_101.  `rows` (a slice) limits the output to those rows."""
    img = np.asarray(img, np.float64)
    h, w = img.shape
    R = (len(taps) - 1) // 2
    r0, r1 = (0, h) if rows is None else (rows.start, rows.stop)
    yi = reflect101(np.arange(r0 - R, r1 + R), h)
    src = img[yi]
    v = np.zeros((r1 - r0, w))
    for j, t in enumerate(taps):
        v += t * src[j:j + r1 - r0]
    xi = reflect101(np.arange(-R, w + R), w)
    src = v[:, xi]
    out = np.zeros((r1 - r0, w))
    for j, t in enumerate(taps):
        out += t * src[:, j:j + w]
    return out


def upsample2x(gray):
    """resize(INTER_LINEAR) by exactly 2 (weights 1/4, 3/4, borders clamped): exact."""
    g = np.asarray(gray, np.float64)

    def up(a, axis):
        n = a.shape[axis]
        i = np.arange(n)
        prev = np.take(a, np.maximum(i - 1, 0), axis=axis)
        nxt = np.take(a, np.minimum(i + 1, n - 1), axis=axis)
        even = 0.25 * prev + 0.75 * a
        odd = 0.75 * a + 0.25 * nxt
        out = np.stack([even, odd], axis=axis + 1)
        shape = list(a.shape)
        shape[axis] = 2 * n
        return out.reshape(shape)

    return up(up(g, 1), 0)


def base_image(gray):
    """createInitialImage(doubleImageSize = true): the upsampled input blurred by the initial sigma."""
    return blur64(upsample2x(gray), all_taps()[0])


def n_octaves(rows, cols):
    """cvRound(log2(min(base side)) - 2) - firstOctave, firstOctave = -1."""
    return int(np.rint(math.log(min(2 * rows, 2 * cols)) / math.log(2.0) - 2)) + 1


def octave_shapes(rows, cols):
    shapes, h, w = [], 2 * rows, 2 * cols
    for _ in range(n_octaves(rows, cols)):
        shapes.append((h, w))
        h, w = h // 2, w // 2
    return shapes


def next_octave_base(g3):
    """resize(INTER_NEAREST) to (cols / 2, rows / 2) of Gaussian 3."""
    h, w = g3.shape
    return g3[: 2 * (h // 2): 2, : 2 * (w // 2): 2][: h // 2, : w // 2]


def gaussian_pyramid(gray):
    """The full float64 pyramid: list over octaves of [6, h, w]."""
    taps = all_taps()
    pyr = []
    g = base_image(gray)
    for o, _ in enumerate(octave_shapes(*gray.shape)):
        if o:
            g = next_octave_base(pyr[-1][N_LAYERS])
        levels = [g]
        for i in range(1, N_GAUSS):
            levels.append(blur64(levels[-1], taps[i]))
        pyr.append(np.stack(levels))
    return pyr


def dog(gauss_octave):
    """DoG of one octave as OpenCV stores it: float32 differences of the Gaussians, [5, h, w]."""
    g = np.asarray(gauss_octave, np.float32)
    return g[1:] - g[:-1]


# ------------------------------------------------------------------ extrema
def extrema(gauss):
    """findScaleSpaceExtrema's pixel test on every octave: int64 array [n, 4] of (octave, layer, row, col), sorted."""
    out = []
    for o, g in enumerate(gauss):
        D = dog(g)
        _, h, w = D.shape
        if h <= 2 * BORDER or w <= 2 * BORDER:
            continue
        mx = ndimage.maximum_filter(D, size=3, mode="nearest")
        mn = ndimage.minimum_filter(D, size=3, mode="nearest")
        for layer in range(1, N_LAYERS + 1):
            v = D[layer, BORDER:h - BORDER, BORDER:w - BORDER]
            a = mx[layer, BORDER:h - BORDER, BORDER:w - BORDER]
            b = mn[layer, BORDER:h - BORDER, BORDER:w - BORDER]
            hit = (np.abs(v) > DOG_THRESHOLD) & (((v > 0) & (v >= a)) | ((v < 0) & (v <= b)))
            r, c = np.nonzero(hit)
            out.append(np.stack([np.full_like(r, o), np.full_like(r, layer), r + BORDER, c + BORDER], 1))
    if not out:
        return np.zeros((0, 4), np.int64)
    a = np.concatenate(out).astype(np.int64)
    return a[np.lexsort(a.T[::-1])]


def decode_candidates(keys):
    """The kernel's candidate words (octave << 56 | layer << 48 | row << 24 | col) as sorted [n, 4] rows."""
    k = np.asarray(keys, np.uint64)
    a = np.stack([(k >> np.uint64(56)), (k >> np.uint64(48)) & np.uint64(0xFF), (k >> np.uint64(24)) & np.uint64(0xFFFFFF),
                  k & np.uint64(0xFFFFFF)], 1).astype(np.int64)
    return a[np.lexsort(a.T[::-1])] if len(a) else a.reshape(0, 4)


# ------------------------------------------------------------------ refinement
def _derivs(D, l, r, c):
    """dD, the 3x3 Hessian and the centre value at integer positions (vectorised over candidates)."""
    v = D[l, r, c]
    dx = (D[l, r, c + 1] - D[l, r, c - 1]) * 0.5 / 255
    dy = (D[l, r + 1, c] - D[l, r - 1, c]) * 0.5 / 255
    ds = (D[l + 1, r, c] - D[l - 1, r, c]) * 0.5 / 255
    dxx = (D[l, r, c + 1] + D[l, r, c - 1] - 2 * v) / 255
    dyy = (D[l, r + 1, c] + D[l, r - 1, c] - 2 * v) / 255
    dss = (D[l + 1, r, c] + D[l - 1, r, c] - 2 * v) / 255
    dxy = (D[l, r + 1, c + 1] - D[l, r + 1, c - 1] - D[l, r - 1, c + 1] + D[l, r - 1, c - 1]) * 0.25 / 255
    dxs = (D[l + 1, r, c + 1] - D[l + 1, r, c - 1] - D[l - 1, r, c + 1] + D[l - 1, r, c - 1]) * 0.25 / 255
    dys = (D[l + 1, r + 1, c] - D[l + 1, r - 1, c] - D[l - 1, r + 1, c] + D[l - 1, r - 1, c]) * 0.25 / 255
    H = np.stack([np.stack([dxx, dxy, dxs], -1), np.stack([dxy, dyy, dys], -1), np.stack([dxs, dys, dss], -1)], -2)
    return np.stack([dx, dy, ds], -1), H, v


def refine(gauss, cand):
    """adjustLocalExtrema on every candidate row (octave, layer, row, col).  Returns a dict of arrays over the
    candidates that survive: octave index o, layer, r, c (final integer position), xi, xr, xc, contr, the keypoint
    fields x, y, size, response, octave word, and `margin`: the smallest relative distance of any decision taken for
    that candidate (step / stop at 0.5, the rounding of a step, the contrast and edge tests, det > 0) from its
    threshold, divided by the condition number of the Hessian; `kappa`: that condition number at the final position.
    `rejected_margin`: the same for the candidates that
    did not survive (o, layer, r, c of the start, margin)."""
    cand = np.asarray(cand, np.int64).reshape(-1, 4)
    res = {k: [] for k in ("o", "layer", "r", "c", "xi", "xr", "xc", "contr", "margin", "kappa")}
    rej = {k: [] for k in ("o", "layer", "r", "c", "margin")}
    for o, g in enumerate(gauss):
        sel = cand[:, 0] == o
        if not sel.any():
            continue
        D = dog(g).astype(np.float64)
        _, h, w = D.shape
        l0, r0, c0 = cand[sel, 1].copy(), cand[sel, 2].copy(), cand[sel, 3].copy()
        l, r, c = l0.copy(), r0.copy(), c0.copy()
        n = len(l)
        X = np.zeros((n, 3))
        margin = np.full(n, np.inf)
        active = np.ones(n, bool)          # still stepping
        alive = np.ones(n, bool)
        for _ in range(MAX_INTERP_STEPS):
            idx = np.nonzero(active)[0]
            if not len(idx):
                break
            dD, H, _ = _derivs(D, l[idx], r[idx], c[idx])
            det = np.linalg.det(H)
            ok = det != 0
            x = np.zeros((len(idx), 3))
            if ok.any():
                x[ok] = np.linalg.solve(H[ok], dD[ok][..., None])[..., 0]
            kappa = np.ones(len(idx))
            if ok.any():
                kappa[ok] = np.linalg.cond(H[ok])
            X[idx] = -x
            xc, xr, xi = -x[:, 0], -x[:, 1], -x[:, 2]
            ax = np.abs(np.stack([xc, xr, xi], 1))
            # step / stop: every |offset| against 0.5; the rounding of a step: the fractional part against 0.5
            m = np.min(np.abs(ax - 0.5) / 0.5, 1)
            stop = (ax < 0.5).all(1)
            frac = np.abs(np.abs(ax - np.floor(ax)) - 0.5)
            m_round = np.where(stop, np.inf, np.min(np.where(ax >= 0.5, frac, np.inf), 1))
            margin[idx] = np.minimum(margin[idx], np.minimum(m, m_round) / kappa)
            huge = (ax > float(np.float32(2147483647 / 3))).any(1) & ~stop
            alive[idx[huge]] = False
            active[idx[stop | huge]] = False
            mv = idx[~stop & ~huge]
            if len(mv):
                xs = X[mv]
                c[mv] += cv_round(xs[:, 0])
                r[mv] += cv_round(xs[:, 1])
                l[mv] += cv_round(xs[:, 2])
                out = (l[mv] < 1) | (l[mv] > N_LAYERS) | (c[mv] < BORDER) | (c[mv] >= w - BORDER) | (r[mv] < BORDER) | \
                      (r[mv] >= h - BORDER)
                alive[mv[out]] = False
                active[mv[out]] = False
        alive &= ~active                    # not converged within MAX_INTERP_STEPS
        idx = np.nonzero(alive)[0]
        if len(idx):
            dD, H, v = _derivs(D, l[idx], r[idx], c[idx])
            xc, xr, xi = X[idx, 0], X[idx, 1], X[idx, 2]
            t = dD[:, 0] * xc + dD[:, 1] * xr + dD[:, 2] * xi
            contr = v / 255 + t * 0.5
            ok = np.abs(contr) * N_LAYERS >= CONTRAST_THR
            kappa = np.linalg.cond(H)
            kappa = np.where(np.isfinite(kappa), kappa, 1e30)
            m_contr = np.abs(np.abs(contr) * N_LAYERS - CONTRAST_THR) / CONTRAST_THR
            dxx, dyy, dxy = H[:, 0, 0], H[:, 1, 1], H[:, 0, 1]
            tr, dt = dxx + dyy, dxx * dyy - dxy * dxy
            scale = np.maximum(np.abs(dxx * dyy), dxy * dxy) + 1e-300
            m_det = np.abs(dt) / scale
            lhs, rhs = tr * tr * EDGE_THR, (EDGE_THR + 1) ** 2 * dt
            m_edge = np.abs(lhs - rhs) / (np.abs(lhs) + np.abs(rhs) + 1e-300)
            ok &= (dt > 0) & (lhs < rhs)
            margin[idx] = np.minimum(margin[idx], np.minimum(m_contr, np.where(np.abs(contr) * N_LAYERS >= CONTRAST_THR,
                                                                             np.minimum(m_det, m_edge), np.inf)) / kappa)
            alive[idx[~ok]] = False
            good = idx[ok]
            res["o"].append(np.full(len(good), o))
            res["layer"].append(l[good]); res["r"].append(r[good]); res["c"].append(c[good])
            res["xc"].append(X[good, 0]); res["xr"].append(X[good, 1]); res["xi"].append(X[good, 2])
            res["contr"].append(contr[ok]); res["margin"].append(margin[good]); res["kappa"].append(kappa[ok])
        bad = np.nonzero(~alive)[0]
        rej["o"].append(np.full(len(bad), o)); rej["layer"].append(l0[bad]); rej["r"].append(r0[bad])
        rej["c"].append(c0[bad]); rej["margin"].append(margin[bad])
    cat = lambda d: {k: (np.concatenate(v) if v else np.zeros(0)) for k, v in d.items()}
    res, rej = cat(res), cat(rej)
    for k in ("o", "layer", "r", "c"):
        res[k] = res[k].astype(np.int64)
        rej[k] = rej[k].astype(np.int64)
    s = 2.0 ** res["o"]
    res["x"] = (res["c"] + res["xc"]) * s
    res["y"] = (res["r"] + res["xr"]) * s
    res["size"] = SIGMA * 2.0 ** ((res["layer"] + res["xi"]) / N_LAYERS) * s * 2
    res["response"] = np.abs(res["contr"])
    res["octave"] = res["o"] + (res["layer"] << 8) + (cv_round((res["xi"] + 0.5) * 255) << 16)
    return res, rej


# ------------------------------------------------------------------ orientation
def fast_atan2_deg(y, x):
    """cv::fastAtan2's polynomial (degrees, [0, 360)), evaluated in float64."""
    y = np.asarray(y, np.float64)
    x = np.asarray(x, np.float64)
    sc = 180.0 / math.pi
    p1, p3, p5, p7 = 0.9997878412794807 * sc, -0.3258083974640975 * sc, 0.1555786518463281 * sc, -0.04432655554792128 * sc
    ax, ay = np.abs(x), np.abs(y)
    eps = 2.220446049250313e-16
    big = ax >= ay
    cc = np.where(big, ay / (ax + eps), ax / (ay + eps))
    c2 = cc * cc
    p = (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * cc
    a = np.where(big, p, 90.0 - p)
    a = np.where(x < 0, 180.0 - a, a)
    return np.where(y < 0, 360.0 - a, a)


def _ori_samples(img, r, c, radius, sig):
    """calcOrientationHist's samples for keypoints sharing one radius: (ori, weight * mag, valid) [K, (2R + 1)^2]."""
    h, w = img.shape[-2:]
    d = np.arange(-radius, radius + 1)
    ii, jj = np.meshgrid(d, d, indexing="ij")
    ii, jj = ii.ravel(), jj.ravel()
    y = r[:, None] + ii[None]
    x = c[:, None] + jj[None]
    valid = (y > 0) & (y < h - 1) & (x > 0) & (x < w - 1)
    yc, xc = np.clip(y, 1, h - 2), np.clip(x, 1, w - 2)
    dx = img[yc, xc + 1] - img[yc, xc - 1]
    dy = img[yc - 1, xc] - img[yc + 1, xc]
    wgt = np.exp((ii * ii + jj * jj)[None] * (-1.0 / (2.0 * sig[:, None] ** 2)))
    return fast_atan2_deg(dy, dx), wgt * np.hypot(dx, dy), valid


def _smooth(hist):
    h = hist
    return (np.roll(h, 2, -1) + np.roll(h, -2, -1)) * (1 / 16) + (np.roll(h, 1, -1) + np.roll(h, -1, -1)) * (4 / 16) + h * (6 / 16)


def _peaks(sm):
    """(bin index, interpolated angle, margin) of every accepted peak of one smoothed histogram; margin: the smallest
    relative distance of a peak decision (> left, > right, >= 0.8 max) from its threshold, over all 36 bins."""
    n = ORI_BINS
    mx = sm.max()
    thr = mx * ORI_PEAK_RATIO
    left, right = np.roll(sm, 1), np.roll(sm, -1)
    acc = (sm > left) & (sm > right) & (sm >= thr)
    scale = max(mx, 1e-300)
    cond = np.stack([sm - left, sm - right, sm - thr]) / scale
    live = cond.min(0) > -1e-4                  # bins that are peaks, or miss by a near-tie only
    m = float(np.abs(cond[:, live]).min()) if live.any() else np.inf
    out = []
    for j in np.nonzero(acc)[0]:
        den = left[j] - 2 * sm[j] + right[j]
        b = j + 0.5 * (left[j] - right[j]) / den
        b = n + b if b < 0 else (b - n if b >= n else b)
        ang = 360.0 - (360.0 / n) * b
        if abs(ang - 360.0) < FLT_EPSILON:
            ang = 0.0
        out.append((j, ang, sm[j] / max(abs(den), 1e-300)))
    return out, m


def orientations(gauss, ref, envelope=False):
    """calcOrientationHist + the peak loop for the refined keypoints `ref` (refine()'s dict).  Returns KP_DTYPE-like
    float64 fields as a dict of arrays (one row per accepted peak) with `src` (the refined keypoint's index), `hmargin`
    (peak-decision margin of its histogram) and `gain` (peak height over the interpolation denominator: how much an
    error in the histogram moves the angle).  envelope=True adds `amin`, `amax`: the range of the angle of the same peak
    when any one sample whose bin position 0.1 * ori lies within 1e-4 of a rounding boundary goes to the other bin."""
    n = len(ref["x"])
    rows = {k: [] for k in ("src", "angle", "hmargin", "gain", "amin", "amax")}
    if not n:
        return {k: np.zeros(0) for k in rows}
    scl_octv = ref["size"] * 0.5 / 2.0 ** ref["o"]
    radius = cv_round(ORI_RADIUS * scl_octv)
    sig = ORI_SIG_FCTR * scl_octv
    hists = np.zeros((n, ORI_BINS))
    amb = {}
    for (o, layer, R) in set(zip(ref["o"].tolist(), ref["layer"].tolist(), radius.tolist())):
        sel = np.nonzero((ref["o"] == o) & (ref["layer"] == layer) & (radius == R))[0]
        img = np.asarray(gauss[o][layer], np.float64)
        ori, wm, valid = _ori_samples(img, ref["r"][sel], ref["c"][sel], R, sig[sel])
        pos = ori * (ORI_BINS / 360.0)
        b = cv_round(pos) % ORI_BINS
        b = np.where(b < 0, b + ORI_BINS, b)
        wm = np.where(valid, wm, 0.0)
        hists[sel] = np.stack([np.bincount(b[k], wm[k], ORI_BINS) for k in range(len(sel))])
        if envelope:
            near = valid & (np.abs(np.abs(pos - np.floor(pos)) - 0.5) < 1e-4)
            for k, s in zip(*np.nonzero(near)):
                p = pos[k, s]
                other = int(np.floor(p)) if b[k, s] == int(np.ceil(p)) % ORI_BINS else int(np.ceil(p))
                amb.setdefault(int(sel[k]), []).append((int(b[k, s]), other % ORI_BINS, wm[k, s]))
    for i in range(n):
        sm = _smooth(hists[i])
        peaks, m = _peaks(sm)
        variants = []
        for (fr, to, v) in amb.get(i, []):
            h2 = hists[i].copy()
            h2[fr] -= v
            h2[to] += v
            variants.append(_peaks(_smooth(h2))[0])
        for (j, ang, gain) in peaks:
            alts = [ang] + [a for var in variants for (jj, a, _) in var if jj == j]
            rows["src"].append(i); rows["angle"].append(ang); rows["hmargin"].append(m); rows["gain"].append(gain)
            rows["amin"].append(min(alts)); rows["amax"].append(max(alts))
    return {k: np.asarray(v) for k, v in rows.items()}


def keypoints_before_selection(gauss, cand):
    """refine + orientations as a KP_DTYPE array (what the refine kernel emits, before duplicate removal)."""
    ref, _ = refine(gauss, cand)
    ori = orientations(gauss, ref)
    src = ori["src"].astype(np.int64)
    out = np.zeros(len(src), KP_DTYPE)
    for f in ("x", "y", "size", "response", "octave"):
        out[f] = ref[f][src]
    out["angle"] = ori["angle"]
    return out


# ------------------------------------------------------------------ selection
def order(kps):
    """KeyPoint_LessThan: x asc, y asc, size desc, angle asc, response desc, octave desc (a stable index order)."""
    return np.lexsort((-kps["octave"].astype(np.int64), -kps["response"].astype(np.float64), kps["angle"],
                       -kps["size"].astype(np.float64), kps["y"], kps["x"]))


def select(kps, rows, size_ratio=0.0, nfeatures=N_FEATURES):
    """removeDuplicatedSorted, retainBest(nfeatures) keeping ties, the firstOctave = -1 rescale (x 0.5 and the octave
    word) and the reference's relative-size filter (size < float(rows * ratio)); float32 fields in and out, in
    KeyPoint_LessThan order."""
    k = np.asarray(kps, KP_DTYPE)[order(np.asarray(kps, KP_DTYPE))]
    if len(k) > 1:
        # equal (x, y, size, angle) are adjacent in this order: comparing with the previous entry is comparing with
        # the last one kept
        same = np.ones(len(k) - 1, bool)
        for f in ("x", "y", "size", "angle"):
            same &= k[f][1:] == k[f][:-1]
        k = k[np.concatenate([[True], ~same])]
    if nfeatures > 0 and len(k) > nfeatures:
        thr = np.sort(k["response"])[::-1][nfeatures - 1]
        k = k[k["response"] >= thr]
    k = k.copy()
    k["octave"] = (k["octave"] & ~255) | ((k["octave"] - 1) & 255)
    for f in ("x", "y", "size"):
        k[f] = k[f] * np.float32(0.5)
    if size_ratio > 0:
        k = k[k["size"] < np.float32(np.float32(rows) * np.float32(size_ratio))]
    return k


# ------------------------------------------------------------------ descriptors
def unpack_octave(word):
    word = np.asarray(word, np.int64)
    o = word & 255
    layer = (word >> 8) & 255
    o = np.where(o < 128, o, o - 256)
    return o, layer


def descriptors(gauss, kps):
    """calcDescriptors / calcSIFTDescriptor for final keypoints (input-image coordinates, octave word of
    firstOctave = -1): the real-valued 128-D descriptors before the saturate_cast to u8, float64 [n, 128]."""
    kps = np.asarray(kps)
    d, nb = DESCR_WIDTH, DESCR_BINS
    n = len(kps)
    out = np.zeros((n, d * d * nb))
    if not n:
        return out
    o, layer = unpack_octave(kps["octave"])
    scale = np.where(o >= 0, 1.0 / 2.0 ** np.maximum(o, 0), 2.0 ** np.maximum(-o, 0))
    size = kps["size"].astype(np.float64) * scale
    px, py = kps["x"].astype(np.float64) * scale, kps["y"].astype(np.float64) * scale
    ori = 360.0 - kps["angle"].astype(np.float64)
    ori = np.where(np.abs(ori - 360.0) < FLT_EPSILON, 0.0, ori)
    scl = size * 0.5
    hist_width = DESCR_SCL_FCTR * scl
    radius = cv_round(hist_width * math.sqrt(2.0) * (d + 1) * 0.5)
    oi = o + 1                                  # octave index in the pyramid (firstOctave = -1)
    hist_len = (d + 2) * (d + 2) * (nb + 2)
    for key in set(zip(oi.tolist(), layer.tolist(), radius.tolist())):
        oo, ll, R0 = key
        sel = np.nonzero((oi == oo) & (layer == ll) & (radius == R0))[0]
        img = np.asarray(gauss[oo][ll], np.float64)
        h, w = img.shape
        R = min(R0, int(math.sqrt(float(w) * w + float(h) * h)))
        dd = np.arange(-R, R + 1)
        ii, jj = np.meshgrid(dd, dd, indexing="ij")
        ii, jj = ii.ravel()[None], jj.ravel()[None]
        cos_t = np.cos(np.radians(ori[sel]))[:, None] / hist_width[sel][:, None]
        sin_t = np.sin(np.radians(ori[sel]))[:, None] / hist_width[sel][:, None]
        c_rot = jj * cos_t - ii * sin_t
        r_rot = jj * sin_t + ii * cos_t
        rbin = r_rot + d / 2 - 0.5
        cbin = c_rot + d / 2 - 0.5
        pty, ptx = cv_round(py[sel])[:, None], cv_round(px[sel])[:, None]
        r = pty + ii
        c = ptx + jj
        valid = (rbin > -1) & (rbin < d) & (cbin > -1) & (cbin < d) & (r > 0) & (r < h - 1) & (c > 0) & (c < w - 1)
        rc, cc = np.clip(r, 1, h - 2), np.clip(c, 1, w - 2)
        dx = img[rc, cc + 1] - img[rc, cc - 1]
        dy = img[rc - 1, cc] - img[rc + 1, cc]
        wgt = np.exp((c_rot * c_rot + r_rot * r_rot) * (-1.0 / (d * d * 0.5)))
        obin = (fast_atan2_deg(dy, dx) - ori[sel][:, None]) * (nb / 360.0)
        mag = np.where(valid, np.hypot(dx, dy) * wgt, 0.0)
        r0, c0, o0 = np.floor(rbin), np.floor(cbin), np.floor(obin)
        fr, fc, fo = rbin - r0, cbin - c0, obin - o0
        r0, c0, o0 = r0.astype(np.int64), c0.astype(np.int64), o0.astype(np.int64)
        o0 = np.where(o0 < 0, o0 + nb, o0)
        o0 = np.where(o0 >= nb, o0 - nb, o0)
        r0 = np.where(valid, r0, 0)
        c0 = np.where(valid, c0, 0)
        base = ((r0 + 1) * (d + 2) + c0 + 1) * (nb + 2) + o0
        K = len(sel)
        hist = np.zeros((K, hist_len))
        rowoff = (np.arange(K) * hist_len)[:, None]
        for dr in (0, 1):
            wr = fr if dr else 1 - fr
            for dc in (0, 1):
                wc = fc if dc else 1 - fc
                for do in (0, 1):
                    wo = fo if do else 1 - fo
                    idx = base + dr * (d + 2) * (nb + 2) + dc * (nb + 2) + do
                    hist += np.bincount((rowoff + idx).ravel(), (mag * wr * wc * wo).ravel(), K * hist_len).reshape(K, hist_len)
        hist = hist.reshape(K, d + 2, d + 2, nb + 2)
        core = hist[:, 1:d + 1, 1:d + 1, :].copy()
        core[..., 0] += core[..., nb]
        core[..., 1] += core[..., nb + 1]
        v = core[..., :nb].reshape(K, -1)
        thr = np.sqrt((v * v).sum(1)) * DESCR_MAG_THR
        v = np.minimum(v, thr[:, None])
        nrm = INT_DESCR_FCTR / np.maximum(np.sqrt((v * v).sum(1)), FLT_EPSILON)
        out[sel] = v * nrm[:, None]
    return out


def quantize(desc):
    """saturate_cast<uchar>: round half to even, clamp to 0..255."""
    return np.clip(np.rint(desc), 0, 255).astype(np.uint8)


# ------------------------------------------------------------------ the whole operation
def detect_and_compute(gray, size_ratio=0.0):
    """The float64 pipeline end to end: (keypoints KP_DTYPE in KeyPoint_LessThan order, real descriptors [n, 128])."""
    gray = np.asarray(gray, np.uint8)
    gauss = gaussian_pyramid(gray)
    pre = keypoints_before_selection(gauss, extrema(gauss))
    kps = select(pre, gray.shape[0], size_ratio)
    return kps, descriptors(gauss, kps)
