"""K11 (csrc/sift.cu) stage by stage against the float64 restatement tests/sift_ref.py, each stage conditioned on the
kernel's own input to it (vstab_b200.k_sift_stages reads every stage back): Gaussian pyramid, DoG candidates,
refinement + orientation, selection, descriptors; determinism of the output (order and bits) over plans and graph
replays; the 4096-pair fit (fit_kernel<kOrbMaxKp>) against cv2.estimateAffinePartial2D."""
import cv2
import numpy as np
import pytest
from scipy.spatial import cKDTree

import sift_ref as R
import vstab_b200 as vs
from conftest import render_clip

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -24


# ------------------------------------------------------------------ images
def _gray(frame, W=None, H=None):
    g = cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY)
    return g if W is None else cv2.resize(g, (W, H), interpolation=cv2.INTER_AREA)


def _lattice(W, H, period=8):
    """Identical blobs on a power-of-two grid: every octave's decimation keeps them identical, so interior keypoints
    tie exactly in response (and there are more than 2500 of them)."""
    yy, xx = np.mgrid[0:H, 0:W]
    d2 = (yy % period - period // 2) ** 2 + (xx % period - period // 2) ** 2
    return np.clip(50 + 150 * np.exp(-d2 / 4.5), 0, 255).astype(np.uint8)


def _border_blobs(W, H):
    """Blobs centred 6 px from the edges: their orientation and descriptor windows are clipped by the image."""
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    img = np.full((H, W), 90.0)
    for cy, cx, s in [(6, 6, 2.0), (H - 7, 6, 1.5), (6, W - 7, 2.5), (H - 7, W - 7, 1.8), (H // 2, 6, 2.2), (6, W // 2, 1.6)]:
        img += 120 * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * s * s))
    return img.astype(np.uint8)


IMAGES = {
    "render640": lambda t: _gray(render_clip(t, 1280, 720, 1, start=7)[0], 640, 360),
    "noise640": lambda t: np.random.default_rng(7).integers(0, 256, (360, 640), dtype=np.uint8),
    "render333": lambda t: _gray(render_clip(t, 333, 250, 1, start=3)[0]),
    "render97": lambda t: _gray(render_clip(t, 97, 61, 1, start=5)[0]),
    "render128": lambda t: _gray(render_clip(t, 128, 72, 1, start=9)[0]),
    "render1920": lambda t: _gray(render_clip(t, 1920, 1080, 1, start=11)[0]),
    "noise4k": lambda t: np.random.default_rng(8).integers(0, 256, (2160, 3840), dtype=np.uint8),
    "flat": lambda t: np.full((360, 640), 117, np.uint8),
    "lattice": lambda t: _lattice(640, 360),
    "border": lambda t: _border_blobs(128, 72),
}
SMALL = ["render640", "noise640", "render333", "render97", "render128", "lattice", "border"]
_cache = {}


def stages(texture, name, size_ratio=0.0):
    key = (name, size_ratio)
    if key not in _cache:
        gray = IMAGES[name](texture)
        _cache.clear()                                   # one image at a time: the 4K pyramid is 1 GB
        _cache[key] = (gray, vs.k_sift_stages(gray, size_ratio))
    return _cache[key]


def _bands(h, big):
    if not big:
        return [slice(0, h)]
    b = 48
    return [slice(0, b), slice(h // 2 - b // 2, h // 2 + b // 2), slice(h - b, h)]


def blur_bound(R_, vmax=255.0):
    """Two float32 passes of 2R + 1 taps: each output within (2R + 2) * 2^-24 * vmax of the exact sum of the float32
    products, plus one rounding of the taps' sum."""
    return (2 * (2 * R_ + 2) + 2) * EPS32 * vmax


# ------------------------------------------------------------------ pyramid
@pytest.mark.parametrize("name", SMALL + ["render1920", "noise4k"])
def test_pyramid_stages(texture, name):
    gray, S = stages(texture, name)
    big = gray.shape[0] > 1000
    assert [g.shape[1:] for g in S.pyr] == R.octave_shapes(*gray.shape)
    taps = R.all_taps()
    worst = {}
    for o, g in enumerate(S.pyr):
        h = g.shape[1]
        for i in range(R.N_GAUSS):
            if i == 0 and o > 0:                          # next octave: nearest decimation, bit-exact
                assert np.array_equal(g[0], R.next_octave_base(S.pyr[o - 1][R.N_LAYERS])), (o,)
                continue
            for rows in _bands(h, big and o == 0):
                want = R.blur64(R.upsample2x(gray), taps[0], rows) if i == 0 else R.blur64(g[i - 1], taps[i], rows)
                err = float(np.abs(g[i][rows] - want).max())
                rad = (len(taps[i]) - 1) // 2
                worst[rad] = max(worst.get(rad, 0.0), err / blur_bound(rad))
                assert err <= blur_bound(rad), (o, i, rows, err, blur_bound(rad))
    print(f"{name}: blur error / bound by radius " + ", ".join(f"R{r}: {v:.3f}" for r, v in sorted(worst.items())))


@pytest.mark.parametrize("name", ["render333", "render97", "render128", "border"])
def test_pyramid_end_to_end(texture, name):
    gray, S = stages(texture, name)
    ref = R.gaussian_pyramid(gray)
    err = max(float(np.abs(a - b).max()) for a, b in zip(S.pyr, ref))
    print(f"{name}: pyramid chained from u8, max |diff| {err:.2e}")
    assert err < 1e-2


# ------------------------------------------------------------------ DoG candidates
@pytest.mark.parametrize("name", SMALL + ["render1920", "noise4k", "flat"])
def test_extrema_exact(texture, name):
    gray, S = stages(texture, name)
    print(f"{name}: {S.n_cand} candidates (capacity {S.cand_cap}), {S.n_kp} keypoints before selection "
          f"(capacity {S.kp_cap}), {len(S.kps)} out")
    assert S.n_cand < S.cand_cap and S.n_kp < S.kp_cap            # nothing dropped at either list
    got = R.decode_candidates(S.cand)
    if name == "noise4k":
        # octave 0 at 4K is 7680 x 4320 x 5 DoG levels: compared on row bands at the top, middle and bottom, the other
        # octaves whole
        g0 = S.pyr[0]
        h = g0.shape[1]
        for a, b in [(R.BORDER, R.BORDER + 48), (h // 2 - 24, h // 2 + 24), (h - R.BORDER - 48, h - R.BORDER)]:
            band = got[(got[:, 0] == 0) & (got[:, 2] >= a) & (got[:, 2] < b)]
            assert np.array_equal(band, _extrema_rows(g0, a, b)), (a, b)
        got = got[got[:, 0] > 0]
        want = R.extrema([np.zeros((6, 1, 1))] + S.pyr[1:])
    else:
        want = R.extrema(S.pyr)
    assert got.shape == want.shape and np.array_equal(got, want)
    if name == "flat":
        assert S.n_cand == 0 and len(S.kps) == 0


def _extrema_rows(g, a, b):
    """R.extrema's rows a .. b - 1 of octave 0 (BORDER <= a < b <= h - BORDER), from rows a - 1 .. b of its DoG."""
    sub = np.asarray(g[:, a - 1:b + 1], np.float32)
    D = sub[1:] - sub[:-1]
    w = D.shape[2]
    from scipy import ndimage
    mx = ndimage.maximum_filter(D, size=3, mode="nearest")
    mn = ndimage.minimum_filter(D, size=3, mode="nearest")
    out = []
    for layer in range(1, R.N_LAYERS + 1):
        v = D[layer, 1:-1, R.BORDER:w - R.BORDER]
        hit = (np.abs(v) > R.DOG_THRESHOLD) & (((v > 0) & (v >= mx[layer, 1:-1, R.BORDER:w - R.BORDER])) |
                                               ((v < 0) & (v <= mn[layer, 1:-1, R.BORDER:w - R.BORDER])))
        r, c = np.nonzero(hit)
        out.append(np.stack([np.zeros_like(r), np.full_like(r, layer), r + a, c + R.BORDER], 1))
    rows = np.concatenate(out).astype(np.int64)
    return rows[np.lexsort(rows.T[::-1])]


def _planted_pyramid(rows, cols, seed):
    """A Gaussian pyramid of the geometry of a rows x cols input whose DoG stays within +-0.3 except at planted 3x3x3
    extrema of exactly +-1.0 (the contrast threshold: not candidates) and +-(1 + 2^-23) (candidates)."""
    rng = np.random.default_rng(seed)
    pyr, planted = [], []
    for o, (h, w) in enumerate(R.octave_shapes(rows, cols)):
        g = np.empty((6, h, w), np.float32)
        g[0] = rng.uniform(0.0, 0.3, (h, w))
        for i in range(1, 6):
            g[i] = g[i - 1] + rng.uniform(-0.1, 0.1, (h, w)).astype(np.float32)
        if h > 2 * R.BORDER + 8 and w > 2 * R.BORDER + 8:
            k = 0
            for r in range(R.BORDER + 2, h - R.BORDER - 2, 7):
                for c in range(R.BORDER + 2 + (r % 3), w - R.BORDER - 2, 9):
                    layer = 1 + k % 3
                    lo, hi = [(np.float32(0.5), np.float32(1.5)), (np.float32(0.5), np.float32(1.5) + np.float32(2 ** -23)),
                              (np.float32(1.5), np.float32(0.5)), (np.float32(1.5) + np.float32(2 ** -23), np.float32(0.5))][k % 4]
                    g[layer, r, c], g[layer + 1, r, c] = lo, hi
                    planted.append((o, layer, r, c, k % 4))
                    k += 1
        pyr.append(g)
    return pyr, planted


@pytest.mark.parametrize("rows,cols", [(90, 121), (64, 128), (61, 97)])
def test_extrema_at_threshold(rows, cols):
    """|DoG| > threshold is strict: an extremum of exactly 1.0 is not a candidate, one of 1 + 2^-23 is.  Both load paths
    of the tile kernel see planted values: octave widths that are multiples of 4 (float4 rows) and that are not."""
    pyr, planted = _planted_pyramid(rows, cols, rows + cols)
    want = R.extrema(pyr)
    wset = set(map(tuple, want.tolist()))
    n_exact = 0
    for (o, layer, r, c, kind) in planted:
        D = R.dog(pyr[o])
        v = D[layer, r, c]
        nb = D[layer - 1:layer + 2, r - 1:r + 2, c - 1:c + 2]
        is_ext = v == (nb.max() if v > 0 else nb.min())
        assert is_ext and abs(v) in (np.float32(1.0), np.float32(1.0) + np.float32(2 ** -23))
        assert ((o, layer, r, c) in wset) == (kind % 2 == 1)
        n_exact += kind % 2 == 0
    assert n_exact >= 8
    cand, n, cap = vs.k_sift_extrema(pyr, rows, cols)
    assert n < cap
    assert np.array_equal(R.decode_candidates(cand), want)


# ------------------------------------------------------------------ refinement + orientation
def _group(kp):
    return (kp["octave"] & 0xFFFF).astype(np.int64)                 # octave index + layer << 8


@pytest.mark.parametrize("name", SMALL + ["render1920"])
def test_refine_orientation(texture, name):
    gray, S = stages(texture, name)
    cand = R.decode_candidates(S.cand)
    ref, rej = R.refine(S.pyr, cand)
    ori = R.orientations(S.pyr, ref, envelope=True)
    src = ori["src"].astype(np.int64)
    rm = ref["margin"][src]
    fragile = (rm < 1e-5) | (ori["hmargin"] < 1e-5)
    ker = S.kps_pre
    assert len(ker) == S.n_kp
    o_ref = ref["o"][src]
    scale = 2.0 ** o_ref
    rgroup = (ref["octave"][src] & 0xFFFF)
    kgroup = _group(ker)
    used = np.zeros(len(ker), bool)
    unmatched_ref, dpos, dang, drel = [], 0.0, 0.0, 0.0
    trees = {g: (np.nonzero(kgroup == g)[0], cKDTree(np.stack([ker["x"][kgroup == g], ker["y"][kgroup == g]], 1)))
             for g in np.unique(kgroup)}
    for i in range(len(src)):
        g = int(rgroup[i])
        if g not in trees:
            unmatched_ref.append(i)
            continue
        idxs, tree = trees[g]
        # refinement values: the position tolerance scales with the Hessian's conditioning at that octave
        kap = float(ref["kappa"][src[i]])
        tol = max(1e-4, 1e-4 * kap) * scale[i]
        best = None
        for j in tree.query_ball_point([ref["x"][src[i]], ref["y"][src[i]]], tol):
            k = idxs[j]
            if used[k]:
                continue
            a = float(ker["angle"][k])
            ta = 1e-3
            lo, hi = ori["amin"][i] - ta, ori["amax"][i] + ta
            ok = lo <= a <= hi or lo <= a - 360 <= hi or lo <= a + 360 <= hi
            if ok:
                best = k
                break
        if best is None:
            unmatched_ref.append(i)
            continue
        used[best] = True
        dpos = max(dpos, max(abs(ker["x"][best] - ref["x"][src[i]]), abs(ker["y"][best] - ref["y"][src[i]])) / scale[i])
        dang = max(dang, abs((float(ker["angle"][best]) - ori["angle"][i] + 180) % 360 - 180))
        for f in ("size", "response"):
            rel = abs(float(ker[f][best]) - ref[f][src[i]]) / abs(ref[f][src[i]])
            drel = max(drel, rel)
            assert rel < 1e-5 + 1e-7 * kap, (name, f, rel)
        assert int(ker["octave"][best]) == int(ref["octave"][src[i]]) or fragile[i], (name, i)
    bad_ref = [i for i in unmatched_ref if not fragile[i]]
    # a keypoint only the kernel has must come from a decision the reference shows as a near-tie
    rej_frag = rej["margin"] < 1e-5
    extra = np.nonzero(~used)[0]
    bad_ker = []
    for k in extra:
        o = int(ker["octave"][k] & 255)
        x, y = float(ker["x"][k]), float(ker["y"][k])
        near_ref = fragile & (o_ref == o) & (np.abs(ref["x"][src] - x) <= 2 * 2.0 ** o) & (np.abs(ref["y"][src] - y) <= 2 * 2.0 ** o)
        near_rej = rej_frag & (rej["o"] == o) & (np.abs(rej["c"] * 2.0 ** o - x) <= 6 * 2.0 ** o) & \
            (np.abs(rej["r"] * 2.0 ** o - y) <= 6 * 2.0 ** o)
        if not (near_ref.any() or near_rej.any()):
            bad_ker.append(k)
    print(f"{name}: {len(ker)} kernel / {len(src)} reference keypoints before selection, {int(fragile.sum())} near-ties, "
          f"{len(unmatched_ref)} reference-only, {len(extra)} kernel-only; max position diff {dpos:.2e} px (octave "
          f"units), max angle diff {dang:.2e} deg, max size / response rel diff {drel:.2e}")
    assert not bad_ref and not bad_ker, (name, bad_ref[:5], bad_ker[:5])


# ------------------------------------------------------------------ selection
@pytest.mark.parametrize("name,ratio", [(n, 0.0) for n in SMALL + ["render1920", "noise4k", "flat"]] + [("render640", 0.05)])
def test_selection_exact(texture, name, ratio):
    gray, S = stages(texture, name, ratio)
    assert S.n_kp <= S.kp_cap
    want = R.select(S.kps_pre, gray.shape[0], ratio)
    assert S.n_sel == len(want)
    if name == "lattice":
        # every blob of the lattice gives the same responses: retainBest(2500) keeps all the ties, more than the 4096
        # rows of the output, which keeps the first 4096 in order
        assert len(want) > 4096
    want = want[:4096]
    got = np.zeros(len(S.kps), R.KP_DTYPE)
    for j, f in enumerate(("x", "y", "size", "angle", "response")):
        got[f] = S.kps[:, j]
    got["octave"] = S.kps[:, 5].astype(np.int64)
    assert len(got) == len(want), (len(got), len(want))
    assert got.tobytes() == want.tobytes()                          # values, bits and order
    if name == "lattice":
        thr = np.sort(R.select(S.kps_pre, gray.shape[0], nfeatures=0)["response"])[::-1]
        print(f"lattice: {len(thr)} after duplicates, {len(got)} kept, ties at the threshold "
              f"{int((thr == thr[2499]).sum()) if len(thr) > 2500 else 0}")


# ------------------------------------------------------------------ descriptors
DESC_DELTA = 0.06


@pytest.mark.parametrize("name", SMALL + ["render1920", "noise4k"])
def test_descriptors(texture, name):
    gray, S = stages(texture, name)
    kps = np.zeros(len(S.kps), R.KP_DTYPE)
    for j, f in enumerate(("x", "y", "size", "angle", "response")):
        kps[f] = S.kps[:, j]
    kps["octave"] = S.kps[:, 5].astype(np.int64)
    ref = np.clip(R.descriptors(S.pyr, kps), 0, 255)
    err = np.abs(S.desc.astype(np.float64) - ref)
    worst = float(err.max()) if err.size else 0.0
    print(f"{name}: {len(kps)} descriptors, max |q - r| {worst:.4f} (bound 0.5 + {DESC_DELTA})")
    assert worst <= 0.5 + DESC_DELTA


# ------------------------------------------------------------------ determinism
def test_output_deterministic_over_plans_and_graph_replays(texture):
    for name in ("noise640", "render640", "lattice"):
        gray = IMAGES[name](texture)
        runs = [vs.k_sift_stages(gray, calls=c) for c in (1, 3, 1, 2)]
        for r in runs[1:]:
            assert r.kps.tobytes() == runs[0].kps.tobytes(), name
            assert np.array_equal(r.desc, runs[0].desc), name
            assert np.array_equal(R.decode_candidates(r.cand), R.decode_candidates(runs[0].cand))
        assert np.array_equal(runs[0].kps, vs.k_sift(gray)[0])


def test_sift_lock_streaming_deterministic(texture):
    frames = render_clip(texture, 640, 360, 10, start=2)
    outs = []
    for _ in range(2):
        st = vs.Stabilizer(3, 2, 360, device=0)
        st.set_stabilization_mode(vs.SIFT_FULL_LOCK)
        o = [st.stabilize_frame(f).copy() for f in frames]
        st.close()
        outs.append(o)
    for a, b in zip(*outs):
        assert np.array_equal(a, b)


# ------------------------------------------------------------------ fit_kernel<kOrbMaxKp>
@pytest.mark.parametrize("n", [10, 500, 1300, 1301, 2500, 4096])
def test_fit_large_matches_opencv_ransac(n):
    corners = np.array([[0, 0, 1], [640, 0, 1], [0, 360, 1], [640, 360, 1]], float).T
    rng = np.random.default_rng(n)
    for frac in (0.0, 0.05, 0.3, 0.6):
        p = np.stack([rng.uniform(0, 640, n), rng.uniform(0, 360, n)], 1).astype(np.float32)
        th = rng.uniform(-0.03, 0.03)
        A = (1.0 + rng.uniform(-0.01, 0.01)) * np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
        q = (p @ A.T + rng.uniform(-8, 8, 2) + rng.normal(0, 0.5, (n, 2))).astype(np.float32)
        bad = rng.random(n) < frac
        q[bad] += rng.uniform(-60, 60, (int(bad.sum()), 2)).astype(np.float32)
        st = (rng.random(n) > 0.03).astype(np.uint8)
        keep = st == 1
        Mr, inl = cv2.estimateAffinePartial2D(p[keep].reshape(-1, 1, 2), q[keep].reshape(-1, 1, 2), method=cv2.RANSAC,
                                              ransacReprojThreshold=5.0)
        M, T, cnt = vs.k_fit_large(p, q, st, 640, 360, thresh=5.0)
        if int(keep.sum()) < 10:
            assert np.array_equal(T, np.eye(3)) and cnt == (int(keep.sum()), 0)
            continue
        assert cnt == (int(keep.sum()), int(inl.sum())), (n, frac)
        assert np.abs(M @ corners - Mr @ corners).max() < 1e-6, (n, frac)
        if n <= 1300:
            M2, T2, cnt2 = vs.k_fit(p, q, st, 640, 360, thresh=5.0)
            assert cnt2 == cnt and np.array_equal(M2, M) and np.array_equal(T2, T)
