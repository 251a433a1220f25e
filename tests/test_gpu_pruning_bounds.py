"""Exactness of the chunk pruning on inputs built to sit on its bounds.

A pruning group skips a target chunk when the chunk's circle lies beyond the group's `reach`: the
group's moved circle (radius = stretch(T) x the untransformed radius) plus the largest upper bound of
its points, plus rounding terms.  Every case below places the true nearest neighbour of one point in
a chunk just outside what an unsound bound would reach, and holds every engine variant to the same
verdict:

* the first pass's correspondences equal an fp64 brute force in numpy (the reference's rounding,
  (dx*dx) + (dy*dy), and np.argmin's first index);
* multi-pass runs give the pass counts and correspondences of the C oracle (not its transforms to
  1e-9: a 2 mm segment 1e5 m from the origin leaves the fitted rotation to rounding, in the oracle
  as in the kernel);
* pruned, exhaustive, large-scan and cluster runs give the same bits.

Families:
  A  non-rigid initial guesses R(theta) diag(1 + delta, 1) R(phi) (optionally reflected) for which an
     fp32 evaluation of the largest singular value cancels catastrophically, plus degenerate linear
     parts (shear, reflection, rank 1, zero, scale 1e3 / 1e-3, near-singular);
  B  rigid transforms with the nearest neighbour a few fp32 ulps nearer than the best target the
     first-pass upper bound sees, over coordinate offsets 0 ... 1e7 and group radii 1e-3 ... 1e3;
  C  the coordinate and initial-guess magnitude contract of include/icpb.h: inputs beyond it are
     rejected with ValueError (a list of scans while the library packs it, everything else before any
     launch), inputs just inside it still match the oracle.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MAX_COORD = 1e10          # ICPB_MAX_COORD
MAX_LINEAR = 1e3          # ICPB_MAX_GUESS_LINEAR
MAX_SHIFT = 1e12          # ICPB_MAX_GUESS_SHIFT
REPEAT = 16               # copies of a 16-point group: 256 source points = 4 tiles of 64


@pytest.fixture(scope="module")
def gicp():
    from icp_slam_b200 import icp as m
    return m


@pytest.fixture(scope="module")
def c_oracle():
    from oracle import c_oracle as m
    m.build()
    return m


@pytest.fixture(scope="module")
def eng(gicp):
    e = gicp.IcpEngine()
    yield e
    e.close()


def hom(s):
    return np.c_[s, np.ones(len(s))]


def rot(t):
    c, s = np.cos(t), np.sin(t)
    return np.array([[c, -s], [s, c]])


def affine(A, t=(0.0, 0.0)):
    T = np.eye(3)
    T[:2, :2] = A
    T[:2, 2] = t
    return T


# ---- a float32 copy of the stretch bound the alignment kernel used before its cancellation-free form ----
# (as compiled for sm_100a: the sums of products contracted into FFMA).  It only selects inputs.
def _fma32(x, y, z):
    return (x.astype(np.float64) * y.astype(np.float64) + z.astype(np.float64)).astype(np.float32)


def fp32_stretch_estimate(M):
    f = np.float32
    a, b, c, d = (M[:, 0, 0].astype(f), M[:, 0, 1].astype(f), M[:, 1, 0].astype(f), M[:, 1, 1].astype(f))
    f2 = _fma32(a, a, b * b)
    f2 = _fma32(c, c, f2)
    det = _fma32(a, d, -(b * c))
    f2 = _fma32(d, d, f2)
    disc = np.maximum(_fma32(f2, f2, det * (det * f(-4.0))), f(0.0))
    s = np.sqrt(f(0.5) * (f2 + np.sqrt(disc)))
    return _fma32(s, np.full_like(s, f(1.00002)), np.full_like(s, f(1e-30))).astype(np.float64)


def near_conformal_matrices(n, seed):
    """The n matrices R(theta) diag(1 + delta, 1) R(phi) [diag(1, -1)] whose fp32 stretch estimate
    falls furthest below the true largest singular value (all by more than 2.1e-4 relative: the
    multiplicative slack of the chunk test)."""
    rng = np.random.default_rng(seed)
    N = 60000
    th, ph = rng.uniform(-np.pi, np.pi, N), rng.uniform(-np.pi, np.pi, N)
    de = rng.uniform(4e-4, 8e-4, N)
    c1, s1, c2, s2 = np.cos(th), np.sin(th), np.cos(ph), np.sin(ph)
    R1 = np.stack([np.stack([c1, -s1], -1), np.stack([s1, c1], -1)], -2)
    R2 = np.stack([np.stack([c2, -s2], -1), np.stack([s2, c2], -1)], -2)
    D = np.zeros((N, 2, 2))
    D[:, 0, 0], D[:, 1, 1] = 1.0 + de, 1.0
    M = R1 @ D @ R2
    flip = rng.random(N) < 0.5
    M[flip] = M[flip] @ np.diag([1.0, -1.0])
    under = 1.0 - fp32_stretch_estimate(M) / np.linalg.svd(M, compute_uv=False)[:, 0]
    keep = np.argsort(-under)[:n]
    assert under[keep].min() > 2.1e-4
    return M[keep]


def boundary_pair(T, centre, radius, d, margin, n_star=16):
    """Source: 16 points on a segment of half-length `radius` around `centre`, repeated REPEAT times
    (every group of every tile is the same group).  Targets, one chunk each:
      filler beyond point 0 | decoys: moved point k + 0.3 d across the segment, the end
      point's decoy at d + margin | filler | n_star copies of T* = moved end point + d along the segment.
    With the decoy chunk the nearest chunk to the group centre, the end point's first-pass upper bound
    is d + margin, while its nearest neighbour T* is d away, at distance radius + d from the moved
    centre: a chunk that only a sound stretch bound reaches.  The direction is the image's largest
    singular direction, so the moved segment has half-length stretch x radius."""
    A, t = T[:2, :2], T[:2, 2]
    U, S, Vt = np.linalg.svd(A)
    u1, u2, v1 = U[:, 0], U[:, 1], Vt[0]
    if S[0] == 0.0:
        u1, u2, v1 = np.array([1.0, 0.0]), np.array([0.0, 1.0]), np.array([1.0, 0.0])
    p = centre + np.linspace(-radius, radius, 16)[:, None] * v1
    mp = p @ A.T + t
    mc = centre @ A.T + t
    far = np.tile(mc - (S[0] * radius + 4.0 * (d + margin)) * u1, (16, 1))
    dec = mp + 0.3 * d * u2
    dec[15] = mp[15] + (d + margin) * u2
    star = np.tile(mp[15] + d * u1, (n_star, 1))
    return np.tile(p, (REPEAT, 1)), np.concatenate([far, dec, far, star])


def brute_force(src, dst, T):
    """First-pass correspondences in fp64 with the reference's rounding and np.argmin's first index."""
    P = src @ T[:2, :2].T + T[:2, 2]
    dx = dst[None, :, 0] - P[:, None, 0]
    dy = dst[None, :, 1] - P[:, None, 1]
    return np.argmin(dx * dx + dy * dy, axis=1)


VARIANTS = (("pruned", None, False), ("exhaustive", None, True), ("large", ("large", 1), False),
            ("cluster2", ("cluster", 2), False), ("cluster4", ("cluster", 4), False))
RESET = {"large": -1, "cluster": -1}


def run_variants(e, scans, pairs, init, **kw):
    """Every engine variant on the same resident table; returns {name: BatchResult}."""
    e.set_scans(scans)
    out = {}
    for name, tune, exhaustive in VARIANTS:
        if tune:
            e.set_tuning(*tune)
        try:
            out[name] = e.run(pairs, init, return_correspondences=True, exhaustive=exhaustive, **kw)
        finally:
            if tune:
                e.set_tuning(tune[0], RESET[tune[0]])
    ref = out["pruned"]
    for name, r in out.items():
        for field in ("T", "error", "iters", "correspondences"):
            np.testing.assert_array_equal(getattr(r, field), getattr(ref, field), err_msg=f"{name}: {field}")
    return ref


def check_family(gicp, c_oracle, e, scans, pairs, init, iteration_every=1):
    """The common verdict for a batch of pairs (pair b = scans 2b -> 2b + 1)."""
    # first pass: every variant, against the fp64 brute force
    first = run_variants(e, scans, pairs, init, epsilon=np.inf, max_iters=0)
    assert np.all(first.iters == 1)
    for b, (s, d) in enumerate(pairs):
        want = brute_force(scans[s], scans[d], init[b])
        np.testing.assert_array_equal(first.correspondences[b, :len(want)], want, err_msg=f"pair {b}")
        if b % iteration_every == 0:
            _, corr, _ = gicp.icp_iteration(hom(scans[s]), hom(scans[d]), init[b].copy())
            np.testing.assert_array_equal(corr, want, err_msg=f"icp_iteration, pair {b}")
    # later passes (the upper bound is the previous match): every variant, against the C oracle
    kw = dict(epsilon=0.0, stopping_thresh=0.0, max_iters=5)
    multi = run_variants(e, scans, pairs, init, **kw)
    batch = gicp.icp_batch(scans, pairs, init, return_correspondences=True, **kw)
    np.testing.assert_array_equal(batch.T, multi.T)
    np.testing.assert_array_equal(batch.correspondences, multi.correspondences)
    for b, (s, d) in enumerate(pairs):
        T, err, passes, corr = c_oracle.icp_pair(scans[s], scans[d], init[b], **kw)
        assert multi.iters[b] == passes, b
        np.testing.assert_array_equal(multi.correspondences[b, :len(corr)], corr, err_msg=f"pair {b}")


# ------------------------------------------------------------------------------------- family A
def test_family_a_near_conformal_guesses(gicp, c_oracle, eng):
    """A few hundred non-rigid guesses whose fp32 stretch estimate undershoots by more than the
    chunk test's slack; one 1,000 m pair per matrix, all in one batch."""
    Ms = near_conformal_matrices(256, seed=4242)
    rng = np.random.default_rng(4243)
    scans, init = [], []
    for M in Ms:
        t = rng.uniform(-5.0, 5.0, 2)
        T = affine(M, t)
        src, dst = boundary_pair(T, np.zeros(2), 1000.0 / np.linalg.norm(M, 2), 0.5, 0.005)
        scans += [src, dst]
        init.append(T)
    pairs = np.arange(2 * len(Ms), dtype=np.int32).reshape(-1, 2)
    check_family(gicp, c_oracle, eng, scans, pairs, np.stack(init), iteration_every=16)


def _degenerate_cases():
    th = 0.37
    return {
        "shear": np.array([[1.0, 0.8], [0.0, 1.0]]),
        "reflection": rot(th) @ np.diag([1.0, -1.0]),
        "rank1": np.outer([np.cos(th), np.sin(th)], [0.6, -0.8]) * 1.3,
        "zero": np.zeros((2, 2)),
        "scale1e3": 1e3 * rot(th),
        "scale1e-3": 1e-3 * rot(-th),
        "near_singular": rot(th) @ np.diag([1.0, 1e-8]) @ rot(0.2),
    }


def test_family_a_degenerate_linear_parts(gicp, c_oracle, eng):
    """Shear, reflection (det < 0), rank 1, a zero linear part (every point maps to the translation: a
    single matched target, the identity-rotation fit), uniform scale 1e3 and 1e-3, det ~ 1e-8: as
    boundary pairs and as plain scan-like pairs."""
    rng = np.random.default_rng(77)
    scans, init = [], []
    for name, A in _degenerate_cases().items():
        T = affine(A, rng.uniform(-3.0, 3.0, 2))
        span = np.linalg.norm(A, 2)
        src, dst = boundary_pair(T, rng.uniform(-2.0, 2.0, 2), 10.0 / span if span > 0.0 else 10.0, 0.5, 0.005)
        scans += [src, dst]
        init.append(T)
        # a plain pair: a noisy polyline and its image under T, with n2 not a multiple of 16
        u = np.sort(rng.uniform(0.0, 20.0, 300))
        src = np.stack((u, np.sin(u) + 0.3 * np.floor(u)), axis=1)
        dst = (src @ A.T + T[:2, 2])[rng.permutation(300)[:203]] + rng.normal(0.0, 1e-3, (203, 2))
        scans += [src, dst]
        init.append(T)
    pairs = np.arange(len(scans), dtype=np.int32).reshape(-1, 2)
    check_family(gicp, c_oracle, eng, scans, pairs, np.stack(init))


# ------------------------------------------------------------------------------------- family B
OFFSETS = (0.0, 1e3, 1e5, 1e6, 1e7)
RADII = (1e-3, 1e-1, 10.0, 1e3)


def test_family_b_rigid_reach_boundary(gicp, c_oracle, eng):
    """Rigid transforms; T* is the end point's nearest neighbour by a few fp32 ulps of the coordinate
    magnitude and sits at distance radius + d from the moved group centre.  n2 = 53: the T* chunk is
    partial, so padding targets share it.  This pins the absolute terms of the bound (the rounding of
    centres and differences, the tolerance of the filter, the radius term of the group circle)."""
    rng = np.random.default_rng(99)
    scans, init = [], []
    for off in OFFSETS:
        for r in RADII:
            T = affine(rot(rng.uniform(-np.pi, np.pi)), rng.uniform(-1.0, 1.0, 2) * r)
            centre = np.array([off, -0.6 * off])
            mag = 1.2 * abs(off) + 3.0 * r + 1.0
            ulp = float(np.spacing(np.float32(mag)))
            d = 0.05 * r
            src, dst = boundary_pair(T, centre, r, d, 3.0 * ulp, n_star=5)
            assert len(dst) % 16 != 0
            scans += [src, dst]
            init.append(T)
    pairs = np.arange(len(scans), dtype=np.int32).reshape(-1, 2)
    check_family(gicp, c_oracle, eng, scans, pairs, np.stack(init))


# ------------------------------------------------------------------------------------- family C
def _plain_scans(rng, offset, n=300):
    u = np.sort(rng.uniform(0.0, 60.0, n))
    dst = np.stack((u, 3.0 * np.sin(u / 4.0) + 0.2 * np.floor(u)), axis=1)
    src = (dst[rng.permutation(n)[:250]] - [0.05, -0.03]) @ rot(0.02) + rng.normal(0.0, 0.01, (250, 2))
    return [src + offset, dst + offset]


def test_family_c_out_of_range_inputs_are_rejected(gicp, eng):
    """Coordinates beyond ICPB_MAX_COORD (and NaN) and initial guesses beyond the guess bounds raise
    ValueError from every entry point -- before any launch, except for a list of scans, which the
    library checks while it packs the upload -- and the handle keeps working."""
    rng = np.random.default_rng(5)
    good = _plain_scans(rng, np.zeros(2))
    pairs = np.array([[0, 1]], dtype=np.int32)
    want = eng.align(good, pairs, None, epsilon=0.0, max_iters=5)
    for bad_value in (1.0001 * MAX_COORD, -2.0 * MAX_COORD, 1e15, np.nan):
        bad = [good[0].copy(), good[1]]
        bad[0][17, 1] = bad_value
        launches = eng.launch_count
        with pytest.raises(ValueError):
            gicp.icp(hom(bad[0]), hom(bad[1]))
        with pytest.raises(ValueError):
            gicp.icp(hom(bad[1]), hom(bad[0]))
        with pytest.raises(ValueError):
            gicp.icp_iteration(hom(bad[0]), hom(bad[1]), np.eye(3))
        with pytest.raises(ValueError):
            gicp.ScanTable(bad)
        with pytest.raises(ValueError):                      # packed-table path (upload + run)
            gicp.icp_batch(bad, pairs, return_correspondences=True)
        with pytest.raises(ValueError):
            eng.set_scans(bad)
        assert eng.launch_count == launches
        with pytest.raises(ValueError):                      # list of arrays: checked while packing
            gicp.icp_batch(bad, pairs)
        with pytest.raises(ValueError):
            eng.align(bad, pairs, None)
        again = eng.align(good, pairs, None, epsilon=0.0, max_iters=5)
        np.testing.assert_array_equal(again.T, want.T)
    for T in (affine(np.eye(2), (1.0001 * MAX_SHIFT, 0.0)), affine(np.diag([1.0, -1.0001 * MAX_LINEAR])),
              affine(np.array([[1.0, np.inf], [0.0, 1.0]]))):
        launches = eng.launch_count
        with pytest.raises(ValueError):
            gicp.icp(hom(good[0]), hom(good[1]), T)
        with pytest.raises(ValueError):
            gicp.icp_batch(good, pairs, T[None])
        with pytest.raises(ValueError):
            gicp.icp_batch(good, pairs, T[None], return_correspondences=True)
        with pytest.raises(ValueError):
            eng.align(good, pairs, T[None])
        assert eng.launch_count == launches
        np.testing.assert_array_equal(eng.run(pairs, None, epsilon=0.0, max_iters=5).T, want.T)


def replay_passes(gicp, c_oracle, src, dst, starts):
    """Every pass replayed from the kernel's own starting transform: its correspondences equal the fp64
    brute force and the oracle's from the same start (the fit arithmetic of kernel and oracle may
    differ in the last bits, which far from the origin can move later passes apart)."""
    corr = None
    for T0 in starts:
        _, corr, _ = gicp.icp_iteration(hom(src), hom(dst), T0.copy())
        np.testing.assert_array_equal(corr, brute_force(src, dst, T0))
        _, _, _, want = c_oracle.icp_pair(src, dst, T0, epsilon=np.inf, max_iters=0)
        np.testing.assert_array_equal(corr, want)
    return corr


def test_family_c_just_inside_the_bound(gicp, c_oracle, eng):
    """Scans whose largest coordinate is just under ICPB_MAX_COORD (fp32 cannot tell points apart
    there; the fp64 decision does all the work) and the largest guesses allowed: every pass is exact,
    through the packed and the list-of-arrays paths and every engine variant."""
    rng = np.random.default_rng(6)
    scans = []
    for off in (np.array([MAX_COORD - 100.0, -(MAX_COORD - 100.0)]), np.array([0.5 * MAX_COORD, 7.0])):
        scans += _plain_scans(rng, off)
    pairs = np.array([[0, 1], [2, 3]], dtype=np.int32)
    init = np.stack([affine(np.eye(2), (0.02, -0.01)), affine(np.eye(2), (0.02, -0.01))])
    assert np.abs(np.concatenate(scans)).max() <= MAX_COORD
    kw = dict(epsilon=0.0, stopping_thresh=0.0, max_iters=8)
    res = run_variants(eng, scans, pairs, init, **kw)
    listed = eng.align(scans, pairs, init, **kw)
    np.testing.assert_array_equal(listed.T, res.T)
    np.testing.assert_array_equal(listed.iters, res.iters)
    hist = gicp.icp_batch(scans, pairs, init, return_history=True, **kw)
    np.testing.assert_array_equal(hist.T, res.T)
    for b, (s, d) in enumerate(pairs):
        _, _, passes, _ = c_oracle.icp_pair(scans[s], scans[d], init[b], **kw)
        assert res.iters[b] == passes
        starts = [init[b]] + list(hist.history[b, :passes - 1])
        last = replay_passes(gicp, c_oracle, scans[s], scans[d], starts)
        np.testing.assert_array_equal(res.correspondences[b, :len(last)], last)
    # the largest guesses allowed: a translation of MAX_SHIFT and linear entries of MAX_LINEAR
    small = _plain_scans(rng, np.zeros(2))
    for T in (affine(np.eye(2), (MAX_SHIFT, -MAX_SHIFT)), affine(np.diag([MAX_LINEAR, -MAX_LINEAR]), (3.0, 4.0))):
        first = run_variants(eng, small, np.array([[0, 1]], dtype=np.int32), T[None], epsilon=np.inf, max_iters=0)
        last = replay_passes(gicp, c_oracle, small[0], small[1], [T])
        np.testing.assert_array_equal(first.correspondences[0, :len(last)], last)
