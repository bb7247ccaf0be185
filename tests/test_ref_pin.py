"""Pins the restated oracles against the reference's OWN code.

oracle/_ref/liblexp_ref.so is the reference's CostVolumeEnergy / NaiveStereoEnergy / FastGuidedImageFilter<double> /
LayerManager / RandomProposer compiled from the reference's headers (oracle/build_ref.py) over the cv:: layer of
oracle/cvshim/.  Two kinds of checks:
  * the cv:: layer's primitives against the real OpenCV (cv2): box filter, warpAffine, getAffineTransform, cvtColor, Sobel;
  * the numpy oracle and the C oracle against the compiled reference: costs, masks, statistics, cell geometry, random labels.
CPU only.  What the compiled reference returned for these very inputs is stored in tests/golden/ref_pin.npz (tests/ref_golden.py),
so the comparisons run without the reference's sources."""
import numpy as np
import pytest

from oracle import build_ref
from oracle import lexp_oracle as O
from lexp_testlib import make_scene
import ref_golden

R = ref_golden.reference()
thin, kept = ref_golden.thin, ref_golden.kept


@pytest.fixture(scope="module", autouse=True)
def _minted_golden():
    yield
    if ref_golden.MINT:
        ref_golden.store().save()


@pytest.fixture(autouse=True)
def _reference_calls_of(request):
    """The stored reference results are found by the test's name and the order of its calls."""
    st = ref_golden.store()
    st.test, st.n = request.node.name, 0
    yield
    st.test = None

INVALID = np.float32(O.COST_FOR_INVALID)


# ------------------------------------------------------------------------------------------------------------------
# the cv:: layer against the real library
# ------------------------------------------------------------------------------------------------------------------
def test_shim_box_filter_equals_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(0)
    for (h, w, R_) in [(57, 83, 5), (30, 41, 10), (9, 9, 10), (100, 100, 16), (1, 50, 3), (50, 1, 3)]:
        X = rng.random((h, w))
        ref = cv2.boxFilter(X, -1, (2 * R_ + 1, 2 * R_ + 1), None, (-1, -1), False, cv2.BORDER_CONSTANT)
        got = R.shim_box_sum(X, R_, _keep=thin)
        assert np.abs(got - ref)[kept(got)].max() < 1e-10
        Xf = X.astype(np.float32)
        reff = cv2.boxFilter(Xf, -1, (2 * R_ + 1, 2 * R_ + 1), None, (-1, -1), False, cv2.BORDER_CONSTANT)
        got = R.shim_box_sum(Xf, R_, _keep=thin)
        assert np.array_equal(got[kept(got)], reff[kept(got)])


def test_shim_image_kernels_equal_cv2():
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(1)
    I = O.synthetic_image(70, 90, 8).astype(np.float32)
    gray = R.shim_bgr2gray(I, _keep=thin)
    assert np.abs(gray - cv2.cvtColor(I, cv2.COLOR_BGR2GRAY))[kept(gray)].max() < 5e-5  # cv2 4.x uses FMAs here: <= 1 ulp of 255
    g = (rng.random((40, 60)) * 255).astype(np.float32)
    sob = R.shim_sobel_x(g, 0.5, _keep=thin)
    assert np.array_equal(sob[kept(sob)], cv2.Sobel(g, cv2.CV_32F, 1, 0, ksize=1, scale=0.5, borderType=cv2.BORDER_REPLICATE)[kept(sob)])
    src = (rng.random((40, 60, 4)) * 100).astype(np.float32)
    nd = npx = 0
    for _ in range(40):
        s3 = (rng.random((3, 2)) * 40).astype(np.float32)
        s3[1, 1] += 30; s3[2, 0] += 30  # keep the triangle well conditioned
        d3 = np.array([[0, 0], [0, 40], [45, 0]], np.float32)
        M = R.shim_get_affine(s3, d3)
        Mref = cv2.getAffineTransform(s3, d3)
        assert np.abs(M - Mref).max() <= 1e-12 * max(1.0, np.abs(Mref).max())
        a = R.shim_warp_affine(src, Mref, 45, 40, _keep=thin)  # same matrix in: the sampler must agree bit for bit
        b = cv2.warpAffine(src, Mref, (45, 40), flags=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)
        assert np.array_equal(a[kept(a)], b[kept(a)])
        c = R.shim_warp_affine(src, M, 45, 40, _keep=thin)      # own matrix: may differ at exact 1/32-pixel rounding ties only
        nd += int((np.abs(c - b) > 1e-4)[kept(c)].sum()); npx += int(kept(c).sum())
    assert nd / npx < 1e-3


# ------------------------------------------------------------------------------------------------------------------
# CostVolumeEnergy + FastGuidedImageFilter<double>
# ------------------------------------------------------------------------------------------------------------------
SCENE = dict(H=96, W=128, D=16, windR=20, eps=1e-4, th_col=0.5)


@pytest.fixture(scope="module")
def cv_pair():
    s = SCENE
    imL, imR, volL, volR = make_scene(s["H"], s["W"], s["D"], seed=3)
    ref = R.RefEnergy(imL, imR, volL, volR, windR=s["windR"], eps=s["eps"], th_col=s["th_col"], max_disp=s["D"] - 1, min_disp=0, kind=0)
    ora = O.CostVolumeEnergyOracle(imL, imR, volL, volR, s["windR"], s["eps"], s["th_col"], float(s["D"] - 1))
    return ref, ora, (imL, imR, volL, volR)


def _special_planes(D):
    return [np.array(p, np.float32) for p in [
        (0, 0, 5.25, 0), (0, 0, 0, 0), (0, 0, D - 1, 0), (0, 0, D - 1.5, 0), (0, 0, -3, 0), (0, 0, D + 4, 0),
        (0.4, -0.3, 4, 0), (-0.11, 0.07, 9.5, 0), (3.0, 0, -100, 0), (0, 2.5, -80, 0),
        (np.nan, 0, 3, 0), (0, 0, np.inf, 0), (np.inf, 0, 0, 0), (1e-3, 1e-3, D - 1.05, 0)]]


def test_guided_filter_statistics_equal_the_reference(cv_pair):
    ref, ora, _ = cv_pair
    for mode in (0, 1):
        st = ref.stats(mode, _keep=thin)
        mine = np.stack(list(ora.filter[mode].mean) + list(ora.filter[mode].inv))
        k = kept(st)
        # same formulas in the same order; the only freedom is the summation order inside the box sums, which the
        # cancellation in var = E[II] - E[I]E[I] amplifies to ~1e-9 relative on the inverse covariance
        assert np.abs(st - mine)[k].max() <= 1e-7 * np.abs(st[k]).max()
        assert np.abs(st[:3] - mine[:3])[k[:3]].max() < 1e-13


def test_numpy_oracle_equals_the_reference_on_every_cell_class(cv_pair):
    ref, ora, _ = cv_pair
    s = SCENE
    rng = O.CvRNG(11)
    worst = 0.0
    n = 0
    for unit in (5, 10, 30):
        lay = O.make_layer(s["W"], s["H"], s["windR"], unit)
        nc = len(lay["unit"])
        wb = lay["widthBlocks"]
        picks = sorted({0, wb - 1, wb, nc // 2, nc - wb, nc - 1, nc - 2})
        for ci in picks:
            fr, tr, un = lay["filter"][ci], lay["shared"][ci], lay["unit"][ci]
            k = rng.uniform_int(0, un[2] * un[3])
            planes = [O.create_random_label(rng, un[0] + k % un[2], un[1] + k // un[2], 0.0, float(s["D"] - 1))]
            planes += [_special_planes(s["D"])[(ci + j) % 14] for j in range(2)]
            for pl in planes:
                for mode in (0, 1):
                    for chk in (True, False):
                        a = ref.unary_target(fr, tr, pl, mode, chk, _keep=thin)
                        b = (ora.compute_unary_potential if chk else ora.compute_unary_potential_without_check)(fr, tr, pl, mode)
                        inv = a == INVALID
                        assert np.array_equal(inv, b == INVALID), (unit, ci, pl, mode, chk)
                        ok = ~inv & np.isfinite(a) & kept(a)
                        assert np.array_equal(np.isfinite(a), np.isfinite(b))
                        if ok.any():
                            worst = max(worst, float((np.abs(a[ok].astype(np.float64) - b[ok]) / np.maximum(np.abs(b[ok]), 1e-3)).max()))
                        n += 1
    assert n > 200
    assert worst <= 1e-6, worst  # (measured: 0 -- bit identical; the slack allows another libm/compiler)


def test_reference_writes_only_the_target_rectangle(cv_pair):
    ref, ora, _ = cv_pair
    fr, tr = (10, 8, 80, 70), (30, 28, 30, 20)
    pl = np.array([0.05, -0.02, 6.0, 0], np.float32)
    out = ref.unary(fr, tr, pl, 0, True, fill=-7.0)
    m = np.zeros(out.shape, bool)
    m[tr[1] - fr[1]:tr[1] - fr[1] + tr[3], tr[0] - fr[0]:tr[0] - fr[0] + tr[2]] = True
    assert (out[~m] == -7.0).all() and (out[m] != -7.0).all()


def test_validity_mask_equals_the_reference(cv_pair):
    ref, ora, _ = cv_pair
    s = SCENE
    rng = O.CvRNG(5)
    rects = [(0, 0, s["W"], s["H"]), (17, 9, 40, 33), (100, 60, 28, 36), (5, 5, 1, 1), (0, 90, 128, 6)]
    planes = _special_planes(s["D"]) + [O.create_random_label(rng, 64, 48, 0.0, float(s["D"] - 1)) for _ in range(20)]
    # planes that graze the bounds: d = MAX exactly at one corner
    planes += [np.array([0.1, 0.0, (s["D"] - 1) - 0.1 * 60 - 0.5, 0], np.float32), np.array([0.0, -0.1, 0.5 + 0.1 * 40, 0], np.float32)]
    nb = 0
    for pl in planes:
        for r in rects:
            a = ref.valid_mask(pl, r)
            b = O.is_valid_label(pl, r, np.float32(0), np.float32(s["D"] - 1))
            assert np.array_equal(a != 0, b), (pl, r)
            nb += int(b.any() and not b.all())
    assert nb >= 3  # some masks really are mixed


def test_c_oracle_equals_the_reference(cv_pair):
    from oracle.c_oracle import COracle
    ref, ora, (imL, imR, volL, volR) = cv_pair
    s = SCENE
    Cc = COracle(s["H"], s["W"], s["D"], s["windR"], s["eps"], s["th_col"], s["D"] - 1)
    Cc.set_image(0, imL); Cc.set_image(1, imR)
    Cc.set_volume(0, volL); Cc.set_volume(1, volR)
    lay = O.make_layer(s["W"], s["H"], s["windR"], 10)
    rng = O.CvRNG(21)
    worst = 0.0
    for ci in (0, 7, len(lay["unit"]) // 2, len(lay["unit"]) - 1):
        fr, tr, un = lay["filter"][ci], lay["shared"][ci], lay["unit"][ci]
        for pl in [O.create_random_label(rng, un[0], un[1], 0.0, float(s["D"] - 1)), _special_planes(s["D"])[6], _special_planes(s["D"])[8]]:
            for mode in (0, 1):
                a = ref.unary_target(fr, tr, pl, mode, True)
                b = Cc.unary(mode, fr, tr, pl, True)
                inv = a == INVALID
                assert np.array_equal(inv, b == INVALID)
                if (~inv).any():
                    worst = max(worst, float((np.abs(a[~inv].astype(np.float64) - b[~inv]) / np.maximum(np.abs(a[~inv]), 1e-3)).max()))
    assert worst <= 1e-6, worst


def test_group_loop_equals_cell_by_cell(cv_pair):
    """ref_unary_group is FastGCStereo.h:30-49 (OpenMP over the cells of a disjoint group, Reusable kept across proposals)."""
    ref, ora, _ = cv_pair
    s = SCENE
    lay = O.make_layer(s["W"], s["H"], s["windR"], 10)
    g = lay["groups"][3]
    fr = [lay["filter"][i] for i in g]
    tr = [lay["shared"][i] for i in g]
    rng = O.CvRNG(2)
    K = 3
    planes = np.stack([np.stack([O.create_random_label(rng, lay["unit"][i][0], lay["unit"][i][1], 0.0, float(s["D"] - 1)) for _ in range(K)]) for i in g])
    img = ref.unary_group(fr, tr, planes, 0, True, nthreads=2)
    for j, i in enumerate(g):
        x, y, w, h = tr[j]
        assert np.array_equal(img[y:y + h, x:x + w], ora.compute_unary_potential(fr[j], tr[j], planes[j, K - 1], 0))


def test_nonzero_min_disparity():
    H, W, D = 64, 80, 12
    imL, imR, volL, volR = make_scene(H, W, D, seed=9)
    mn, mx = -4.0, 7.0  # D0 = 4, vol index = int(d) + 4
    ref = R.RefEnergy(imL, imR, volL, volR, windR=10, eps=1e-3, th_col=0.7, max_disp=mx, min_disp=mn, kind=0)
    ora = O.CostVolumeEnergyOracle(imL, imR, volL, volR, 10, 1e-3, 0.7, mx, mn)
    fr, tr = (0, 0, 60, 50), (10, 10, 30, 25)
    for pl in [(0, 0, -3.5, 0), (0.1, 0.05, -2.0, 0), (0, 0, 6.9, 0), (-0.2, 0.1, 3, 0), (0, 0, -0.5, 0)]:
        pl = np.array(pl, np.float32)
        a = ref.unary_target(fr, tr, pl, 0, True)
        b = ora.compute_unary_potential(fr, tr, pl, 0)
        assert np.array_equal(a == INVALID, b == INVALID)
        ok = a != INVALID
        assert np.abs(a[ok] - b[ok]).max() <= 1e-6 if ok.any() else True


# ------------------------------------------------------------------------------------------------------------------
# NaiveStereoEnergy
# ------------------------------------------------------------------------------------------------------------------
def test_naive_energy_equals_the_reference():
    H, W = 75, 90
    imL = O.synthetic_image(H, W, 8)
    imR = O.synthetic_image(H, W, 9)
    kw = dict(windR=20, eps=1e-4 * 255 * 255 / (255 * 255), th_col=10.0, th_grad=2.0, alpha=0.9)
    ref = R.RefEnergy(imL, imR, windR=20, eps=kw["eps"], th_col=10.0, th_grad=2.0, alpha=0.9, max_disp=31.0, min_disp=0.0, kind=1)
    ora = O.NaiveStereoEnergyOracle(imL, imR, 20, kw["eps"], 10.0, 2.0, 0.9, 31.0)
    for m in (0, 1):
        exi = ref.exi(m, _keep=thin)
        assert np.array_equal(exi[kept(exi)], ora.ExI[m][kept(exi)])  # cvtColor / Sobel / scale chain, bit for bit
    rng = O.CvRNG(3)
    nbad = ntot = 0
    for _ in range(25):
        fx, fy = rng.uniform_int(0, 40), rng.uniform_int(0, 30)
        fr = (fx, fy, 45, 40)
        tr = (fx + 10, fy + 10, 20, 15)
        pl = O.create_random_label(rng, fx + 20, fy + 20, 0.0, 31.0)
        for mode in (0, 1):
            a = ref.unary_target(fr, tr, pl, mode, True, _keep=thin)
            b = ora.compute_unary_potential(fr, tr, pl, mode)
            assert np.array_equal(a == INVALID, b == INVALID)
            ok = (a != INVALID) & kept(a)
            # the oracle repeats getAffineTransform's LU solve + warpAffine's inversion operation by operation, so every
            # 1/32-pixel source coordinate equals the reference's: the same tolerance as everywhere else, no outlier budget
            err = np.abs(a[ok].astype(np.float64) - b[ok]) / np.maximum(np.abs(b[ok]), 1e-3)
            nbad += int((err > 1e-4).sum()); ntot += int(ok.sum())
    assert ntot > 5000 // 32 and nbad == 0, (nbad, ntot)


# ------------------------------------------------------------------------------------------------------------------
# LayerManager, Plane, cv::RNG-driven labels
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("W,H,windR,unit", [(128, 96, 20, 5), (128, 96, 20, 10), (130, 97, 20, 15), (450, 375, 20, 5), (450, 375, 20, 15),
                                             (450, 375, 20, 25), (2048, 1536, 20, 20), (2048, 1536, 20, 61), (2048, 1536, 20, 184),
                                             (718, 496, 10, 25), (101, 103, 7, 50), (64, 64, 20, 16)])
def test_layer_geometry_equals_layer_manager(W, H, windR, unit):
    a = R.layer(W, H, windR, unit)
    b = O.make_layer(W, H, windR, unit)
    assert (a["heightBlocks"], a["widthBlocks"]) == (b["heightBlocks"], b["widthBlocks"])
    for k in ("unit", "shared", "filter"):
        assert [tuple(r) for r in a[k]] == [tuple(int(v) for v in r) for r in b[k]], k
    assert a["groups"] == [list(g) for g in b["groups"]]


def test_plane_helpers_equal_the_reference():
    rng = np.random.default_rng(4)
    for _ in range(200):
        n = rng.standard_normal(3).astype(np.float32)
        n[2] = abs(n[2]) + np.float32(0.05)
        z, x, y = np.float32(rng.uniform(0, 60)), np.float32(rng.integers(0, 2000)), np.float32(rng.integers(0, 1500))
        a = R.create_plane(n, z, x, y)
        b = O.create_plane(n[0], n[1], n[2], z, x, y)
        assert np.array_equal(a, b)
        assert np.array_equal(R.plane_normal(a), O.plane_normal(b))


def test_random_labels_and_proposals_equal_the_reference(cv_pair):
    ref, ora, _ = cv_pair
    s = SCENE
    R.rng_seed(12345)
    rng = O.CvRNG(12345)
    for i in range(50):
        x, y = (7 * i) % s["W"], (11 * i) % s["H"]
        a = ref.create_random_label(x, y)
        b = O.create_random_label(rng, x, y, 0.0, float(s["D"] - 1))
        assert np.array_equal(a, b), i
    assert R.rng_state() == rng.state
    # RandomProposer over a unit region of a labeling (Proposer.h:120-148), as FastGCStereo.h:39-46 drives it
    lab = np.zeros((s["H"], s["W"], 4), np.float32)
    r2 = O.CvRNG(99)
    for yy in range(0, s["H"], 8):
        for xx in range(0, s["W"], 8):
            lab[yy:yy + 8, xx:xx + 8] = O.create_random_label(r2, xx, yy, 0.0, float(s["D"] - 1))
    unit = (40, 24, 10, 10)
    for outer in (0, 1, 3):
        R.rng_seed(777 + outer)
        rng = O.CvRNG(777 + outer)
        got = R.random_proposals(lab, unit, outer, 7, float(s["D"] - 1), 0.0)
        dz = lambda m: np.float32(np.float32(s["D"] - 1) * np.float32(np.power(np.float32(0.5), m + 1)))
        want = []
        it = 0
        while it < 7 and not (dz(outer + it) < 0.1):            # isContinued (Proposer.h:149-152)
            k = rng.uniform_int(0, unit[2] * unit[3])           # selectRandomPixelInRect (:38-45)
            px, py = k % unit[2], k // unit[2]
            src = lab[unit[1] + py, unit[0] + px]
            want.append(O.random_proposal(rng, src, unit[0] + px, unit[1] + py, outer + it, 0.0, float(s["D"] - 1)))
            it += 1
        assert len(got) == len(want) and len(got) > 0
        got, want = np.asarray(got), np.stack(want)
        # plane normals go through sqrt/sin/cos in double and a float division: allow 2 ulp on a, b and the c they feed
        assert np.allclose(got, want, rtol=3e-6, atol=1e-6), (outer, np.abs(got - want).max())
        assert R.rng_state() == rng.state


def test_adapter_compiles_against_the_reference_headers_and_harness_self_check():
    """oracle/_ref/dropin_check = the reference's FastGCStereo loop + include/CudaCostVolumeEnergy.h compiled against the REAL
    StereoEnergy.h (not the stub of tests/cxx) and linked with liblexp_cuda.so.  Without a GPU only its CPU self-check can run:
    the reference's CPU energy on both sides, which validates the harness the GPU test relies on."""
    import json
    import os
    import subprocess
    if build_ref.build() is None:
        pytest.skip("compiles the reference's own sources, which are not on this machine")
    if not os.path.exists(build_ref.DROPIN):
        pytest.skip("liblexp_cuda.so is not built yet")
    for extra in ([], ["--naive"]):
        res = subprocess.run([build_ref.DROPIN, "--cpu-self-check", "--W", "96", "--H", "80"] + extra, capture_output=True, text=True, timeout=600)
        d = json.loads(res.stdout.strip().splitlines()[-1])
        assert res.returncode == 0 and d["ok"] is True and d["out_of_tolerance"] == 0 and d["move_calls"] > 1000, d


# ------------------------------------------------------------------------------------------------------------------
# PatchMatch phase: the oracle's step-wise restatement against the reference's own loop, proposers and energy
# ------------------------------------------------------------------------------------------------------------------
def test_pm_phase_oracle_equals_the_reference_loop():
    """oracle.pm_step / pm_proposal (what the device path is compared with) vs oracle/_ref's ref_pm_group: the body of
    FastGCStereo::localExpansionMovesForLayer_CPU with doGC == false (FastGCStereo.h:30-61) driving the reference's own
    ExpansionProposer / RandomProposer / CostVolumeEnergy, with cv::theRNG() started from the same per-(cell, step) states.
    Same proposals bit for bit, same currentLabeling_ and the same currentCost_ (to 1 float ulp) after two groups of two layers."""
    H, W, D, windR = 72, 96, 12, 12
    imL, imR, volL, volR = make_scene(H, W, D)
    ref = R.RefEnergy(imL, imR, volL, volR, windR=windR, eps=1e-4, th_col=0.5, max_disp=D - 1, min_disp=0.0, kind=0)
    ora = O.CostVolumeEnergyOracle(imL, imR, volL, volR, windR, 1e-4, 0.5, D - 1)
    try:
        rng = O.CvRNG(21)
        lay0 = O.make_layer(W, H, windR, 8)
        units0 = lay0["unit"]
        labels = np.stack([O.create_random_label(rng, u[0] + rng.uniform_int(0, u[2]), u[1] + rng.uniform_int(0, u[3]), 0.0, D - 1.0) for u in units0])
        state = {}
        for who in ("ref", "ora"):
            state[who] = (np.full((H, W), np.inf, np.float32), np.zeros((H, W, 4), np.float32))
        ref.pm_init(units0, labels, windR, *state["ref"])
        fr0 = [(max(x - windR, 0), max(y - windR, 0), min(x + w + windR, W) - max(x - windR, 0), min(y + h + windR, H) - max(y - windR, 0)) for (x, y, w, h) in units0]
        O.pm_step(ora, units0, units0, fr0, 0, 0, 0, None, *state["ora"], planes=labels, init=True)
        assert np.array_equal(state["ref"][0], state["ora"][0]) and np.array_equal(state["ref"][1], state["ora"][1])
        list_rng = O.CvRNG(77)
        for li, (u, proposers) in enumerate([(8, [(1, 1), (0, 1), (2, 3)]), (22, [(1, 2), (0, 1)])]):   # Expansion, replayed list (Ransac slot), Random
            lay = O.make_layer(W, H, windR, u)
            for gi in (0, 5):
                cells = lay["groups"][gi]
                us = [lay["unit"][r] for r in cells]; ts = [lay["shared"][r] for r in cells]; fs = [lay["filter"][r] for r in cells]
                steps = [(k, m) for k, K in proposers for m in range(K)]       # outer_iter = 1 below: Random m = 1 + iter
                seeds = [1000 * li + 10 * gi + s for s in range(len(steps))]
                states = np.array([[O.pm_rng_state(seeds[s], 100 * li + r) for s in range(len(steps))] for r in cells], dtype=np.uint64)
                lists = np.stack([[O.create_random_label(list_rng, u_[0], u_[1], 0.0, D - 1.0)] for u_ in us])   # [n][1][4]
                planes_ref, nsteps = ref.pm_group(us, ts, fs, proposers, 1, states, *state["ref"], list_planes=lists)
                assert (nsteps == len(steps)).all()
                for s, (kind, it) in enumerate(steps):
                    used = O.pm_step(ora, us, ts, fs, kind, 1 + it, seeds[s], [100 * li + r for r in cells], *state["ora"],
                                     planes=lists[:, 0] if kind == 0 else None)
                    assert np.array_equal(used, planes_ref[:, s]), f"layer {li} group {gi} step {s}: proposals differ"
                # the oracle's double guided filter equals the reference's up to 1 float ulp of the stored cost (summation order
                # of the box filter); the labels -- the decisions `cur > prop` -- must be identical
                assert np.allclose(state["ref"][0], state["ora"][0], rtol=2.5e-7, atol=0), f"layer {li} group {gi}: currentCost differs"
                assert np.array_equal(state["ref"][1], state["ora"][1]), f"layer {li} group {gi}: currentLabeling differs"
        assert np.isfinite(state["ora"][0]).all()
    finally:
        ref.close()


# ------------------------------------------------------------------------------------------------------------------
# Pairwise terms and the graph-cut move: the oracle's restatement against the reference's own StereoEnergy and
# FastGCStereo::expansionMoveBK (compiled from FastGCStereo.h over oracle/maxflow/graph.h)
# ------------------------------------------------------------------------------------------------------------------
def test_smoothness_oracle_equals_the_reference():
    """oracle.smoothness_coeff / smoothness_terms_expansion / smoothness_cost vs the reference's initSmoothnessCoeff,
    computeSmoothnessTermsExpansion (as expansionMoveBK calls it) and computeSmoothnessCost: coefficients to 1 ulp of exp(),
    zero pattern identical; with the same coefficients the three cost maps are bit-identical on interior and border regions."""
    H, W, D, windR = 60, 84, 10, 12
    imL, imR, volL, volR = make_scene(H, W, D, seed=6)
    ref = R.RefEnergy(imL, imR, volL, volR, windR=windR, eps=1e-4, th_col=0.5, max_disp=D - 1, min_disp=0.0, kind=0)
    try:
        rng = O.CvRNG(12)
        lab = np.zeros((H, W, 4), np.float32)
        for y in range(0, H, 6):
            for x in range(0, W, 6):
                lab[y:y + 6, x:x + 6] = O.create_random_label(rng, x, y, 0.0, D - 1.0)
        for (lam, omega, th, eps) in ((1.0, 10.0, 1.0, 0.01), (0.35, 4.0, 0.6, 0.1)):
            ref.set_smoothness(lam, omega, th, eps)
            for mode, im in ((0, imL), (1, imR)):
                co_r, co_o = ref.smooth_coeff(mode), O.smoothness_coeff(im, omega, eps)
                assert np.array_equal(co_r == 0, co_o == 0)
                assert np.allclose(co_r, co_o, rtol=1e-6, atol=0)   # float exp of the shim vs exp in double
                for region in [(10, 8, 25, 21), (0, 0, 19, 14), (W - 13, H - 17, 13, 17), (0, 0, W, H), (5, 5, 1, 1)]:
                    plane = O.create_random_label(rng, region[0], region[1], 0.0, D - 1.0)
                    got = O.smoothness_terms_expansion(lab, plane, region, co_r, lam, th)
                    want = ref.smooth_terms_expansion(lab, plane, region, mode, _keep=lambda t: tuple(thin(x) for x in t))
                    for g, w_ in zip(got, want):
                        assert np.array_equal(g[kept(w_)], w_[kept(w_)]), (region, np.abs(g - w_)[kept(w_)].max())
                assert abs(O.smoothness_cost(lab, co_r, lam, th) - ref.smoothness_cost(lab, mode)) <= 1e-6 * ref.smoothness_cost(lab, mode)
    finally:
        ref.close()


def test_graph_cut_oracle_equals_the_reference_loop():
    """oracle.gc_step (numpy graph of expansion_graph + the C grid minimum cut) vs oracle/_ref's ref_gc_group: the body of
    FastGCStereo::localExpansionMovesForLayer_CPU with doGC == true driving the reference's own proposers, CostVolumeEnergy and
    FastGCStereo::expansionMoveBK.  Same proposals, the same minimum-cut energy of every move (1e-6: only the order of the
    double-precision flow sums differs), identical currentLabeling_, currentCost_ equal to 1 ulp -- over two iterations of two
    layers, including the first groups whose current costs still hold COST_FOR_INVALID next to the pairwise terms."""
    H, W, D, windR = 72, 96, 12, 12
    imL, imR, volL, volR = make_scene(H, W, D)
    ref = R.RefEnergy(imL, imR, volL, volR, windR=windR, eps=1e-4, th_col=0.5, max_disp=D - 1, min_disp=0.0, kind=0)
    ora = O.CostVolumeEnergyOracle(imL, imR, volL, volR, windR, 1e-4, 0.5, D - 1)
    lam, omega, th, eps = 0.7, 10.0, 1.0, 0.01
    try:
        ref.set_smoothness(lam, omega, th, eps)
        coeff = ref.smooth_coeff(0)
        rng = O.CvRNG(21)
        lay0 = O.make_layer(W, H, windR, 8)
        units0 = lay0["unit"]
        labels = np.stack([O.create_random_label(rng, u[0] + rng.uniform_int(0, u[2]), u[1] + rng.uniform_int(0, u[3]), 0.0, D - 1.0) for u in units0])
        cost_r, lab_r = np.full((H, W), np.inf, np.float32), np.zeros((H, W, 4), np.float32)
        ref.pm_init(units0, labels, windR, cost_r, lab_r)
        cost_o, lab_o = cost_r.copy(), lab_r.copy()
        n_moves = 0
        for it in range(2):
            for li, (u, proposers) in enumerate([(8, [(1, 1), (2, 2)]), (22, [(1, 2)])]):
                lay = O.make_layer(W, H, windR, u)
                for gi, cells in enumerate(lay["groups"]):
                    us = [lay["unit"][r] for r in cells]; ts = [lay["shared"][r] for r in cells]; fs = [lay["filter"][r] for r in cells]
                    steps = [(k, (it + j if k == 2 else 0)) for k, K in proposers for j in range(K)]
                    seeds = [10000 * it + 1000 * li + 10 * gi + s for s in range(len(steps))]
                    states = np.array([[O.pm_rng_state(seeds[s], 100 * li + r) for s in range(len(steps))] for r in cells], dtype=np.uint64)
                    planes, nsteps, flows = ref.gc_group(us, ts, fs, proposers, it, states, cost_r, lab_r)
                    assert (nsteps == len(steps)).all()
                    for s, (kind, m) in enumerate(steps):
                        used, fl = O.gc_step(ora, us, ts, fs, kind, m, seeds[s], [100 * li + r for r in cells], cost_o, lab_o, coeff, lam, th)
                        assert np.allclose(used, planes[:, s], rtol=3e-6, atol=1e-6)
                        assert (np.abs(fl - flows[:, s]) <= 1e-6 * np.maximum(np.abs(flows[:, s]), 1e-3)).all(), (it, li, gi, s)
                        n_moves += len(cells)
            assert np.array_equal(lab_r, lab_o), (it, int((lab_r != lab_o).any(axis=2).sum()))
            assert np.abs(cost_r - cost_o).max() <= 1e-6
        assert n_moves > 500
    finally:
        ref.close()


def test_maxflow_stand_in_on_random_graphs():
    """oracle/maxflow/graph.h (the interface of the un-vendored BK library, used by the compiled reference) and the C grid minimum
    cut of the oracle are two independent implementations: on random expansion-move-shaped grids they report the same flow and the
    same SOURCE segment, and the cut they report has the value of the flow (max-flow = min-cut)."""
    from oracle import c_oracle
    rng = np.random.default_rng(5)
    for (h, w) in [(1, 1), (1, 7), (6, 1), (9, 13), (24, 31)]:
        for trial in range(3):
            tr = (rng.random((h, w)) - 0.5).astype(np.float32) * np.float32(4)
            cap = (rng.random((4, h, w)) * (rng.random((4, h, w)) < 0.8)).astype(np.float32)
            mask, flow = c_oracle.grid_mincut(tr, cap)
            # value of the cut (SOURCE = mask): source arcs into the sink side + sink arcs out of the source side + forward arcs S -> T
            cut = float(np.maximum(tr, 0)[~mask].sum() + np.maximum(-tr, 0)[mask].sum())
            for d, (dx, dy) in enumerate([(1, 0), (0, 1), (-1, 1), (1, 1)]):
                for y in range(h):
                    for x in range(w):
                        xx, yy = x + dx, y + dy
                        if 0 <= xx < w and yy < h and mask[y, x] and not mask[yy, xx]:
                            cut += float(cap[d, y, x])
            assert abs(cut - flow) <= 1e-4 * max(1.0, flow), (h, w, trial, cut, flow)
            m2, f2 = R.shim_grid_mincut(tr, cap)
            assert abs(f2 - flow) <= 1e-5 * max(1.0, flow) and np.array_equal(m2, mask), (h, w, trial)


def test_file_formats_equal_the_reference(tmp_path):
    """The product's PFM writer, volume-file reader and disparity map against the reference's own cvutils::io::save_pfm_file /
    read_pfm_file / loadMatBinary and StereoEnergy::computeDisparities (compiled in oracle/_ref): byte-identical PFM file, the file
    the reference reads back, the same volume from the same `.acrt` bytes.  (Host-side functions of the product library: the
    emulator build of the same source is loaded here; no kernel runs except the disparity map's.)"""
    import os
    from emu import emu_lib
    import localexpstereo_b200 as L
    H, W, D, windR = 40, 56, 9, 8
    imL, imR, volL, volR = make_scene(H, W, D, seed=3)
    ref = R.RefEnergy(imL, imR, volL, volR, windR=windR, eps=1e-4, th_col=0.5, max_disp=D - 1, min_disp=0.0, kind=0)
    with emu_lib.emulated():
        E = L.CostVolumeEnergy(imL, None, volL, None, L.Parameters(windR=windR, filterName="GF", filter_param1=1e-4, th_col=0.5), D - 1)
        try:
            rng = O.CvRNG(9)
            lab = np.zeros((H, W, 4), np.float32)
            for y in range(0, H, 4):
                for x in range(0, W, 8):
                    lab[y:y + 4, x:x + 8] = O.create_random_label(rng, x, y, 0.0, D - 1.0)
            E.pm_begin(0, np.zeros((H, W), np.float32), lab)
            disp = E.computeDisparities(0)
            assert np.array_equal(disp, ref.disparities(lab))
            a, b = os.path.join(str(tmp_path), "a.pfm"), os.path.join(str(tmp_path), "b.pfm")
            L.save_pfm_file(a, disp)
            R.save_pfm(b, disp)
            assert open(a, "rb").read() == open(b, "rb").read()
            assert np.array_equal(R.read_pfm(a, H, W), disp)
            acrt = os.path.join(str(tmp_path), "im0.acrt")
            volL.tofile(acrt)
            vol = R.load_acrt(acrt, D, H, W, _keep=thin)
            assert np.array_equal(vol[kept(vol)], volL[kept(vol)])          # what the reference would have loaded
            E.set_volume_file(0, acrt)                                          # and what the product ingests from the same bytes
            f, t = (4, 4, 40, 30), (10, 8, 20, 16)
            p = np.array([0.02, -0.01, 3.5, 0], np.float32)
            img = np.zeros((H, W), np.float32)
            E.ComputeUnaryPotential(f, t, img[f[1]:f[1] + f[3], f[0]:f[0] + f[2]], p)
            got = img[t[1]:t[1] + t[3], t[0]:t[0] + t[2]]
            want = ref.unary_target(f, t, p)
            assert np.allclose(got, want, rtol=1e-4, atol=1e-7)
        finally:
            E.close()
            ref.close()
