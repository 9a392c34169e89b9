"""CPU tests: pin the oracle (oracle/b2o_oracle.c) against the reference's own known-answer vectors and
against the committed golden fixtures, which hold what oracle/_ref (the reference's im2col.cpp compiled
verbatim) computed.  No GPU needed."""
import json
import os

import numpy as np
import pytest

import oracle as o
from cases import ALL_CASES, REF_IM2COL_SHAPES, REF_TEST_CASES, digest, make, tensors, rel_err

GOLD = os.path.join(os.path.dirname(__file__), "golden")


# ---- test_util_blas.cpp:19-175 integer known answers (EXPECT_EQ -> exact) -----------------------
def test_gemm_known_answers():
    data = np.arange(1, 13, dtype=np.float32)
    A, B = data[:6], data
    At = np.array([1, 4, 2, 5, 3, 6], np.float32)
    Bt = np.array([1, 5, 9, 2, 6, 10, 3, 7, 11, 4, 8, 12], np.float32)
    want = np.array([38, 44, 50, 56, 83, 98, 113, 128], np.float32)
    z = np.zeros(8, np.float32)
    for acc64 in (False, True):
        assert np.array_equal(o.gemm(0, 0, 2, 4, 3, 1.0, A, B, 0.0, z, acc64), want)
        assert np.array_equal(o.gemm(1, 0, 2, 4, 3, 1.0, At, B, 0.0, z, acc64), want)
        assert np.array_equal(o.gemm(1, 1, 2, 4, 3, 1.0, At, Bt, 0.0, z, acc64), want)
        assert np.array_equal(o.gemm(0, 1, 2, 4, 3, 1.0, A, Bt, 0.0, z, acc64), want)


def test_gemm_beta1_known_answer():
    A = np.array([1, 2, 3, 4, 5, 6], np.float32)
    B = np.array([1, 2], np.float32)
    res = np.array([5, 11, 17], np.float32)
    assert np.array_equal(o.gemm(0, 0, 3, 1, 2, 1.0, A, B, 1.0, res), res * 2)


def test_gemv_known_answers():
    A = np.arange(1, 7, dtype=np.float32)
    assert np.array_equal(o.gemv(0, 2, 3, 1.0, A, A[:3], 0.0, np.zeros(2, np.float32)), [14, 32])
    assert np.array_equal(o.gemv(1, 2, 3, 1.0, A, A[:2], 0.0, np.zeros(3, np.float32)), [9, 12, 15])
    assert np.array_equal(o.gemv(0, 3, 2, 1.0, A, A[:2], 0.0, np.zeros(3, np.float32)), [5, 11, 17])
    assert np.array_equal(o.gemv(1, 3, 2, 1.0, A, A[:3], 0.0, np.zeros(2, np.float32)), [22, 28])


# ---- im2col: bit for bit against the reference source compiled verbatim (test_im2col_kernel.cu:102-212 shapes) ----
# tests/golden/im2col_ref_digests.json holds the sha256 of every output oracle/_ref produced from these seeded inputs
def ref_digests():
    with open(os.path.join(GOLD, "im2col_ref_digests.json")) as f:
        return json.load(f)


@pytest.mark.parametrize("shape", REF_IM2COL_SHAPES)
def test_im2col_col2im_bit_exact_vs_reference_source(rng, shape):
    Cc, H, W, k, s, p, d = shape
    want = ref_digests()[repr(shape)]
    im = rng.standard_normal((Cc, H, W)).astype(np.float32)
    col = o.im2col(im, k, s, p, d)
    colr = rng.standard_normal(col.shape).astype(np.float32)
    assert (digest(im), digest(colr)) == (want["im"], want["colr"]), "seeded inputs differ from the recorded ones"
    assert digest(col) == want["col"]
    back = o.col2im(colr, (Cc, H, W), k, s, p, d)
    assert digest(back) == want["col2im"]
    # N-D restatement against the reference N-D source and against the 2-D path (TestNDAgainst2D :606)
    coln = o.im2col_nd(im, k, s, p, d)
    assert digest(coln) == want["col_nd"] and np.array_equal(coln, col)
    backn = o.col2im_nd(colr, (Cc, H, W), k, s, p, d)
    assert digest(backn) == want["col2im_nd"]


def test_im2col_3d_nd(rng):
    # 3 spatial axes (TestSimple3DConvolution :352 uses the N-D path)
    im = rng.standard_normal((2, 5, 6, 4)).astype(np.float32)
    k, s, p, d = (3, 2, 3), (2, 1, 1), (1, 0, 1), (1, 2, 1)
    col = o.im2col_nd(im, k, s, p, d)
    # brute-force definition
    out = [(im.shape[1 + a] + 2 * p[a] - (d[a] * (k[a] - 1) + 1)) // s[a] + 1 for a in range(3)]
    want = np.zeros((2 * 18, *out), np.float32)
    for c in range(2):
        for a in range(3):
            for b in range(2):
                for e in range(3):
                    r = ((c * 3 + a) * 2 + b) * 3 + e
                    for x in range(out[0]):
                        for y in range(out[1]):
                            for z in range(out[2]):
                                i0, i1, i2 = x * s[0] - p[0] + a * d[0], y * s[1] - p[1] + b * d[1], z * s[2] - p[2] + e * d[2]
                                if 0 <= i0 < 5 and 0 <= i1 < 6 and 0 <= i2 < 4:
                                    want[r, x, y, z] = im[c, i0, i1, i2]
    assert np.array_equal(col, want)
    ref = ref_digests()["3d"]
    assert digest(im) == ref["im"] and digest(col) == ref["col_nd"]


def test_im2col_layer_known_positions(rng):
    # test_im2col_layer.cpp:63-77: top-left 3x3 block of the first output location equals the image patch
    im = rng.standard_normal((3, 6, 5)).astype(np.float32)
    col = o.im2col(im, 3, 2, 0, 1)
    for c in range(3):
        for i in range(3):
            for j in range(3):
                assert col[(c * 3 + i) * 3 + j, 0, 0] == im[c, i, j]


# ---- forward: vs the independent direct definition (caffe_conv's role, tol 1e-4 :255) ------------
@pytest.mark.parametrize("name,case", ALL_CASES, ids=[c[0] for c in ALL_CASES])
def test_forward_matches_direct_definition(rng, name, case):
    prm = make(o, case)
    x, w, b, _ = tensors(rng, prm)
    y = o.conv_forward(prm, x, w, b)
    yd = o.conv_direct(prm, x, w, b)
    assert y.shape == prm.y_shape()
    assert np.abs(y - yd).max() <= 1e-4 * max(1.0, float(np.abs(yd).max()))


def test_sobel_known_answer(rng):
    # test_convolution_layer.cpp:511-604: 3x3 Sobel == (3x1 [1 2 1], stride (2,1)) then (1x3 [-1 0 1], stride (1,2))
    x = rng.standard_normal((2, 3, 6, 4)).astype(np.float32)
    w = np.tile(np.array([-1, 0, 1, -2, 0, 2, -1, 0, 1], np.float32), 3).reshape(1, 3, 3, 3)
    y = o.conv_forward(o.ConvParams.make(2, 3, 6, 4, 1, 3, 2, 0, 1, 1, False), x, w)
    w1 = np.tile(np.array([1, 2, 1], np.float32), 3).reshape(1, 3, 3, 1)
    t = o.conv_forward(o.ConvParams.make(2, 3, 6, 4, 1, (3, 1), (2, 1), 0, 1, 1, False), x, w1)
    w2 = np.array([-1, 0, 1], np.float32).reshape(1, 1, 1, 3)
    y2 = o.conv_forward(o.ConvParams.make(2, 1, t.shape[2], t.shape[3], 1, (1, 3), (1, 2), 0, 1, 1, False), t, w2)
    assert y.shape == y2.shape
    assert np.abs(y - y2).max() <= 1e-4


# ---- backward: finite differences like GradientChecker (step 1e-2, threshold 1e-3) --------------
@pytest.mark.parametrize("name,case", REF_TEST_CASES, ids=[c[0] for c in REF_TEST_CASES])
def test_backward_gradient_check(rng, name, case):
    prm = make(o, case)
    x, w, b, _ = tensors(rng, prm, scale_w=1.0)
    # objective = 0.5*||y||^2 -> dy = y   (test_gradient_check_util.hpp:71-172)
    y = o.conv_forward(prm, x, w, b, acc64=True)
    dw, db, dx = o.conv_backward(prm, x, w, y, acc64=True)

    def loss(xx, ww, bb):
        yy = o.conv_forward(prm, xx, ww, bb, acc64=True).astype(np.float64)
        return 0.5 * float((yy * yy).sum())

    step, thr = 1e-2, 1e-3
    for arr, grad, which in ((x, dx, 0), (w, dw, 1), (b, db, 2)):
        if arr is None:
            continue
        flat = arr.reshape(-1)
        for idx in rng.choice(flat.size, size=min(12, flat.size), replace=False):
            old = flat[idx]
            flat[idx] = old + step
            lp = loss(x, w, b)
            flat[idx] = old - step
            lm = loss(x, w, b)
            flat[idx] = old
            est = (lp - lm) / (2 * step)
            got = float(grad.reshape(-1)[idx])
            scale = max(abs(est), abs(got), 1.0)
            assert abs(est - got) <= thr * scale * 5, (which, idx, est, got)


def test_backward_accumulates_param_diffs_and_overwrites_bottom(rng):
    prm = o.ConvParams.make(2, 3, 6, 4, 4, 3, 2, 0, 1, 1, True)
    x, w, b, dy = tensors(rng, prm)
    dw0, db0, dx0 = o.conv_backward(prm, x, w, dy)
    dw1, db1, dx1 = o.conv_backward(prm, x, w, dy, dw=dw0, db=db0)
    assert np.allclose(dw1, 2 * dw0, rtol=1e-6, atol=1e-6) and np.allclose(db1, 2 * db0, rtol=1e-6, atol=1e-6)
    assert np.array_equal(dx0, dx1)


# ---- SGD / LR ---------------------------------------------------------------------------------
def test_sgd_update_closed_form(rng):
    # GradientBasedSolverTest closed form (test_gradient_based_solver.cpp:228-364): with momentum m, lr, decay wd:
    #   h' = m*h + lr*(g + wd*w);  w' = w - h'
    n = 1001
    g, w, h = (rng.standard_normal(n).astype(np.float32) for _ in range(3))
    for l2 in (True, False):
        for clear in (True, False):
            g2, w2, h2 = o.sgd_update(g, w, h, 0.9, 0.01, 0.0005, l2=l2, clear_grads=clear)
            reg = w if l2 else np.sign(w)
            hh = 0.9 * h.astype(np.float64) + 0.01 * (g.astype(np.float64) + 0.0005 * reg)
            assert np.allclose(h2, hh, rtol=1e-6, atol=1e-7)
            assert np.allclose(w2, w - hh, rtol=1e-6, atol=1e-6)
            assert np.array_equal(g2, np.zeros_like(g2)) if clear else np.array_equal(g2, h2)
    # iter_size accumulation normalisation and 1/solver_count folding
    g2, w2, h2 = o.sgd_update(g, w, h, 0.0, 1.0, 0.0, grad_scale=0.25, iter_size=2)
    assert np.allclose(h2, g * 0.125, rtol=1e-6)


def test_learning_rate_policies():
    assert o.learning_rate("fixed", 10, 0.1) == pytest.approx(0.1)
    assert o.learning_rate("step", 25, 0.1, gamma=0.5, stepsize=10) == pytest.approx(0.1 * 0.25)
    assert o.learning_rate("exp", 3, 0.1, gamma=0.9) == pytest.approx(0.1 * 0.9 ** 3, rel=1e-6)
    assert o.learning_rate("inv", 100, 0.01, gamma=1e-4, power=0.75) == pytest.approx(0.01 * (1 + 1e-4 * 100) ** -0.75, rel=1e-6)
    # resnet50 solver: poly, power 2
    assert o.learning_rate("poly", 1200000, 0.001, power=2.0, max_iter=2400000) == pytest.approx(0.001 * 0.25, rel=1e-6)
    assert o.learning_rate("multistep", 5, 0.1, gamma=0.1, current_step=2) == pytest.approx(0.001, rel=1e-5)
    assert o.learning_rate("fixed", 5, 0.1, rampup_interval=10, rampup_lr=0.0) == pytest.approx(0.05)


def test_allreduce_avg(rng):
    bufs = [rng.standard_normal(77).astype(np.float32) for _ in range(4)]
    out = o.allreduce_avg(bufs)
    want = (bufs[0] + bufs[1] + bufs[2] + bufs[3]) * np.float32(0.25)
    for b in out:
        assert np.allclose(b, want, rtol=1e-6, atol=1e-7)


# ---- golden fixtures produced from oracle/_ref (tests/golden/make_golden.py) -----------------------
def test_oracle_matches_golden_fixtures():
    path = os.path.join(GOLD, "conv_ref_golden.npz")
    assert os.path.exists(path), "golden fixture missing: run tests/golden/make_golden.py in the build container"
    z = np.load(path)
    names = sorted(set(k.split("/")[0] for k in z.files))
    assert len(names) >= 6
    for nm in names:
        c = {k: int(v) for k, v in zip(z[nm + "/keys"], z[nm + "/vals"])}
        prm = o.ConvParams(*[c[f] for f, _ in o.ConvParams._fields_])
        x, w, dy = z[nm + "/x"], z[nm + "/w"], z[nm + "/dy"]
        b = z[nm + "/b"] if prm.has_bias else None
        y = o.conv_forward(prm, x, w, b)
        dw, db, dx = o.conv_backward(prm, x, w, dy)
        # reference leg used OpenBLAS sgemm (different summation order): fp32 round-off tolerance
        assert rel_err(y, z[nm + "/y"]) < 2e-6, nm
        assert rel_err(dw, z[nm + "/dw"]) < 5e-6, nm
        assert rel_err(dx, z[nm + "/dx"]) < 2e-6, nm
        if prm.has_bias:
            assert rel_err(db, z[nm + "/db"]) < 5e-6, nm
        # im2col part of the fixture is bit-exact (pure copy)
        col = o.im2col(x[0], (prm.kh, prm.kw), (prm.sh, prm.sw), (prm.ph, prm.pw), (prm.dh, prm.dw))
        assert np.array_equal(col, z[nm + "/col0"]), nm
