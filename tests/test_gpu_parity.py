"""GPU parity tests (run with -m gpu on the B200 box): every CUDA path behind include/b2c.h against the
CPU oracle on the same seeded inputs, through the C ABI.

Tolerances: index/copy work (im2col, col2im) is BIT-EXACT; integer-valued GEMM/GEMV known answers are
exact; floating-point conv/GEMM results are compared to the oracle with double accumulation using the
blob-level relative error  max|a-ref| / max|ref| <= 1e-3  (BASELINE.json north_star; DESIGN.md states
why blob-level).  In the default FP32 math mode the observed error is ~1e-6, so the FP32-mode bar used
below is 2e-5; the 1e-3 bar is what the TF32 mode is held to."""
import os

import numpy as np
import pytest

import oracle as o
from cases import ALL_CASES, EDGE_CASES, FULL_SIZE_CASES, MODEL_CASES, REF_TEST_CASES, full_size_inputs, make, sample_index, tensors, rel_err

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import caffe_mpi_b200 as m  # noqa: E402
from caffe_mpi_b200 import capi  # noqa: E402

TOL_FP32 = 1e-4   # 3xTF32: tensor-core accumulator rounding grows with K (3e-5 at K=4608), DESIGN.md
TOL_SIMT = 2e-5
TOL_TF32 = 1e-3
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def dev(a):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    torch.cuda.synchronize()
    return t.cpu().numpy()


# ---------------------------------------------------------------------------------------------- im2col
IM2COL_SHAPES = [
    (500, 15, 15, (3, 3), (2, 2), (0, 0), (3, 3)),   # test_im2col_kernel.cu:102-156
    (3, 6, 5, (3, 3), (2, 2), (0, 0), (1, 1)),
    (4, 9, 11, (3, 5), (2, 1), (1, 2), (1, 1)),
    (2, 12, 10, (3, 3), (1, 2), (2, 1), (2, 3)),
    (64, 56, 56, (3, 3), (1, 1), (1, 1), (1, 1)),
    (3, 224, 224, (7, 7), (2, 2), (3, 3), (1, 1)),
    (1, 5, 5, (3, 3), (1, 1), (3, 3), (1, 1)),
]


@pytest.mark.parametrize("shape", IM2COL_SHAPES)
def test_im2col_col2im_bit_exact(rng, shape):
    Cc, H, W, k, s, p, d = shape
    im = rng.standard_normal((Cc, H, W)).astype(np.float32)
    want = o.im2col(im, k, s, p, d)
    col = torch.empty(want.shape, device="cuda")
    capi.im2col(dev(im), col, k, s, p, d)
    assert np.array_equal(host(col), want)
    coln = torch.empty(want.shape, device="cuda")
    capi.im2col_nd(dev(im), coln, k, s, p, d)          # TestNDAgainst2D :606
    assert np.array_equal(host(coln), want)
    colr = rng.standard_normal(want.shape).astype(np.float32)
    want_im = o.col2im(colr, (Cc, H, W), k, s, p, d)
    back = torch.full((Cc, H, W), 7.0, device="cuda")   # must be overwritten, not accumulated
    capi.col2im(dev(colr), back, k, s, p, d)
    assert np.array_equal(host(back), want_im)
    backn = torch.full((Cc, H, W), 7.0, device="cuda")
    capi.col2im_nd(dev(colr), backn, k, s, p, d)
    assert np.array_equal(host(backn), want_im)


def test_im2col_nd_3d(rng):
    im = rng.standard_normal((2, 5, 6, 4)).astype(np.float32)
    k, s, p, d = (3, 2, 3), (2, 1, 1), (1, 0, 1), (1, 2, 1)
    want = o.im2col_nd(im, k, s, p, d)
    col = torch.empty(want.shape, device="cuda")
    capi.im2col_nd(dev(im), col, k, s, p, d)
    assert np.array_equal(host(col), want)
    colr = rng.standard_normal(want.shape).astype(np.float32)
    back = torch.empty(im.shape, device="cuda")
    capi.col2im_nd(dev(colr), back, k, s, p, d)
    assert np.array_equal(host(back), o.col2im_nd(colr, im.shape, k, s, p, d))


# ---------------------------------------------------------------------------------------------- BLAS
def test_sgemm_known_answers():
    data = np.arange(1, 13, dtype=np.float32)
    At = np.array([1, 4, 2, 5, 3, 6], np.float32)
    Bt = np.array([1, 5, 9, 2, 6, 10, 3, 7, 11, 4, 8, 12], np.float32)
    want = np.array([38, 44, 50, 56, 83, 98, 113, 128], np.float32)
    for tA, tB, A, B in ((0, 0, data[:6], data), (1, 0, At, data), (1, 1, At, Bt), (0, 1, data[:6], Bt)):
        Cm = torch.zeros(8, device="cuda")
        capi.sgemm(tA, tB, 2, 4, 3, 1.0, dev(A), dev(B), 0.0, Cm)
        assert np.array_equal(host(Cm), want)
    res = np.array([5, 11, 17], np.float32)
    Cm = dev(res.copy())
    capi.sgemm(0, 0, 3, 1, 2, 1.0, dev(data[:6]), dev(data[:2]), 1.0, Cm)
    assert np.array_equal(host(Cm), res * 2)


def test_sgemv_known_answers():
    A = np.arange(1, 7, dtype=np.float32)
    for tA, M, N, x, want in ((0, 2, 3, A[:3], [14, 32]), (1, 2, 3, A[:2], [9, 12, 15]),
                              (0, 3, 2, A[:2], [5, 11, 17]), (1, 3, 2, A[:3], [22, 28])):
        y = torch.zeros(len(want), device="cuda")
        capi.sgemv(tA, M, N, 1.0, dev(A), dev(x), 0.0, y)
        assert np.array_equal(host(y), np.array(want, np.float32))


GEMM_SHAPES = [(64, 3136, 576), (256, 196, 2304), (20, 576, 25), (127, 65, 33), (1, 1, 1), (512, 49, 4608),
               (128, 1200, 729), (96, 3025, 363)]


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
@pytest.mark.parametrize("tA,tB", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_sgemm_random_vs_oracle(rng, M, N, K, tA, tB):
    A = rng.standard_normal((K, M) if tA else (M, K)).astype(np.float32)
    B = rng.standard_normal((N, K) if tB else (K, N)).astype(np.float32)
    C0 = rng.standard_normal((M, N)).astype(np.float32)
    for alpha, beta in ((1.0, 0.0), (1.0, 1.0), (0.5, -2.0)):
        want = o.gemm(tA, tB, M, N, K, alpha, A, B, beta, C0, acc64=True)
        Cm = dev(C0.copy())
        capi.sgemm(tA, tB, M, N, K, alpha, dev(A), dev(B), beta, Cm)
        # NoTrans x Trans products with alpha = 1 and beta in {0, 1} (InnerProduct forward) may run on the tensor cores with the
        # fp32-equivalent bf16x3 split (1e-4 bar, like the convolutions); everything else is the exact-fp32 FFMA kernel
        tc = (tA, tB) == (0, 1) and K % 4 == 0 and K >= 64 and alpha == 1.0 and beta in (0.0, 1.0)
        assert rel_err(host(Cm), want) < (TOL_FP32 if tc else TOL_SIMT)


@pytest.mark.parametrize("M,N,K", [(64, 1000, 2048), (32, 512, 4096), (256, 10, 800), (64, 500, 800), (7, 130, 68)])
def test_sgemm_ex_split_k_vs_oracle(rng, M, N, K):
    """InnerProduct forward shapes (y = x W^T) through b2c_sgemm_ex with its workspace: the K loop is split over CTAs and the partial
    tiles reduced in a fixed order -- same tolerance as the unsplit tensor-core path, and bit-reproducible run to run."""
    A = rng.standard_normal((M, K)).astype(np.float32)
    B = (rng.standard_normal((N, K)) * (2.0 / K) ** 0.5).astype(np.float32)
    C0 = rng.standard_normal((M, N)).astype(np.float32)
    for beta in (0.0, 1.0):
        want = o.gemm(0, 1, M, N, K, 1.0, A, B, beta, C0, acc64=True)
        outs = []
        for _ in range(2):
            Cm = dev(C0.copy())
            _, nbytes = capi.sgemm_ex(0, 1, M, N, K, 1.0, dev(A), dev(B), beta, Cm)
            outs.append(host(Cm))
        assert rel_err(outs[0], want) < TOL_FP32
        assert np.array_equal(outs[0], outs[1])
    assert nbytes > 0 or K < 512


# ---------------------------------------------------------------------------------------------- conv
ENGINES = [("caffe", capi.ENGINE_CAFFE, None), ("implicit_simt", capi.ENGINE_CUDNN, capi.ALGO_SIMT),
           ("implicit_auto", capi.ENGINE_DEFAULT, capi.ALGO_AUTO)]


def run_conv(prm_case, engine, algo, math, rng):
    po, pc = make(o, prm_case), make(capi, prm_case)
    x, w, b, dy = tensors(rng, po)
    want_y = o.conv_forward(po, x, w, b, acc64=True)
    dw0 = rng.standard_normal(po.w_shape()).astype(np.float32) * 0.1      # pre-existing diffs: must be ADDED to
    db0 = rng.standard_normal(po.O).astype(np.float32) * 0.1 if po.has_bias else None
    want_dw, want_db, want_dx = o.conv_backward(po, x, w, dy, dw=dw0, db=db0, acc64=True)
    d = m.ConvDesc(pc, engine, math=math, algo=algo)
    X, Wt, Bv, DY = dev(x), dev(w), dev(b), dev(dy)
    Y = dev(np.full(po.y_shape(), 3.0, np.float32))
    d.forward(X, Wt, Bv, Y)
    DX = dev(np.full(po.x_shape(), 3.0, np.float32))
    d.backward_data(DY, Wt, DX)
    DW = dev(dw0.copy())
    d.backward_filter(X, DY, DW)
    got = dict(y=host(Y), dx=host(DX), dw=host(DW))
    want = dict(y=want_y, dx=want_dx, dw=want_dw)
    if po.has_bias:
        DB = dev(db0.copy())
        d.backward_bias(DY, DB)
        got["db"], want["db"] = host(DB), want_db
    return got, want, d


@pytest.mark.parametrize("ename,engine,algo", ENGINES, ids=[e[0] for e in ENGINES])
@pytest.mark.parametrize("name,case", ALL_CASES, ids=[c[0] for c in ALL_CASES])
def test_conv_forward_backward_vs_oracle_fp32(rng, name, case, ename, engine, algo):
    got, want, _ = run_conv(case, engine, algo, capi.MATH_FP32, rng)
    for k in want:
        assert got[k].shape == want[k].shape
        assert rel_err(got[k], want[k]) < TOL_FP32, (k, rel_err(got[k], want[k]))


@pytest.mark.parametrize("name,case", MODEL_CASES + EDGE_CASES, ids=[c[0] for c in MODEL_CASES + EDGE_CASES])
def test_conv_tf32_mode_within_1e3(rng, name, case):
    got, want, _ = run_conv(case, capi.ENGINE_DEFAULT, capi.ALGO_AUTO, capi.MATH_TF32, rng)
    for k in want:
        assert rel_err(got[k], want[k]) < TOL_TF32, (k, rel_err(got[k], want[k]))


PREP_CASES = ["resnet_res2_3x3", "resnet_res2_1x1_expand", "resnet_res3_1x1_s2", "alexnet_conv2_g2", "resnet_stem", "resnet_res5_3x3",
              "staged_5x5_c32", "lenet_conv1"]


@pytest.mark.parametrize("name", PREP_CASES)
def test_prepared_filter_cache_is_bitwise_equivalent(rng, name):
    """b2c_conv_prepare_filter + bind: forward / backward_data read the cached GEMM-ordered filter instead of re-deriving it;
    results must be bit-identical to the self-contained calls, and a stale cache must be the caller's problem only (new
    weights + re-prepare == fresh result)."""
    case = dict(ALL_CASES)[name]
    po, pc = make(o, case), make(capi, case)
    x, w, b, dy = tensors(rng, po)
    X, Wt, Bv, DY = dev(x), dev(w), dev(b), dev(dy)
    plain, cached = m.ConvDesc(pc), m.ConvDesc(pc)
    Y0, Y1 = torch.empty(po.y_shape(), device="cuda"), torch.empty(po.y_shape(), device="cuda")
    DX0, DX1 = torch.empty(po.x_shape(), device="cuda"), torch.empty(po.x_shape(), device="cuda")
    plain.forward(X, Wt, Bv, Y0); plain.backward_data(DY, Wt, DX0)
    has_cache = cached.prepare_filter(Wt)
    assert has_cache == (capi.ALGO_TCGEN05 in (cached.algo_used(0), cached.algo_used(1)))
    before = m.lib().b2c_launch_count()
    cached.forward(X, Wt, Bv, Y1); cached.backward_data(DY, Wt, DX1)
    launched = m.lib().b2c_launch_count() - before
    assert torch.equal(Y0, Y1) and torch.equal(DX0, DX1)
    if has_cache and cached.algo_used(0) == capi.ALGO_TCGEN05 and cached.algo_used(1) == capi.ALGO_TCGEN05:
        assert launched <= 3          # two conv kernels (+ the memset-free scatter path's none): no per-call prepass
    W2 = dev((w * 0.5 + 0.01).astype(np.float32))
    cached.prepare_filter(W2)
    plain.forward(X, W2, Bv, Y0); cached.forward(X, W2, Bv, Y1)
    assert torch.equal(Y0, Y1)
    cached.unbind_filter_cache()
    cached.forward(X, Wt, Bv, Y1); plain.forward(X, Wt, Bv, Y0)
    assert torch.equal(Y0, Y1)


ACC_CASES = dict(ALL_CASES)
ACC_CASES["staged_5x5_o64"] = dict(N=5, Cin=32, H=10, W=14, O=64, k=5, s=1, p=2, d=1, G=1, bias=True)   # dgrad reduces over O: O % 32 == 0


@pytest.mark.parametrize("name", ["resnet_res2_3x3", "resnet_res2_1x1_expand", "resnet_res4_3x3", "staged_5x5_o64", "resnet_res3_3x3"])
def test_backward_data_accumulate(rng, name):
    """dx += dgrad through the TMA reduce-add store == (dx0 + dgrad) computed separately, bit for bit (one fp32 add either way);
    covers tiles inside one image (TMA path) and tiles that span two (read-modify-write path)."""
    case = ACC_CASES[name]
    po, pc = make(o, case), make(capi, case)
    x, w, b, dy = tensors(rng, po)
    d = m.ConvDesc(pc)
    assert d.backward_data_accumulate_supported()
    dx0 = rng.standard_normal(po.x_shape()).astype(np.float32)
    Wt, DY = dev(w), dev(dy)
    DX = torch.empty(po.x_shape(), device="cuda")
    d.backward_data(DY, Wt, DX)
    want = dev(dx0) + DX
    ACC = dev(dx0)
    d.backward_data_accumulate(DY, Wt, ACC)
    assert torch.equal(ACC, want)
    # a layer the staged kernel does not take reports so, and the call refuses instead of silently overwriting
    d2 = m.ConvDesc(make(capi, dict(ALL_CASES)["resnet_res3_1x1_s2"]))
    assert not d2.backward_data_accumulate_supported()


def test_sobel_known_answer(rng):
    # test_convolution_layer.cpp:511-604 / CuDNN variant :1013-1110, tol 1e-4
    x = rng.standard_normal((2, 3, 6, 4)).astype(np.float32)
    w = np.tile(np.array([-1, 0, 1, -2, 0, 2, -1, 0, 1], np.float32), 3).reshape(1, 3, 3, 3)
    w1 = np.tile(np.array([1, 2, 1], np.float32), 3).reshape(1, 3, 3, 1)
    w2 = np.array([-1, 0, 1], np.float32).reshape(1, 1, 1, 3)
    for engine in (capi.ENGINE_CAFFE, capi.ENGINE_CUDNN):
        d = m.ConvDesc(capi.ConvParams.make(2, 3, 6, 4, 1, 3, 2, 0, 1, 1, False), engine)
        y = torch.empty(d.params.y_shape(), device="cuda")
        d.forward(dev(x), dev(w), None, y)
        d1 = m.ConvDesc(capi.ConvParams.make(2, 3, 6, 4, 1, (3, 1), (2, 1), 0, 1, 1, False), engine)
        t = torch.empty(d1.params.y_shape(), device="cuda")
        d1.forward(dev(x), dev(w1), None, t)
        d2 = m.ConvDesc(capi.ConvParams.make(2, 1, t.shape[2], t.shape[3], 1, (1, 3), (1, 2), 0, 1, 1, False), engine)
        y2 = torch.empty(d2.params.y_shape(), device="cuda")
        d2.forward(t, dev(w2), None, y2)
        assert y.shape == y2.shape
        assert np.abs(host(y) - host(y2)).max() <= 1e-4


def test_golden_fixtures_from_reference_build():
    z = np.load(os.path.join(GOLD, "conv_ref_golden.npz"))
    names = sorted(set(k.split("/")[0] for k in z.files))
    for nm in names:
        c = {k: int(v) for k, v in zip(z[nm + "/keys"], z[nm + "/vals"])}
        prm = capi.ConvParams(*[c[f] for f, _ in capi.ConvParams._fields_])
        for engine in (capi.ENGINE_CAFFE, capi.ENGINE_DEFAULT):
            d = m.ConvDesc(prm, engine)
            X, Wt, DY = dev(z[nm + "/x"]), dev(z[nm + "/w"]), dev(z[nm + "/dy"])
            Bv = dev(z[nm + "/b"]) if prm.has_bias else None
            Y = torch.empty(prm.y_shape(), device="cuda")
            d.forward(X, Wt, Bv, Y)
            DX = torch.empty(prm.x_shape(), device="cuda")
            d.backward_data(DY, Wt, DX)
            DW = torch.zeros(prm.w_shape(), device="cuda")
            d.backward_filter(X, DY, DW)
            assert rel_err(host(Y), z[nm + "/y"]) < TOL_FP32, nm
            assert rel_err(host(DX), z[nm + "/dx"]) < TOL_FP32, nm
            assert rel_err(host(DW), z[nm + "/dw"]) < TOL_FP32, nm
            if prm.has_bias:
                DB = torch.zeros(prm.O, device="cuda")
                d.backward_bias(DY, DB)
                assert rel_err(host(DB), z[nm + "/db"]) < TOL_FP32, nm


@pytest.mark.parametrize("name,case", FULL_SIZE_CASES, ids=[c[0] for c in FULL_SIZE_CASES])
def test_full_size_vs_reference_loop(rng, name, case):
    """The shapes and batch sizes the benchmark runs (BASELINE.json configs), forward + dgrad + wgrad (+ bias grad) in the
    default fp32-equivalent mode against the reference's own CPU structure -- verbatim im2col.cpp + per-image/per-group
    OpenBLAS sgemm (oracle/_ref) -- at 1e-4.  These launches run several tiles per persistent CTA (up to 3136 tiles on 148
    SMs) and the split-K plans that depend on N, which the small cases above never reach.  The reference's outputs are
    tests/golden/full_size_ref_golden.npz: each kept at the fixed positions cases.sample_index, with its max |value|."""
    z = np.load(os.path.join(GOLD, "full_size_ref_golden.npz"))
    pc = make(capi, case)
    x, w, b, dy, dw0 = full_size_inputs(rng, pc)      # dw0: pre-existing diff, accumulated into
    d = m.ConvDesc(pc)
    strided_k = case["s"] != 1 and case["k"] != 1      # no BASELINE layer of this kind needs a bottom gradient (conv1 only)
    for op in (0, 2) if strided_k else (0, 1, 2):
        assert d.algo_used(op) == capi.ALGO_TCGEN05, "full-size BASELINE layers must run on the tcgen05 kernels"
    X, Wt, Bv, DY = dev(x), dev(w), dev(b), dev(dy)
    Y = torch.full(pc.y_shape(), 3.0, device="cuda")
    d.forward(X, Wt, Bv, Y)
    DX = torch.full(pc.x_shape(), 3.0, device="cuda")
    d.backward_data(DY, Wt, DX)
    DW = dev(dw0)
    d.backward_filter(X, DY, DW)
    # y / dx reduce over K_dim <= 4608 terms: 1e-4.  dW reduces over N*Ho*Wo = 1.3e4 .. 1.6e6 terms in fp32 on BOTH sides (the
    # tensor core's fp32 accumulator here, OpenBLAS sgemm + image-by-image accumulation in the reference), so the two fp32
    # results drift apart with sqrt(terms): measured 1.02e-4 at 1.9e5 terms (AlexNet conv2, N = 256); bar 3e-4, a third of 1e-3.
    for k, got, tol in (("y", Y, TOL_FP32), ("dx", DX, TOL_FP32), ("dw", DW, 3e-4)):
        g = host(got).reshape(-1)[sample_index(got.numel())]
        e = float(np.abs(g.astype(np.float64) - z[f"{name}/{k}"]).max()) / float(z[f"{name}/{k}_absmax"])
        assert e < tol, (name, k, e)
    if pc.has_bias:
        DB = torch.zeros(pc.O, device="cuda")
        d.backward_bias(DY, DB)
        assert rel_err(host(DB), z[f"{name}/db"]) < TOL_FP32
    # run-to-run determinism of the split-K reductions (the reference accumulates in a fixed order too)
    DW2 = dev(dw0)
    d.backward_filter(X, DY, DW2)
    assert torch.equal(DW, DW2)


def test_full_size_properties_resnet50_layer(rng):
    """BASELINE full-size layer (res4 3x3, N=64): size-independent properties instead of the oracle.
    Adjointness <conv(x,w),dy> == <x,dgrad(dy,w)> == <w,wgrad(x,dy)> and linearity in x.
    (Reductions are done with numpy on the host: only this library's kernels run on the GPU.)"""
    prm = capi.ConvParams.make(64, 256, 14, 14, 256, 3, 1, 1, 1, 1, False)
    d = m.ConvDesc(prm)
    xh = rng.standard_normal(prm.x_shape()).astype(np.float32)
    x2h = rng.standard_normal(prm.x_shape()).astype(np.float32)
    wh = (rng.standard_normal(prm.w_shape()) * 0.02).astype(np.float32)
    dyh = rng.standard_normal(prm.y_shape()).astype(np.float32)
    x, x2, w, dy = dev(xh), dev(x2h), dev(wh), dev(dyh)
    y = torch.empty(prm.y_shape(), device="cuda")
    d.forward(x, w, None, y)
    dx = torch.empty(prm.x_shape(), device="cuda")
    d.backward_data(dy, w, dx)
    dw = dev(np.zeros(prm.w_shape(), np.float32))
    d.backward_filter(x, dy, dw)
    yh, dxh, dwh = host(y).astype(np.float64), host(dx).astype(np.float64), host(dw).astype(np.float64)
    a = float((yh * dyh).sum())
    b = float((xh * dxh).sum())
    c = float((wh * dwh).sum())
    scale = float(np.linalg.norm(yh) * np.linalg.norm(dyh))
    assert abs(a - b) / scale < 1e-5 and abs(a - c) / scale < 1e-5
    y2 = torch.empty(prm.y_shape(), device="cuda")
    d.forward(x2, w, None, y2)
    y3 = torch.empty(prm.y_shape(), device="cuda")
    d.forward(dev(2.0 * xh - 0.5 * x2h), w, None, y3)
    y3h = host(y3).astype(np.float64)
    assert np.abs(y3h - (2.0 * yh - 0.5 * host(y2))).max() / np.abs(y3h).max() < 1e-4


# ---------------------------------------------------------------------------------------------- SGD
@pytest.mark.parametrize("n", [1, 7, 1024, 100003])
def test_sgd_update_vs_oracle(rng, n):
    g, w, h = (rng.standard_normal(n).astype(np.float32) for _ in range(3))
    for l2 in (True, False):
        for clear in (True, False):
            want = o.sgd_update(g, w, h, 0.9, 0.01, 0.0005, l2=l2, grad_scale=0.125, clear_grads=clear)
            G, Wt, H = dev(g.copy()), dev(w.copy()), dev(h.copy())
            capi.sgd_update(G, Wt, H, 0.9, 0.01, 0.0005, l2=l2, grad_scale=0.125, clear_grads=clear)
            for a, b in zip((host(G), host(Wt), host(H)), want):
                assert np.allclose(a, b, rtol=2e-6, atol=1e-6)


def test_sgd_update_arena_vs_oracle(rng):
    # 161 segments like ResNet-50's learnable blobs, even-padded slots (net.cpp:1356-1371)
    counts = [int(c) for c in rng.integers(1, 70000, size=161)]
    counts[3], counts[10] = 1, 3
    offs, off = [], 0
    for c in counts:
        offs.append(off)
        off += c + (c & 1)
    total = off
    g, w, h = (rng.standard_normal(total).astype(np.float32) for _ in range(3))
    rates = [0.01 * (1 + (i % 3)) for i in range(len(counts))]
    decays = [0.0005 * (i % 2) for i in range(len(counts))]
    wg, ww, wh = g.copy(), w.copy(), h.copy()
    for of, c, lr, dc in zip(offs, counts, rates, decays):
        a, b, cc = o.sgd_update(g[of:of + c], w[of:of + c], h[of:of + c], 0.9, lr, dc, grad_scale=0.5)
        wg[of:of + c], ww[of:of + c], wh[of:of + c] = a, b, cc
    G, Wt, H = dev(g.copy()), dev(w.copy()), dev(h.copy())
    capi.sgd_update_arena(offs, counts, rates, decays, G, Wt, H, 0.9, grad_scale=0.5)
    for a, b in zip((host(G), host(Wt), host(H)), (wg, ww, wh)):
        assert np.allclose(a, b, rtol=2e-6, atol=1e-6)   # pad elements untouched too


def test_kernels_were_launched_by_this_library():
    before = m.lib().b2c_launch_count()
    y = torch.zeros(2, device="cuda")
    capi.sgemv(0, 2, 3, 1.0, dev(np.arange(1, 7, dtype=np.float32)), dev(np.ones(3, np.float32)), 0.0, y)
    assert m.lib().b2c_launch_count() == before + 1
