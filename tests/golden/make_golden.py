"""Generate the golden fixtures under tests/golden/ from the reference, so that the tests which compare against it run
without it:

  conv     conv_ref_golden.npz         oracle/_ref, i.e. the reference's own src/caffe/util/im2col.cpp compiled verbatim,
                                       driven through the per-image / per-group ConvolutionLayer CPU loop with OpenBLAS
                                       cblas_sgemm/sgemv (the reference's BLAS := open), on small layers
  im2col   im2col_ref_digests.json     sha256 of oracle/_ref's im2col / col2im outputs (test_oracle.py's bit-exact tests)
  full     full_size_ref_golden.npz    the same conv loop on the FULL_SIZE_CASES layers, kept at cases.sample_index
  models   reference_models.json       the reference's models/*.prototxt and solver.prototxt files as this project's parser
                                       reads them (layers, convolutions, learnable parameters, solver settings)

  python tests/golden/make_golden.py [--ref REFERENCE_TREE] [conv] [im2col] [full] [models]      (default: all)

oracle/_ref is built by `make -C oracle ref REF=REFERENCE_TREE`; `models` reads REFERENCE_TREE itself."""
import argparse
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle as o  # noqa: E402
from cases import FULL_SIZE_CASES, REF_IM2COL_SHAPES, digest, full_size_inputs, make, sample_index  # noqa: E402

CASES = [
    ("simple", dict(N=2, Cin=3, H=6, W=4, O=4, k=3, s=2, p=0, d=1, G=1, bias=True)),
    ("group3", dict(N=2, Cin=6, H=6, W=4, O=3, k=3, s=2, p=0, d=1, G=3, bias=True)),
    ("dilated", dict(N=2, Cin=3, H=11, W=9, O=4, k=3, s=1, p=0, d=2, G=1, bias=True)),
    ("one_by_one", dict(N=2, Cin=8, H=6, W=4, O=4, k=1, s=1, p=0, d=1, G=1, bias=True)),
    ("rect", dict(N=2, Cin=4, H=9, W=11, O=5, k=(3, 5), s=(2, 1), p=(1, 2), d=(1, 1), G=1, bias=True)),
    ("res_3x3", dict(N=2, Cin=32, H=14, W=14, O=48, k=3, s=1, p=1, d=1, G=1, bias=False)),
    ("res_1x1_s2", dict(N=2, Cin=32, H=14, W=14, O=24, k=1, s=2, p=0, d=1, G=1, bias=False)),
    ("stem_7x7", dict(N=1, Cin=3, H=30, W=30, O=16, k=7, s=2, p=3, d=1, G=1, bias=False)),
    ("alex_g2", dict(N=2, Cin=16, H=13, W=13, O=24, k=5, s=1, p=2, d=1, G=2, bias=True)),
]

# name, prototxt under the reference tree, batch, parser defaults -- the batches and defaults test_prototxt.py builds the
# generated nets (caffe_mpi_b200/models.py) with
REF_MODELS = [
    ("resnet50", "models/resnet50/train_val.prototxt", 2, {}),
    ("alexnet", "models/bvlc_alexnet/train_val.prototxt", 8, {}),
    ("vgg16", "models/vgg16/train_val.prototxt", 8, {}),
    ("googlenet", "models/bvlc_googlenet/train_val.prototxt", 8, {}),
    ("lenet", "examples/mnist/lenet_train_test.prototxt", 8, dict(default_channels=1, default_size=28)),
]
REF_SOLVERS = [("resnet50", "models/resnet50/solver.prototxt"), ("alexnet", "models/bvlc_alexnet/solver.prototxt"),
               ("vgg16", "models/vgg16/solver.prototxt"), ("lenet", "examples/mnist/lenet_solver.prototxt")]


def conv_golden():
    assert o.ref() is not None and o.ref_blas_open(1), "oracle/_ref or OpenBLAS unavailable"
    rng = np.random.default_rng(1701)
    out = {}
    for name, c in CASES:
        prm = make(o, c)
        x = rng.standard_normal(prm.x_shape()).astype(np.float32)
        w = (rng.standard_normal(prm.w_shape()) * (2.0 / prm.Kd) ** 0.5).astype(np.float32)
        b = (rng.standard_normal(prm.O) * 0.1).astype(np.float32) if prm.has_bias else None
        dy = rng.standard_normal(prm.y_shape()).astype(np.float32)
        y = np.zeros(prm.y_shape(), np.float32)
        dw = np.zeros(prm.w_shape(), np.float32)
        db = np.zeros(prm.O, np.float32)
        dx = np.zeros(prm.x_shape(), np.float32)
        assert o.ref_conv_fwd_bwd(prm, x, w, b, y=y, dy=dy, dw=dw, db=db if prm.has_bias else None, dx=dx) == 0
        col0 = np.empty((prm.C * prm.kh * prm.kw, prm.Ho, prm.Wo), np.float32)
        o.ref().ref_im2col_cpu(np.ascontiguousarray(x[0]), prm.C, prm.H, prm.W, prm.kh, prm.kw, prm.ph, prm.pw,
                               prm.sh, prm.sw, prm.dh, prm.dw, col0)
        keys = [f for f, _ in o.ConvParams._fields_]
        out[name + "/keys"] = np.array(keys)
        out[name + "/vals"] = np.array([getattr(prm, k) for k in keys], np.int64)
        for k, v in (("x", x), ("w", w), ("dy", dy), ("y", y), ("dw", dw), ("dx", dx), ("col0", col0)):
            out[name + "/" + k] = v
        if prm.has_bias:
            out[name + "/b"] = b
            out[name + "/db"] = db
    return "conv_ref_golden.npz", out


def im2col_golden():
    """The inputs are drawn as test_oracle.py draws them (the `rng` fixture: default_rng(1701), fresh per test)."""
    R = o.ref()
    assert R is not None, "oracle/_ref unavailable"
    i32 = lambda v: np.asarray(v, np.int32)
    out = {}
    for shape in REF_IM2COL_SHAPES:
        Cc, H, W, k, s, p, d = shape
        rng = np.random.default_rng(1701)
        im = rng.standard_normal((Cc, H, W)).astype(np.float32)
        Ho = (H + 2 * p[0] - (d[0] * (k[0] - 1) + 1)) // s[0] + 1
        Wo = (W + 2 * p[1] - (d[1] * (k[1] - 1) + 1)) // s[1] + 1
        col = np.empty((Cc * k[0] * k[1], Ho, Wo), np.float32)
        R.ref_im2col_cpu(im, Cc, H, W, k[0], k[1], p[0], p[1], s[0], s[1], d[0], d[1], col)
        colr = rng.standard_normal(col.shape).astype(np.float32)
        back = np.empty_like(im)
        R.ref_col2im_cpu(colr, Cc, H, W, k[0], k[1], p[0], p[1], s[0], s[1], d[0], d[1], back)
        coln, backn = np.empty_like(col), np.empty_like(im)
        R.ref_im2col_nd_cpu(im, 2, i32(im.shape), i32(col.shape), i32(k), i32(p), i32(s), i32(d), coln)
        R.ref_col2im_nd_cpu(colr, 2, i32(im.shape), i32(col.shape), i32(k), i32(p), i32(s), i32(d), backn)
        out[repr(shape)] = dict(im=digest(im), colr=digest(colr), col=digest(col), col2im=digest(back), col_nd=digest(coln),
                                col2im_nd=digest(backn))
    # test_im2col_3d_nd: three spatial axes through the N-D source
    im = np.random.default_rng(1701).standard_normal((2, 5, 6, 4)).astype(np.float32)
    k, s, p, d = (3, 2, 3), (2, 1, 1), (1, 0, 1), (1, 2, 1)
    col = np.empty((2 * 18, 3, 4, 4), np.float32)
    R.ref_im2col_nd_cpu(im, 3, i32(im.shape), i32(col.shape), i32(k), i32(p), i32(s), i32(d), col)
    out["3d"] = dict(im=digest(im), col_nd=digest(col))
    return "im2col_ref_digests.json", out


def full_golden():
    """Inputs drawn as test_gpu_parity.py::test_full_size_vs_reference_loop draws them; every output is kept at
    sample_index(size) together with its max |value| (the denominator of the blob-level relative error), bias grads whole."""
    assert o.ref() is not None and o.ref_blas_open(os.cpu_count() or 1), "oracle/_ref or OpenBLAS unavailable"
    out = {}
    for name, case in FULL_SIZE_CASES:
        po = make(o, case)
        x, w, b, dy, dw0 = full_size_inputs(np.random.default_rng(1701), po)
        y = np.empty(po.y_shape(), np.float32)
        dw = dw0.copy()
        db = np.zeros(po.O, np.float32) if po.has_bias else None
        dx = np.empty(po.x_shape(), np.float32)
        o.ref_conv_fwd_bwd(po, x, w, b, y=y, dy=dy, dw=dw, db=db, dx=dx)
        for k, v in (("y", y), ("dx", dx), ("dw", dw)):
            out[f"{name}/{k}"] = v.reshape(-1)[sample_index(v.size)]
            out[f"{name}/{k}_absmax"] = np.float64(np.abs(v).max())
        if po.has_bias:
            out[f"{name}/db"] = db
        print(name, flush=True)
    return "full_size_ref_golden.npz", out


def models_golden(ref):
    from caffe_mpi_b200 import host_api as h
    fields = lambda p: [getattr(p, f) for f, _ in p._fields_]
    out = {"conv_fields": [f for f, _ in h.capi.ConvParams._fields_], "models": {}, "solvers": {}}
    for name, path, batch, kw in REF_MODELS:
        n = h.Net(os.path.join(ref, path), "TRAIN", batch_override=batch, **kw)
        out["models"][name] = dict(file=path, batch=batch, parser_defaults=kw,
                                   layers=[[nm, t, list(s)] for nm, t, s in n.layers()],
                                   convs=[[nm, fields(p), pd] for nm, p, pd in n.conv_layers()],
                                   params=[list(p) for p in n.learnable_params()])
    for name, path in REF_SOLVERS:
        s, net = h.solver_from_prototxt(os.path.join(ref, path))
        out["solvers"][name] = dict(file=path, net=net, **h.solver_describe(s))
    return "reference_models.json", out


def to_json(v, ind=0):
    """JSON with one table row (a list of lists' element) per line, so that the fixture reads as a table."""
    pad = " " * (ind + 1)
    if isinstance(v, dict):
        return "{\n" + ",\n".join(f"{pad}{json.dumps(k)}: {to_json(x, ind + 1)}" for k, x in sorted(v.items())) + "\n" + " " * ind + "}"
    if isinstance(v, list) and v and isinstance(v[0], list):
        return "[\n" + ",\n".join(pad + json.dumps(r) for r in v) + "\n" + " " * ind + "]"
    return json.dumps(v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", default=os.environ.get("REF", ""), help="the reference tree (needed by `models`)")
    ap.add_argument("which", nargs="*", default=["conv", "im2col", "full", "models"])
    args = ap.parse_args()
    for which in args.which:
        name, out = {"conv": conv_golden, "im2col": im2col_golden, "full": full_golden,
                     "models": lambda: models_golden(args.ref)}[which]()
        path = os.path.join(HERE, name)
        if name.endswith(".npz"):
            np.savez_compressed(path, **out)
        else:
            with open(path, "w") as f:
                f.write(to_json(out) + "\n")
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
