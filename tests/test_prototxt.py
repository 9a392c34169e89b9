"""CPU tests of the text-format prototxt reader and the Net graph builder (host/prototxt.cpp, SURVEY 8(f) rank 1).
Part 1 uses small nets written here; part 2 takes the reference's own models/*.prototxt and solver.prototxt files as this
parser read them UNMODIFIED (tests/golden/reference_models.json, written by tests/golden/make_golden.py) and checks those
inventories against SURVEY Appendix A, against caffe_mpi_b200/shapes.py and against the nets and solvers that
caffe_mpi_b200/models.py generates for bench.py."""
import json
import os

import pytest

from caffe_mpi_b200 import capi, host_api as h
from caffe_mpi_b200.shapes import MODELS, EXTRA_PARAMS

TINY = """
name: "tiny"   # comment
reduce_buckets: 3
layer { name: "data" type: "Data" top: "data" top: "label"
        data_param { source: "x" batch_size: 16 backend: LMDB } transform_param { crop_size: 32 mirror: true }
        include { phase: TRAIN } }
layer { name: "data" type: "Data" top: "data" top: "label" data_param { batch_size: 4 } transform_param { crop_size: 32 }
        include: { phase: TEST } }
layer { name: "conv1" type: "Convolution" bottom: "data" top: "conv1"
        param { lr_mult: 1 decay_mult: 1 } param { lr_mult: 2 decay_mult: 0 }
        convolution_param { num_output: 8 kernel_size: 5 stride: 2 pad: 1 weight_filler { type: "gaussian" std: 0.01 }
                            bias_filler { type: "constant" value: 0.1 } } }
layer { name: "relu1" type: "ReLU" bottom: "conv1" top: "conv1" }
layer { name: "pool1" type: "Pooling" bottom: "conv1" top: "pool1" pooling_param { pool: MAX kernel_size: 3 stride: 2 } }
layer { name: "conv2" type: "Convolution" bottom: "pool1" top: "conv2"
        convolution_param { num_output: 12 kernel_h: 3 kernel_w: 1 pad_h: 1 pad_w: 0 group: 2 bias_term: false engine: CAFFE } }
layer { name: "bn" type: "BatchNorm" bottom: "conv2" top: "bn" batch_norm_param { scale_bias: true eps: 1e-4 } }
layer { name: "sum" type: "Eltwise" bottom: "bn" bottom: "conv2" top: "sum" }
layer { name: "gp" type: "Pooling" bottom: "sum" top: "gp" pooling_param { pool: AVE global_pooling: true } }
layer { name: "fc" type: "InnerProduct" bottom: "gp" top: "fc" inner_product_param { num_output: 10 } }
layer { name: "acc" type: "Accuracy" bottom: "fc" bottom: "label" top: "acc" include { phase: TEST } }
layer { name: "loss" type: "SoftmaxWithLoss" bottom: "fc" bottom: "label" top: "loss" }
"""


def test_parse_tiny_net_train_phase():
    n = h.Net(TINY, "TRAIN", is_text=True)
    layers = n.layers()
    assert [l[0] for l in layers] == ["data", "conv1", "relu1", "pool1", "conv2", "bn", "sum", "gp", "fc", "loss"]   # Accuracy filtered out
    shapes = {l[0]: l[2] for l in layers}
    assert shapes["data"] == (16, 3, 32, 32)
    assert shapes["conv1"] == (16, 8, 15, 15)          # (32 + 2 - 5)/2 + 1, truncating
    assert shapes["pool1"] == (16, 8, 7, 7)            # ceil((15 - 3)/2) + 1
    assert shapes["conv2"] == (16, 12, 7, 7)
    assert shapes["gp"] == (16, 12, 1, 1)
    assert shapes["fc"] == (16, 10)
    assert n.reduce_buckets() == 3
    convs = n.conv_layers()
    assert [c[0] for c in convs] == ["conv1", "conv2"]
    p1, p2 = convs[0][1], convs[1][1]
    assert (p1.kh, p1.kw, p1.sh, p1.ph, p1.has_bias, p1.G) == (5, 5, 2, 1, 1, 1)
    assert (p2.kh, p2.kw, p2.ph, p2.pw, p2.has_bias, p2.G) == (3, 1, 1, 0, 0, 2)
    assert convs[0][2] is False and convs[1][2] is True      # conv1's bottom is data: no bottom gradient (net.cpp:183-191)
    params = n.learnable_params()
    assert [(p[0], p[1]) for p in params] == [("conv1", 8 * 3 * 25), ("conv1", 8), ("conv2", 12 * 4 * 3), ("bn", 12), ("bn", 12),
                                              ("fc", 10 * 12), ("fc", 10)]
    assert params[1][2:] == (2.0, 0.0)                        # ParamSpec of the bias blob


def test_phase_filter_and_batch_override():
    n = h.Net(TINY, "TEST", is_text=True)
    assert "acc" in [l[0] for l in n.layers()]
    assert n.layers()[0][2] == (4, 3, 32, 32)
    n2 = h.Net(TINY, "TRAIN", batch_override=64, is_text=True)   # per-rank batch (parallel.cpp:284-293)
    assert n2.layers()[0][2][0] == 64 and n2.conv_layers()[0][1].N == 64


@pytest.mark.parametrize("bad,msg", [
    ('layer { name: "c" type: "Convolution" bottom: "nope" top: "c" convolution_param { num_output: 1 kernel_size: 1 } }', "Unknown bottom blob"),
    ('layer { name: "x" type: "FancyNewLayer" top: "x" }', "Unknown layer type"),
    ('layer { name: "x" type: "Input" top: "x" ', "missing '}'"),
    ('layer { name: "x" type: "Input" top: "x" input_param { shape { dim: 1 dim: 3 dim: 8 dim: 8 } } }\n'
     'layer { name: "c" type: "Convolution" bottom: "x" top: "c" convolution_param { num_output: 4 kernel_size: 0 } }', "Filter dimensions must be nonzero"),
])
def test_malformed_prototxt_is_fatal(bad, msg):
    with pytest.raises(h.HostError, match=msg):
        h.Net(bad, "TRAIN", is_text=True)


def test_solver_prototxt_text():
    s, net = h.solver_from_prototxt('net: "a/b.prototxt"\nbase_lr: 0.01 momentum: 0.9 weight_decay: 0.0005 lr_policy: "inv" gamma: 0.0001 power: 0.75\n'
                                    'max_iter: 10000 display: 100 solver_mode: GPU # lenet', is_text=True)
    assert net == "a/b.prototxt"
    d = h.solver_describe(s)
    assert d["lr_policy"] == "inv" and d["max_iter"] == 10000 and abs(d["momentum"] - 0.9) < 1e-6
    assert s.lr_at(100) == pytest.approx(0.01 * (1 + 1e-4 * 100) ** -0.75, rel=1e-6)
    with pytest.raises(h.HostError, match="SGD only"):
        h.solver_from_prototxt('type: "Adam" base_lr: 0.1', is_text=True)


# ---------------------------------------------------------------------------------------- the reference's own prototxts
def reference_models():
    with open(os.path.join(os.path.dirname(__file__), "golden", "reference_models.json")) as f:
        r = json.load(f)
    assert r["conv_fields"] == [f for f, _ in capi.ConvParams._fields_]
    return r


REF_MODELS = [
    # name, convs, fwd GF/img, learnable blobs, learnable floats   (SURVEY Appendix A)
    ("resnet50", 53, 7.712, 161, 25557032),
    ("alexnet", 5, 1.332, 16, 60965224),
    ("vgg16", 13, 30.693, 32, 138357544),
    ("googlenet", 59, 3.168, 128, 13378280),
    ("lenet", 2, 0.003776, 8, 431080),
]


@pytest.mark.parametrize("name,nconv,gf,nblobs,nfloats", REF_MODELS, ids=[m[0] for m in REF_MODELS])
def test_reference_model_inventory(name, nconv, gf, nblobs, nfloats):
    r = reference_models()["models"][name]
    convs = [(nm, capi.ConvParams(*v), pd) for nm, v, pd in r["convs"]]
    assert len(convs) == nconv
    assert sum(p.flops() for _, p, _ in convs) / r["batch"] / 1e9 == pytest.approx(gf, rel=2e-3)
    params = r["params"]
    assert len(params) == nblobs and sum(c for _, c, _, _ in params) == nfloats
    assert convs[0][2] is False and all(pd for _, _, pd in convs[1:])
    if name in MODELS:     # the table bench.py uses must be exactly what the prototxt says
        table = []
        for (cnt, C, H, O, k, s, p, G, b) in MODELS[name]:
            table += [(C, H, O, k, s, p, G, int(b))] * cnt
        got = sorted((p.C, p.H, p.O, p.kh, p.sh, p.ph, p.G, p.has_bias) for _, p, _ in convs)
        assert got == sorted(table)
        conv_floats = sum(c for layer, c, _, _ in params if layer in {nm for nm, _, _ in convs})
        assert nfloats - conv_floats == EXTRA_PARAMS[name]


def test_reference_solver_prototxts():
    """The reference's solver files against the solver settings bench.py trains with (caffe_mpi_b200.models.SOLVERS)."""
    from caffe_mpi_b200 import models
    solvers = reference_models()["solvers"]
    assert sorted(solvers) == ["alexnet", "lenet", "resnet50", "vgg16"]
    for name, d in solvers.items():
        assert d["net"].endswith(".prototxt") and d["max_iter"] > 0
        s, net = h.solver_from_prototxt(models.SOLVERS[name], is_text=True)
        assert h.solver_describe(s) == {k: d[k] for k in ("base_lr", "momentum", "weight_decay", "max_iter", "iter_size", "lr_policy")}
    for name, policy, lr in (("resnet50", "poly", 0.001), ("lenet", "inv", 0.01)):
        assert solvers[name]["lr_policy"] == policy and solvers[name]["base_lr"] == pytest.approx(lr)


def test_generated_resnet50_has_the_reference_inventory():
    """caffe_mpi_b200.models.resnet50_prototxt (what bench.py trains) against the inventory of
    models/resnet50/train_val.prototxt: SURVEY Appendix A numbers, and layer by layer."""
    from caffe_mpi_b200 import host_api, models
    net = host_api.Net(models.resnet50_prototxt(2), "TRAIN", is_text=True)
    params = net.learnable_params()
    assert len(net.conv_layers()) == 53 and len(params) == 161
    assert sum(p[1] for p in params) == 25557032
    r = reference_models()["models"]["resnet50"]
    assert r["batch"] == 2
    assert net.layers() == [(n, t, tuple(shp)) for n, t, shp in r["layers"] if t != "Accuracy"]
    assert params == [tuple(p) for p in r["params"]]
    fields = lambda p: [getattr(p, f) for f, _ in p._fields_]
    assert [[n, fields(p), pd] for n, p, pd in net.conv_layers()] == r["convs"]


GENERATED = [("alexnet", {}), ("vgg16", {}), ("googlenet", {}), ("lenet", dict(default_channels=1, default_size=28))]


@pytest.mark.parametrize("name,kw", GENERATED, ids=[g[0] for g in GENERATED])
def test_generated_prototxt_has_the_reference_inventory(name, kw):
    """caffe_mpi_b200/models.py generators (what bench.py trains) against the reference's own model files: same TRAIN-phase
    layer list (name, type), conv shapes and learnable-parameter list."""
    from caffe_mpi_b200 import host_api, models
    r = reference_models()["models"][name]
    assert r["parser_defaults"] == kw
    g = host_api.Net(models.PROTOTXT[name](r["batch"]), is_text=True, **kw)
    fields = lambda p: [getattr(p, f) for f, _ in p._fields_]
    assert r["convs"] == [[n, fields(p), pd] for n, p, pd in g.conv_layers()]
    assert [x[1:] for x in r["params"]] == [list(x[1:]) for x in g.learnable_params()]
    keep = lambda layers: [(n, t) for n, t, _ in layers if t not in ("Accuracy", "Data", "Input")]
    assert keep(r["layers"]) == keep(g.layers())
