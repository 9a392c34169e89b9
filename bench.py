#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native Caffe-MPI training hot path.

Metric (BASELINE.json): images/sec, ResNet-50 fp32 training, batch 64 per GPU, synthetic ImageNet-shaped input.
One "step" = one Solver::Step iteration of the WHOLE prototxt graph (models/resnet50/train_val.prototxt semantics, generated
by caffe_mpi_b200/models.py because the reference tree does not exist on the GPU box): every layer forward and backward
through the C++ host layer (caffe::TrainNet), the bucketed gradient allreduce over the contiguous diff arena through
P2PSync / ReduceScheduler (N > 1, overlapped with the rest of backward) and the fused SGD-momentum update.  Nothing is
left out of the timed region.

  python bench.py --gpus N --steps K --warmup W [--model resnet50|alexnet|vgg16|googlenet|lenet] [--batch B]
                                                            (N>1: launched by torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                      (the reference's CPU conv path + host SGD on the host cores)
  python bench.py ... --dump-outputs DIR                    (also write what the last timed step computed, DIR/<name>.npy)

Prints ONE JSON line on rank 0 (key list in DESIGN.md "Measurement").
"""
import argparse
import csv
import glob
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODEL_TITLES = {"resnet50": "ResNet-50", "alexnet": "AlexNet", "vgg16": "VGG-16", "googlenet": "GoogLeNet", "lenet": "LeNet"}


def metric_name(model):
    return f"images/sec {MODEL_TITLES[model]} fp32 train"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained"),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


# ------------------------------------------------------------------------------------------- reference arm
def conv_inventory(model, batch):
    """[(count, oracle.ConvParams)] of the model's convolution layers, from the generated prototxt (host parser, CPU only)."""
    import oracle as o
    from caffe_mpi_b200 import host_api, models
    kw = dict(default_channels=1, default_size=28) if model == "lenet" else {}
    net = host_api.Net(models.PROTOTXT[model](batch), is_text=True, **kw)
    seen, order = {}, []
    first = True
    for name, p, prop_down in net.conv_layers():
        key = (p.C, p.H, p.W, p.O, p.G, p.kh, p.kw, p.sh, p.sw, p.ph, p.pw, p.has_bias, bool(prop_down))
        if key not in seen:
            seen[key] = [0, p, prop_down]
            order.append(key)
        seen[key][0] += 1
        first = False
    return [(seen[k][0], seen[k][1], seen[k][2]) for k in order]


def learnable_floats(model, batch=8):
    from caffe_mpi_b200 import host_api, models
    kw = dict(default_channels=1, default_size=28) if model == "lenet" else {}
    net = host_api.Net(models.PROTOTXT[model](batch), is_text=True, **kw)
    return sum(p[1] for p in net.learnable_params())


def reference_sample_runner(model):
    """Returns (run(n_images) -> seconds, cores, kind, description).  The reference's CPU ConvolutionLayer path: verbatim
    im2col.cpp (oracle/_ref) + per-image/per-group loop + OpenBLAS sgemm, plus the CPU SGD update of every learnable parameter;
    falls back to the plain-C oracle port when oracle/_ref or OpenBLAS is unavailable."""
    import numpy as np
    import oracle as o
    cores = os.cpu_count() or 1
    use_ref = o.ref() is not None and o.ref_blas_open(cores)
    state = {"threads": cores}
    rng = np.random.default_rng(1701)
    inv = conv_inventory(model, 1)
    nparam = learnable_floats(model)

    def run(nimg):
        t = 0.0
        for (cnt, cp, prop_down) in inv:
            prm = o.ConvParams.make(nimg, cp.C, cp.H, cp.W, cp.O, (cp.kh, cp.kw), (cp.sh, cp.sw), (cp.ph, cp.pw), 1, cp.G, bool(cp.has_bias))
            x = rng.standard_normal(prm.x_shape(), dtype=np.float32)
            w = rng.standard_normal(prm.w_shape(), dtype=np.float32) * np.float32((2.0 / prm.Kd) ** 0.5)
            dy = rng.standard_normal(prm.y_shape(), dtype=np.float32)
            b = np.zeros(prm.O, np.float32) if cp.has_bias else None
            y = np.empty(prm.y_shape(), np.float32)
            dw = np.zeros(prm.w_shape(), np.float32)
            db = np.zeros(prm.O, np.float32) if cp.has_bias else None
            dx = np.empty(prm.x_shape(), np.float32) if prop_down else None
            t0 = time.perf_counter()
            if use_ref:
                o.ref_conv_fwd_bwd(prm, x, w, b, y=y, dy=dy, dw=dw, db=db, dx=dx)
            else:
                o.conv_forward(prm, x, w, b)
                o.conv_backward(prm, x, w, dy, want_dx=bool(prop_down))
            t += (time.perf_counter() - t0) * cnt            # identical layers are timed once and counted `cnt` times
        g = np.zeros(nparam, np.float32); w_ = np.zeros(nparam, np.float32); h = np.zeros(nparam, np.float32)
        t0 = time.perf_counter()
        o.lib().b2o_sgd_update(nparam, g, w_, h, 0.9, 0.001, 1e-4, 1, 1.0, 1, 1)     # CPU branch of ComputeUpdateValue
        t += time.perf_counter() - t0
        return t

    if use_ref:
        # the reference's OpenBLAS uses every core by default, which is far from optimal for its per-image GEMMs on a
        # many-core host; give the CPU arm its best thread count out of {all, 64, 32, 16, 8} (1-image calibration)
        best = None
        for th in sorted({cores, 64, 32, 16, 8} & set(range(1, cores + 1)), reverse=True):
            o.ref_blas_open(th)
            run(1)
            t = run(1)
            if best is None or t < best[0]:
                best = (t, th)
        state["threads"] = best[1]
        o.ref_blas_open(best[1])
    kind = "port"   # the conv loop is a restatement; only im2col.cpp is the reference's own object code
    desc = (f"{MODEL_TITLES[model]} conv stack fwd+bwd (+ host SGD), reference im2col.cpp verbatim + OpenBLAS sgemm per image/group"
            if use_ref else f"{MODEL_TITLES[model]} conv stack fwd+bwd, plain-C oracle port (single thread)")
    if use_ref:
        desc += f" ({state['threads']} OpenBLAS threads = best of calibration, host has {cores} cores)"
    return run, (state["threads"] if use_ref else 1), kind, desc


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    run, cores, kind, desc = reference_sample_runner(args.model)
    run(1)                      # cold start (BLAS threads, page faults) is not the calibration
    t1 = run(1)
    S = max(1, min(8, int(4.0 / max(t1, 1e-3))))
    for _ in range(args.warmup):
        run(S)
    t0 = time.perf_counter()
    tt = 0.0
    for _ in range(args.steps):
        tt += run(S)
    wall = time.perf_counter() - t0
    ips = S * args.steps / tt
    out = {
        "impl": "reference", "metric": metric_name(args.model), "value": ips, "unit": "images/sec", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model} conv fwd+bwd + SGD on the host CPU (the reference's non-conv layers are not built "
                               f"here: the CPU arm is therefore FASTER than a full reference step), {S} images per step (bounded sample)",
                   "per_gpu_batch": args.batch},
        "cpu_baseline": {"value": ips, "unit": "images/sec", "cores": cores, "kind": kind,
                         "sample": f"{desc}; {S} images/step x {args.steps} steps; wall {wall:.1f}s"},
        "e2e": {"value": ips, "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out))


# ------------------------------------------------------------------------------------------- our arm
class ClockSampler:
    def __init__(self, idx):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(idx)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(kernel_substr):
    """DRAM bytes per launch of the kernels whose name contains `kernel_substr`, from the newest committed ncu launch list of
    this round (profiles/r02_*launches*.csv: gpu__time_duration.sum, dram__bytes_read.sum, dram__bytes_write.sum per launch).
    Returns (read_bytes, write_bytes, launches, file) or None."""
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r02_*launches*.csv")))      # r02_final_* sorts after the per-call r02_cN_* lists
    for path in reversed(files):
        try:
            rows = list(csv.reader(l for l in open(path) if l.startswith('"')))
            hdr = rows[0]
            iname, imet, ival, iunit = hdr.index("Kernel Name"), hdr.index("Metric Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
            iid = hdr.index("ID")
            rd, wr, ids = 0.0, 0.0, set()
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "B": 1.0, "KB": 1e3, "MB": 1e6, "GB": 1e9}
            for r in rows[1:]:
                if kernel_substr not in r[iname]:
                    continue
                v = float(r[ival].replace(",", "")) * scale.get(r[iunit], 1.0)
                if r[imet] == "dram__bytes_read.sum":
                    rd += v; ids.add(r[iid])
                elif r[imet] == "dram__bytes_write.sum":
                    wr += v
            if ids:
                return rd / len(ids), wr / len(ids), len(ids), os.path.relpath(path, ROOT)
        except Exception:
            continue
    return None


def run_ours(args):
    import torch
    import torch.distributed as dist
    import caffe_mpi_b200 as m
    from caffe_mpi_b200 import capi, host_api, models

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = m.lib()
    model, N = args.model, args.batch
    math = {"fp32": capi.MATH_FP32, "tf32": capi.MATH_TF32, "3xtf32": capi.MATH_FP32_3XTF32}[args.math]
    kw = dict(default_channels=1, default_size=28, num_classes=10) if model == "lenet" else {}
    net_text = models.PROTOTXT[model](N)
    if args.buckets > 0:
        net_text = f"reduce_buckets: {args.buckets}\n" + net_text
    if args.lmdb:                                    # opt-in: the Data layer reads this database (host/data_layer.cpp) instead of the synthetic source
        os.environ["B2C_DATA"] = "db"
        net_text = net_text.replace('source: "synthetic"', 'source: "%s"' % args.lmdb)
    t = host_api.Trainer(net_text, models.SOLVERS[model], batch=N, seed=1701 + rank, math=math, **kw)   # seed + rank, parallel.cpp:179-187
    if world > 1:
        ids = [t.new_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        t.attach_sync(world, rank, ids[0])           # P2PSync: weights broadcast from rank 0, bucketed allreduce per iteration

    def barrier():
        t.sync()
        if world > 1:
            dist.barrier()

    def mx(ms):
        if world == 1:
            return ms
        v = torch.tensor([ms], device=dev)
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        return float(v.item())

    # ---- headline: K steps, input batch resident in HBM, CUDA events on the net's stream, max over ranks ----------------
    t.step(args.warmup)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = L.b2c_launch_count()
    ms = mx(t.timed_steps(args.steps))
    launches = L.b2c_launch_count() - l0
    clocks = sampler.stop() if sampler else None
    loss = t.loss()
    if args.dump_outputs and rank == 0:
        dump_outputs(t, args.dump_outputs)
    # ---- end to end: every step copies the batch from pinned host memory and reads the loss back ---------------------------
    t.step(1, copy_input=True)
    barrier()
    ms_e2e = mx(t.timed_steps(args.steps, copy_input=True, read_loss=True))
    barrier()
    # ---- per-layer device times of the same step (CUDA events around every layer call), for the roofline block ---------------
    prof = t.profile(2)
    layers = t.layers()
    allreduce = time_allreduce(t, world, dev) if world > 1 else None
    if world > 1:
        # the same exchange inside the step: CUDA events around every bucket's allreduce on the comm stream, 3 steps, max over ranks
        t.bucket_timing(True)
        t.step(1)                         # the first step after the profiled ones starts with the ranks out of step: not recorded
        t.bucket_times()
        barrier()
        nst = 5
        t.step(nst)
        recs = t.bucket_times()
        t.bucket_timing(False)
        nb = len(recs) // nst
        if nb:
            # per bucket: the fastest of the steps (an allreduce cannot finish before the slowest rank has produced its gradients, so
            # every sample contains the ranks' skew; the minimum has the least of it), then the maximum over ranks
            ms_b = torch.tensor([[recs[s_ * nb + b_][1] for b_ in range(nb)] for s_ in range(nst)], device=dev).min(0).values
            dist.all_reduce(ms_b, op=dist.ReduceOp.MAX)
            by_b = [recs[b_][0] for b_ in range(nb)]
            f = 2.0 * (world - 1) / world
            allreduce["in_step_buckets"] = [{"bytes": by_b[b_], "ms": float(ms_b[b_]), "busbw_gbs": by_b[b_] * f / (float(ms_b[b_]) / 1e3) / 1e9}
                                            for b_ in range(nb)]
            allreduce["in_step_busbw_gbs"] = sum(by_b) * f / (float(ms_b.sum()) / 1e3) / 1e9

    if rank == 0:
        pk = peaks()
        imgs = N * world * args.steps
        value = imgs / (ms / 1e3)
        e2e_v = imgs / (ms_e2e / 1e3)
        # conv inventory of the net: FLOPs per layer and pass
        net_desc = host_api.Net(models.PROTOTXT[model](N), is_text=True, **{k: v for k, v in kw.items() if k != "num_classes"})
        conv = {name: (p, pd) for name, p, pd in net_desc.conv_layers()}
        fl = lambda p: 2.0 * p.N * p.O * (p.C // p.G) * p.kh * p.kw * (((p.H + 2 * p.ph - (p.dh * (p.kh - 1) + 1)) // p.sh) + 1) * (((p.W + 2 * p.pw - (p.dw * (p.kw - 1) + 1)) // p.sw) + 1)
        by_type, conv_ms, conv_fl = {}, {"fwd": 0.0, "wgrad": 0.0, "dgrad": 0.0}, {"fwd": 0.0, "wgrad": 0.0, "dgrad": 0.0}
        for li, op, v in prof:
            name, typ = layers[li]
            if typ == "Convolution":
                if op in conv_ms and not (op == "fwd" and False):
                    conv_ms[op] += v
                    conv_fl[op] += fl(conv[name][0])
                if op == "bwd":
                    by_type["Convolution bwd (wgrad + dgrad + bias grad)"] = by_type.get("Convolution bwd (wgrad + dgrad + bias grad)", 0.0) + v
                elif op == "fwd":
                    by_type["Convolution fwd"] = by_type.get("Convolution fwd", 0.0) + v
            elif op in ("fwd", "bwd"):
                by_type[f"{typ} {op}"] = by_type.get(f"{typ} {op}", 0.0) + v
        tf32_peak = pk["bf16_tflops"] / 2.0          # TF32 dense = half the bf16 rate on the same tensor pipe
        fam = {   # kernel families: algorithmic FLOPs / CUDA-event time of their launches inside the step
            "conv forward + data gradient (igemm_stg_kernel / igemm_fwd_kernel)": (conv_fl["fwd"] + conv_fl["dgrad"], conv_ms["fwd"] + conv_ms["dgrad"], "igemm"),
            "conv weight gradient (wgrad1x1_tma_kernel / igemm_wgrad_kernel + reduce)": (conv_fl["wgrad"], conv_ms["wgrad"], "wgrad"),
        }
        dom = max(fam, key=lambda k: fam[k][1])
        ach = fam[dom][0] / (fam[dom][1] / 1e3) / 1e12 if fam[dom][1] > 0 else 0.0
        tr = ncu_traffic("igemm_stg" if fam[dom][2] == "igemm" else "wgrad")
        step_ms = ms / args.steps
        out = {
            "metric": metric_name(model), "value": value, "unit": "images/sec", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "lmdb of raw uint8 datums (--lmdb)" if args.lmdb else "synthetic",
            "config": {"workload": f"{model}: full train_val graph, {len(layers)} layers forward + backward through caffe::TrainNet (C++), "
                                   + (f"bucketed NCCL allreduce of the {t.arena_floats() * 4 / 1e6:.1f} MB diff arena through P2PSync / ReduceScheduler overlapped with backward, "
                                      if world > 1 else "") + f"fused SGD-momentum update of {t.num_learnable()} learnable blobs; N={N}/GPU",
                       "model": model, "per_gpu_batch": N, "global_batch": N * world, "parallelism": f"dp{world}",
                       "reduce_buckets": args.buckets if args.buckets > 0 else 6,
                       "math": {"fp32": "fp32-equivalent: bf16x3 split (staged fwd/dgrad kernel) and 3xTF32 split (all other conv kernels), fp32 accumulate",
                                "tf32": "tf32 single pass (informational)", "3xtf32": "fp32-equivalent: 3xTF32 split everywhere"}[args.math],
                       "l2_policy": f"per-step activation working set {t.activation_floats() * 4 / 1e9:.2f} GB exceeds the 126 MB L2; every layer has its own blobs"},
            "gpu_launches": launches,
            "loss": loss,
            "e2e": {"value": e2e_v, "unit": "images/sec", "h2d_bytes_per_step": t.input_bytes() * world,
                    "d2h_bytes_per_step": 4 * world, "ms_per_step": ms_e2e / args.steps},
            "clocks": clocks,
            "allreduce": allreduce,
            "roofline": {"bound": "tensor", "achieved": ach, "peak": tf32_peak, "unit": "TFLOP/s", "frac": ach / tf32_peak if tf32_peak else None,
                         "kernel": dom,
                         "share_of_step": fam[dom][1] / step_ms if step_ms else None,
                         "traffic": (tr[0] + tr[1]) if tr else None,
                         "traffic_read_write": {"read": tr[0], "write": tr[1], "launches": tr[2], "file": tr[3], "unit": "bytes per launch (mean)"} if tr else None,
                         "peak_source": pk["source"] + ": bf16_tflops/2 (TF32 dense); fp32-equivalent ceilings: 2/3 of this peak for the "
                                        "bf16x3 kernel (three bf16 MMAs = 1.5 TF32 MMAs per MAC), 1/3 for the 3xTF32 kernels",
                         "families": {k: {"tflops": (v[0] / (v[1] / 1e3) / 1e12 if v[1] > 0 else None), "ms_per_step": round(v[1], 3),
                                          "frac": (v[0] / (v[1] / 1e3) / 1e12 / tf32_peak if v[1] > 0 else None)} for k, v in fam.items()},
                         "conv_ms_per_step": {k: round(v, 3) for k, v in conv_ms.items()},
                         # BASELINE.json configs[1] quotes AlexNet as "conv fwd/bwd only": the conv layers' share of this same step
                         "conv_only": {"ms_per_step": round(sum(conv_ms.values()), 3),
                                       "images_per_sec": (N / (sum(conv_ms.values()) / 1e3) if sum(conv_ms.values()) > 0 else None),
                                       "tflops": (sum(conv_fl.values()) / (sum(conv_ms.values()) / 1e3) / 1e12 if sum(conv_ms.values()) > 0 else None)}},
            "layer_ms_per_step": {k: round(v, 3) for k, v in sorted(by_type.items(), key=lambda kv: -kv[1])},
        }
        if world == 1 and not args.no_cpu_baseline:
            run, cores, kind, desc = reference_sample_runner(model)
            run(1)
            t1 = run(1)
            S = max(1, min(8, int(10.0 / max(t1, 1e-3))))
            tt = run(S) if S > 1 else t1
            out["cpu_baseline"] = {"value": S / tt, "unit": "images/sec", "cores": cores, "kind": kind,
                                   "sample": f"{desc}; {S} images once ({tt:.1f}s)"}
        print(json.dumps(out))
    if world > 1:
        barrier()
        dist.destroy_process_group()


DUMP_MAX_VALUES = 1 << 22     # per array: 16 MB of float32, so that a dump stays under 64 MB


def dump_outputs(t, out_dir):
    """What the last timed step handed back: the loss, the trainable parameters after the update and the solver's momentum
    history (the step the update took), each flattened over the blobs in net order, as float32 .npy files.  An array larger
    than DUMP_MAX_VALUES keeps the values at a fixed seeded sample of positions, the same for every run of the same model."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = t.num_params()
    arrays = {"loss": np.array([t.loss()], np.float32),
              "params": np.concatenate([t.get_param(i, 0) for i in range(n)]),
              "history": np.concatenate([t.get_param(i, 2) for i in range(n)])}
    for name, a in arrays.items():
        if a.size > DUMP_MAX_VALUES:
            a = a[np.sort(np.random.default_rng(1701).integers(0, a.size, DUMP_MAX_VALUES))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def time_allreduce(t, world, dev, reps=5):
    """Standalone in-place sum-allreduce of a buffer the size of the diff arena on a second communicator (nccl-tests
    convention for busbw), next to the in-step exchange that the headline already contains."""
    import torch
    import torch.distributed as dist
    from caffe_mpi_b200 import capi
    rank = dist.get_rank()
    ids = [capi.Comm.get_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    comm = capi.Comm(world, rank, ids[0])
    n = t.arena_floats()
    # the buffer the product path uses: ncclMemAlloc memory registered with the communicator (plain cudaMalloc memory if that fails)
    import ctypes as C
    L = capi.lib()
    L.b2c_comm_mem_alloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
    L.b2c_comm_mem_free.argtypes = [C.c_void_p]
    L.b2c_comm_register.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    L.b2c_comm_allreduce_sum.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    st = torch.cuda.Stream(device=dev)
    ptr, registered = C.c_void_p(), False
    if L.b2c_comm_mem_alloc(C.byref(ptr), n * 4) == 0:
        registered = L.b2c_comm_register(comm._h, ptr, n * 4) == 0
        buf = None
    else:
        buf = torch.zeros(n, device=dev)
        ptr = C.c_void_p(buf.data_ptr())
    sp = C.c_void_p(st.cuda_stream)

    comm_allreduce = lambda: capi.check(L.b2c_comm_allreduce_sum(comm._h, ptr, n, sp))
    for _ in range(2):
        comm_allreduce()
    st.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(st)
    for _ in range(reps):
        comm_allreduce()
    b.record(st)
    st.synchronize()
    v = torch.tensor([a.elapsed_time(b) / reps], device=dev)
    dist.all_reduce(v, op=dist.ReduceOp.MAX)
    ms_ = float(v.item())
    comm.destroy()
    if buf is None:
        L.b2c_comm_mem_free(ptr)
    algbw = n * 4 / (ms_ / 1e3) / 1e9
    return {"bytes": n * 4, "ms": ms_, "algbw_gbs": algbw, "busbw_gbs": algbw * 2 * (world - 1) / world, "nvlink_ref_gbs": 900.0,
            "buffer": "ncclMemAlloc + ncclCommRegister" if registered else "cudaMalloc"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="resnet50", choices=sorted(MODEL_TITLES))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the BASELINE.json config of the model)")
    ap.add_argument("--math", default="fp32", choices=["fp32", "tf32", "3xtf32"],
                    help="fp32 = fp32-equivalent split-precision tensor-core math (the headline); tf32 = single-pass TF32 (informational)")
    ap.add_argument("--buckets", type=int, default=0,
                    help="NetParameter.reduce_buckets of the generated prototxt (0 = the reference's default, 6; caffe.proto:140)")
    ap.add_argument("--lmdb", default="", help="train from this LMDB of raw uint8 Datums (tools/make_lmdb.py writes one) instead of the "
                                               "synthetic in-memory source; e2e then includes the parser threads and the database read")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the cpu_baseline leg (N = 1 only)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the loss, parameters and momentum history of the last one to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if not args.batch:
        from caffe_mpi_b200 import models
        args.batch = models.BASELINE_BATCH[args.model]
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
