#!/usr/bin/env python
"""Benchmark of the DINO training step (BASELINE.json metric: DINO train samples/s + roofline fraction, next to the
host-CPU reference path).

    python bench.py --gpus N --steps K --warmup W            # our arm (one process per GPU; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on the host cores
    python bench.py ... --dump-outputs DIR                   # + the last timed step's loss and weights as DIR/<name>.npy

Workload (config.workload): BASELINE.json configs[1] -- multimodal central DINO (CentralMultiModalEncoder, image 28x28 +
spectrogram 112x112, 2 global + 4 local views, tuned YAML augmentations, E=O=256, P=128), default training mode, synthetic
AVMNIST-shaped data, per-GPU batch --batch (weak scaling).  One step = augmentation (device-sampled) + student/teacher
forward + fused DINO loss + centre EMA + teacher EMA + backward + gradient all-reduce (N > 1) + Adam.
Prints ONE JSON line on rank 0.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "DINO train samples/sec"
UNIT = "samples/s"
WORKLOAD = "multi_central DINO step (2 global + 4 local views, img 28x28 + spec 112x112, E=O=256, P=128), default mode"


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm_gbs": float(p["hbm_gbs"]), "tflops": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "source": "measured"}
    except Exception:
        return {"hbm_gbs": 6650.0, "tflops": 1400.0, "source": "fallback"}


def augment_values():
    import yaml
    from multimodal_ssl_avmnist_b200 import augment as A
    cfg = yaml.safe_load(open(os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments", "configs", "config_multimodal_dino.yaml")))
    return A.values_from_config(cfg)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes every tensor of `arrays` as out_dir/<name>.npy (float64 stays float64, everything else becomes float32).  The
    inputs of the timed path are seeded, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    import torch
    host = {name: t.detach().to("cpu", torch.float64 if t.dtype == torch.float64 else torch.float32).numpy() for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_LIMIT_BYTES})")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.proc, self.path = None, None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                                          str(gpu_index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(self.proc.kill)       # never outlives the benchmark, even when it fails before stop()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference(batch, steps, warmup, cores, with_aug=True, kind="multi_central", mode="default"):
    """The reference's CPU path for this workload (oracle port): torchvision-composed augmentation in `cores` worker
    processes + the fp32 torch-CPU step (forward, loss, EMA, backward, Adam) with `cores` intra-op threads.
    Returns (samples/s, ms per step, description)."""
    import torch
    from oracle import augment_tv as TV
    from oracle import dino_ref as R
    from oracle.fixtures import make_masks, synth_views, views_to_vb
    torch.set_num_threads(cores)
    from oracle.fixtures import synth_raw
    if kind.startswith("contrastive"):     # other_ssl/info_nce, other_ssl/multimodal_simclr: the oracle's contrastive_step (no augmentation timed)
        from oracle.fixtures import contrastive_batch
        ck = kind.split("_", 1)[1]
        st = R.ContrastiveState(seed=1)
        img1, spec1, img2, spec2 = contrastive_batch(batch, 0)
        data = (img1, spec1) if ck == "infonce" else (img1, spec1, img2, spec2)
        for i in range(warmup):
            R.contrastive_step(st, ck, data, mode=i % 4)
        t0 = time.perf_counter()
        for i in range(steps):
            R.contrastive_step(st, ck, data, mode=i % 4)
        step_s = (time.perf_counter() - t0) / steps
        rate = batch / step_s
        return rate, 1e3 * step_s, (f"{steps} steps of B={batch} of the {ck} step (fwd+loss+bwd+Adam, fp32 torch CPU, {cores} threads): "
                                    f"{rate:.1f} samples/s; augmentation not timed")
    if kind not in R.KIND_MIX:
        kind = "multi_central"          # (image_simple: the multimodal oracle step stands in; only the headline kinds are compared)
    st = R.CentralDinoState(seed=1, mode=mode, kind=kind)
    img, aud = views_to_vb(*synth_views(batch, seed=1))
    masks = make_masks(seed=2, V=6, Vg=2, B=batch, E=256, hidden=512)
    raw = labels = None
    if mode != "default":
        image, audio, labels = synth_raw(batch, seed=3)
        raw = (image, audio)
    for _ in range(warmup):
        R.central_dino_step(st, img, aud, masks, raw=raw, labels=labels)
    t0 = time.perf_counter()
    for _ in range(steps):
        R.central_dino_step(st, img, aud, masks, raw=raw, labels=labels)
    step_s = (time.perf_counter() - t0) / steps
    step_rate = batch / step_s
    aug_rate = None
    if with_aug:
        per_worker = max(2, min(8, batch // cores))
        aug_rate = TV.time_augmentation(per_worker, cores, augment_values())
    rate = min(step_rate, aug_rate) if aug_rate else step_rate
    desc = (f"{steps} steps of B={batch} (fwd+loss+EMA+bwd+Adam, fp32 torch CPU, {cores} threads): {step_rate:.1f} samples/s; "
            + (f"augmentation (torchvision chains, {cores} worker processes): {aug_rate:.1f} samples/s; value = min of the two" if aug_rate
               else "augmentation not timed"))
    return rate, 1e3 * batch / rate, desc


def run_reference_on_gpu(args):
    """Library-kernel bar (SURVEY 8d): the oracle's restatement of the reference step (the same torch calls as models/dino.py /
    models/unimodal.py) moved to cuda:0 and run the way the reference runs on a GPU -- eager ATen / cuDNN / cuBLAS, fp16
    autocast (run_dino.py:360) unless --reference-fp32.  Inputs are ALREADY-AUGMENTED views resident in HBM: the reference has
    no GPU augmentation (its torchvision chains run in DataLoader workers), so this bar EXCLUDES the augmentation that our step
    includes.  A reported baseline beside the CPU arm, never part of the product path."""
    import torch
    from oracle import dino_ref, fixtures

    def to_cuda(obj):
        if torch.is_tensor(obj):
            return obj.cuda()
        if isinstance(obj, dict):
            return {k: to_cuda(v) for k, v in obj.items()}
        if isinstance(obj, (list, tuple)):
            return type(obj)(to_cuda(v) for v in obj)
        return obj

    torch.backends.cudnn.benchmark = True
    B, V, Vg = args.batch, 6, 2
    st = dino_ref.CentralDinoState(seed=0)
    for name, val in list(vars(st).items()):
        setattr(st, name, to_cuda(val))
    g = torch.Generator(device="cuda").manual_seed(1)
    img = torch.rand(V, B, 1, 28, 28, device="cuda", generator=g)
    aud = torch.rand(V, B, 1, 112, 112, device="cuda", generator=g)
    masks = to_cuda(fixtures.make_masks(3, V, Vg, B, st.E, 512))

    def step():
        with torch.autocast("cuda", dtype=torch.float16, enabled=not args.reference_fp32):
            return dino_ref.central_dino_step(st, img, aud, masks)["loss"]

    for _ in range(max(args.warmup, 3)):
        loss = step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    rate = B / ms * 1e3
    prec = "fp32 (torch defaults)" if args.reference_fp32 else "fp16 autocast (run_dino.py:360)"
    print(json.dumps({"metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
                      "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "f32" if args.reference_fp32 else "f16", "data": "synthetic",
                      "config": {"workload": WORKLOAD, "per_gpu_batch": B, "inputs": "pre-augmented views resident in HBM (no augmentation timed)",
                                 "execution": "stock PyTorch eager kernels (cuDNN / cuBLAS / ATen) on cuda:0, " + prec},
                      "impl": "reference", "library_bar": True, "last_loss": float(loss),
                      "torch": torch.__version__, "cudnn": torch.backends.cudnn.version()}))


REF_SAMPLE_BATCH = 64        # the CPU arm steps on a fixed 64-sample slice of the workload's batch (pinned: same B in every run)


def workload_config(args, world):
    """The `config` object of the JSON line -- identical for our arm and the reference arm."""
    B = per_gpu_batch(args, world)
    if args.kind.startswith("multi"):
        wl = WORKLOAD if args.mode == "default" else WORKLOAD.replace("default mode", args.mode + " mode")
        if args.kind != "multi_central":            # the 3x3 conv encoders of SURVEY 8f-4 (models/dino.py:214-263, 385-452)
            wl = wl.replace("multi_central", args.kind)
    elif args.kind == "contrastive_infonce":
        wl = "stand-alone multimodal InfoNCE step (ImageEncoder + SpectrogramEncoder + 2 projection heads, un-augmented batch)"
    elif args.kind == "contrastive_simclr":
        wl = "multimodal SimCLR step (2 augmented views per modality, random modality pairing, NT-Xent)"
    else:
        wl = "image_simple unimodal DINO step (2 global + 4 local views of 28x28 images, O=256, P=128)"
    return {"workload": wl, "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
            "l2": "inputs larger than L2: the per-step working set (activations) is several GB against the 126 MB L2"}


def per_gpu_batch(args, world):
    if args.global_batch:
        if args.global_batch % world:
            raise SystemExit(f"--global-batch {args.global_batch} is not divisible by {world} GPUs")
        return args.global_batch // world
    return args.batch


def run_reference(args):
    """The reference's own CPU implementation of the path (oracle port; /root/reference does not exist on the GPU box) on all
    host cores.  Same `config` as our arm; every step is a FIXED 64-sample slice of that workload's batch (a bounded sample:
    the CPU rate is flat in B beyond a few dozen samples), steps / warm-up as asked."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if args.reference_device == "gpu":
        return run_reference_on_gpu(args)
    cores = os.cpu_count() or 1
    import torch
    torch.set_num_threads(cores)
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    batch = REF_SAMPLE_BATCH
    rate, ms, desc = cpu_reference(batch, args.steps, args.warmup, cores, kind=args.kind, mode=args.mode)
    line = {"metric": METRIC.replace("DINO", "contrastive") if args.kind.startswith("contrastive") else METRIC, "value": rate, "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args, world), "impl": "reference",
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"each step = a {batch}-sample slice of the workload batch; " + desc},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
def op_cost(name, meta):
    """Algorithmic (flops, bytes) of one op launch from the shapes of its first tensor arguments."""
    import math

    def numel(s):
        return math.prod(s) if s else 0
    ints = ()
    if meta and meta[-1] and meta[-1][0] == "i":
        ints, meta = meta[-1][1:], meta[:-1]
    if name == "conv_tc" and len(meta) >= 3 and len(ints) >= 4:
        # (x8 | quad8, wprep, [bias], out) + (n_per_view, Cout, K, pad): tcgen05 implicit GEMM, bf16 operands, fp32 accumulate
        x, out = meta[0], meta[-1]
        n_per_view, Cout, K, pad = ints[:4]
        if len(x) == 4:               # first layer: quad8 image [N, H, ceil((W + 2 pad) / 4), 8]; square inputs
            N, H, W, Cin = x[0], x[1], x[1], 1
        else:
            N, H, W, Cin = x[0], x[2], x[3], x[1] * 8
        Ho, Wo = H + 2 * pad - K + 1, W + 2 * pad - K + 1
        out_bytes = numel(out) * (4 if len(out) == 4 else 2)
        return 2.0 * N * Cout * Ho * Wo * Cin * K * K, numel(x) * 2.0 + out_bytes
    if name == "conv_tc_pool" and len(meta) >= 5 and len(ints) >= 4:
        # (x8 | quad8, wprep, bias, gamma, [z], e) + (n_per_view, Cout, K, pad): forward conv whose epilogue also emits the 2x2 window
        # extreme e (fp16, a quarter of z); z is only written for the student
        x, e8 = meta[0], meta[-1]
        n_per_view, Cout, K, pad = ints[:4]
        if len(x) == 4:
            N, H, W, Cin = x[0], x[1], x[1], 1
        else:
            N, H, W, Cin = x[0], x[2], x[3], x[1] * 8
        Ho, Wo = H + 2 * pad - K + 1, W + 2 * pad - K + 1
        z_bytes = numel(meta[-2]) * 2.0 if len(meta) >= 6 else 0.0
        return 2.0 * N * Cout * Ho * Wo * Cin * K * K, numel(x) * 2.0 + z_bytes + numel(e8) * 2.0
    if name == "conv_tc_dgrad_bnstat" and len(meta) >= 4 and len(ints) >= 3:
        # (dz8, wprep, dx8, p8) + (n_per_view, K, pad'): data gradient whose epilogue also reads p and accumulates the BN-backward sums
        dz, dx, p8 = meta[0], meta[2], meta[3]
        K = ints[1]
        return 2.0 * dx[0] * dx[1] * 8 * dx[2] * dx[3] * dz[1] * 8 * K * K, (numel(dz) + numel(dx) + numel(p8)) * 2.0
    if name == "bn_relu_apply8" and len(meta) >= 4:
        return 0.0, numel(meta[0]) * 2.0 + numel(meta[3]) * (2.0 if len(meta[3]) == 5 else 4.0)
    if name == "conv_tc_wgrad" and len(meta) >= 3:
        x, dz, dw = meta[0], meta[1], meta[2]
        Cout, Cin, K, _ = dw
        return 2.0 * dz[0] * Cout * dz[2] * dz[3] * Cin * K * K, (numel(x) + numel(dz)) * 2.0
    if name == "bn_relu_pool8_fwd" and len(meta) >= 4:
        return 0.0, numel(meta[0]) * 2.0 + numel(meta[3]) * (2.0 if len(meta[3]) == 5 else 4.0)
    if name == "bn_relu_pool8_bwd_reduce" and len(meta) >= 2:
        return 0.0, numel(meta[0]) * 2.0 + numel(meta[1]) * (2.0 if len(meta[1]) == 5 else 4.0)
    if name == "bn_relu_pool8_bwd_apply" and len(meta) >= 2:
        return 0.0, numel(meta[0]) * 4.0 + numel(meta[1]) * (2.0 if len(meta[1]) == 5 else 4.0)
    if name == "conv_tc_wgrad_l0_fused" and len(meta) >= 3:
        # (quad8 x, z8 fp16, dp8 bf16, ...): BatchNorm-apply + weight gradient, every operand read once; dz never leaves the SM
        x, z, dp = meta[0], meta[1], meta[2]
        K = 5 if x[2] * 4 - x[1] >= 4 else 3
        return 2.0 * z[0] * z[1] * 8 * z[2] * z[3] * K * K, (numel(x) + numel(z) + numel(dp)) * 2.0
    if name in ("pack_shift8", "pack_quad8") and len(meta) >= 2:
        return 0.0, numel(meta[0]) * 4.0 + numel(meta[1]) * 2.0
    if name in ("conv_fwd", "conv_bwd_data", "conv_bwd_weight") and len(meta) >= 2:
        if name == "conv_fwd":
            x, w = meta[0], meta[1]
            N, Cin, H, W = x
            Cout, _, K, _ = w
            z = meta[3] if len(meta) > 3 else (N, Cout, H, W)
            Ho, Wo = z[2], z[3]
        elif name == "conv_bwd_data":
            dz, w, dx = meta[0], meta[1], meta[2]
            N, Cout, Ho, Wo = dz
            _, Cin, K, _ = w
        else:
            x, dz, dw = meta[0], meta[1], meta[2]
            N, Cin, H, W = x
            _, Cout, Ho, Wo = dz
            K = dw[2]
        return 2.0 * N * Cout * Ho * Wo * Cin * K * K, 0.0
    if name == "linear_fwd" and len(meta) >= 2:
        (M, K), (N, _) = meta[0], meta[1]
        return 2.0 * M * N * K, 0.0
    if name == "linear_bwd_data" and len(meta) >= 2:
        (M, N), (_, K) = meta[0], meta[1]
        return 2.0 * M * N * K, 0.0
    if name == "linear_bwd_weight" and len(meta) >= 2:
        (M, N), (_, K) = meta[0], meta[1]
        return 2.0 * M * N * K, 0.0
    if name in ("aug_apply_audio", "aug_apply_image"):
        # source read once (re-reads by the other views hit L2) + every view written once: fp32 [V,B,S,S] or bf16 quad8 [V,B,S,ceil((S+2pad)/4),8]
        src = meta[0]
        out8 = [m for m in meta[1:] if len(m) == 5]                    # bf16 quad8
        out32 = [m for m in meta[1:] if len(m) == 4 and m[-1] == m[-2]]  # fp32 [V,B,S,S]
        out_bytes = sum(numel(m) * 2.0 for m in out8) + sum(numel(m) * 4.0 for m in out32)
        return 0.0, numel(src) * (1.0 if name == "aug_apply_audio" else 4.0) + out_bytes
    if name == "ema_flat":
        return 0.0, 12.0 * numel(meta[0])
    if name == "adam_flat":
        return 0.0, 28.0 * numel(meta[0])
    if name == "dino_loss_fwd_bwd":
        return 0.0, 4.0 * (2 * numel(meta[0]) + numel(meta[1]))
    if name == "bn_relu_pool_fwd":
        return 0.0, 4.0 * numel(meta[0]) * 1.25
    if name == "bn_relu_pool_bwd_reduce":
        return 0.0, 4.0 * numel(meta[0]) * 1.25
    if name == "bn_relu_pool_bwd_apply":
        return 0.0, 4.0 * numel(meta[0]) * 2.25
    return 0.0, 0.0


NCU_EXTRA = {}      # tensor-pipe / l1tex busy % of the roofline kernel from the same committed ncu capture


def ncu_traffic(row, B):
    """dram__bytes_read.sum + dram__bytes_write.sum of this launch from the committed ncu --set full capture
    (profiles/ncu_traffic.json, taken at per-GPU batch 1024; scaled linearly to B), or None if it was not captured."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        return None
    ints = [s_ for s_ in row["shapes"] if s_ and s_[0] == "i"]
    key = row["op"] + ":" + "x".join(str(v) for v in row["shapes"][0]) + (":" + "x".join(str(v) for v in ints[0][1:]) if ints else "")
    ent = table.get("launches", {}).get(key)
    if ent is None:
        return None
    NCU_EXTRA.update({k_: ent[k_] for k_ in ("tensor_pipe_busy_pct", "l1tex_pct") if k_ in ent})
    return ent["dram_bytes"] * B / table.get("per_gpu_batch", 1024)


def profile_ops(engine, images, audios, steps=3, labels=None):
    """Per-op CUDA-event timing (events on the launching stream, side streams switched off so that every op runs alone on the
    current stream).  One un-recorded step first: switching the streams off moves ops onto streams whose scratch buffers do
    not exist yet, and a first-use cudaMalloc between two events would be charged to that op (round 1's 6 ms
    `linear_bwd_weight`).  Per op and shape the MEDIAN over the recorded calls is reported."""
    import statistics
    import torch
    from multimodal_ssl_avmnist_b200 import ops
    overlap, engine.overlap_teacher = engine.overlap_teacher, False      # per-kernel times: no concurrent streams while profiling
    engine._prefetch = None
    engine.train_step(images, audios, labels)                            # un-recorded: allocates the per-stream scratch
    torch.cuda.synchronize()
    rec = ops.start_profile()
    for _ in range(steps):
        engine.train_step(images, audios, labels)
    torch.cuda.synchronize()
    ops.stop_profile()
    engine.overlap_teacher = overlap
    agg = {}
    for name, a, b, meta, *_ in rec:
        agg.setdefault((name, meta), []).append(a.elapsed_time(b))
    rows = []
    for (name, meta), ts in agg.items():
        fl, by = op_cost(name, meta)
        calls = len(ts) / steps
        per = statistics.median(ts)
        rows.append({"op": name, "shapes": [list(s) for s in meta], "calls_per_step": calls, "ms_per_call": per,
                     "ms_per_step": per * calls, "flops": fl, "bytes": by,
                     "tflops": fl / per / 1e9 if per > 0 else 0.0, "gbs": by / per / 1e6 if per > 0 else 0.0})
    rows.sort(key=lambda r: -r["ms_per_step"])
    return rows


def step_work(kind, mode, B):
    """Algorithmic work of ONE step on one GPU (SURVEY 8d): (FLOPs, HBM bytes).  FLOPs: forward MACs x 2 x (6 student views x
    3 [fwd, dgrad, wgrad] + 2 teacher views); the non-default modes add one un-augmented student pass through both conv
    stacks + encoder linears + the two mode heads (x 3).  Bytes: augmentation 373,184 B/sample (21,952 image only), saved
    pre-BatchNorm activations 2 B x (1 write + 1 read) x 6 views, DINO loss 7,168 B/sample, + per step the teacher EMA
    (12 B/param) and Adam (28 B per trainable param)."""
    head = 196_608
    if kind == "multi_central":
        enc, act_elems, aug = 39_770_624, 219_648, 373_184
        n_ema, n_adam = 6_600_580, 1_728_368
        raw_pass = 39_770_624 - 196_608                      # conv stacks + encoder linears, no fusion
    elif kind.startswith("multi"):
        # SimpleMultiModalEncoder family (models/dino.py:18-73, 214-234): image 3 x conv3x3 (1->32->64->128 @28/14/7) + Linear(128,E),
        # audio 4 x conv3x3 (1->32->64->128->256 @112/56/28/14) + Linear(256,E), fusion 2E->E->O; cross attention adds 6 E^2 MACs of
        # projections and 4 B E MACs of batch-wide attention per row
        img = 9 * (28 * 28 * 32 + 14 * 14 * 64 * 32 + 7 * 7 * 128 * 64) + 128 * 256
        aud = 9 * (112 * 112 * 32 + 56 * 56 * 64 * 32 + 28 * 28 * 128 * 64 + 14 * 14 * 256 * 128) + 256 * 256
        raw_pass = img + aud
        enc = raw_pass + 196_608 + (6 * 256 * 256 + 4 * B * 256 if kind == "multi_cross_attention" else 0)
        act_elems = (32 * 784 + 64 * 196 + 128 * 49) + (32 * 12544 + 64 * 3136 + 128 * 784 + 256 * 196)
        aug = 373_184
        import numpy as np
        from multimodal_ssl_avmnist_b200.engine import MULTI_KINDS, head_params, simple_multi_params
        n_adam = sum(int(np.prod(sh)) if sh else 1 for _, sh in simple_multi_params(256, 256, MULTI_KINDS[kind])[0] + head_params(256, 128))
        n_ema = n_adam
    else:
        enc = 225_792 + 3_612_672 + 3_612_672 + 128 * 512 + 512 * 256       # 3 x conv3x3 + Linear(128,512) + Linear(512,256)
        act_elems, aug = 32 * 28 * 28 + 64 * 14 * 14 + 128 * 7 * 7, 21_952
        n_ema, n_adam = 488_768, 488_768
        raw_pass = 0
    macs = 20 * (enc + head)
    extra_bytes = 0.0
    if mode != "default":
        out = 10 if mode == "semi_supervised" else 128
        macs += 3 * (raw_pass + 2 * (256 * 512 + 512 * out))
        n_adam += 2 * (256 * 512 + 512 + 1024 + 512 * out + out)
        extra_bytes += act_elems * 4.0                       # the 7th view-call's saved activations
        if mode == "infonce":
            macs += 3 * B * 128                              # per sample: B x 128 similarity MACs, forward + two gradient GEMMs
    flops = 2.0 * macs * B
    byts = B * (aug + act_elems * 6 * 4.0 + 7168 + extra_bytes) + 12.0 * n_ema + 28.0 * n_adam
    return flops, byts


def run_module_path(args, B, steps, warmup):
    """Throughput of the DROP-IN path (reference flow run_dino.py:356-373): `Trainer.fit(MultiModalDINOLightning,
    AVMNISTDinoDataModule)` from the API mirror -- training_step -> loss.backward() -> B200Adam.step() per batch, batches
    gathered from the HBM-resident split (DeviceResidentLoader), augmentation on the device.  Timed with CUDA events recorded
    from a Trainer callback after `warmup` batches.  Returns a dict for the JSON line."""
    import shutil
    import tempfile
    import torch
    mirror = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
    if mirror not in sys.path:
        sys.path.insert(0, mirror)
    import models.dino as md
    import utils.get_data as gd
    from _compat import pl
    Callback = pl.Callback
    tmp = tempfile.mkdtemp(prefix="avmnist_bench_") + "/"
    try:
        n_batches = warmup + steps
        n_train = (n_batches * B * 12 + 10) // 11 + B          # the data module keeps 55000/60000 of the train file for training
        gd.write_synthetic_avmnist(tmp, n_train=n_train, n_test=16)
        aug = gd.MultiModalAugmentation(2, 4, augment_values=augment_values())
        dm = gd.AVMNISTDinoDataModule(data_dir=tmp, batch_size=B, num_workers=0, type="burst_noise", augmentations=aug, device_resident=True)
        dm.probe_dataloaders = None            # no per-epoch linear probe here: only the training steps are timed
        lit = md.MultiModalDINOLightning(data_dir=tmp, encoder_class=md.CentralMultiModalEncoder, projection_dim=128, output_dim=256,
                                         encoder_output_dim=256, learning_rate=1e-4, num_epochs=1, weight_decay=1e-6, dropout=0.3)

        class Timer(Callback):
            def __init__(self):
                self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                self.n = 0

            def on_train_batch_start(self, trainer, pl_module, batch, batch_idx):
                if batch_idx == warmup:
                    torch.cuda.synchronize()
                    self.e0.record()

            def on_train_batch_end(self, trainer, pl_module, outputs, batch, batch_idx):
                if batch_idx >= warmup:
                    self.n += 1
                if batch_idx == warmup + steps - 1:
                    self.e1.record()

        timer = Timer()
        tr = pl.Trainer(max_epochs=1, limit_train_batches=n_batches, callbacks=[timer], logger=None, log_every_n_steps=10 ** 9,
                        devices=1, accelerator="gpu", precision="16-mixed")
        tr.fit(lit, datamodule=dm)
        torch.cuda.synchronize()
        if timer.n != steps:
            return {"error": f"module path ran {timer.n} timed steps, wanted {steps}"}
        ms = timer.e0.elapsed_time(timer.e1) / steps
        return {"value": B / (ms / 1e3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "warmup": warmup, "per_gpu_batch": B,
                "api": "Trainer.fit(MultiModalDINOLightning(CentralMultiModalEncoder), AVMNISTDinoDataModule(device_resident=True)): "
                       "training_step -> loss.backward() -> B200Adam.step(), reference flow run_dino.py:356-373",
                "fused_graph_step": bool(lit.model.engine is not None and lit.model.engine._graph is not None),
                "last_loss": float(tr.callback_metrics.get("train_loss", float("nan")))}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from multimodal_ssl_avmnist_b200 import ops
    from multimodal_ssl_avmnist_b200.engine import DinoStepEngine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B = per_gpu_batch(args, world)
    eng = DinoStepEngine(kind=args.kind, mode=args.mode, augment_values=augment_values() if args.kind.startswith("multi") else None,
                         seed=1 + rank, device=dev, fused_pool=not args.no_fused_pool, fused_bnstat=args.fused_bnstat)
    g = torch.Generator().manual_seed(1 + rank)
    img_h = torch.rand(B, 28, 28, generator=g).pin_memory()
    aud_h = torch.randint(0, 256, (B, 112, 112), generator=g, dtype=torch.uint8).pin_memory() if args.kind.startswith("multi") else None
    img_d, aud_d = img_h.to(dev), (aud_h.to(dev) if aud_h is not None else None)
    lab_h = torch.randint(0, 10, (B,), generator=g).pin_memory() if args.mode == "semi_supervised" else None
    lab_d = lab_h.to(dev) if lab_h is not None else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (also sizes the workspaces) ----
    for _ in range(max(args.warmup, 3)):
        eng.train_step(img_d, aud_d, lab_d)
        eng.prefetch_augment(img_d, aud_d)
    barrier()
    use_graph = bool(args.graph)             # data parallel too: the NCCL all-reduces (C ABI) are captured with the kernels
    graph_launches = None
    if use_graph:
        eng._prefetch = None
        lg = ops.launch_count()
        eng.capture_train_step(B)               # 2 warm-up bodies + the captured one
        graph_launches = (ops.launch_count() - lg) // 3
        for _ in range(3):
            eng.graph_step(img_d, aud_d, lab_d)
        barrier()
    # ---- timed region 1: inputs resident in HBM ----
    clocks = ClockSampler(local) if rank == 0 else None
    l0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        if use_graph:
            loss = eng.graph_step(img_d, aud_d, lab_d)
        else:
            loss = eng.train_step(img_d, aud_d, lab_d)
            eng.prefetch_augment(img_d, aud_d)  # the next step's views, on the augmentation stream (input pipeline overlap)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / args.steps
    launches = graph_launches if use_graph else (ops.launch_count() - l0) // args.steps
    if args.dump_outputs and rank == 0:     # the last timed step's loss and the weights it left (trainable parameters)
        n = eng.n_trainable_prefix
        outputs = {"loss": loss, "center": eng.center, "student": eng.student.flat[:n], "teacher": eng.teacher.flat[:n]}
        if eng.aux_range:
            outputs["student_aux_heads"] = eng.student.flat[eng.aux_range[0]:eng.aux_range[1]]
        dump_outputs(args.dump_outputs, outputs)
    # ---- timed region 2: end to end through the host-facing call (pinned host buffers in, loss out); every step copies its
    #      batch host->device and reads its loss back; the NEXT batch's copy + augmentation are enqueued before the read-back ----
    nxt = ((img_h, aud_h) + ((lab_h,) if lab_h is not None else ())) if aud_h is not None else (img_h,)
    def host_step():
        if not use_graph:       # every step: H2D of its batch, the step, D2H of its loss (read one call later: the host never stalls)
            return eng.train_step_host(img_h, aud_h, lab_h, next_batch=nxt, lagged_loss=True)
        img_d.copy_(img_h, non_blocking=True)   # H2D of this step's batch, graph replay, D2H of the loss
        if aud_h is not None:
            aud_d.copy_(aud_h, non_blocking=True)
        if lab_h is not None:
            lab_d.copy_(lab_h, non_blocking=True)
        return float(eng.graph_step(img_d, aud_d, lab_d)[3].item())

    for _ in range(2):
        host_step()
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    last = None
    for _ in range(args.steps):
        last = host_step()
    if not use_graph:
        last = eng.flush_loss()                 # the final step's loss is read inside the timed region too
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3) / args.steps
    clk = clocks.stop() if clocks is not None else None
    t = torch.tensor([ms, ms_e2e], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    # launches per step, COUNTED: the kernel nodes of the step captured as one CUDA graph (all streams; NCCL kernels when N > 1);
    # the per-wrapper tally above stays as a cross-check
    launch_detail = {"tally_from_wrappers": int(launches)}
    try:
        if world > 1 and not use_graph:
            raise RuntimeError("census skipped at N > 1 (a capture that failed on one rank only would desynchronise the collectives)")
        if not use_graph:
            eng._prefetch = None
            eng.capture_train_step(B)
        counts = eng.graph_node_counts()
        launch_detail.update(counts, source="census of one training step captured as a CUDA graph (cudaGraphGetNodes): `kernels` = every kernel "
                                            "node of the step = this library's launches (the wrapper tally, reported as gpu_launches) + the "
                                            "handful of ATen fill / copy / add kernels the engine uses for zeroing and the loss total")
        if counts["kernels"] < launches:        # the tally may never exceed what the graph really contains
            launches = counts["kernels"]
    except Exception as exc:
        launch_detail["source"] = f"per-wrapper tally ({exc})"
    eng.release_graph()                         # the per-op profile below steps eagerly
    # per-op profile; every rank runs it (the step contains collectives when N > 1).  Consistency gate: with the side streams
    # off the per-op times must add up to about the step time (<= 1.3 x: the overlapped step hides ~15 %); otherwise a stall sat
    # between two events (allocation, clock ramp) and the profile is taken again.
    for attempt in range(3):
        rows = profile_ops(eng, img_d, aud_d, steps=3, labels=lab_d)
        step_ms_prof = sum(r["ms_per_step"] for r in rows)
        if step_ms_prof <= 1.3 * ms + 0.3:
            break
    profile_ok = step_ms_prof <= 1.3 * ms + 0.3
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = load_peaks()
    # (i) the whole step against both rooflines (SURVEY 8d algorithmic work / the timed ms_per_step / measured peaks)
    fl_step, by_step = step_work(args.kind, args.mode, B)
    t_tensor_step, t_hbm_step = fl_step / (peaks["tflops"] * 1e9), by_step / (peaks["hbm_gbs"] * 1e6)       # ms
    whole = {"algorithmic_tflop": fl_step / 1e12, "algorithmic_gb": by_step / 1e9, "tflops": fl_step / ms / 1e9, "gbs": by_step / ms / 1e6,
             "frac_tensor": fl_step / ms / 1e9 / peaks["tflops"], "frac_hbm": by_step / ms / 1e6 / peaks["hbm_gbs"],
             "ideal_ms": max(t_tensor_step, t_hbm_step), "achieved_over_ideal": max(t_tensor_step, t_hbm_step) / ms}
    # (ii) the dominant kernel = the largest launch of the kernel family with the largest share of the step
    costed = [r for r in rows if r["flops"] > 0 or r["bytes"] > 0]
    fam = {}
    for r in costed:
        fam[r["op"]] = fam.get(r["op"], 0.0) + r["ms_per_step"]
    top_op = max(fam, key=fam.get)
    top = max((r for r in costed if r["op"] == top_op), key=lambda r: r["ms_per_call"])
    shapes = [s_ for s_ in top["shapes"] if not (s_ and s_[0] == "i")][:3]
    # the binding roofline of a kernel = whichever of (FLOPs / tensor peak, bytes / HBM peak) takes longer
    t_tensor = top["flops"] / (peaks["tflops"] * 1e9)          # ms
    t_hbm = top["bytes"] / (peaks["hbm_gbs"] * 1e6)            # ms
    if top["flops"] > 0 and t_tensor >= t_hbm:
        roof = {"bound": "tensor", "kernel": f"{top['op']} {shapes}", "achieved": top["tflops"], "peak": peaks["tflops"], "unit": "TFLOP/s",
                "frac": top["tflops"] / peaks["tflops"], "traffic": None, "peak_source": peaks["source"] + " (cuBLAS bf16, sustained)",
                "share_of_step": top["ms_per_step"] / step_ms_prof, "algorithmic_gflop_per_launch": top["flops"] / 1e9,
                "algorithmic_gbs": top["gbs"], "hbm_frac": top["gbs"] / peaks["hbm_gbs"]}
    else:
        roof = {"bound": "hbm", "kernel": f"{top['op']} {shapes}", "achieved": top["gbs"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": top["gbs"] / peaks["hbm_gbs"], "traffic": None, "peak_source": peaks["source"],
                "share_of_step": top["ms_per_step"] / step_ms_prof, "algorithmic_mb_per_launch": top["bytes"] / 1e6}
        if top["flops"] > 0:
            roof["tflops"] = top["tflops"]
            roof["note"] = ("tcgen05 implicit-GEMM convolution whose FLOPs need less time at the tensor peak than its act8 bytes need at the "
                            "HBM peak: HBM is the binding roofline")
    roof["us_per_launch"] = 1e3 * top["ms_per_call"]
    roof["family_share_of_step"] = fam[top_op] / step_ms_prof
    roof["profile"] = {"sum_of_op_ms": step_ms_prof, "ms_per_step": ms, "consistent": profile_ok}
    roof["whole_step"] = whole
    roof["traffic"] = ncu_traffic(top, B)
    if NCU_EXTRA:       # from the same committed ncu --set full capture (profiles/ncu_traffic.json)
        roof["ncu"] = dict(NCU_EXTRA)
        if NCU_EXTRA.get("tensor_pipe_busy_pct", 0) > 80:
            roof["note"] = (roof.get("note", "") + "; ncu: the tensor pipe is busy %.0f %% of the time (a UMMA occupies it for its shared-memory operand "
                            "fetch whatever its N): the kernel's real ceiling" % NCU_EXTRA["tensor_pipe_busy_pct"]).lstrip("; ")
    tc_rows = [r for r in rows if r["op"] in ("conv_tc", "conv_tc_pool", "conv_tc_dgrad_bnstat", "conv_tc_wgrad")]
    if tc_rows:
        tc_ms = sum(r["ms_per_step"] for r in tc_rows)
        tc_fl = sum(r["flops"] * r["calls_per_step"] for r in tc_rows)
        roof["all_tensor_core_convs"] = {"tflops": tc_fl / tc_ms / 1e9, "share_of_step": tc_ms / step_ms_prof}
    hbm = {}
    for r in rows:
        if r["bytes"] > 0 and r["flops"] == 0:
            k = r["op"]
            if k not in hbm or r["ms_per_step"] > hbm[k]["_ms"]:
                hbm[k] = {"gbs": round(r["gbs"], 1), "frac": round(r["gbs"] / peaks["hbm_gbs"], 3), "us": round(1e3 * r["ms_per_call"], 1),
                          "_ms": r["ms_per_step"]}
    for v in hbm.values():
        v.pop("_ms")
    for k in ("aug_apply_audio", "aug_apply_image"):
        if k in hbm:        # listed for completeness: HBM is not what bounds these kernels (DESIGN 4.4)
            hbm[k]["note"] = ("instruction-issue bound, not HBM bound: up to ten dependent passes over each view in shared memory (~270 "
                              "thread-instructions per pixel; ncu 77 % issue-active), 373 KB of HBM traffic per sample; runs on the "
                              "augmentation stream beside the step")
    if "dino_loss_fwd_bwd" in hbm:
        hbm["dino_loss_fwd_bwd"]["note"] = "launch-latency regime (7 MB per launch)"
    if args.ops_out:
        with open(args.ops_out, "w") as f:
            json.dump({"ms_per_step": ms, "profiled_ms_per_step": step_ms_prof, "ops": rows}, f, indent=1)
    cpu = None
    if world == 1 and not args.no_cpu_baseline and args.kind.startswith("multi") and args.mode == "default":
        cores = os.cpu_count() or 1
        rate, _, desc = cpu_reference(REF_SAMPLE_BATCH, 3, 1, cores, kind=args.kind)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"each step = a {REF_SAMPLE_BATCH}-sample slice of the workload batch; " + desc}
    drop_in = None
    if world == 1 and args.kind == "multi_central" and args.mode == "default" and not args.no_module_path:
        try:
            del eng
            torch.cuda.empty_cache()
            drop_in = run_module_path(args, B, min(args.steps, 20), 3)
        except Exception as exc:        # reported, never hidden: the engine numbers above stand on their own
            drop_in = {"error": f"{type(exc).__name__}: {exc}"}
    h2d = img_h.numel() * 4 + (aud_h.numel() if aud_h is not None else 0)
    # the ONE published throughput of the reference for a configuration this repo runs (BASELINE.md section 1, row 1): the semi-supervised
    # SimpleMultiModalEncoder DINO step at B = 128, 1.74 it/s = 223 samples/s on an unnamed single GPU
    # (archive/semi-supervised_dino/semi-supervised_dino.ipynb:153).  Every other configuration has no published number: null.
    vs_base = None
    if world == 1 and args.kind == "multi_simple" and args.mode == "semi_supervised" and B == 128:
        vs_base = B * world / (ms / 1e3) / 223.0
    line = {"metric": METRIC, "value": B * world / (ms / 1e3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak", "vs_baseline": vs_base,
            "dtype": "bf16", "data": "synthetic",
            "config": workload_config(args, world),
            "details": {"execution": "one CUDA graph replay per step (device-side step counters)" if use_graph else "eager launches on 6 streams",
                        "precision": "bf16 tensor-core convolutions (fp16 pre-BatchNorm z, bf16 activations / gradients), fp32 accumulate, "
                                     "statistics, linears, losses, EMA, Adam"},
            "e2e": {"value": B * world / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e, "last_loss": last,
                    "note": "every step: H2D of its raw batch from pinned memory + D2H of its total loss (fp32 scalar, read back one "
                            "call later so that the host never waits for the step it has just enqueued)"},
            "gpu_launches": int(launches), "gpu_launches_detail": launch_detail, "clocks": clk, "roofline": roof, "hbm_kernels": hbm, "cpu_baseline": cpu, "drop_in_module_path": drop_in,
            "impl": "ours"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def run_contrastive(args):
    """The stand-alone contrastive steps of the reference's other_ssl/ modules (SURVEY 8f-4, BASELINE config 4): kind contrastive_infonce =
    other_ssl/info_nce/info_nce.py (InfoNCE between the modalities of the un-augmented batch), contrastive_simclr =
    other_ssl/multimodal_simclr/multimodal_simclr.py (two augmented views, random modality pairing, NT-Xent).  One GPU; `value` with
    the raw batch resident in HBM, `e2e` with the pinned host batch copied in and the loss read back every step."""
    import torch
    from multimodal_ssl_avmnist_b200 import ops
    from multimodal_ssl_avmnist_b200.contrastive import ContrastiveStepEngine
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    kind = args.kind.split("_", 1)[1]
    B = args.batch
    torch.manual_seed(1 + rank)
    eng = ContrastiveStepEngine(kind=kind, device=dev, seed=1)          # replicated weights (same seed), rank-local data below
    g = torch.Generator().manual_seed(1 + rank)
    img_h = torch.rand(B, 28, 28, generator=g).pin_memory()
    aud_h = torch.randint(0, 256, (B, 112, 112), generator=g, dtype=torch.uint8).pin_memory()
    img_d, aud_d = img_h.to(dev), aud_h.to(dev)
    W = max(args.warmup, 3)
    use_graph = bool(args.graph) and kind == "infonce" and world == 1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if use_graph:
        eng.capture_train_step(B)
    step = eng.graph_step if use_graph else eng.train_step
    for _ in range(W):
        loss = step(img_d, aud_d)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step(img_d, aud_d)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / args.steps
    launches = (ops.launch_count() - l0) // args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss, "params": eng.student.flat[:eng.student.size]})
    if use_graph:                       # a replay issues no wrapper calls: count one eager step of the same engine state instead
        eng2 = ContrastiveStepEngine(kind=kind, device=dev, seed=1)
        eng2.train_step(img_d, aud_d)
        l1 = ops.launch_count()
        eng2.train_step(img_d, aud_d)
        launches = ops.launch_count() - l1
        del eng2
    buf_i, buf_a = torch.empty_like(img_d), torch.empty_like(aud_d)
    e0.record()
    for _ in range(args.steps):
        buf_i.copy_(img_h, non_blocking=True)
        buf_a.copy_(aud_h, non_blocking=True)
        last = float(step(buf_i, buf_a)[3].item())
    e1.record()
    barrier()
    ms_e2e = e0.elapsed_time(e1) / args.steps
    if world > 1:                       # max over ranks (device-timed)
        t = torch.tensor([ms, ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    clk = sampler.stop() if sampler is not None else None
    if rank != 0:
        dist.destroy_process_group()
        return
    # algorithmic FLOPs per sample: ImageEncoder 7.65 M + head, SpectrogramEncoder 177.1 M + head MACs per encoder call, x3 (fwd, dgrad, wgrad)
    img_macs = 9 * (28 * 28 * 32 + 14 * 14 * 64 * 32 + 7 * 7 * 128 * 64) + 128 * 512 + 512 * 256 + 256 * 512 + 512 * 256
    aud_macs = 9 * (112 * 112 * 32 + 56 * 56 * 64 * 32 + 28 * 28 * 128 * 64 + 14 * 14 * 256 * 128) + 256 * 256 + 256 * 512 + 512 * 256
    per_sample = (img_macs + aud_macs) * 6.0        # infonce: one call of each encoder; simclr: two calls, on average one of each
    published = {("infonce", 128): (2180.0, "other_ssl/info_nce/info_nce.ipynb:156"), ("simclr", 256): (790.0, "other_ssl/multimodal_simclr/multimodal_simclr.ipynb:87")}
    pub = published.get((kind, B)) if world == 1 else None
    rate = B * world / (ms / 1e3)
    wl = ("stand-alone multimodal InfoNCE step (ImageEncoder + SpectrogramEncoder + 2 projection heads, un-augmented batch)" if kind == "infonce" else
          "multimodal SimCLR step (2 augmented views per modality, random modality pairing, NT-Xent)")
    print(json.dumps({"metric": METRIC.replace("DINO", "contrastive"), "value": rate, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
                      "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": (rate / pub[0]) if pub else None,
                      "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": wl, "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
                                 "published_reference": ({"samples_per_s": pub[0], "source": pub[1], "hardware": "unnamed single GPU"} if pub else None),
                                 "l2": "activations of a step exceed the 126 MB L2"},
                      "e2e": {"value": B * world / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": img_h.numel() * 4 + aud_h.numel(), "d2h_bytes_per_step": 4,
                              "ms_per_step": ms_e2e, "last_loss": last},
                      "details": {"execution": "one CUDA graph replay per step" if use_graph else "eager launches"},
                      "gpu_launches": int(launches), "clocks": clk,
                      "roofline": {"bound": "tensor", "kernel": "whole step", "achieved": per_sample * B / ms / 1e9, "peak": load_peaks()["tflops"], "unit": "TFLOP/s",
                                   "frac": per_sample * B / ms / 1e9 / load_peaks()["tflops"], "traffic": None,
                                   "note": "per GPU; whole-step algorithmic FLOPs (6 x forward MACs of one call of each encoder + head) over the step time"},
                      "cpu_baseline": None, "impl": "ours"}))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=1024, help="per-GPU batch (weak scaling)")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="STRONG scaling: total batch over all GPUs (per-GPU batch = global / N); overrides --batch")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (loss, updated weights) as DIR/<name>.npy")
    ap.add_argument("--ops-out", metavar="FILE", help="write the per-op profile of the step as JSON to FILE")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-module-path", action="store_true", help="skip the Trainer.fit (drop-in module path) throughput measurement")
    ap.add_argument("--reference-device", default="cpu", choices=["cpu", "gpu"],
                    help="--impl reference only: 'gpu' times the same oracle step with stock PyTorch kernels on cuda:0 (library bar)")
    ap.add_argument("--reference-fp32", action="store_true", help="library bar without fp16 autocast")
    ap.add_argument("--no-fused-pool", action="store_true",
                    help="A/B: the round-1 forward (full-resolution z -> bn_relu_pool8_fwd) instead of the fused max-pool epilogue")
    ap.add_argument("--fused-bnstat", action="store_true",
                    help="A/B: BN-backward sums in the data-gradient epilogue instead of separate bn_pool8_bwd_reduce_p passes (measured slower)")
    ap.add_argument("--graph", action="store_true",
                    help="replay the whole step from one CUDA graph (meant for small per-GPU batches, where the ~165 host-side "
                         "launches bound the step; with N > 1 the all-reduces are captured too)")
    ap.add_argument("--kind", default="multi_central", choices=["multi_central", "image_simple", "multi_simple", "multi_simple_gated", "multi_cross_attention", "contrastive_infonce",
                             "contrastive_simclr"],
                    help="image_simple = BASELINE.json configs[0] (unimodal image DINO); multi_simple* / multi_cross_attention = the 3x3 conv "
                         "encoders of SURVEY 8f-4; the headline line is multi_central")
    ap.add_argument("--mode", default="default", choices=["default", "semi_supervised", "infonce", "mse"],
                    help="training mode (BASELINE.json configs 2-5); the headline line is --mode default")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    elif args.kind.startswith("contrastive"):
        run_contrastive(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
