"""Throughput of the unimodal DINO steps (DinoStepEngine kinds 'spectrogram_simple', 'image_simple', 'image_central' and
'spectrogram_central') on one GPU, with multi_central at B = 1024 as the reference point of the CentralNet rows.

    python tools/bench_unimodal.py [--steps 50] [--warmup 5] [--kinds KIND ...] [--out FILE.json] [--no-profile]

Method as in bench.py: seeded synthetic raw batches resident in HBM (images fp32 in [0, 1], spectrograms uint8), the default
augmentation chains sampled and applied on the device inside every step, warm-up steps first, then CUDA events around >= 50 timed
steps.  Eager rows step with train_step() and prefetch the next step's views on the augmentation stream like bench.py; graph rows
replay the whole step captured as one CUDA graph (capture_train_step / graph_step).  Prints one JSON line per configuration and a
summary line with the GPU's name and power limit; --out writes everything as one JSON document.  --kinds keeps the rows of the
given kinds only.

Every row also carries the step's algorithmic FLOP count and rate, computed from the layer shapes (step_flops): forward MACs per
view-call = the convolutions (Ho*Wo*Cout*Cin*K*K each) + the trainable linears of the encoder and the projection head (SURVEY 8a
a3 / a4 for the CentralNet stacks); the backward costs twice the forward except for the first convolution of a stack, which has no
data gradient; the student runs forward + backward on all views, the teacher forward on the global views; 1 MAC = 2 FLOP.

A separate torch.profiler pass (CUDA activity, after the timed runs) lists the kernels of two eager steps of each profiled kind and
which of them are not this library's (b200::*) kernels, and compares that list with spectrogram_simple's.  Nothing is written into
the source tree unless --out points there."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from multimodal_ssl_avmnist_b200.engine import DinoStepEngine  # noqa: E402

CONFIGS = [("spectrogram_simple", 1024, False), ("spectrogram_simple", 128, False), ("spectrogram_simple", 128, True),
           ("image_simple", 1024, False), ("image_simple", 128, False), ("image_simple", 128, True),
           ("image_central", 256, False), ("image_central", 256, True), ("image_central", 1024, False),
           ("spectrogram_central", 1024, False), ("spectrogram_central", 128, False), ("spectrogram_central", 128, True),
           ("multi_central", 1024, False)]
PROFILED = ["spectrogram_central", "image_central"]
CENSUS_BASELINE = "spectrogram_simple"          # a kind whose step's kernel list is on record (profiles/r3a_bench_unimodal.json)


def gpu_info():
    info = {"name": torch.cuda.get_device_name(), "power_limit_w": None, "max_sm_clock_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
        p, c = (x.strip() for x in out.splitlines()[0].split(","))
        info["power_limit_w"], info["max_sm_clock_mhz"] = float(p), float(c)
    except Exception as exc:            # reported, not guessed
        info["query_error"] = f"{type(exc).__name__}: {exc}"
    return info


def batch(eng, B, seed=1):
    """Seeded raw batch of the modalities the engine encodes (None for the other one)."""
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(B, 28, 28, generator=g).cuda()
    aud = torch.randint(0, 256, (B, 112, 112), generator=g, dtype=torch.uint8).cuda()
    return (img if eng.img_layers else None), (aud if eng.aud_layers else None)


def step_flops(eng):
    """Algorithmic FLOP per sample of one training step (see the module docstring), from the engine's layer tables and arena shapes."""
    fwd = first = 0
    for layers in (eng.img_layers, eng.aud_layers):
        for li, (conv, bn, ci, co, hw, k, pad) in enumerate(layers):
            ho = hw + 2 * pad - k + 1
            macs = ho * ho * co * ci * k * k
            fwd += macs
            if li == 0:
                first += macs
    for name, shape in eng.student.spec:          # linears that take part in the step (the trainable prefix; not fc1 / fc2)
        if len(shape) == 2 and name.endswith(".weight") and eng.student.offsets[name][0] < eng.n_trainable_prefix:
            fwd += shape[0] * shape[1]
    bwd = 2 * fwd - first
    return {"fwd_macs_per_view": fwd, "step_flop_per_sample": 2 * (eng.V * (fwd + bwd) + eng.Vg * fwd)}


def run(kind, B, graph, steps, warmup):
    eng = DinoStepEngine(kind=kind, seed=1, device="cuda")
    img, aud = batch(eng, B)
    for _ in range(max(warmup, 3)):
        eng.train_step(img, aud)
        eng.prefetch_augment(img, aud)
    torch.cuda.synchronize()
    if graph:
        eng._prefetch = None
        eng.capture_train_step(B)
        for _ in range(3):
            eng.graph_step(img, aud)
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        if graph:
            loss = eng.graph_step(img, aud)
        else:
            loss = eng.train_step(img, aud)
            eng.prefetch_augment(img, aud)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    fl = step_flops(eng)
    row = {"kind": kind, "batch": B, "execution": "cuda_graph" if graph else "eager", "steps": steps, "warmup": max(warmup, 3),
           "ms_per_step": ms, "samples_per_s": B / (ms / 1e3), "last_loss": [float(x) for x in loss.tolist()],
           "precision": eng.precision, "tensor_core_convs": {m: list(map(bool, v)) for m, v in eng.tc.items() if v},
           "fused_pool": {r: {m: list(map(bool, v)) for m, v in eng.pool[r].items() if v} for r in ("s", "t")},
           **fl, "algorithmic_tflop_per_s": fl["step_flop_per_sample"] * B / (ms / 1e3) / 1e12}
    if graph:
        row["graph_nodes"] = eng.graph_node_counts()
    del eng
    torch.cuda.empty_cache()
    return row


def kernel_census(kind="spectrogram_simple", B=128, steps=2):
    """Kernel names of `steps` eager steps (after warm-up) from torch.profiler; library kernels live in namespace b200."""
    from torch.profiler import ProfilerActivity, profile
    eng = DinoStepEngine(kind=kind, seed=1, device="cuda", cosine_loss_alpha=0.3)
    img, aud = batch(eng, B)
    for _ in range(3):
        eng.train_step(img, aud)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            eng.train_step(img, aud)
        torch.cuda.synchronize()
    names = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            names[ev.name] = names.get(ev.name, 0) + 1
    lib = {n: c for n, c in names.items() if "b200::" in n}
    other = {n: c for n, c in names.items() if "b200::" not in n}
    return {"kind": kind, "batch": B, "steps": steps, "cosine_loss_alpha": 0.3, "library_kernel_launches": sum(lib.values()) // steps,
            "library_kernels": sorted({n.replace("(anonymous namespace)::", "").split("(")[0] for n in lib}), "other_device_activity": {n: c // steps for n, c in sorted(other.items())}}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--kinds", nargs="+", choices=sorted({k for k, _, _ in CONFIGS}), help="time only these kinds' rows")
    ap.add_argument("--out", metavar="FILE")
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args(argv)
    if args.steps < 50:
        raise SystemExit("bench_unimodal.py: time at least 50 steps")
    if not torch.cuda.is_available():
        raise SystemExit("bench_unimodal.py: no CUDA device (the step has no CPU fallback)")
    gpu = gpu_info()
    rows = []
    for kind, B, graph in CONFIGS:
        if args.kinds and kind not in args.kinds:
            continue
        row = run(kind, B, graph, args.steps, args.warmup)
        row["gpu"] = gpu
        rows.append(row)
        print(json.dumps(row), flush=True)
    doc = {"gpu": gpu, "rows": rows}
    if not args.no_profile:
        base = kernel_census(CENSUS_BASELINE)
        doc["kernel_census"] = [base]
        for kind in PROFILED:
            c = kernel_census(kind)
            # device activity outside the library that the baseline kind's step does not have as well
            c["other_beyond_" + CENSUS_BASELINE] = sorted(set(c["other_device_activity"]) - set(base["other_device_activity"]))
            doc["kernel_census"].append(c)
        for c in doc["kernel_census"]:
            print(json.dumps(c), flush=True)
    print(json.dumps({"gpu": gpu["name"], "power_limit_w": gpu["power_limit_w"],
                      "summary": {f"{r['kind']} B={r['batch']} {r['execution']}": round(r["samples_per_s"]) for r in rows}}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
