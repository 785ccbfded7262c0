"""Time of one epoch of the downstream MLP probe (train_downstream's inner loop) on one GPU, for the kinds multi_central,
image_simple and spectrogram_central at B = 128 and 1024 (the default), and on request for the stand-alone contrastive
containers contrastive_infonce / contrastive_simclr (is_dino_based=False).

    python tools/bench_downstream.py [--samples 55000] [--warmup 8] [--kinds KIND ...] [--batches B ...] [--out FILE.json] [--no-profile]

Data: a seeded synthetic AVMNIST-shaped labelled split resident in HBM (images fp32 in [0, 1], spectrograms uint8, labels int64),
55 000 samples by default (the reference's training split), consumed in order; a batch is a slice, the last one is ragged.  The
DINO model is a freshly initialised one (a probe's cost does not depend on the weights' values).  Three paths per configuration:
  torch       -- _DinoLightningBase.probe_accuracy's training loop: DownstreamClassifier (CUDA encoder features, torch head),
                 torch.optim.AdamW, CrossEntropyLoss, float(loss) per batch;
  session     -- probe.ProbeSession eagerly: encode -> probe kernel -> AdamW kernels on the device, one host read per epoch;
  session_graph -- the same step captured once per batch size and replayed as one CUDA graph (the ragged last batch runs eagerly).
Each path runs `--warmup` batches first (the graph is captured there), then one timed epoch between CUDA events ending in a device
synchronise.  `encoder_share` = the time of an epoch of train-mode encode_features alone over the path's epoch time.  A separate
torch.profiler pass (CUDA activity) lists the kernels of two graph-path batches and which of them are not this library's (b200::*).
The contrastive kinds (an InfoNCEModel / MultiModalSimCLRModel fresh from its Lightning module, bf16 path) add two rows that
time the frozen-feature extraction of the same split in eval mode, as the kNN evaluation does it:
  knn_features    -- feature_extraction_loop over FeatureExtractor(model, is_dino_based=False): the library path;
  module_features -- cat([model.image_encoder(x), model.audio_encoder(spectrogram / 255)], 1) through the containers' own
                     module-by-module forward (exact-fp32 kernels, no probe-private BatchNorm copy), then one torch.cat;
and a census of their own.
Prints one JSON line per row and a summary line with the GPU's name and power limit; nothing is written into the source tree
unless --out points there."""
import argparse
import json
import os
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MIRROR = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments")
for p in (ROOT, MIRROR, os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)

import models.dino as md  # noqa: E402
from bench_unimodal import gpu_info  # noqa: E402
from other_ssl.info_nce.info_nce import MultiModalInfoNCELightning  # noqa: E402
from other_ssl.multimodal_simclr.multimodal_simclr import MultiModalSimCLRLightning  # noqa: E402
from training_structures.dino_train import feature_extraction_loop  # noqa: E402
from multimodal_ssl_avmnist_b200.binding import contrastive_binding  # noqa: E402
from multimodal_ssl_avmnist_b200.probe import ProbeSession  # noqa: E402

KINDS = {"multi_central": md.CentralMultiModalEncoder, "image_simple": md.ImageEncoder, "spectrogram_central": md.SpectrogramEncoderCentral}
CONTRASTIVE = {"contrastive_infonce": MultiModalInfoNCELightning, "contrastive_simclr": MultiModalSimCLRLightning}
PATHS = ("torch", "session", "session_graph")


def dino_model(kind):
    torch.manual_seed(0)
    if kind in CONTRASTIVE:
        model = CONTRASTIVE[kind](projection_dim=256, output_dim=256).model.cuda()
        contrastive_binding(model).ensure_eval()
        return model
    if kind.startswith("multi"):
        lit = md.MultiModalDINOLightning(data_dir="x/", encoder_class=KINDS[kind], projection_dim=128, output_dim=256, encoder_output_dim=256)
    else:
        lit = md.UniModalDINOLightning(encoder_class=KINDS[kind], data_dir="x/", projection_dim=128, output_dim=256)
    lit = lit.cuda()
    lit.model._b200.ensure(torch.device("cuda"))
    return lit.model


def data(n, seed=1):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(n, 1, 28, 28, generator=g).cuda()
    aud = torch.randint(0, 256, (n, 1, 112, 112), generator=g, dtype=torch.uint8).cuda()
    lab = torch.randint(0, 10, (n,), generator=g).cuda()
    return img, aud, lab


def slices(n, B):
    return [(i, min(n, i + B)) for i in range(0, n, B)]


class TorchProbe:
    """probe_accuracy's training loop body, one batch at a time."""

    def __init__(self, model):
        self.probe = md.DownstreamClassifier(model, trainable_encoder=False, is_dino_based=model_is_dino(model)).cuda().train()
        self.opt = torch.optim.AdamW(self.probe.classifier.parameters(), lr=1e-3)
        self.crit = nn.CrossEntropyLoss()
        self.total = 0.0

    def train_batch(self, images, audios, labels):
        self.opt.zero_grad()
        loss = self.crit(self.probe(images, audios), labels)
        loss.backward()
        self.opt.step()
        self.total += float(loss)

    def end_epoch(self):
        return self.total


def model_is_dino(model):
    return hasattr(model, "_b200")


def engine(model):
    return model._b200.ensure(torch.device("cuda")) if model_is_dino(model) else contrastive_binding(model).ensure_eval()


def make(path, model):
    if path == "torch":
        return TorchProbe(model)
    return ProbeSession(model, lr=1e-3, graph=path == "session_graph")


def timed(fn):
    """Milliseconds of fn() between CUDA events, ending in a device synchronise."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def run(kind, B, n, warmup):
    model = dino_model(kind)
    img, aud, lab = data(n)
    spans = slices(n, B)
    eng = engine(model)
    token = eng.begin_probe()

    def encode_epoch(spans=spans):
        for lo, hi in spans:
            eng.encode_features(img[lo:hi], aud[lo:hi], train=True, probe=token)

    encode_epoch(spans[:warmup] + spans[-1:])
    enc_ms = timed(encode_epoch)
    rows = []
    for path in PATHS:
        p = make(path, model)

        def epoch(spans=spans, p=p):
            for lo, hi in spans:
                p.train_batch(img[lo:hi], aud[lo:hi], lab[lo:hi])
            p.end_epoch()                 # the epoch's read-back is part of the epoch

        epoch(spans[:warmup] + spans[-1:])
        ms = timed(epoch)
        rows.append({"kind": kind, "batch": B, "path": path, "samples": n, "batches": len(spans), "warmup_batches": warmup,
                     "epoch_ms": ms, "ms_per_batch": ms / len(spans), "samples_per_s": n / (ms / 1e3),
                     "encoder_epoch_ms": enc_ms, "encoder_share": enc_ms / ms, "precision": eng.precision})
        del p
    if not model_is_dino(model):
        rows += feature_rows(kind, B, model, img, aud, lab, spans, warmup, eng.precision)
    del model, eng
    torch.cuda.empty_cache()
    return rows


def feature_rows(kind, B, model, img, aud, lab, spans, warmup, precision):
    """Eval-mode feature extraction of the whole split: the library path and the containers' module-by-module forward."""
    n = img.shape[0]
    fx = md.FeatureExtractor(model, is_dino_based=False)

    def library(spans=spans):
        feature_extraction_loop("cuda", fx, [(img[lo:hi], aud[lo:hi], lab[lo:hi]) for lo, hi in spans])

    @torch.no_grad()
    def module(spans=spans):
        model.eval()
        torch.cat([torch.cat([model.image_encoder(img[lo:hi], None), model.audio_encoder(None, aud[lo:hi].float() / 255.0)], 1)
                   for lo, hi in spans])

    rows = []
    for path, fn in (("knn_features", library), ("module_features", module)):
        fn(spans[:warmup] + spans[-1:])
        ms = timed(fn)
        rows.append({"kind": kind, "batch": B, "path": path, "samples": n, "batches": len(spans),
                     "warmup_batches": warmup, "epoch_ms": ms, "ms_per_batch": ms / len(spans), "samples_per_s": n / (ms / 1e3),
                     "precision": precision if path == "knn_features" else "fp32"})
    return rows


def kernel_census(kind="multi_central", B=128, batches=2):
    """Kernel names of `batches` graph-path probe batches (after capture and warm-up) from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    model = dino_model(kind)
    img, aud, lab = data(B * (batches + 4))
    s = ProbeSession(model, lr=1e-3, graph=True)
    for i in range(4):
        s.train_batch(img[i * B:(i + 1) * B], aud[i * B:(i + 1) * B], lab[i * B:(i + 1) * B])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(4, 4 + batches):
            s.train_batch(img[i * B:(i + 1) * B], aud[i * B:(i + 1) * B], lab[i * B:(i + 1) * B])
        torch.cuda.synchronize()
    names = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            names[ev.name] = names.get(ev.name, 0) + 1
    lib = {k: c for k, c in names.items() if "b200::" in k}
    other = {k: c for k, c in names.items() if "b200::" not in k}
    return {"kind": kind, "batch": B, "path": "session_graph", "batches": batches, "library_kernel_launches_per_batch": sum(lib.values()) / batches,
            "library_kernels": sorted({k.replace("(anonymous namespace)::", "").split("(")[0] for k in lib}),
            "other_device_activity_per_batch": {k: c / batches for k, c in sorted(other.items())}}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=55000)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--kinds", nargs="+", choices=list(KINDS) + list(CONTRASTIVE), default=list(KINDS))
    ap.add_argument("--batches", nargs="+", type=int, default=[128, 1024])
    ap.add_argument("--out", metavar="FILE")
    ap.add_argument("--no-profile", action="store_true")
    args = ap.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_downstream.py: no CUDA device (the probe has no CPU fallback)")
    gpu = gpu_info()
    rows = []
    for kind in args.kinds:
        for B in args.batches:
            for row in run(kind, B, args.samples, args.warmup):
                row["gpu"] = gpu
                rows.append(row)
                print(json.dumps(row), flush=True)
    doc = {"gpu": gpu, "rows": rows}
    if not args.no_profile:
        doc["kernel_census"] = [kernel_census()] + [kernel_census(kind) for kind in args.kinds if kind in CONTRASTIVE]
        for c in doc["kernel_census"]:
            print(json.dumps(c), flush=True)
    print(json.dumps({"gpu": gpu["name"], "power_limit_w": gpu["power_limit_w"],
                      "summary": {f"{r['kind']} B={r['batch']} {r['path']}": round(r["samples_per_s"]) for r in rows}}))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
