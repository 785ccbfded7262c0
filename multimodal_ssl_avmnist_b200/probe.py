"""Downstream MLP probe on the device: the frozen features of a DINO student or of a contrastive container's two encoders ->
DownstreamClassifier's head Linear(O, 128) -> ReLU -> Linear(128, C), trained with CrossEntropyLoss and torch.optim.AdamW semantics
(DESIGN.md sections 4.11 and 4.12).

A training batch is encode_features(train=True, probe=token) -> b200_probe_mlp_fwd_bwd -> b200_adam_bias_dev + b200_adamw_flat_dev ->
b200_counters_advance, all on the device.  The head's parameters, gradient and AdamW moments live in flat arenas laid out as
[W1 | b1 | W2 | b2]; the loss sum and correct count accumulate on the device and are read back once per epoch.  The dropout
position and the AdamW step are device counters, so the same launches can be captured once per batch size and replayed as one
CUDA graph: eager and graph steps are bit-identical.
"""
import torch
import torch.nn as nn

from . import ops
from ._lib import B200Error
from .binding import contrastive_binding

HIDDEN = 128


def make_head(in_dim, num_classes):
    """DownstreamClassifier's head (same layers, same draws from the global RNG)."""
    return nn.Sequential(nn.Linear(in_dim, HIDDEN), nn.ReLU(), nn.Linear(HIDDEN, num_classes))


class ProbeSession:
    """One probe run on a frozen DINO model (anything with a `_b200` DINO binding: MultiModalDINO / UniModalDINO) or a stand-alone
    contrastive container (InfoNCEModel / MultiModalSimCLRModel, whose features are its two encoders' outputs side by side, O = 2 *
    its output_dim).

    head: the nn.Sequential whose initial weights the arena starts from (a fresh make_head() if None); export_head() writes the
    trained weights back into it.  probe: the engine's begin_probe() token -- the probe's private copy of the BatchNorm running
    statistics (a fresh one if None).  graph=True: the training step of the first batch size seen is captured once and replayed;
    other batch sizes (a ragged last batch) run the same launches eagerly."""

    def __init__(self, dino_model, num_classes=10, lr=1e-3, weight_decay=1e-2, graph=True, head=None, probe=None):
        if hasattr(dino_model, "_b200"):
            self.device = dino_model.center.device
            self.eng = dino_model._b200.ensure(self.device)
            self.O = int(dino_model.student.output_dim)
        else:
            binding = contrastive_binding(dino_model)
            if binding is None:
                raise B200Error("ProbeSession needs a DINO model with a compiled B200 step or a contrastive container")
            self.eng = binding.ensure_eval()
            self.device = self.eng.device
            self.O = 2 * int(dino_model.output_dim)
        self.C = int(num_classes)
        self.lr, self.weight_decay, self.use_graph = float(lr), float(weight_decay), bool(graph)
        self.head = head if head is not None else make_head(self.O, self.C)
        self.token = probe if probe is not None else self.eng.begin_probe()
        O, C, dev = self.O, self.C, self.device
        sizes = [HIDDEN * O, HIDDEN, C * HIDDEN, C]
        self._offsets = [sum(sizes[:i]) for i in range(4)]
        self._sizes = sizes
        n = (sum(sizes) + 3) // 4 * 4
        self.params = torch.zeros(n, device=dev)
        self.grad = torch.zeros(n, device=dev)
        self.exp_avg = torch.zeros(n, device=dev)
        self.exp_avg_sq = torch.zeros(n, device=dev)
        self.load_head(self.head)
        # [0] the dropout position of the next train-mode encode (the token's host counter + 1), [1] the AdamW steps taken
        self._ctr = torch.tensor([self.token["step"] + 1, 0], dtype=torch.int64, device=dev)
        self._step0 = self.token["step"]
        self._bc = torch.zeros(3, device=dev)
        self.loss_sum = torch.zeros(1, dtype=torch.float64, device=dev)
        self.correct = torch.zeros(1, dtype=torch.int64, device=dev)
        self.steps = 0
        self._n_epoch = 0
        self._work = {}
        self._graph = None

    # ---- parameters ---------------------------------------------------------------------------------------------------------
    def _views(self, flat):
        shapes = [(HIDDEN, self.O), (HIDDEN,), (self.C, HIDDEN), (self.C,)]
        return [flat[o:o + n].view(s) for o, n, s in zip(self._offsets, self._sizes, shapes)]

    def _head_tensors(self, module):
        lin1, lin2 = module[0], module[2]
        if tuple(lin1.weight.shape) != (HIDDEN, self.O) or tuple(lin2.weight.shape) != (self.C, HIDDEN):
            raise B200Error(f"head shape mismatch: expected Linear({self.O}, {HIDDEN}) -> Linear({HIDDEN}, {self.C})")
        return [lin1.weight, lin1.bias, lin2.weight, lin2.bias]

    @torch.no_grad()
    def load_head(self, module):
        """Copy an nn.Sequential head's weights into the parameter arena."""
        for dst, src in zip(self._views(self.params), self._head_tensors(module)):
            dst.copy_(src.detach())

    @torch.no_grad()
    def export_head(self, module=None):
        """Copy the trained weights into `module` (default: the session's head); returns the module."""
        module = self.head if module is None else module
        for dst, src in zip(self._head_tensors(module), self._views(self.params)):
            dst.copy_(src.to(dst.device))
        return module

    # ---- training ---------------------------------------------------------------------------------------------------------
    def _to_dev(self, t, dtype=None):
        if t is None:
            return None
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        return t.to(self.device, non_blocking=t.device.type == "cpu" and t.is_pinned())

    def _work_for(self, B):
        w = self._work.get(B)
        if w is None:
            w = self._work[B] = torch.empty(ops.probe_work_floats(B, self.C), device=self.device)
        return w

    def _batch_size(self, images, audios):
        return self.eng._batch_size(images, audios)

    def _step(self, images, audios, labels):
        """The training step's launches; every per-step scalar comes from a device counter."""
        feats = self.eng.encode_features(images, audios, train=True, probe=self.token, step_dev=self._ctr[0:1])
        B = feats.shape[0]
        w1, b1, w2, b2 = self._views(self.params)
        ops.probe_mlp_fwd_bwd(feats.contiguous(), w1, b1, w2, b2, labels, self._work_for(B), self.loss_sum, self.correct,
                              grad=self.grad, train=True)
        ops.adam_bias_dev(self._ctr[1:2], self._bc)
        ops.adamw_flat_dev(self.params, self.grad, self.exp_avg, self.exp_avg_sq, self._bc, self.lr, weight_decay=self.weight_decay)
        ops.counters_advance(self._ctr)

    def _state_tensors(self):
        ts = [self.params, self.exp_avg, self.exp_avg_sq, self.loss_sum, self.correct, self._ctr]
        for bn in self.token["bns"].values():
            ts += [bn.running_mean, bn.running_var, bn.num_batches_tracked]
        return ts

    def _capture(self, images, audios):
        """Capture _step for this batch's size and dtypes into one CUDA graph (warm-up and capture leave the state untouched)."""
        B = self._batch_size(images, audios)
        g = {"B": B}
        for name, t in (("img", images), ("aud", audios)):
            if t is not None:
                g[name] = torch.empty(t.shape, dtype=torch.float32 if t.is_floating_point() else t.dtype, device=self.device)
                g[name].copy_(t)
        g["lab"] = torch.zeros(B, dtype=torch.int64, device=self.device)
        state = self._state_tensors()
        snap = [t.clone() for t in state]
        host_step = self.token["step"]

        def body():
            self._step(g.get("img"), g.get("aud"), g["lab"])

        def restore():
            for t, c in zip(state, snap):
                t.copy_(c)
            self.token["step"] = host_step

        side = torch.cuda.Stream(device=self.device)      # warm-up off the capture stream: workspaces, one-time attributes
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            body()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize(self.device)
        restore()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            body()
        restore()
        torch.cuda.synchronize(self.device)
        g["graph"] = graph
        self._graph = g

    def train_batch(self, images, audios, labels):
        """One probe training step on a labelled batch (images [B,1,28,28] / audios [B,1,112,112], host or device; labels [B])."""
        images, audios = self._to_dev(images), self._to_dev(audios)
        labels = self._to_dev(labels, torch.int64)
        B = self._batch_size(images, audios)
        if self.use_graph and self._graph is None:
            self._capture(images, audios)
        g = self._graph
        if g is not None and g["B"] == B:
            for name, t in (("img", images), ("aud", audios)):
                if name in g:
                    g[name].copy_(t.reshape(g[name].shape))
            g["lab"].copy_(labels)
            g["graph"].replay()
        else:
            self._step(images, audios, labels)
        self.steps += 1
        self._n_epoch += B
        self.token["step"] = self._step0 + self.steps

    def end_epoch(self):
        """(mean training loss per sample, training accuracy in %) of the batches since the last call; resets the accumulators.
        The only host read of the epoch."""
        loss, correct = torch.cat([self.loss_sum, self.correct.double()]).tolist()
        n = max(self._n_epoch, 1)
        self.loss_sum.zero_()
        self.correct.zero_()
        self._n_epoch = 0
        return loss / n, 100.0 * correct / n

    # ---- evaluation -------------------------------------------------------------------------------------------------------
    @torch.no_grad()
    def evaluate(self, loader, predictions=False):
        """Eval-mode features (the probe copy's running statistics, no dropout) -> the forward-only kernel over every batch of
        `loader`.  Returns {"loss": mean per sample, "accuracy": fraction, "confusion_matrix": int64 numpy [C, C] (rows = labels),
        "n": samples[, "predictions": int64 device tensor [n]]}; one host read at the end."""
        C, dev = self.C, self.device
        loss_sum = torch.zeros(1, dtype=torch.float64, device=dev)
        correct = torch.zeros(1, dtype=torch.int64, device=dev)
        conf = torch.zeros(C, C, dtype=torch.int64, device=dev)
        w1, b1, w2, b2 = self._views(self.params)
        preds, n = [], 0
        for batch in loader:
            images, audios = self._to_dev(batch[0]), self._to_dev(batch[1])
            labels = self._to_dev(batch[2], torch.int64)
            feats = self.eng.encode_features(images, audios, train=False, probe=self.token)
            B = feats.shape[0]
            p = torch.empty(B, dtype=torch.int64, device=dev) if predictions else None
            ops.probe_mlp_fwd_bwd(feats.contiguous(), w1, b1, w2, b2, labels, self._work_for(B), loss_sum, correct, preds=p,
                                  confusion=conf, train=False)
            if predictions:
                preds.append(p)
            n += B
        loss, ncorrect = torch.cat([loss_sum, correct.double()]).tolist()
        out = {"loss": loss / max(n, 1), "accuracy": ncorrect / max(n, 1), "confusion_matrix": conf.cpu().numpy(), "n": n}
        if predictions:
            out["predictions"] = torch.cat(preds) if preds else torch.empty(0, dtype=torch.int64, device=dev)
        return out
