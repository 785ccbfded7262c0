"""CPU: the oracle (oracle/) against the golden fixtures generated from the imported reference
(tests/golden/make_golden.py) and the known answers of SURVEY.md §8c."""
import os
import random
import re

import numpy as np
import pytest
import torch
import yaml

from oracle import augment_ref as AR
from oracle import dino_ref as R
from oracle.fixtures import make_masks, summaries_close, summarize, synth_raw, synth_views, views_to_vb
from multimodal_ssl_avmnist_b200 import augment as A

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = os.path.join(ROOT, "multimodal_ssl_avmnist_b200", "AVMNIST_Experiments", "configs")


def _kat_inputs():
    torch.manual_seed(7)
    return torch.randn(6, 4, 128), torch.randn(2, 4, 128)


def test_loss_known_answers(golden):
    S, T = _kat_inputs()
    g = golden["losses"]
    assert abs(float(R.dino_loss_multimodal(S, T)) - g["dino_multimodal"]) < 2e-6
    assert abs(float(R.dino_loss_unimodal(S, T)) - g["dino_unimodal"]) < 2e-6
    assert abs(float(R.infonce_loss(S[0], S[1])) - g["infonce"]) < 2e-6
    assert abs(float(R.mse_align_loss(S[0], S[1])) - g["mse"]) < 1e-8
    assert abs(float(R.cosine_consistency_loss(S)) - g["cosine_consistency"]) < 2e-6
    lab = torch.tensor([3, 1, 4, 1])
    assert abs(float(R.supervised_loss(S[0][:, :10], S[1][:, :10], lab)) - g["supervised"]) < 2e-6
    # SURVEY §8c literal values
    assert abs(g["dino_multimodal"] - 5.20687056) < 1e-6 and abs(g["dino_unimodal"] - 5.19582653) < 1e-6
    assert abs(g["infonce"] - 1.38977242) < 1e-6 and abs(g["mse"] - 0.01482718) < 1e-7


def test_ntxent_known_answer(golden):
    """SimCLR NT-Xent (SURVEY 8f-4): the oracle's restatement against the reference's own nt_xent_loss on cat([S[0], S[1]])."""
    S, _ = _kat_inputs()
    reps = torch.cat([S[0], S[1]]).clone().requires_grad_(True)
    loss = R.ntxent_loss(reps)
    assert abs(float(loss.detach()) - golden["losses"]["ntxent"]) < 1e-6
    loss.backward()
    assert abs(float(reps.grad.abs().sum()) - golden["losses"]["ntxent_grad_abs_sum"]) < 1e-4 * golden["losses"]["ntxent_grad_abs_sum"]
    assert torch.allclose(reps.grad.flatten()[:8], torch.tensor(golden["losses"]["ntxent_grad_first8"]), rtol=1e-4, atol=1e-7)


def test_loss_gradient_known_answer(golden):
    S, T = _kat_inputs()
    Sg = S.clone().requires_grad_(True)
    R.dino_loss_multimodal(Sg, T).backward()
    g = golden["losses"]
    assert abs(float(Sg.grad.abs().sum()) - g["dino_multimodal_grad_abs_sum"]) < 1e-5
    np.testing.assert_allclose(Sg.grad.flatten()[:8].numpy(), g["dino_multimodal_grad_first8"], rtol=1e-4, atol=1e-8)


def test_ema_bit_exact(golden):
    gen = torch.Generator().manual_seed(11)
    t = {"w": torch.randn(1000, generator=gen)}
    s = {"w": torch.randn(1000, generator=gen)}
    R.ema_update(t, s, 0.996)
    assert t["w"][:8].tolist() == golden["losses"]["ema_first8"]
    assert float(t["w"].double().sum()) == golden["losses"]["ema_sum64"]


def _chains(tag):
    ig, il = A.image_chains()
    if tag == "default":
        ag, al = A.default_audio_chains()
    else:
        name = {"tuned": "config_multimodal_dino.yaml", "old": "config_multimodal_dino_old_augments.yaml"}[tag]
        cfg = yaml.safe_load(open(os.path.join(CFG, name)))
        from multimodal_ssl_avmnist_b200.augment import values_from_config
        ag, al = A.audio_chains_from_values(values_from_config(cfg))
    return ig, il, ag, al


def _oracle_views(tag, data_seed, rng_seed):
    ig, il, ag, al = _chains(tag)
    g = torch.Generator().manual_seed(data_seed)
    img = torch.rand(1, 28, 28, generator=g)[0].numpy()
    aud = torch.rand(1, 112, 112, generator=g)[0].numpy()
    torch.manual_seed(rng_seed)
    random.seed(rng_seed)
    hs = A.HostSampler()
    out = {"gi": [], "ga": [], "li": [], "la": []}
    for ki, ka, ci, ca, n in (("gi", "ga", ig, ag, 2), ("li", "la", il, al, 4)):
        for _ in range(n):
            ops, b, nz = hs.sample_view(ci, 28, 28)
            out[ki].append(AR.apply_chain(img, ops, b, None if nz is None else nz.numpy()))
            ops, b, nz = hs.sample_view(ca, 112, 112)
            out[ka].append(AR.apply_chain(aud, ops, b, None if nz is None else nz.numpy()))
    return {k: np.stack(v) for k, v in out.items()}


@pytest.mark.parametrize("tag", ["tuned", "old", "default"])
def test_augment_against_reference_outputs(tag, golden, golden_aug):
    sums = golden["augment"][tag]["sums"]
    for s in range(8):
        o = _oracle_views(tag, 1000 + s, s)
        for k, ref in zip(("gi", "ga", "li", "la"), sums[s]):
            assert abs(float(o[k].astype(np.float64).sum()) - ref) < 2e-3 * max(1.0, abs(ref)) * 1e-2, (tag, s, k)
        if s < 2:
            np.testing.assert_allclose(o["gi"][:, None], golden_aug[f"{tag}_{s}_gi"], atol=1e-6, rtol=0)
            np.testing.assert_allclose(o["li"][:, None], golden_aug[f"{tag}_{s}_li"], atol=1e-6, rtol=0)
            for nm in ("ga", "la"):
                a = o[nm][:, None]
                np.testing.assert_allclose(a[:, :, ::4, 1::4], golden_aug[f"{tag}_{s}_{nm}_dec"], atol=1e-6, rtol=0)
                np.testing.assert_allclose(a.astype(np.float64).sum(-1), golden_aug[f"{tag}_{s}_{nm}_rows"], atol=2e-3)
                np.testing.assert_allclose(a.astype(np.float64).sum(-2), golden_aug[f"{tag}_{s}_{nm}_cols"], atol=2e-3)


def test_augment_survey_known_answer(golden):
    o = _oracle_views("old", 1234, 1)
    for k, ref in zip(("gi", "ga", "li", "la"), (723.604126, 11128.843750, 1186.044312, 15762.379883)):
        assert abs(float(o[k].sum(dtype=np.float64)) - ref) < 2e-2, k
    np.testing.assert_allclose(golden["augment"]["survey_kat_sums"], [723.604126, 11128.843750, 1186.044312, 15762.379883], rtol=1e-6)


def test_affine_index_map_matches_torchvision():
    """Bit-exact integer gather maps for NEAREST rotate/affine (SURVEY Appendix A1).  tests/golden/affine_torchvision.json holds
    the SHA-256 of torchvision 0.26's map (int64, -1 = fill) for each case below, so the check needs no torchvision; where
    torchvision is installed its maps are compared directly as well."""
    import hashlib
    import json
    try:
        import torchvision.transforms.functional as F
        from torchvision.transforms import InterpolationMode
    except ImportError:
        F = None
    with open(os.path.join(ROOT, "tests", "golden", "affine_torchvision.json")) as f:
        digests = json.load(f)["sha256"]
    rng = np.random.default_rng(3)
    i = 0
    for S in (28, 112):
        img = (torch.arange(S * S, dtype=torch.float32) + 1).view(1, S, S)
        for t in range(40):
            ang = float(rng.uniform(-15, 15))
            tx, ty = int(rng.integers(-S // 5, S // 5 + 1)), int(rng.integers(-S // 5, S // 5 + 1))
            sc = float(rng.uniform(0.7, 1.3))
            if t % 2:
                m = AR.inverse_affine_matrix(-ang, 0, 0, 1.0)
            else:
                m = AR.inverse_affine_matrix(ang, tx, ty, sc)
            got = AR.affine_index_map(m, S, S).astype(np.int64)
            assert hashlib.sha256(got.tobytes()).hexdigest() == digests[i], (S, t)
            i += 1
            if F is None:
                continue
            if t % 2:
                out = F.rotate(img, ang, interpolation=InterpolationMode.NEAREST, fill=[0.0])
            else:
                out = F.affine(img, ang, [tx, ty], sc, [0.0, 0.0], interpolation=InterpolationMode.NEAREST, fill=[0.0])
            ref = out.numpy().reshape(S, S).astype(np.int64) - 1
            assert np.array_equal(ref, got)
    assert i == len(digests)


def _bias_cancelled_by_bn(name):
    """A bias that feeds straight into a train-mode BatchNorm has an exactly-zero gradient; what the reference
    (and we) produce is rounding noise, so it is checked for smallness, not equality."""
    import re
    return re.search(r"(\.conv[1-4]\.bias|mlp\.0\.bias|student\.fusion\.3\.bias|student\.projection\.0\.bias|(student|teacher)\.encoder\.[048]\.bias|(image|audio)_encoder\.(0|4|8|12)\.bias)$", name) is not None


def _check_group(got, want, rtol, atol, what, noise=1e-4):
    for name, ref in want.items():
        mine = summarize(got[name])
        if "grad" in what and _bias_cancelled_by_bn(name):
            assert mine["abs_sum"] < noise and ref["abs_sum"] < noise, f"{what}:{name}"
            continue
        if "adam" in what and _bias_cancelled_by_bn("student." + name):
            # Adam normalises the rounding-noise gradient of these biases to a full +-lr step per iteration
            ok, why = summaries_close(mine, ref, rtol, 1e-3)
            assert ok, f"{what}:{name}: {why}"
            continue
        ok, why = summaries_close(mine, ref, rtol, atol)
        assert ok, f"{what}:{name}: {why}"


SIMPLE_CASES = ["multi_simple/default", "multi_simple/mse", "multi_simple_gated/default", "multi_simple_gated/semi_supervised",
                "multi_cross_attention/default", "multi_cross_attention/infonce"]


@pytest.mark.parametrize("case", SIMPLE_CASES)
def test_simple_family_step_against_reference(case, golden_simple):
    """SURVEY 8f-4: the oracle's SimpleMultiModalEncoder / GatedMultiModalEncoder / CrossAttentionMultiModalEncoder steps against the
    training_step of the imported reference (tests/golden/golden_simple.json)."""
    kind, mode = case.split("/")
    # step 0 is held to the same 2e-4 as the central encoder; at step 1 the seven-BatchNorm 3x3 stacks amplify the +-lr Adam noise on
    # the BatchNorm-cancelled conv biases through more max-pool arg-max flips than the LeNet stacks do: 5e-2 on single gradient values
    # (and the Adam update of step 1, ~lr * g / |g|, moves by that fraction of lr = 1e-4); the exactly-cancelled conv-bias gradients are
    # rounding noise of up to 1e-3 summed over a layer in the reference's own run (InfoNCE's 1 / 0.07 logits), and the two-path
    # gradients of the encoder linears in the non-default modes agree to 1e-3
    _step_against_reference(golden_simple[case], mode, kind, step0_rtol=1e-3, step1_rtol=5e-2, adam1_atol=1e-5, loss1_rtol=5e-5)


@pytest.mark.parametrize("mode", ["default", "semi_supervised", "infonce", "mse"])
def test_step_against_reference(mode, golden):
    _step_against_reference(golden["steps"][mode], mode, "multi_central")


def _step_against_reference(fx, mode, kind, step0_rtol=2e-4, step1_rtol=1e-2, noise=1e-4, adam1_atol=1e-6, loss1_rtol=5e-6):
    B = fx["B"]
    st = R.CentralDinoState(seed=fx["seed"], mode=mode, kind=kind)
    for it, rec in enumerate(fx["steps"]):
        img, aud = views_to_vb(*synth_views(B, seed=100 + it))
        masks = make_masks(seed=200 + it, V=6, Vg=2, B=B, E=256, hidden=512)
        raw = labels = None
        if mode != "default":
            image, audio, labels = synth_raw(B, seed=300 + it)
            raw = (image, audio)
        out = R.central_dino_step(st, img, aud, masks, raw=raw, labels=labels)
        ltol = 5e-6 if it == 0 else loss1_rtol
        assert abs(float(out["loss"]) - rec["loss"]) < ltol * max(1.0, abs(rec["loss"])), (mode, it, float(out["loss"]), rec["loss"])
        ok, why = summaries_close(summarize(st.center), rec["center"], 1e-5, 1e-7)
        assert ok, why
        grads = {}
        for k, v in out["grads"]["student"].items():
            grads[f"model.student.{k}"] = v
        for k, v in out["grads"]["student_head"].items():
            grads[f"model.student_projection.{k}"] = v
        aux_names = {"semi_supervised": ("image_classifier", "audio_classifier")}.get(mode, ("image_projection_head", "audio_projection_head"))
        for m, nm in zip(("image", "audio"), aux_names):
            for k, v in out["grads"].get(m, {}).items():
                grads[f"model.{nm}.{k}"] = v
        assert set(grads) == set(rec["grads"]), set(grads) ^ set(rec["grads"])
        # step 0 agrees to rounding; from step 1 on, the +-lr Adam noise on BN-cancelled biases perturbs
        # pre-BN activations at the 1e-7 level, which flips a few max-pool arg-maxes (1e-3 relative on grads)
        _check_group(grads, rec["grads"], step0_rtol if it == 0 else step1_rtol, 1e-8 if it == 0 else 1e-6, f"{mode} step{it} grad",
                     max(noise, 1e-5 * max(v["abs_sum"] for v in rec["grads"].values())))    # rounding noise scales with the gradient magnitude
        ta = 1e-9 if it == 0 else 2e-6     # step>0: the EMA ingests the noise-stepped biases (see above)
        _check_group(st.teacher, rec["teacher"], 1e-6, ta, "teacher")
        _check_group(st.teacher_head, rec["teacher_head"], 1e-6, ta, "teacher_head")
        _check_group(st.student, rec["student_after_adam"], 1e-5, 1e-7 if it == 0 else adam1_atol, "student_after_adam")
        bn = {k: v for k, v in st.student_buf.items()}
        ba = 1e-7 if it == 0 else 4e-4     # running_mean contains the conv bias
        _check_group(bn, rec["student_bn"], 1e-5, ba, "student_bn")
        _check_group(st.teacher_buf, rec["teacher_bn"], 1e-5, ba, "teacher_bn")
        _check_group(st.student_head_buf, rec["student_head_bn"], 1e-5, ba, "head_bn")


@pytest.mark.parametrize("key,alpha", [("unimodal_image_simple", 0.0), ("unimodal_image_simple_cosine", 0.3)])
def test_unimodal_step_loss_and_gradients_against_reference(key, alpha, golden):
    """UniModalDINOLightning.training_step of the imported reference on ImageEncoder (BASELINE config 1), with and without the
    cosine-consistency term: the oracle's pieces (image_simple_encoder, projection_head, dino_loss_unimodal,
    cosine_consistency_loss) reproduce its loss and parameter gradients."""
    fx = golden[key]
    B = fx["B"]
    spec, hspec = R.image_simple_spec(256), R.head_spec(256, 128)
    sp = {k: v.clone().requires_grad_(True) for k, v in R.make_params(spec, fx["seed"]).items()}
    hp = {k: v.clone().requires_grad_(True) for k, v in R.make_params(hspec, fx["seed"] + 1).items()}
    bufs = [R.make_bn_buffers(spec, R.image_simple_bn_names()) for _ in range(2)] + [R.make_bn_buffers(hspec, ["mlp.1"]) for _ in range(2)]
    gi, ga, li, la = synth_views(B, seed=100)
    img, _ = views_to_vb(gi, ga, li, la)
    m = make_masks(seed=200, V=6, Vg=2, B=B, E=256, hidden=512)
    feats = torch.cat([R.image_simple_encoder(img[v], sp, bufs[0]) for v in range(6)])
    with torch.no_grad():
        tfeat = torch.cat([R.image_simple_encoder(img[v], {k: v_.detach() for k, v_ in sp.items()}, bufs[1]) for v in range(2)])
        tproj = R.projection_head(tfeat, {k: v_.detach() for k, v_ in hp.items()}, bufs[3], None, 0.0)
    sproj = R.projection_head(feats, hp, bufs[2], m["student_head"], 0.3)
    loss = R.dino_loss_unimodal(sproj.view(6, B, -1), tproj.view(2, B, -1))        # centre is zero on the first step
    if alpha > 0:
        loss = loss + alpha * R.cosine_consistency_loss(feats.view(6, B, -1))
    assert abs(float(loss.detach()) - fx["loss"]) < 1e-5 * fx["loss"], (float(loss.detach()), fx["loss"])
    loss.backward()
    checked = 0
    for k, ref in fx["grads"].items():
        if k.startswith("model.student_projection."):
            g = hp[k[len("model.student_projection."):]].grad
        elif k.startswith("model.student."):
            g = sp[k[len("model.student."):]].grad
        else:
            continue
        if g is None:
            continue
        ok, why = summaries_close(summarize(g), ref, 2e-4, 1e-7)
        # conv biases in front of a train-mode BatchNorm: mathematically zero gradient, pure rounding noise on both sides
        if not ok and k.endswith(".bias") and ref["abs_sum"] < 1e-4 * ref["n"]:
            continue
        assert ok, (k, why)
        checked += 1
    assert checked >= 10


def test_simclr_augmentation_against_reference_fixture():
    """SURVEY 8f-4: SimCLRMultiModalAugmentation (utils/get_data.py:299-408: RandomResizedCrop, rotation, affine, ElasticTransform,
    GaussianBlur on the image; crop, time-warp, masks, Gaussian noise on the spectrogram; one parameter set per BATCH).  The host
    sampler replays the reference's RNG order, the numpy oracle applies the records: against the imported reference's outputs
    (tests/golden/simclr_aug.npz) 2e-6 abs (ATen's 3x3 blur / grid-sampler accumulation order is not reproduced bit for bit)."""
    import random
    import numpy as np
    from multimodal_ssl_avmnist_b200 import augment as A
    from oracle import augment_ref as AR
    fx = np.load(os.path.join(ROOT, "tests", "golden", "simclr_aug.npz"))
    img_chain, aud_chain = A.simclr_chains()
    kinds = set()
    B = 3
    for s in range(8):
        g = torch.Generator().manual_seed(2000 + s)
        img = torch.rand(B, 1, 28, 28, generator=g)
        aud = torch.rand(B, 1, 112, 112, generator=g)
        torch.manual_seed(s)
        random.seed(s)
        hs = A.HostSampler()
        # reference call order: image view 1, image view 2, spectrogram view 1, spectrogram view 2
        recs = []
        for chain, size in ((img_chain, 28), (img_chain, 28), (aud_chain, 112), (aud_chain, 112)):
            ops_, bits, noise = hs.sample_view(chain, size, size, batch=B)
            recs.append((ops_, noise, hs.last_grid))
            kinds |= {k for k, _ in ops_}
        for v, name in ((0, "i1"), (1, "i2")):
            ops_, _, grid = recs[v]
            for b in range(B):
                got = AR.apply_chain(img[b, 0].numpy(), ops_, None, None, grid=grid)
                np.testing.assert_allclose(got, fx[f"s{s}_{name}"][b, 0], rtol=0, atol=2e-6)
        for v, name in ((2, "a1"), (3, "a2")):
            ops_, noise, _ = recs[v]
            for b in range(B):
                got = AR.apply_chain(aud[b, 0].numpy(), ops_, None, None if noise is None else noise[b].numpy())
                np.testing.assert_allclose(got[::4, 1::4], fx[f"s{s}_{name}_dec"][b, 0], rtol=0, atol=2e-6)
                np.testing.assert_allclose(got.astype(np.float64).sum(-1), fx[f"s{s}_{name}_rows"][b, 0], rtol=0, atol=2e-3)
    assert {A.OP_ELASTIC, A.OP_BLUR3, A.OP_NOISE, A.OP_TIME_WARP} <= kinds          # the seeds exercise every new op


from oracle.fixtures import contrastive_batch  # noqa: E402


@pytest.mark.parametrize("kind", ["infonce", "simclr"])
def test_contrastive_step_against_reference(kind, golden_contrastive):
    """other_ssl/info_nce/info_nce.py and other_ssl/multimodal_simclr/multimodal_simclr.py (SURVEY 8f-4, BASELINE config 4): the oracle's
    contrastive_step against training_step -> backward -> Adam.step of the imported Lightning modules, incl. the SimCLR modality pairing
    (all four modes) and Adam's per-parameter step counts (a branch without gradients is skipped)."""
    fx = golden_contrastive[kind]
    B = fx["B"]
    st = R.ContrastiveState(seed=fx["seed"])
    for it, rec in enumerate(fx["steps"]):
        img1, spec1, img2, spec2 = contrastive_batch(B, it)
        if kind == "infonce":
            out = R.contrastive_step(st, "infonce", (img1, spec1))
        else:
            out = R.contrastive_step(st, "simclr", (img1, spec1, img2, spec2), mode=fx["modes"][it])
        assert abs(float(out["loss"]) - rec["loss"]) < (5e-6 if it == 0 else 1e-4) * max(1.0, abs(rec["loss"])), (kind, it, float(out["loss"]), rec["loss"])
        grads = {f"{m}.{k}": v for m in R.CONTRASTIVE_MODULES for k, v in out["grads"][m].items()}
        assert set(grads) == set(rec["grads"]), (kind, it, set(grads) ^ set(rec["grads"]))
        noise = max(1e-4, 1e-5 * max(v["abs_sum"] for v in rec["grads"].values()))
        for name, ref in rec["grads"].items():
            mine = summarize(grads[name])
            if re.search(r"(encoder\.(0|4|8|12|14|18)\.bias|projection\.0\.bias|mlp\.0\.bias)$", name):      # feeds a BatchNorm: exact gradient 0
                assert mine["abs_sum"] < noise and ref["abs_sum"] < noise, (kind, it, name)
                continue
            ok, why = summaries_close(mine, ref, 1e-3 if it == 0 else 5e-2, 1e-8 if it == 0 else 1e-6)
            assert ok, (kind, it, name, why)
        for name, ref in rec["params_after_adam"].items():
            # Adam's first steps are ~lr * sign(g): an element whose gradient is rounding noise (dead unit, cancelled bias) may land
            # 2 * lr = 2e-4 away; everything else agrees to fp32 rounding
            m, k = name.split(".", 1)
            ok, why = summaries_close(summarize(st.params[m][k]), ref, 1e-5, 2.5e-4 * (it + 1))
            assert ok, (kind, it, name, why)
        for name, ref in rec["bn"].items():
            m, k = name.split(".", 1)
            ok, why = summaries_close(summarize(st.buf[m][k]), ref, 1e-5, 1e-7 if it == 0 else 4e-4)
            assert ok, (kind, it, name, why)
