"""CPU tests: the oracle restatement (oracle/vit_oracle.py) against the golden vectors generated from the REAL
reference (oracle/make_golden.py), plus the pins of oracle/make_golden_pins.py against the reference outputs they store."""
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import vit_oracle as vo  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def _check_pin(pin):
    """The oracle against the reference's side of one pin, stored by oracle/make_golden_pins.py where the two were
    bit-identical: every output and parameter gradient, by its L2 norm and by its values at the stored positions (a
    different CPU / torch build may reorder fp32 sums, and bf16 autocast roundings differ with the CPU's instruction set)."""
    import make_golden_pins as mgp

    rec = torch.load(os.path.join(GOLDEN, "reference_pins.pt"), weights_only=True)
    threads = torch.get_num_threads()
    torch.set_num_threads(mgp.THREADS)
    try:
        outputs = {mode: mgp.oracle_outputs(pin, mode, rec.get("unet_shapes", ())) for mode in rec["pins"][pin]}
    finally:
        torch.set_num_threads(threads)
    for mode, ref in rec["pins"][pin].items():
        ours = mgp.summarize(outputs[mode])
        assert (ours["keys"], ours["numel"], ours["lengths"]) == (ref["keys"], ref["numel"], ref["lengths"])
        tol = 1e-4 if mode == "fp32" else 3e-2
        values = zip(ours["values"].split(ref["lengths"]), ref["values"].split(ref["lengths"]))
        for k, n, o_norm, r_norm, (o, r) in zip(ref["keys"], ref["numel"], ours["norm"], ref["norm"], values):
            # (absolute floor: gradients whose true value is 0 hold rounding noise, see the UNet test below)
            assert abs(o_norm - r_norm) <= tol * r_norm + 1e-5 * n ** 0.5, (pin, mode, k, o_norm.item(), r_norm.item())
            assert (o - r).norm() <= tol * r.norm() + 1e-5 * r.numel() ** 0.5, (pin, mode, k, o, r)


@pytest.fixture(scope="module")
def fixture():
    return torch.load(os.path.join(GOLDEN, "vit_tiny_reference.pt"), weights_only=False)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_oracle_matches_reference_golden(fixture, mode):
    cfg = vo.vit_config(fixture["config_name"])
    sd = vo.init_state_dict(cfg, seed=fixture["weights_seed"])
    x, y = vo.synthetic_batch(cfg, fixture["batch"], seed=fixture["data_seed"])
    assert torch.equal(x, fixture["x"]) and torch.equal(y, fixture["labels"])
    loss, grads, taps = vo.train_step(sd, x, y, cfg, autocast_bf16=(mode == "bf16"), want_taps=True)
    ref = fixture["reference"][mode]
    # same torch build -> bit-identical; a different CPU / torch build may reorder fp32 sums, so allow a few ulps
    tol = dict(rtol=1e-5, atol=1e-6) if mode == "fp32" else dict(rtol=2e-2, atol=2e-3)
    assert torch.allclose(taps["encoded"].float(), ref["encoded"].float(), **tol)
    assert torch.allclose(taps["logits"].float(), ref["logits"].float(), **tol)
    assert torch.allclose(loss.float(), ref["loss"].float(), **tol)
    assert set(grads) == set(ref["grads"])
    for k, g in ref["grads"].items():
        err = (grads[k] - g).norm() / g.norm().clamp_min(1e-20)
        assert err < (1e-4 if mode == "fp32" else 2e-2), (k, err.item())


def test_state_dict_contract_matches_reference_vit_b16():
    with open(os.path.join(GOLDEN, "vit_b16_state_dict_keys.json")) as f:
        golden = json.load(f)
    cfg = vo.vit_config("vit_b16")
    spec = {k: list(s) for k, s in vo.state_dict_spec(cfg) if not k.startswith("head.linear")}
    assert spec == golden["keys"]
    assert golden["num_params"] == 85798656  # SURVEY.md finding 5


def test_loss_known_answer():
    # CrossEntropyLoss semantics (losses/basic.py:137-141): uniform logits -> log(C)
    logits = torch.zeros(5, 7)
    labels = torch.arange(5)[:, None]
    assert abs(vo.cross_entropy(logits, labels).item() - torch.log(torch.tensor(7.0)).item()) < 1e-6


def test_live_pin_against_reference():
    import make_golden

    make_golden.known_answer_attention()
    _check_pin("vit")


# ---- FCNN (BASELINE.json configs[0]) ----------------------------------------------------------------------------
def test_fcnn_oracle_matches_reference_golden():
    """oracle/fcnn_oracle.py vs the fixture written from the REAL reference FCNN + MAELoss + MSELoss (bit-exact)."""
    import fcnn_oracle as fo

    torch.set_num_threads(1)
    g = torch.load(os.path.join(GOLDEN, "fcnn_reference.pt"))
    assert g["keys"] == [k for k, _ in fo.state_dict_spec(10, 1)]
    x_all, y_all = fo.toy_data()
    assert torch.equal(x_all[:128], g["x"]) and torch.equal(y_all[:128], g["y"])  # examples/ml/simple/toy.py recipe
    sd = fo.init_state_dict(10, 1, seed=g["weights_seed"])
    loss, pred, grads = fo.train_step(sd, g["x"], g["y"])
    assert torch.equal(pred, g["pred"])
    assert torch.equal(loss, g["loss"])
    assert abs((g["mae"] + g["mse"]).item() - g["loss"].item()) <= 1e-6 * abs(g["loss"].item())
    for k, v in g["grads"].items():
        assert torch.equal(grads[k], v), k


def test_fcnn_live_pin_against_reference():
    _check_pin("fcnn")


# ---- CLIP vision tower (SURVEY.md 8a row a16, vision half) ------------------------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_clip_vision_oracle_matches_reference_golden(mode):
    """The oracle with CLIP._init_vision's options (no conv bias, embedding_norm, QuickGELU, eps 1e-5, head_norm after the
    cls pick, output_projection) vs the fixture written from the REAL reference ViTEncoder."""
    fx = torch.load(os.path.join(GOLDEN, "clip_vision_tiny_reference.pt"), weights_only=False)
    with open(os.path.join(GOLDEN, "clip_vision_tiny_keys.json")) as f:
        keys = json.load(f)["keys"]
    cfg = vo.vit_config(fx["config_name"])
    assert [[k, list(s)] for k, s in vo.state_dict_spec(cfg)] == keys
    sd = vo.init_state_dict(cfg, seed=fx["weights_seed"])
    out, grads, _ = vo.encoder_train_step(sd, fx["x"], fx["upstream"], cfg, autocast_bf16=(mode == "bf16"))
    ref = fx["reference"][mode]
    tol = dict(rtol=1e-5, atol=1e-6) if mode == "fp32" else dict(rtol=2e-2, atol=2e-3)
    assert out.dtype == ref["out"].dtype and torch.allclose(out.float(), ref["out"].float(), **tol)
    for k, g in ref["grads"].items():
        err = (grads[k] - g).norm() / g.norm().clamp_min(1e-20)
        assert err < (1e-4 if mode == "fp32" else 2e-2), (k, err.item())


def test_clip_vision_live_pin_against_reference():
    _check_pin("clip_vision")


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_clip_text_stack_oracle_matches_reference_golden(mode):
    """TeTEncoder as CLIP._init_text builds it (causal mask, QuickGELU, eps 1e-5): oracle vs the real-reference fixture."""
    fx = torch.load(os.path.join(GOLDEN, "clip_text_tiny_reference.pt"), weights_only=False)
    cfg = vo.tet_config(fx["config_name"])
    sd = vo.tet_init_state_dict(cfg, seed=fx["weights_seed"])
    out, dx, grads = vo.tet_train_step(sd, fx["x"], fx["upstream"], cfg, autocast_bf16=(mode == "bf16"))
    ref = fx["reference"][mode]
    tol = dict(rtol=1e-5, atol=1e-6) if mode == "fp32" else dict(rtol=2e-2, atol=2e-3)
    assert torch.allclose(out, ref["out"], **tol)
    assert (dx - ref["dx"]).norm() / ref["dx"].norm() < (1e-4 if mode == "fp32" else 2e-2)
    for k, g in ref["grads"].items():
        err = (grads[k] - g).norm() / g.norm().clamp_min(1e-20)
        assert err < (1e-4 if mode == "fp32" else 2e-2), (k, err.item())


def test_clip_text_stack_live_pin_against_reference():
    _check_pin("tet")


# ---- full CLIP forward (both towers + embedding / arg-max pooling / projection / l2-normalise / logits) ---------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_clip_oracle_matches_reference_golden(mode):
    """oracle/clip_oracle.py vs the fixture written from the REAL reference CLIP module (oracle/make_golden_clip.py);
    the token-embedding gather and the arg-max token pooling are integer ops: their gradients land on exactly the
    rows that were looked up."""
    import clip_oracle as co

    fx = torch.load(os.path.join(GOLDEN, "clip_tiny_reference.pt"), weights_only=False)
    cfg = co.clip_config(fx["config_name"])
    sd = co.init_state_dict(cfg, seed=fx["weights_seed"])
    x, ids = co.synthetic_batch(cfg, fx["x"].shape[0], seed=3)
    assert torch.equal(x, fx["x"]) and torch.equal(ids, fx["ids"])
    logits, grads = co.train_step(sd, x, ids, fx["upstream"], cfg, autocast_bf16=(mode == "bf16"))
    ref = fx["reference"][mode]
    tol = dict(rtol=1e-5, atol=1e-6) if mode == "fp32" else dict(rtol=2e-2, atol=2e-2)
    assert logits.dtype == ref["logits"].dtype and torch.allclose(logits.float(), ref["logits"].float(), **tol)
    for k, g in ref["grads"].items():
        err = (grads[k] - g).norm() / g.norm().clamp_min(1e-20)
        assert err < (1e-4 if mode == "fp32" else 3e-2), (k, err.item())
    # integer paths: exactly the embedding rows looked up at positions <= the pooled (arg-max) position receive gradient --
    # the causal mask keeps later tokens out of the pooled feature -- and never the padding row 0
    ge = grads["token_embedding.weight"]
    used = torch.zeros(cfg["vocab_size"], dtype=torch.bool)
    pooled = ids.argmax(-1)
    for b in range(ids.shape[0]):
        used[ids[b, : pooled[b] + 1]] = True
    assert torch.equal(ge.abs().sum(1) > 0, used & (torch.arange(cfg["vocab_size"]) != 0))
    assert (ids.argmax(-1) >= 1).all() and (ids.max(-1).values == cfg["vocab_size"] - 1).all()
    assert abs(co.symmetric_cross_entropy(torch.zeros(5, 5)).item() - torch.log(torch.tensor(5.0)).item()) < 1e-6


def test_clip_live_pin_against_reference():
    _check_pin("clip")


# ---- SD-v1.5 UNet (BASELINE.json configs[4]; oracle prepared ahead of the kernels) ---------------------------------------
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_unet_oracle_matches_reference_golden(mode):
    """oracle/unet_oracle.py (structure read off the state_dict keys) vs the fixture written from the REAL reference
    UNetDiffuser (oracle/make_golden_unet.py)."""
    import unet_oracle as uo

    fx = torch.load(os.path.join(GOLDEN, "unet_tiny_reference.pt"), weights_only=False)
    cfg = uo.unet_config(fx["config_name"])
    sd = uo.synthetic_state_dict([(k, tuple(s)) for k, s in fx["shapes"]], seed=fx["weights_seed"])
    out, grads = uo.train_step(sd, fx["x"], fx["timesteps"], fx["context"], fx["upstream"], cfg, autocast_bf16=(mode == "bf16"))
    ref = fx["reference"][mode]
    tol = dict(rtol=1e-5, atol=1e-5) if mode == "fp32" else dict(rtol=3e-2, atol=3e-2)
    assert out.dtype == ref["out"].dtype and torch.allclose(out.float(), ref["out"].float(), **tol)
    for k, g in ref["grads"].items():
        # (absolute floor: e.g. the last ResBlock's conv2.bias feeds a per-channel GroupNorm, its true gradient is 0 and
        # the fp32 value is rounding noise ~1e-6 that changes with the thread count)
        diff = (grads[k] - g).norm().item()
        assert diff < (1e-4 if mode == "fp32" else 3e-2) * g.norm().item() + 1e-5 * g.numel() ** 0.5, (k, diff, g.norm().item())
    # timestep embedding known answer (unet.py:53-77): cos block first, then sin; t = 0 -> (1, ..., 1, 0, ..., 0)
    e = uo.timestep_embedding(torch.tensor([0, 7]), 8, torch.float32)
    assert torch.equal(e[0], torch.tensor([1.0, 1, 1, 1, 0, 0, 0, 0])) and abs(e[1, 0].item() - torch.cos(torch.tensor(7.0)).item()) < 1e-6


def test_unet_live_pin_against_reference():
    _check_pin("unet")


def test_input_pipeline_oracle_known_values():
    """oracle/input_oracle.py (SURVEY.md N4): static_normalize + imagenet_normalize + hwc_to_chw on hand-computed pixels."""
    import numpy as np

    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import input_oracle as io

    x = np.zeros((1, 2, 2, 3), dtype=np.uint8)
    x[0, 0, 0] = (255, 0, 128)
    x[0, 1, 1] = (51, 102, 204)
    out = io.input_pipeline(x, 255.0, io.IMAGENET_MEAN, io.IMAGENET_STD)
    assert out.dtype == torch.float32 and tuple(out.shape) == (1, 3, 2, 2)
    want = torch.tensor([(1.0 - 0.485) / 0.229, (0.0 - 0.456) / 0.224, (128 / 255 - 0.406) / 0.225], dtype=torch.float64).float()
    assert torch.equal(out[0, :, 0, 0], want)
    want2 = torch.tensor([(0.2 - 0.485) / 0.229, (0.4 - 0.456) / 0.224, (0.8 - 0.406) / 0.225], dtype=torch.float64).float()
    assert torch.equal(out[0, :, 1, 1], want2)
    plain = io.input_pipeline(x)  # division only
    assert torch.equal(plain[0, :, 0, 0], torch.tensor([1.0, 0.0, 128 / 255], dtype=torch.float64).float())


def test_mixing_block_ops_is_the_same_computation_as_mixing_block():
    """oracle/vit_oracle.py::mixing_block_ops (op boundaries exposed for the per-op parity tests) == mixing_block, bit for bit,
    in fp32 and under bf16 autocast."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vit_oracle as vo

    cfg = vo.vit_config("vit_tiny")
    sd = vo.init_state_dict(cfg, seed=0)
    x = torch.randn(3, 5, cfg["latent_dim"], generator=torch.Generator().manual_seed(1))
    for autocast in (False, True):
        with torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
            a = vo.mixing_block(sd, 1, x, cfg["latent_dim"] // 64, 1e-6)
            b = vo.mixing_block_ops(sd, 1, x, cfg["latent_dim"] // 64, 1e-6)["out"]
        assert torch.equal(a, b)
