"""TEST INFRASTRUCTURE ONLY -- re-runs the bit-for-bit pins of the oracle against the real reference at the sizes the CPU
tests check (make_golden*.py ``pin*``, imported unmodified through oracle/load_reference.py) and writes
tests/golden/reference_pins.pt, plus tests/golden/reference_host_logic.json (``host_logic_reference``), so that the
tests can repeat each comparison without the reference tree.

Run where the reference project is checked out (oracle/load_reference.py, CFLEARN_REFERENCE_ROOT):
    python oracle/make_golden_pins.py

Stored per pin and mode, for every output and every parameter gradient of the reference: its L2 norm and at most
``SAMPLE`` of its values at fixed seeded positions (``summarize``).  ``oracle_outputs`` is the oracle's side of each pin on
the same seeded inputs; ``main`` checks it equals the reference's side bit for bit before anything is written.
"""
from __future__ import annotations

import os
import sys
from typing import Dict, List, Tuple

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)

import clip_oracle as co  # noqa: E402
import fcnn_oracle as fo  # noqa: E402
import unet_oracle as uo  # noqa: E402
import vit_oracle as vo  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(HERE), "tests", "golden")
PATH = os.path.join(GOLDEN, "reference_pins.pt")
SAMPLE = 16
THREADS = 1  # CPU bf16 autocast results change with the thread count: pins are stored and checked single-threaded
# pin -> (config name, batch); the unet pin runs 8x8 latents with a 3-token context
PINS: Dict[str, Tuple[str, int]] = {"vit": ("vit_tiny", 2), "clip_vision": ("clip_vision_tiny", 2), "tet": ("clip_text_tiny", 2),
                                    "clip": ("clip_tiny", 3), "unet": ("unet_tiny", 2), "fcnn": ("toy", 128)}
MODES = {"vit": ("fp32", "bf16"), "clip_vision": ("fp32", "bf16"), "tet": ("fp32", "bf16"), "clip": ("fp32", "bf16"),
         "unet": ("fp32", "bf16"), "fcnn": ("fp32",)}


def summarize(outputs: Dict[str, torch.Tensor]) -> Dict:
    """Per output (sorted by name): its element count, its L2 norm and its values -- all of them up to SAMPLE, else SAMPLE at
    positions drawn from a fixed seed -- concatenated into one tensor."""
    keys = sorted(outputs)
    flat = [outputs[k].detach().float().reshape(-1) for k in keys]
    values = [t if t.numel() <= SAMPLE else t[torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:SAMPLE]]
              for t in flat]
    return {"keys": keys, "numel": [t.numel() for t in flat], "norm": torch.stack([t.norm() for t in flat]),
            "lengths": [v.numel() for v in values], "values": torch.cat(values)}


def oracle_outputs(pin: str, mode: str, unet_shapes: List[Tuple[str, Tuple[int, ...]]] = ()) -> Dict[str, torch.Tensor]:
    """The oracle's outputs and parameter gradients for one pin, on the seeded inputs the matching ``pin*`` uses."""
    name, batch = PINS[pin]
    bf16 = mode == "bf16"
    if pin == "vit":
        cfg = vo.vit_config(name)
        x, y = vo.synthetic_batch(cfg, batch, seed=1)
        loss, grads, taps = vo.train_step(vo.init_state_dict(cfg, seed=0), x, y, cfg, autocast_bf16=bf16, want_taps=True)
        return {"encoded": taps["encoded"], "logits": taps["logits"], "loss": loss, **grads}
    if pin == "clip_vision":
        cfg = vo.vit_config(name)
        g = torch.Generator().manual_seed(5)
        x = torch.randn(batch, cfg["in_channels"], cfg["img_size"], cfg["img_size"], generator=g)
        up = torch.randn(batch, cfg["output_dim"], generator=g)
        out, grads, _ = vo.encoder_train_step(vo.init_state_dict(cfg, seed=0), x, up, cfg, autocast_bf16=bf16)
        return {"out": out, **grads}
    if pin == "tet":
        cfg = vo.tet_config(name)
        g = torch.Generator().manual_seed(7)
        x = torch.randn(batch, cfg["context_length"], cfg["latent_dim"], generator=g) * 0.5
        up = torch.randn(batch, cfg["context_length"], cfg["latent_dim"], generator=g)
        out, dx, grads = vo.tet_train_step(vo.tet_init_state_dict(cfg, seed=0), x, up, cfg, autocast_bf16=bf16)
        return {"out": out, "dx": dx, **grads}
    if pin == "clip":
        cfg = co.clip_config(name)
        x, ids = co.synthetic_batch(cfg, batch, seed=3)
        up = torch.randn(batch, batch, generator=torch.Generator().manual_seed(9))
        logits, grads = co.train_step(co.init_state_dict(cfg, seed=0), x, ids, up, cfg, autocast_bf16=bf16)
        return {"logits": logits, **grads}
    if pin == "unet":
        cfg = uo.unet_config(name)
        g = torch.Generator().manual_seed(11)
        x = torch.randn(batch, cfg["in_channels"], 8, 8, generator=g)
        ts = torch.randint(0, 1000, (batch,), generator=g)
        ctx = torch.randn(batch, 3, cfg["context_dim"], generator=g)
        up = torch.randn(batch, cfg["out_channels"], 8, 8, generator=g)
        out, grads = uo.train_step(uo.synthetic_state_dict(list(unet_shapes), seed=0), x, ts, ctx, up, cfg, autocast_bf16=bf16)
        return {"out": out, **grads}
    if pin == "fcnn":
        x_all, y_all = fo.toy_data()
        loss, pred, grads = fo.train_step(fo.init_state_dict(10, 1, seed=0), x_all[:batch], y_all[:batch])
        return {"pred": pred, "loss": loss, **grads}
    raise KeyError(pin)


def reference_outputs(pin: str, mode: str):
    """The reference's side of each pin (the ``pin*`` functions assert the oracle matches it bit for bit)."""
    import make_golden
    import make_golden_clip
    import make_golden_fcnn
    import make_golden_unet

    name, batch = PINS[pin]
    bf16 = mode == "bf16"
    if pin == "vit":
        make_golden.known_answer_attention()
        _, _, _, _, enc, logits, loss, grads = make_golden.pin(name, batch, bf16)
        return {"encoded": enc, "logits": logits, "loss": loss, **grads}, None
    if pin == "clip_vision":
        _, _, _, out, grads = make_golden.pin_clip_vision(name, batch, bf16)
        return {"out": out, **grads}, None
    if pin == "tet":
        _, _, _, out, dx, grads = make_golden.pin_tet(name, batch, bf16)
        return {"out": out, "dx": dx, **grads}, None
    if pin == "clip":
        _, _, _, _, logits, grads = make_golden_clip.pin(name, batch, bf16)
        return {"logits": logits, **grads}, None
    if pin == "unet":
        _, shapes, _, _, _, _, out, grads = make_golden_unet.pin(name, batch, 8, 3, bf16)
        return {"out": out, **grads}, shapes
    if pin == "fcnn":
        make_golden_fcnn.main()  # (rewrites tests/golden/fcnn_reference.pt with the same run)
        g = torch.load(os.path.join(GOLDEN, "fcnn_reference.pt"))
        return {"pred": g["pred"], "loss": g["loss"], **g["grads"]}, None
    raise KeyError(pin)


def host_logic_reference() -> Dict:
    """What the host-logic tests compare with: per-tensor (mean, std) of the reference ViTEncoder's own initialisation under
    seed 0, and the learning rates its default WarmupScheduler (multiplier 3 over 4 steps, then StepLR(2, 0.5)) writes into
    a torch.optim.Adam over 10 steps."""
    import importlib

    from load_reference import load_modules

    mods = load_modules()
    torch.manual_seed(0)
    enc = mods.build_encoder("vit", config=dict(img_size=64, patch_size=16, in_channels=3, latent_dim=256, num_layers=2))
    stats = {k: [v.float().mean().item(), v.float().std().item()] for k, v in enc.state_dict().items()}
    sch = importlib.import_module("cflearn.schedulers")
    adam = torch.optim.Adam([torch.nn.Parameter(torch.zeros(3))], lr=1e-3)
    s = sch.WarmupScheduler(adam, multiplier=3.0, warmup_step=4, scheduler_afterwards_base=torch.optim.lr_scheduler.StepLR,
                            scheduler_afterwards_config=dict(step_size=2, gamma=0.5))
    lrs = []
    for _ in range(10):
        adam.step()
        s.step()
        lrs.append(adam.param_groups[0]["lr"])
    return {"vit_init_stats_seed0": stats, "warmup_scheduler_lrs": lrs}


def main() -> None:
    import json

    torch.set_num_threads(THREADS)
    with open(os.path.join(GOLDEN, "reference_host_logic.json"), "w") as f:
        json.dump(host_logic_reference(), f, indent=1)
    record: Dict = {"pins": {}}
    for pin in PINS:
        for mode in MODES[pin]:
            ref, shapes = reference_outputs(pin, mode)
            if shapes is not None:
                record["unet_shapes"] = shapes
            ours = oracle_outputs(pin, mode, record.get("unet_shapes", ()))
            assert set(ours) == set(ref), (pin, mode, set(ours) ^ set(ref))
            for k, v in ref.items():
                assert torch.equal(ours[k], v.detach()), f"{pin} {mode}: {k} differs from the reference"
            record["pins"].setdefault(pin, {})[mode] = summarize(ref)
    torch.save(record, PATH)
    print(f"wrote {PATH} and reference_host_logic.json")


if __name__ == "__main__":
    main()
