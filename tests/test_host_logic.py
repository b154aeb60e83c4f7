"""CPU tests (no GPU, no compute calls into the CUDA library): C-ABI export table, registry / module surface,
parameter arena, data-parallel bucket layout and the world_size=2 gloo run of the bucket reducer."""
import json
import os
import re
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import cflearn_b200  # noqa: E402
from cflearn_b200 import _cabi, dp, registry, vit  # noqa: E402


def _header_functions():
    text = open(os.path.join(ROOT, "include", "b200_cflearn.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200_[a-z0-9_]+)\s*\(", text)))


def test_library_loads_and_exports_every_declared_symbol():
    assert _cabi.available(), _cabi.load_error()
    declared = _header_functions()
    assert declared, "no declarations parsed from include/b200_cflearn.h"
    exported = set(_cabi.exported_symbols())
    assert set(declared) == set(_cabi.SIGNATURES), (set(declared) ^ set(_cabi.SIGNATURES))
    assert not [n for n in declared if n not in exported]
    assert _cabi.lib().b200_abi_version() == 4
    assert _cabi.lib().b200_gemm_pick_splits(768, 768, 50432) >= 1


def test_product_path_fails_loudly_without_gpu():
    m = registry.build_module("cv_clf", config=dict(in_channels=3, num_classes=8, img_size=32, latent_dim=64, encoder="vit",
                                                    encoder_config=dict(patch_size=16, num_layers=1)))
    with pytest.raises(cflearn_b200.B200Error):
        m(torch.randn(2, 3, 32, 32))  # CPU tensor: no fallback
    with pytest.raises(cflearn_b200.B200Error):
        vit.cross_entropy(torch.zeros(2, 8), torch.zeros(2, dtype=torch.long))


def test_missing_library_is_reported(tmp_path, monkeypatch):
    monkeypatch.setattr(_cabi, "LIB_PATH", str(tmp_path / "libb200_cflearn.so"))
    monkeypatch.setattr(_cabi, "_lib", None)
    monkeypatch.setattr(_cabi, "_load_error", None)
    assert not _cabi.available()
    with pytest.raises(_cabi.B200Error, match="no CPU fallback"):
        _cabi.lib()


def test_registry_semantics_mirror_reference():
    # unknown keys are dropped (safe_execute), config is deep-copied, kwargs override the config
    cfg = dict(img_size=32, patch_size=16, in_channels=3, latent_dim=128, num_layers=1, something_else=3)
    e = registry.build_module("encoders.vit", config=cfg, num_layers=2)
    assert e.geo.L == 2 and cfg["num_layers"] == 1
    assert registry.encoders.has("vit") and registry.encoders.get("vit_b200") is vit.ViTEncoderB200
    with pytest.raises(KeyError):
        registry.build_module("no_such_module")
    fake_reference_dict = {"encoders.vit": object, "cv_clf": object}
    replaced = registry.install_into(fake_reference_dict)
    assert fake_reference_dict["encoders.vit"] is vit.ViTEncoderB200 and replaced["cv_clf"] is object
    for bad in (dict(dropout=0.1), dict(drop_path_rate=0.1), dict(norm_type="batch"), dict(output_dim=100),
                dict(feedforward_kwargs={"activation": "geglu"}), dict(to_patches_config={"padding": 1}),
                dict(embedding_norm=torch.nn.BatchNorm1d(128))):
        with pytest.raises(NotImplementedError):
            registry.build_module("encoders.vit", config=dict(img_size=32, patch_size=16, in_channels=3, latent_dim=128, **bad))


def test_fcnn_surface_mirrors_reference():
    # registry name, constructor defaults (fcnn.py:29-31), state_dict keys (golden fixture from the real reference)
    g = torch.load(os.path.join(ROOT, "tests", "golden", "fcnn_reference.pt"))
    m = registry.build_module("fcnn", config=dict(input_dim=10, output_dim=1, not_a_kwarg=1))
    assert list(m.state_dict().keys()) == g["keys"] and m.hidden_units == [32, 32]
    assert [tuple(v.shape) for v in m.state_dict().values()] == [(32, 10), (32,), (32, 32), (32,), (1, 32), (1,)]
    assert registry.build_module("fcnn", input_dim=600, output_dim=3).hidden_units == [1024, 1024]
    assert list(registry.build_module("fcnn", input_dim=4, output_dim=2, bias=False).state_dict()) == [
        "net.0.linear.linear.weight", "net.1.linear.linear.weight", "net.2.weight"]
    for bad in (dict(batch_norm=True), dict(dropout=0.3), dict(activation="GELU"), dict(mapping_type="res"), dict(rank=4)):
        with pytest.raises(NotImplementedError):
            registry.build_module("fcnn", input_dim=10, output_dim=1, **bad)
    with pytest.raises(cflearn_b200.B200Error):
        m(torch.randn(4, 10))  # CPU tensor: no fallback


def test_clip_vision_tower_options_mirror_reference_keys():
    # the ViTEncoder that CLIP._init_vision builds (multimodal/clip.py:121-135): key names AND order of the real reference
    with open(os.path.join(ROOT, "tests", "golden", "clip_vision_tiny_keys.json")) as f:
        golden = json.load(f)
    m = registry.build_module("encoders.vit", config=dict(
        img_size=64, patch_size=32, in_channels=3, latent_dim=128, to_patches_config={"bias": False}, num_layers=2,
        norm_kwargs={"eps": 1e-5}, embedding_norm=torch.nn.LayerNorm(128, 1e-5), attention_kwargs={"num_heads": 2},
        feedforward_kwargs={"activation": "quick_gelu"}, norm_after_head=True, output_dim=64))
    assert [[k, list(v.shape)] for k, v in m.state_dict().items()] == golden["keys"]
    assert m.geo.quick_gelu and m.geo.emb_eps == 1e-5 and m.geo.eps == 1e-5 and not m.geo.conv_bias


def test_tet_encoder_surface_mirrors_reference():
    # key names / order pinned by oracle/make_golden.py::pin_tet against the real TeTEncoder (buffer first, then parameters)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import vit_oracle as vo

    cfg = vo.tet_config("clip_text_tiny")
    m = registry.build_module("tet", config=dict(latent_dim=128, context_length=12, use_triu_attn_mask=True, num_layers=2,
                                                 norm_kwargs={"eps": 1e-5}, attention_kwargs={"num_heads": 2},
                                                 feedforward_kwargs={"activation": "quick_gelu"}, head_pooler=None))
    sd = m.state_dict()
    assert list(sd)[0] == "attention_mask" and sd["attention_mask"].dtype == torch.bool
    assert torch.equal(sd["attention_mask"], torch.ones(12, 12, dtype=torch.bool).triu(1))
    assert [(k, tuple(v.shape)) for k, v in list(sd.items())[1:]] == vo.tet_state_dict_spec(cfg)
    assert m.geo.causal and m.geo.tokens and m.geo.quick_gelu
    for bad in (dict(head_pooler="mean"), dict(dropout=0.1), dict(norm_position="post_norm"), dict(attention_kwargs={"num_heads": 6})):
        with pytest.raises(NotImplementedError):
            registry.build_module("tet", latent_dim=128, context_length=12, **bad)
    with pytest.raises(NotImplementedError):
        m(torch.zeros(1, 12, 128), mask=torch.zeros(12, 12, dtype=torch.bool))


def test_clip_module_surface_mirrors_reference():
    # CLIP.__init__ keywords, state_dict keys / order (pinned to the real reference CLIP by oracle/make_golden_clip.py)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import clip_oracle as co

    cfg = co.clip_config("clip_tiny")
    v, t = cfg["vision"], cfg["text"]
    m = registry.build_module("clip", config=dict(
        img_size=v["img_size"], latent_dim=cfg["latent_dim"], vision_latent_dim=v["latent_dim"], vision_patch_size=v["patch_size"],
        vision_num_heads=2, vision_num_layers=v["num_layers"], vocab_size=cfg["vocab_size"], context_length=t["context_length"],
        text_latent_dim=t["latent_dim"], text_num_heads=2, text_num_layers=t["num_layers"]))
    keys = [(k, tuple(p.shape)) for k, p in m.state_dict().items()]
    i = [k for k, _ in keys].index("text_transformer.attention_mask")
    assert keys[i - 1][0] == "token_embedding.weight"  # the buffer sits where the reference has it
    assert [kv for kv in keys if kv[0] != "text_transformer.attention_mask"] == co.state_dict_spec(cfg)
    assert abs(m.logit_scale.item() - 2.6592600) < 1e-5 and m.token_embedding.padding_idx == 0
    for bad in (dict(use_text=False), dict(token_type_size=2), dict(text_dropout=0.1), dict(text_head_pooler="mean")):
        with pytest.raises(NotImplementedError):
            registry.build_module("clip", img_size=64, latent_dim=64, vision_latent_dim=128, text_latent_dim=128, text_num_heads=2,
                                  vision_num_heads=2, **bad)
    with pytest.raises(cflearn_b200.B200Error):
        m(torch.zeros(1, 3, v["img_size"], v["img_size"]), torch.ones(1, t["context_length"], dtype=torch.long))  # CPU: no fallback


def test_param_arena_views_and_state_dict_roundtrip():
    m = registry.build_module("cv_clf", config=dict(in_channels=3, num_classes=16, img_size=32, latent_dim=128, encoder="vit",
                                                    encoder_config=dict(patch_size=16, num_layers=2)))
    a = m.arena
    for k, p in m.named_arena_parameters():
        assert p.data_ptr() == a.flat.data_ptr() + 4 * a.offsets[k]
        assert a.offsets[k] % 64 == 0
    # the module's own names are the reference cv_clf's: "encoder." + <ViTEncoder key>, then head.linear.*
    assert [k for k, _ in m.named_parameters()] == [("encoder." + k if not k.startswith("head.linear") else k) for k, _ in m.named_arena_parameters()]
    sd = {k: torch.randn_like(v) for k, v in m.state_dict().items()}
    m.load_state_dict(sd)
    a.ensure()
    bare = {(k[len("encoder."):] if k.startswith("encoder.") else k): v for k, v in sd.items()}
    for k in bare:
        assert torch.equal(a.p(k), bare[k])  # load_state_dict copies in place: the arena sees the new values
    m2 = m.double().float()  # _apply() re-allocates every parameter: views are broken, ensure() must repair them
    m2.arena.ensure()
    for k, p in m2.named_arena_parameters():
        assert p.data_ptr() == m2.arena.flat.data_ptr() + 4 * m2.arena.offsets[k]
        assert torch.equal(p, bare[k])
    m.load_reference_state_dict(sd)  # reference cv_clf checkpoint layout == our own state_dict layout
    m.load_state_dict(bare, strict=True)  # bare ViTEncoder keys + head.linear.* (what oracle/vit_oracle.py emits) are accepted too


def test_bucket_layout_covers_arena_without_overlap():
    m = registry.build_module("cv_clf", config=dict(in_channels=3, num_classes=16, img_size=32, latent_dim=128, encoder="vit",
                                                    encoder_config=dict(patch_size=16, num_layers=3)))
    red = dp.GradBucketReducer(m.arena, 3)
    spans = sorted(red.buckets.values())
    assert spans[0][0] == 0 and spans[-1][1] == m.arena.total
    for (lo0, hi0), (lo1, hi1) in zip(spans, spans[1:]):
        assert hi0 == lo1
    assert list(dp.shard_indices(10, 1, 4)) == [1, 5, 9]


def _worker(rank, world, port, total, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    assert dp.ddp_info() == (rank, world, rank)
    torch.manual_seed(0)
    m = registry.build_module("cv_clf", config=dict(in_channels=3, num_classes=16, img_size=32, latent_dim=128, encoder="vit",
                                                    encoder_config=dict(patch_size=16, num_layers=2)))
    with torch.no_grad():
        m.arena.flat.add_(rank)  # replicas differ until the broadcast
    dp.broadcast_parameters(m, src=0)
    red = dp.attach_reducer(m)
    g = m.arena.grad
    g.copy_(torch.arange(g.numel(), dtype=torch.float32) * (rank + 1))
    # the engine signals buckets in backward order: tail, blocks L-1..0, stem
    for key in ["tail", 1, 0, "stem"]:
        red.ready(key, g)
    red.finish()
    q.put((rank, m.arena.flat.sum().item(), g.clone()))
    dist.barrier()
    dist.destroy_process_group()


def test_world2_gloo_bucket_allreduce_matches_mean():
    world, port = 2, 29577
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, 0, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = [q.get(timeout=120) for _ in range(world)]
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (_, s0, g0), (_, s1, g1) = sorted(results, key=lambda t: t[0])
    assert s0 == s1  # parameters identical after the broadcast
    expect = torch.arange(g0.numel(), dtype=torch.float32) * 1.5  # mean of 1x and 2x
    assert torch.equal(g0, g1) and torch.allclose(g0, expect)


# ------------------------------------------------------------------------------------------------------------------
# initialisation statistics (SURVEY.md 8a row a15) and the optimizer's host surface
# ------------------------------------------------------------------------------------------------------------------
def _stats(t):
    t = t.detach().float()
    return t.mean().item(), t.std().item(), t.abs().max().item()


def test_vit_init_statistics_follow_reference():
    """mixed_stacks/api.py:405-417 (`_init_weights`: trunc_normal(0.02) Linear weights, zero biases, LayerNorm 1 / 0),
    api.py:205 and :405 (pos-enc / head token trunc_normal(0.02)), attentions.py:108-110 (in_w trunc_normal(0.02), zero
    qkv_bias), convs/basic.py:56,94-97 (xavier_normal, gain = sqrt 2 / sqrt 2 = 1 for the patch conv).  trunc_normal_ truncates at the
    ABSOLUTE bounds [-2, 2], so with std 0.02 the sample std is 0.02 and |w| stays far below 2."""
    torch.manual_seed(0)
    m = registry.build_module("cv_clf", config=dict(in_channels=3, num_classes=100, img_size=64, latent_dim=256, encoder="vit",
                                                    encoder_config=dict(patch_size=16, num_layers=2)))
    P = dict(m.named_arena_parameters())
    for k, p in P.items():
        mean, std, mx = _stats(p)
        if k.endswith("norm.weight") or k.endswith("norms.0.weight"):
            assert torch.equal(p.detach(), torch.ones_like(p)), k
        elif k.endswith("bias"):
            assert torch.equal(p.detach(), torch.zeros_like(p)), k
        elif k == "to_patches.projection.weight":
            fan_in, fan_out = 3 * 16 * 16, 256 * 16 * 16
            want = (2.0 / (fan_in + fan_out)) ** 0.5
            assert abs(std - want) < 0.03 * want and abs(mean) < 0.05 * want, (k, std, want)
        else:  # Linear weights, in_w, head token, positional encoding
            tol = 0.25 if p.numel() < 1000 else 0.05
            assert abs(std - 0.02) < tol * 0.02 and abs(mean) < 0.004 and mx < 0.2, (k, mean, std, mx)


def _reference_host_logic():
    with open(os.path.join(ROOT, "tests", "golden", "reference_host_logic.json")) as f:
        return json.load(f)


def test_vit_init_matches_reference_distribution_live():
    """Same statistics as the real ViTEncoder built under seed 0 (stored by oracle/make_golden_pins.py; not the same values --
    parity always injects identical weights -- but the same per-tensor std to a few percent)."""
    ref = _reference_host_logic()["vit_init_stats_seed0"]
    torch.manual_seed(1)
    ours = registry.build_module("encoders.vit", config=dict(img_size=64, patch_size=16, in_channels=3, latent_dim=256, num_layers=2))
    osd = ours.state_dict()
    assert list(ref.keys()) == list(osd.keys())
    for k, (rm, rs) in ref.items():
        om, os_, _ = _stats(osd[k])
        if rs == 0.0:
            assert os_ == 0.0 and rm == om, k
        else:
            tol = 0.3 if osd[k].numel() < 1000 else 0.06
            assert abs(os_ - rs) < tol * rs, (k, os_, rs)


def test_clip_text_tower_init_follows_reset_parameters():
    """multimodal/clip.py:188-207: std 0.01 positions, d^-0.5 in_w, d^-0.5 (2L)^-0.5 out / mlp[3], (2d)^-0.5 mlp[0]."""
    torch.manual_seed(0)
    m = registry.build_module("clip", config=dict(img_size=64, latent_dim=64, vision_latent_dim=128, vision_patch_size=32,
                                                  vision_num_heads=2, vision_num_layers=1, vocab_size=512, context_length=16,
                                                  text_latent_dim=128, text_num_heads=2, text_num_layers=3))
    P = m.text_transformer.arena.params
    d, L = 128, 3
    want = {"token_mixing.net.in_w": d ** -0.5, "token_mixing.net.out_linear.linear.weight": d ** -0.5 * (2 * L) ** -0.5,
            "channel_mixing.net.0.linear.weight": (2 * d) ** -0.5, "channel_mixing.net.3.linear.weight": d ** -0.5 * (2 * L) ** -0.5}
    for i in range(L):
        for suffix, std in want.items():
            _, s, _ = _stats(P[f"encoder.mixing_blocks.{i}.{suffix}"])
            assert abs(s - std) < 0.05 * std, (i, suffix, s, std)
    assert abs(_stats(P["encoder.pos_encoding.pos_encoding"])[1] - 0.01) < 0.002
    assert abs(_stats(m.token_embedding.weight)[1] - 0.02) < 0.002
    assert abs(_stats(m.text_projection.weight)[1] - d ** -0.5) < 0.05 * d ** -0.5 and torch.equal(m.text_projection.bias.detach(), torch.zeros(64))
    # the vision tower keeps the encoder's trunc_normal(0.02)
    assert abs(_stats(m.vit.arena.params["encoder.mixing_blocks.0.token_mixing.net.in_w"])[1] - 0.02) < 0.002


def test_arena_adam_host_surface():
    """param_groups / set_lr / state_dict round trip (what LR schedulers and checkpoints touch) -- no GPU involved."""
    from cflearn_b200.optim import ArenaAdam

    m = registry.build_module("cv_clf", config=dict(in_channels=3, num_classes=8, img_size=32, latent_dim=64, encoder="vit",
                                                    encoder_config=dict(patch_size=16, num_layers=1)))
    opt = ArenaAdam(m, lr=1e-3, betas=(0.9, 0.99), weight_decay=0.01)
    assert len(opt.param_groups) == 1 and len(opt.param_groups[0]["params"]) == len(list(m.parameters()))
    opt.set_lr(5e-4)
    assert opt.lr == 5e-4 and opt.param_groups[0]["lr"] == 5e-4
    opt.param_groups[0]["lr"] = 2.5e-4  # how torch.optim.lr_scheduler writes it
    assert opt.lr == 2.5e-4 and opt._hyper_tuple()[:5] == (2.5e-4, 0.9, 0.99, 1e-8, 0.01)


def test_cv_clf_state_dict_layout_is_the_reference_cv_clf_layout():
    """ADVICE r1: keys must be `encoder.<ViTEncoder keys>` + `head.linear.*`, in the reference's order."""
    with open(os.path.join(ROOT, "tests", "golden", "cv_clf_vit_tiny_keys.json")) as f:
        golden = json.load(f)["keys"]
    m = registry.build_module("cv_clf", config=dict(in_channels=3, num_classes=10, img_size=32, latent_dim=128, encoder="vit",
                                                    encoder_config=dict(patch_size=16, num_layers=2)))
    assert [[k, list(v.shape)] for k, v in m.state_dict().items()] == golden
    assert [k for k, _ in m.named_parameters()] == [k for k, _ in golden]
    # a bare-encoder-style checkpoint (ViTEncoder keys + head.linear.*) is accepted as well
    bare = {(k[len("encoder."):] if k.startswith("encoder.") else k): v.clone() for k, v in m.state_dict().items()}
    m.load_state_dict(bare, strict=True)


def test_build_module_merges_nested_kwargs_like_update_dict():
    """cflearn/modules/common.py:50-52: `update_dict(shallow_copy_dict(kwargs), kw)` merges nested dicts key by key."""
    cfg = dict(in_channels=3, num_classes=8, img_size=32, latent_dim=64, encoder="vit", encoder_config=dict(patch_size=16, num_layers=3))
    m = registry.build_module("cv_clf", config=cfg, encoder_config=dict(num_layers=1))
    assert m.geo.L == 1 and m.geo.patch == 16 and cfg["encoder_config"]["num_layers"] == 3  # nested key overridden, sibling kept, config untouched
    ln = torch.nn.LayerNorm(64, 1e-5)
    e = registry.build_module("encoders.vit", config=dict(img_size=32, patch_size=16, in_channels=3, latent_dim=64, num_layers=1, embedding_norm=ln))
    assert e.geo.emb_eps == 1e-5  # leaves (modules) are shared, not deep-copied


def test_install_into_the_real_reference_registry():
    """VERDICT r1 item 7: drop the B200 classes into a registry shaped like the reference's ``module_dict`` (name -> class)
    and build through its entries: class identity, the displaced entries handed back, and the state_dict layout of the
    reference's own ``cv_clf`` / ``ViTEncoder`` (stored from the real modules in tests/golden/cv_clf_vit_tiny_keys.json), which
    a checkpoint in that layout loads into with ``load_state_dict(strict=True)``."""
    with open(os.path.join(ROOT, "tests", "golden", "cv_clf_vit_tiny_keys.json")) as f:
        ref_keys = [(k, tuple(s)) for k, s in json.load(f)["keys"]]
    ref_enc_keys = [(k[len("encoder."):], s) for k, s in ref_keys if k.startswith("encoder.")]
    ref_dict = {name: type(name, (), {}) for name in ("cv_clf", "encoders.vit", "fcnn", "tet", "clip", "encoders.other")}
    before = dict(ref_dict)
    cfg = dict(in_channels=3, num_classes=10, img_size=32, latent_dim=128, encoder="vit", encoder_config=dict(patch_size=16, num_layers=2))
    replaced = registry.install_into(ref_dict)
    assert replaced == {k: v for k, v in before.items() if k != "encoders.other"}
    assert ref_dict["encoders.other"] is before["encoders.other"]
    for name in ("encoders.vit_b200", "cv_clf_b200", "fcnn_b200", "tet_b200", "clip_b200", "encoders.vit", "cv_clf", "fcnn", "tet", "clip"):
        assert ref_dict[name] is registry.module_dict[name], name
    after = registry._safe_execute(ref_dict["cv_clf"], dict(cfg))                   # what the reference's build_module does
    assert type(after) is vit.VanillaClassifierB200
    assert [(k, tuple(v.shape)) for k, v in after.state_dict().items()] == ref_keys
    ckpt = {k: torch.randn(s) for k, s in ref_keys}
    after.load_state_dict(ckpt, strict=True)                                         # reference checkpoint -> drop-in, strict
    assert all(torch.equal(after.state_dict()[k], v) for k, v in ckpt.items())
    enc = registry._safe_execute(ref_dict["encoders.vit"], dict(img_size=32, patch_size=16, in_channels=3, latent_dim=128, num_layers=2))
    assert type(enc) is vit.ViTEncoderB200
    assert [(k, tuple(v.shape)) for k, v in enc.state_dict().items()] == ref_enc_keys
    enc.load_state_dict({k: ckpt["encoder." + k] for k, _ in ref_enc_keys}, strict=True)
    ref_dict.update(replaced)
    assert {k: ref_dict[k] for k in before} == before


def test_reference_warmup_scheduler_drives_arena_adam():
    """N2 / ADVICE r1: the reference's default scheduler policy (cflearn/schedulers.py:126-171 ``WarmupScheduler``, multiplier 3
    over 4 steps, then a StepLR(2, 0.5) follow-up; pipeline/blocks/basic.py:334-352), expressed with torch's own LambdaLR,
    drives ``ArenaAdam`` (a real torch Optimizer) through the same learning rates as ``torch.optim.Adam`` -- the sequence
    the reference scheduler itself wrote into a torch Adam (tests/golden/reference_host_logic.json)."""
    from cflearn_b200.optim import ArenaAdam

    want = _reference_host_logic()["warmup_scheduler_lrs"]
    m = registry.build_module("cv_clf", config=dict(in_channels=3, num_classes=8, img_size=32, latent_dim=64, encoder="vit",
                                                    encoder_config=dict(patch_size=16, num_layers=1)))
    ours = ArenaAdam(m, lr=1e-3, capturable=False)
    assert isinstance(ours, torch.optim.Optimizer)
    ref = torch.optim.Adam([torch.nn.Parameter(torch.zeros(3))], lr=1e-3)

    def factor(epoch):
        return 1.0 + (3.0 - 1.0) * epoch / 4 if epoch <= 4 else 3.0 * 0.5 ** ((epoch - 5) // 2)

    s_ours, s_ref = torch.optim.lr_scheduler.LambdaLR(ours, factor), torch.optim.lr_scheduler.LambdaLR(ref, factor)
    seq_o, seq_r = [], []
    for _ in range(10):
        if hasattr(ours, "_opt_called"):
            ours._opt_called = True  # (no GPU here: tell the scheduler a step happened without launching the kernel)
        ref.step()
        s_ours.step()
        s_ref.step()
        seq_o.append(ours.lr)
        seq_r.append(ref.param_groups[0]["lr"])
    assert seq_o == seq_r and seq_o == pytest.approx(want, rel=1e-12) and max(seq_o) == pytest.approx(3e-3) and seq_o[-1] < 1e-3
    assert ours._hyper_tuple()[0] == seq_o[-1]  # what the next step pushes to the device


def test_persistent_cta_bound_is_a_plain_host_setting():
    """``b200_set_persistent_ctas`` (grid bound of the persistent kernels while an all-reduce holds SMs) touches no device: it
    returns the previous bound, 0 / negative clears it."""
    lib = _cabi.lib()
    first = lib.b200_set_persistent_ctas(132, 0)
    try:
        assert lib.b200_set_persistent_ctas(140, 3) == 132
        assert lib.b200_set_persistent_ctas(0, 0) == 140
        assert lib.b200_set_persistent_ctas(-5, 7) == 0
        assert lib.b200_set_persistent_ctas(0, 0) == 0
    finally:
        lib.b200_set_persistent_ctas(first, 0)


def test_bench_dp_mode_auto_resolves_by_world_size(monkeypatch):
    """``bench.py --dp-mode auto``: the in-graph bucketed exchange up to 2 GPUs, one all-reduce behind the graph from 3 GPUs up
    (what measured best at each size, DESIGN.md section 4)."""
    import importlib
    import sys as _sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    if root not in _sys.path:
        _sys.path.insert(0, root)
    bench = importlib.import_module("bench")
    seen = {}
    monkeypatch.setattr(bench, "run_b200", lambda args: seen.update(mode=args.dp_mode, flat=args.flat_allreduce))
    for world, mode, flat in (("1", "graph", False), ("2", "graph", False), ("4", "flat", True), ("8", "flat", True)):
        monkeypatch.setenv("WORLD_SIZE", world)
        monkeypatch.setattr(_sys, "argv", ["bench.py"])
        bench.main()
        assert seen == dict(mode=mode, flat=flat), (world, seen)
    monkeypatch.setattr(_sys, "argv", ["bench.py", "--dp-mode", "graph"])
    bench.main()
    assert seen["mode"] == "graph"


def test_header_is_plain_c():
    """The boundary is a C ABI: ``include/b200_cflearn.h`` must parse as C99 on its own (no CUDA headers, no C++), which is what a
    cgo / JNI / ctypesgen consumer would feed it to."""
    import shutil
    import subprocess

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([gcc, "-x", "c", "-std=c99", "-pedantic", "-Wall", "-Werror", "-fsyntax-only", os.path.join(root, "include", "b200_cflearn.h")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_product_code_never_touches_the_oracle():
    """``oracle/`` is test infrastructure: nothing under the package may import, read or execute it, and the package has no CPU
    path to fall back to (a CPU tensor raises)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pkg = os.path.join(root, "carefree-learn_b200")
    offenders = []
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                for m in re.finditer(r"^\s*(?:from|import)\s+([\w\.]*oracle[\w\.]*)|oracle/|vit_oracle|clip_oracle|unet_oracle|fcnn_oracle", text, re.M):
                    line = text[: m.start()].count("\n") + 1
                    src = text.splitlines()[line - 1]
                    if "import" in src or "open(" in src or "sys.path" in src:
                        offenders.append((f, line, src.strip()))
    assert not offenders, offenders
    import torch

    from cflearn_b200 import ops
    from cflearn_b200._cabi import B200Error

    with pytest.raises(B200Error):
        ops.gemm(torch.zeros(8, 8, dtype=torch.bfloat16), torch.zeros(8, 8, dtype=torch.bfloat16))


def test_bench_dump_outputs_writes_fixed_float32_samples(tmp_path, monkeypatch):
    """``bench.py --dump-outputs DIR``: loss, parameters and gradients as float32 .npy; an arena longer than DUMP_SAMPLE is cut
    to the same seeded positions on every run (two builds compare output for output); --steps below 1 is refused."""
    import importlib
    import types

    import numpy as np

    bench = importlib.import_module("bench")
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 64)
    small = types.SimpleNamespace(flat=torch.arange(10.0), grad=-torch.arange(10.0))
    big = types.SimpleNamespace(flat=torch.arange(1000.0), grad=torch.arange(1000.0) * 2)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), torch.tensor(1.5), [("small_", small), ("big_", big)])
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == ["big_grads.npy", "big_params.npy", "loss.npy", "small_grads.npy", "small_params.npy"]
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype == np.float32 and np.array_equal(a, b), n
    assert np.array_equal(np.load(tmp_path / "a" / "small_grads.npy"), -np.arange(10.0, dtype=np.float32))
    p, g = np.load(tmp_path / "a" / "big_params.npy"), np.load(tmp_path / "a" / "big_grads.npy")
    assert p.shape == (64,) and np.array_equal(g, 2 * p) and np.all(np.diff(p) >= 0)  # same sorted positions in both arrays
    assert np.load(tmp_path / "a" / "loss.npy").tolist() == [1.5]
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit):
        bench.main()
