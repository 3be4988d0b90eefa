"""CPU: the oracle (oracle/clipvip_oracle.py) replays the golden vectors that
tests/golden/make_golden.py produced from the real reference modules."""
import os

import pytest
import torch

from oracle import clipvip_oracle as O


def _rel(a, b):
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _cfg(meta):
    return O.ClipVipCfg(vision=O.TowerCfg(768, 12, meta["vision_layers"], 3072),
                        text=O.TowerCfg(512, 8, meta["text_layers"], 2048))


def _replay(gold, need_grads):
    meta = gold["meta"]
    cfg = _cfg(meta)
    sd = O.init_state_dict(cfg, seed=meta["weight_seed"])
    video, ids, mask = O.synthetic_batch(meta["B"], meta["T"], meta["Lt"], cfg, seed=meta["data_seed"],
                                         ragged_text=meta["ragged"])
    assert torch.equal(ids, gold["input_ids"]) and torch.equal(mask, gold["attention_mask"])
    assert abs(float(video.double().sum()) - gold["video_checksum"]) < 1e-6 * video.numel() ** 0.5
    if need_grads:
        sd = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    return cfg, sd, video, ids, mask


def test_depth2_ragged_forward_hidden_and_grads(golden_dir):
    gold = torch.load(os.path.join(golden_dir, "depth2_b3_t12_ragged.pt"), weights_only=False)
    cfg, sd, video, ids, mask = _replay(gold, need_grads=True)
    pooled_v, vh = O.vision_tower(sd, video, cfg, return_hidden=True)
    pooled_t, th = O.text_tower(sd, ids, mask, cfg, return_hidden=True)
    got_rows = torch.stack([torch.cat([h[:, :8], h[:, -4:]], 1).detach() for h in vh])
    assert _rel(got_rows, gold["vision_hidden_rows"]) < 1e-5
    assert _rel(torch.stack([h.detach() for h in th]), gold["text_hidden"]) < 1e-5
    out = O.clip_vip_forward(sd, video, ids, mask, cfg)
    assert _rel(out["vis_features"].detach(), gold["vis_features"]) < 1e-5
    assert _rel(out["text_features"].detach(), gold["text_features"]) < 1e-5
    loss = O.nce_learnable_temp_loss(out["vis_features"], out["text_features"], sd["logit_scale"])
    assert abs(float(loss) - float(gold["loss"])) < 1e-5 * abs(float(gold["loss"]))
    loss.backward()
    for k, gn in gold["grad_norms"].items():
        if gn > 1e-5:
            assert abs(float(sd[k].grad.norm()) - gn) < 1e-3 * gn, k
    for k, sample in gold["grad_samples"].items():
        assert _rel(sd[k].grad.flatten()[:256], sample) < 1e-3, k


@pytest.mark.timeout(600)
def test_cfg1_full_depth_forward(golden_dir):
    """BASELINE.json configs[0]: ViT-B/16, B=2, T=4 (temporal interpolation 12 -> 4), 32 tokens, fp32 CPU."""
    gold = torch.load(os.path.join(golden_dir, "cfg1_b2_t4.pt"), weights_only=False)
    cfg, sd, video, ids, mask = _replay(gold, need_grads=False)
    with torch.no_grad():
        out = O.clip_vip_forward(sd, video, ids, mask, cfg)
        loss = O.nce_learnable_temp_loss(out["vis_features"], out["text_features"], sd["logit_scale"])
    assert _rel(out["vis_features"], gold["vis_features"]) < 1e-5
    assert _rel(out["text_features"], gold["text_features"]) < 1e-5
    assert abs(float(loss) - float(gold["loss"])) < 1e-5 * abs(float(gold["loss"]))


def test_nce_loss_gather_and_closed_form(golden_dir):
    gold = torch.load(os.path.join(golden_dir, "nce_loss_w4.pt"), weights_only=False)
    V = O.gather_rank_major(gold["vis_per_rank"])
    T = O.gather_rank_major(gold["txt_per_rank"])
    loss = O.nce_learnable_temp_loss(V, T, gold["logit_scale"])
    assert abs(float(loss) - float(gold["loss"])) < 1e-6
    dv, dt, dl = O.nce_closed_form_grads(V, T, gold["logit_scale"])
    assert _rel(dv, gold["d_vis"]) < 1e-5 and _rel(dt, gold["d_txt"]) < 1e-5
    assert abs(float(dl) - float(gold["d_logit_scale"])) < 1e-5


def test_vip_attention_equals_block_masked_dense():
    """forward2 == dense attention under allow[i,j] = global(i) | global(j) | frame(i)==frame(j) (SURVEY Appendix A)."""
    torch.manual_seed(3)
    heads, C, M, T, L = 2, 32, 4, 3, 5
    S = M + T * L
    sd = {}
    for n in ("q_proj", "k_proj", "v_proj", "out_proj"):
        sd[f"a.{n}.weight"] = torch.randn(C, C, dtype=torch.float64) * 0.2
        sd[f"a.{n}.bias"] = torch.randn(C, dtype=torch.float64) * 0.1
    x = torch.randn(2, S, C, dtype=torch.float64)
    got = O.vip_attention(sd, x, "a.", heads, (M, T, L))
    frame = torch.cat([torch.full((M,), -1), torch.arange(T).repeat_interleave(L)])
    allow = (frame[:, None] < 0) | (frame[None, :] < 0) | (frame[:, None] == frame[None, :])
    add = torch.zeros(S, S, dtype=torch.float64).masked_fill(~allow, float("-inf"))[None, None]
    want = O.dense_attention(sd, x, "a.", heads, add)
    assert _rel(got, want) < 1e-12


def test_flop_model_matches_baseline_md():
    f = O.flops_per_pair(O.ClipVipCfg(), T=12, Lt=32)
    assert abs(f["fwd"] / 1e9 - 423.12) < 0.05
    assert abs(f["train"] / 1e9 - 1266.58) < 0.2
    assert abs(f["vip_block_fwd"] / 1e9 - 34.825) < 0.01


# ------------------------------------------------------------------ config #4: HD-VILA TimeSformer
def _tsf_replay(gold):
    from oracle import timesformer_oracle as TO

    cfg = TO.TimeSformerCfg(**gold["cfg"])
    sd = {k: v.clone().requires_grad_(True) for k, v in TO.init_state_dict(cfg, seed=gold["weight_seed"]).items()}
    x = TO.synthetic_input(gold["B"], gold["T"], gold["H"], gold["W"], cfg, seed=gold["data_seed"]).requires_grad_(True)
    g = torch.Generator().manual_seed(gold["data_seed"] + 1)
    w_out = torch.randn(gold["out"].shape, generator=g) / (gold["B"] * gold["T"] * gold["H"] * gold["W"]) ** 0.5
    return TO, cfg, sd, x, w_out


@pytest.mark.parametrize("name", ["timesformer_interp_b2", "timesformer_native_b2"])
def test_timesformer_oracle_replays_reference_golden(golden_dir, name):
    gold = torch.load(os.path.join(golden_dir, name + ".pt"), weights_only=False)
    TO, cfg, sd, x, w_out = _tsf_replay(gold)
    out, hidden = TO.timesformer_forward(sd, x, cfg, return_hidden=True)
    assert out.shape == gold["out"].shape
    assert _rel(out.detach(), gold["out"]) < 1e-5
    assert _rel(torch.stack([h[:, :6].detach() for h in hidden]), gold["hidden_rows"]) < 1e-5
    loss = (out * w_out).sum()
    assert abs(float(loss) - float(gold["loss"])) < 1e-5 * max(1.0, abs(float(gold["loss"])))
    loss.backward()
    assert _rel(x.grad[:, 0], gold["dx_t0"]) < 1e-4
    for n, ref in gold["grads"].items():
        got = sd[n].grad[:8] if ref.dim() == 2 else sd[n].grad
        assert float((got - ref).norm()) < 1e-4 * gold["grad_norms"][n] + 1e-9, n
    assert sd["norm.weight"].grad is None      # constructed but never applied (timesformer.py:451)


def test_timesformer_flop_model_matches_baseline_md():
    from oracle import timesformer_oracle as TO

    cfg = TO.TimeSformerCfg()
    assert abs(TO.flops_per_sample(cfg, 7, 10, 16) / 1e9 - 162.78) < 0.01     # BASELINE.md §2
    assert abs(TO.flops_per_sample(cfg, 8, 7, 7) / 1e9 - 56.27) < 0.01
    assert abs(TO.flops_per_sample(cfg, 8, 28, 28) / 1e9 - 975.81) < 0.01


# ------------------------------------------------------------------ SURVEY §8(f).1: optimizer step
def test_adamw_oracle_replays_reference_trajectory(golden_dir):
    from oracle import adamw_oracle as AO

    gold = torch.load(os.path.join(golden_dir, "adamw_8steps.pt"), weights_only=False)
    cfg, shapes = gold["cfg"], gold["shapes"]
    g0 = torch.Generator().manual_seed(0)
    p = {n: torch.randn(s, generator=g0) for n, s in shapes.items()}
    m = {n: torch.zeros_like(v) for n, v in p.items()}
    v = {n: torch.zeros_like(x) for n, x in p.items()}
    named = [(n, torch.nn.Parameter(p[n].clone())) for n in shapes]
    groups = AO.param_groups(named, cfg["learning_rate"], cfg["weight_decay"], cfg["lr_mul"], cfg["lr_mul_prefix"])
    name_of = {id(q): n for n, q in named}
    assert [[name_of[id(q)] for q in g["params"]] for g in groups] == gold["group_names"]
    for step in range(1, cfg["steps"] + 1):
        lr = AO.lr_schedule(step, cfg["decay"], cfg["learning_rate"], cfg["num_train_steps"], cfg["warmup_ratio"])
        assert lr == gold["lrs"][step - 1]
        scale = 0.01 if step % 3 == 0 else 1.0
        grads = {n: torch.randn(s, generator=torch.Generator().manual_seed(1000 * step + i)) * scale
                 for i, (n, s) in enumerate(shapes.items())}
        total, coef = AO.clip_coef([grads[n] for n in shapes], cfg["grad_norm"])
        assert abs(float(total) - gold["norms"][step - 1]) < 1e-5 * gold["norms"][step - 1]
        for gi, g in enumerate(groups):
            for q in g["params"]:
                n = name_of[id(q)]
                AO.adamw_step(p[n], grads[n] * coef, m[n], v[n], step, cfg["lr_mul"] * lr if gi < 2 else lr,
                              tuple(cfg["betas"]), 1e-6, g["weight_decay"], True)
    for n in shapes:
        assert torch.equal(p[n], gold["final_p"][n]) and torch.equal(m[n], gold["final_m"][n]), n
        assert torch.equal(v[n], gold["final_v"][n]), n


def test_timesformer_oracle_training_mode_drop_path_golden(golden_dir):
    """Training mode (stochastic depth): the oracle with the factors the reference drew reproduces the reference's
    train() forward and gradients; and re-drawing them under the stored torch seed gives the same factors."""
    from oracle import timesformer_oracle as TO

    gold = torch.load(os.path.join(golden_dir, "timesformer_train_droppath.pt"), weights_only=False)
    cfg = TO.TimeSformerCfg(**gold["cfg"])
    B, T, H, W = gold["B"], gold["T"], gold["H"], gold["W"]
    torch.manual_seed(gold["torch_seed"])
    redraw = TO.draw_drop_masks(cfg, B, T, H, W, gold["rate"])
    for a, b in zip(redraw, gold["masks"]):
        assert (a is None) == (b is None)
        if a is not None:
            assert all(torch.equal(u, v) for u, v in zip(a, b))
    sd = {k: v.clone().requires_grad_(True) for k, v in TO.init_state_dict(cfg, seed=gold["weight_seed"]).items()}
    x = TO.synthetic_input(B, T, H, W, cfg, seed=gold["data_seed"]).requires_grad_(True)
    g = torch.Generator().manual_seed(gold["data_seed"] + 1)
    w_out = torch.randn(gold["out"].shape, generator=g) / (B * T * H * W) ** 0.5
    out = TO.timesformer_forward(sd, x, cfg, drop_masks=gold["masks"])
    assert _rel(out.detach(), gold["out"]) < 1e-5
    (out * w_out).sum().backward()
    assert _rel(x.grad[:, 0], gold["dx_t0"]) < 1e-4
    for n, ref in gold["grads"].items():
        got = sd[n].grad[:8] if ref.dim() == 2 else sd[n].grad
        assert float((got - ref).norm()) < 1e-4 * gold["grad_norms"][n] + 1e-9, n


def test_nce_vsc_fc_oracle_replays_reference_golden(golden_dir):
    gold = torch.load(os.path.join(golden_dir, "nce_vsc_fc_n24.pt"), weights_only=False)
    feats = [gold[k].clone().requires_grad_(True) for k in ("vis", "txt", "img", "cap")]
    temp = gold["logit_scale"].clone().requires_grad_(True)
    loss = O.nce_vsc_fc_loss(*feats, temp)
    loss.backward()
    assert abs(float(loss) - float(gold["loss"])) < 1e-5 * abs(float(gold["loss"]))
    for f, k in zip(feats, ("d_vis", "d_txt", "d_img", "d_cap")):
        assert _rel(f.grad, gold[k]) < 1e-5
    assert abs(float(temp.grad) - float(gold["d_logit_scale"])) < 1e-5 * abs(float(gold["d_logit_scale"]))


def test_retrieval_metrics_oracle_replays_reference_golden(golden_dir):
    """§8(f).3: similarity, DSL re-weighting and compute_metrics (with its tie quirk) vs the reference's own numpy code."""
    import numpy as np
    from oracle import metrics_oracle as MO

    gold = torch.load(os.path.join(golden_dir, "retrieval_metrics_n57.pt"), weights_only=False)
    txt, vis = gold["txt"].numpy(), gold["vis"].numpy()
    sim = MO.cal_cossim(txt, vis)
    assert np.allclose(sim, gold["sim"].numpy(), rtol=0, atol=1e-6)       # BLAS summation order may differ between hosts
    sim = gold["sim"].numpy()                                             # integer logic below: on the stored matrix, exact
    for kind, m in (("simple", sim), ("DSL", MO.dsl(sim, 100.0))):
        for direction, x in (("t2v", m), ("v2t", m.T)):
            g, e = MO.rank_counts(x)
            assert np.array_equal(g, gold[f"{kind}_{direction}_greater"].numpy()), (kind, direction)
            assert np.array_equal(e, gold[f"{kind}_{direction}_equal"].numpy())
            assert tuple(float(v) for v in MO.compute_metrics(x)) == gold[f"{kind}_{direction}"]
    assert int(gold["simple_t2v_equal"].max()) >= 2                       # the fixture really contains ties


# ------------------------------------------------------------------ config #5: LF-VILA Swin-3D video encoder
@pytest.mark.parametrize("name", ["swin3d_small_b2", "swin3d_padded_b1", "swin3d_train_droppath"])
def test_swin3d_oracle_replays_reference_golden(golden_dir, name):
    from oracle import swin3d_oracle as SO

    gold = torch.load(os.path.join(golden_dir, name + ".pt"), weights_only=False)
    cfg = SO.Swin3DCfg(**gold["cfg"])
    sd = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v)
          for k, v in SO.init_state_dict(cfg, seed=gold["weight_seed"]).items()}
    video = SO.synthetic_video(gold["B"], gold["D"], gold["H"], gold["W"], cfg, seed=gold["data_seed"])
    if gold["train_rate"]:                       # the DropPath factors the reference drew are reproduced from its torch seed
        torch.manual_seed(gold["torch_seed"])
        masks = SO.draw_drop_masks(cfg, gold["B"], gold["train_rate"])
        for a, b in zip(masks, gold["masks"]):
            assert (a is None) == (b is None) and (a is None or all(torch.equal(u, v) for u, v in zip(a, b)))
    out, stages = SO.swin3d_forward(sd, video, cfg, drop_masks=gold["masks"], return_stages=True)
    assert out.shape == gold["out"].shape and _rel(out.detach(), gold["out"]) < 1e-5
    for s, ref in zip(stages, gold["stage_rows"]):
        assert _rel(s.flatten(0, 3)[:4].detach(), ref) < 1e-5
    g = torch.Generator().manual_seed(gold["data_seed"] + 1)
    w_out = torch.randn(out.shape, generator=g) / out[0].numel() ** 0.5
    (out * w_out).sum().backward()
    for n, ref in gold["grads"].items():
        got = sd[n].grad if ref.shape == sd[n].grad.shape else sd[n].grad[:8]
        assert float((got - ref).norm()) < 1e-4 * gold["grad_norms"][n] + 1e-9, n
    assert sd["norm_local.weight"].grad is None and sd["local_feat_proj.reduction.weight"].grad is None   # (x, x) quirk


def test_swin3d_flop_and_parameter_model_matches_baseline_md():
    from oracle import swin3d_oracle as SO

    cfg = SO.Swin3DCfg()
    assert sum(v.numel() for v in SO.init_state_dict(cfg).values() if v.is_floating_point()) == 89_229_448   # BASELINE.md §2
    assert abs(SO.flops_per_sample(cfg, 32, 224, 224, include_dead_local_proj=True) / 1e9 - 327.14) < 0.01
    assert abs(SO.flops_per_sample(cfg, 32, 192, 320, include_dead_local_proj=True) / 1e9 - 313.63) < 0.01


@pytest.mark.timeout(900)
def test_full_depth_t12_golden_with_whole_gradient_tensors(golden_dir):
    """The BENCH model (12 + 12 layers, T = 12, ragged text) with the gradients the GPU parity test is calibrated on
    (tests/golden/make_golden.py full12, made from the real reference modules): the oracle replays features, loss, at
    least 4096 elements of each of fifteen weight-gradient tensors (first and last row whole, the rest a fixed, seeded
    sample) and every bias / LayerNorm gradient vector whole (both stored as fp16 after max-normalisation: 2^-11 per
    element) in fp32 on the CPU."""
    gold = torch.load(os.path.join(golden_dir, "full12_b4_t12_ragged.pt"), weights_only=False)
    meta = gold["meta"]
    cfg = O.ClipVipCfg()
    sd = O.init_state_dict(cfg, seed=meta["weight_seed"])
    video, ids, mask = O.synthetic_batch(meta["B"], meta["T"], meta["Lt"], cfg, seed=meta["data_seed"], ragged_text=True)
    assert torch.equal(ids, gold["input_ids"]) and torch.equal(mask, gold["attention_mask"])
    assert abs(float(video.double().sum()) - gold["video_checksum"]) < 1e-6
    sd = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    out = O.clip_vip_forward(sd, video, ids, mask, cfg)
    assert _rel(out["vis_features"].detach(), gold["vis_features"]) < 2e-5
    assert _rel(out["text_features"].detach(), gold["text_features"]) < 2e-5
    loss = O.nce_learnable_temp_loss(out["vis_features"], out["text_features"], sd["logit_scale"])
    assert abs(float(loss.detach()) - float(gold["loss"])) < 2e-5 * abs(float(gold["loss"]))
    loss.backward()
    assert len(gold["grad_full"]) >= 12
    for k, ent in gold["grad_full"].items():
        want = ent["data"].float() * ent["scale"]
        got = sd[k].grad.flatten()[ent["index"].long()]
        assert _rel(got, want) < 1e-3, (k, _rel(got, want))       # fp16 storage of the golden: ~3e-4
    ref_norm = gold["grad_norms"]["logit_scale"]
    for k, ent in gold["grad_vectors"].items():
        g = ent["data"].float() * ent["scale"]
        if float(g.norm()) > 1e-3 * ref_norm:
            assert _rel(sd[k].grad, g) < 1e-3, (k, _rel(sd[k].grad, g))
