"""B200: the CUDA path (VidCLIP module -> C ABI kernels) against the CPU oracle and the golden vectors that were
generated from the real reference (tests/golden/make_golden.py).

Tolerances (bf16 compute, fp32 oracle).  BASELINE.md §3 calibrates what bf16 costs the REFERENCE ITSELF
(autocast vs its own fp32, 12 layers): embeddings rel-L2 4.4e-3 (video) / 7.9e-3 (text), loss rel-err 9.4e-4.
SURVEY.md §8c sets the bar at 2x that for tensors and cosine >= 1 - 1e-3 per row.  Integer paths (patch /
sequence order, EOS argmax, token gather) are bit-exact and covered in test_gpu_kernels.py.
"""
import os
from types import SimpleNamespace

import pytest
import torch

pytestmark = pytest.mark.gpu

# Small-golden bars.  Calibrated on this pool's B200 (profiles/r02_pytest_gpu_parity_v2_fp32_residual.log): the reference's own
# bf16-autocast run deviates from its fp32 output by 3.8e-3 (video) / 7.7e-3 (text) at full depth; ours by 3.6e-3 / 7.3e-3.
EMB_REL_L2 = 1.2e-2      # 1.5 x the reference's bf16 deviation of the text tower (the larger one)
ROW_COSINE = 1.0 - 1e-3
LOSS_REL = 1e-2          # a 2..4-pair loss at logit scale ~100 is one sample of the logits error (see _assert_calibrated)
GRAD_COSINE = 0.97


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a B200")
    return torch.device("cuda", 0)


def _rel(a, b):
    return float((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-30))


def _args(cfg):
    from xpretrain_b200.modeling.clip_vip import ClipVipConfig, TowerConfig
    add = SimpleNamespace(type="ViP", temporal_size=cfg.temporal_size, if_use_temporal_embed=1,
                          logit_scale_init_value=cfg.logit_scale_init, add_cls_num=cfg.add_cls_num)
    mc = ClipVipConfig(vision=TowerConfig(768, 12, cfg.vision.layers, 3072), text=TowerConfig(512, 8, cfg.text.layers, 2048))
    return SimpleNamespace(clip_config=mc, clip_weights="", clip_vision_additional_config=add)


def _build(cfg, sd, dev):
    from xpretrain_b200.modeling import VidCLIP
    model = VidCLIP(_args(cfg))
    missing, unexpected = model.clipmodel.load_state_dict(sd, strict=False)
    assert not unexpected and not missing, (missing, unexpected)      # state_dict names == the reference's
    return model.to(dev)


def _run_case(gold, dev, check_grads):
    from oracle import clipvip_oracle as O
    from xpretrain_b200.optimization.loss import build_loss_func
    meta = gold["meta"]
    cfg = O.ClipVipCfg(vision=O.TowerCfg(768, 12, meta["vision_layers"], 3072), text=O.TowerCfg(512, 8, meta["text_layers"], 2048))
    sd = O.init_state_dict(cfg, seed=meta["weight_seed"])
    video, ids, mask = O.synthetic_batch(meta["B"], meta["T"], meta["Lt"], cfg, seed=meta["data_seed"], ragged_text=meta["ragged"])
    assert torch.equal(ids, gold["input_ids"])
    model = _build(cfg, sd, dev)
    out = model(video=video.to(dev), text_input_ids=ids.to(dev), text_input_mask=mask.to(dev))
    loss_fn = build_loss_func({"loss_name": "NCELearnableTempLoss"})
    loss = loss_fn(out["vis_features"], out["text_features"], model.clipmodel.logit_scale)
    vis, txt = out["vis_features"].detach().cpu(), out["text_features"].detach().cpu()
    e_v, e_t = _rel(vis, gold["vis_features"]), _rel(txt, gold["text_features"])
    cos_v = torch.nn.functional.cosine_similarity(vis, gold["vis_features"]).min()
    cos_t = torch.nn.functional.cosine_similarity(txt, gold["text_features"]).min()
    e_l = abs(float(loss) - float(gold["loss"])) / abs(float(gold["loss"]))
    print(f"[{meta['name']}] vs reference golden: vis rel-L2 {e_v:.2e} (min cos {cos_v:.6f})  txt rel-L2 {e_t:.2e} "
          f"(min cos {cos_t:.6f})  loss {float(loss):.5f} vs {float(gold['loss']):.5f} (rel {e_l:.2e})")
    assert e_v < EMB_REL_L2 and e_t < EMB_REL_L2
    assert cos_v > ROW_COSINE and cos_t > ROW_COSINE
    assert e_l < LOSS_REL
    if not check_grads:
        return
    loss.backward()
    torch.cuda.synchronize()
    named = dict(model.clipmodel.named_parameters())
    worst = (1.0, None)
    for k, gn in gold["grad_norms"].items():
        g = named[k].grad
        assert g is not None, k
        if gn < 1e-4:
            continue
        ratio = float(g.norm()) / gn
        assert 0.85 < ratio < 1.15, (k, ratio)
    for k, sample in gold["grad_samples"].items():
        got = named[k].grad.detach().flatten()[:256].cpu()
        if sample.norm() < 1e-6:
            continue
        cos = float(torch.nn.functional.cosine_similarity(got, sample, dim=0))
        if cos < worst[0]:
            worst = (cos, k)
        assert cos > GRAD_COSINE, (k, cos)
    print(f"  gradients: worst sampled cosine {worst[0]:.5f} at {worst[1]}")


def test_depth2_ragged_against_reference_golden(dev, golden_dir):
    gold = torch.load(os.path.join(golden_dir, "depth2_b3_t12_ragged.pt"), weights_only=False)
    _run_case(gold, dev, check_grads=True)


def test_cfg1_full_depth_against_reference_golden(dev, golden_dir):
    """BASELINE.json configs[0]: ViT-B/16, batch 2, 4 frames (temporal interpolation 12 -> 4), 32 tokens."""
    gold = torch.load(os.path.join(golden_dir, "cfg1_b2_t4.pt"), weights_only=False)
    _run_case(gold, dev, check_grads=True)


def _unpack(e):
    return e["data"].float() * e["scale"]


def _errors_vs_full_golden(gold, vis, txt, loss, grads):
    """Relative L2 errors against the fp32 reference golden (features, logits, loss, every kept gradient: the stored sample of
    each weight gradient, every bias / LayerNorm gradient vector whole)."""
    e = {"vis": _rel(vis, gold["vis_features"]), "txt": _rel(txt, gold["text_features"]),
         "logits": _rel(vis @ txt.t(), gold["vis_features"] @ gold["text_features"].t()),
         "loss": abs(loss - float(gold["loss"])) / abs(float(gold["loss"]))}
    for k, ent in gold["grad_full"].items():
        e["d " + k] = _rel(grads[k].flatten()[ent["index"].long()], _unpack(ent))
    vectors = {k: _unpack(ent) for k, ent in gold["grad_vectors"].items()}
    vec = [(k, g) for k, g in vectors.items() if float(g.norm()) > 1e-3 * gold["grad_norms"]["logit_scale"] and "k_proj.bias" not in k]
    e["d vectors (worst)"] = max(_rel(grads[k], g) for k, g in vec)
    e["d vectors (median)"] = sorted(_rel(grads[k], g) for k, g in vec)[len(vec) // 2]
    return e


CALIBRATION = 1.5      # ours may deviate from the fp32 reference by at most 1.5 x what the reference's own bf16 run deviates


def _full12_case(dev, golden_dir, pad_to):
    """T = 12, 12 + 12 layers, ragged text — the BENCH model — against the golden made from the real reference
    (tests/golden/make_golden.py full12): full-tensor relative L2 of the features and the logits matrix, relative L2 over
    at least 4096 elements of each of fifteen weight-gradient tensors (first and last row whole, the rest a fixed, seeded
    sample) and over every bias / LayerNorm gradient vector whole, each CALIBRATED against the deviation the reference
    algorithm itself shows in bf16 on the same inputs on this GPU (autocast and all-bf16), not against a hand-set number.
    With pad_to = 64 the golden batch occupies rows 0..3 of a 64-pair batch (BASELINE.json configs[1]'s per-GPU batch):
    the loss is taken on those rows only, so every gradient must still equal the reference's."""
    from oracle import clipvip_oracle as O
    from xpretrain_b200.optimization.loss import build_loss_func
    gold = torch.load(os.path.join(golden_dir, "full12_b4_t12_ragged.pt"), weights_only=False)
    meta = gold["meta"]
    cfg = O.ClipVipCfg()
    sd = O.init_state_dict(cfg, seed=meta["weight_seed"])
    video, ids, mask = O.synthetic_batch(meta["B"], meta["T"], meta["Lt"], cfg, seed=meta["data_seed"], ragged_text=True)
    assert torch.equal(ids, gold["input_ids"]) and abs(float(video.double().sum()) - gold["video_checksum"]) < 1e-6
    B = meta["B"]
    model = _build(cfg, sd, dev)
    v_in, i_in, m_in = video, ids, mask
    if pad_to > B:
        v2, i2, m2 = O.synthetic_batch(pad_to - B, meta["T"], meta["Lt"], cfg, seed=777, ragged_text=True)
        v_in, i_in, m_in = torch.cat([video, v2]), torch.cat([ids, i2]), torch.cat([mask, m2])
    out = model(video=v_in.to(dev), text_input_ids=i_in.to(dev), text_input_mask=m_in.to(dev))
    vis, txt = out["vis_features"][:B], out["text_features"][:B]
    loss = build_loss_func({"loss_name": "NCELearnableTempLoss"})(vis, txt, model.clipmodel.logit_scale)
    loss.backward()
    torch.cuda.synchronize()
    grads = {n: p.grad.detach().float().cpu() for n, p in model.clipmodel.named_parameters()}
    ours = _errors_vs_full_golden(gold, vis.detach().float().cpu(), txt.detach().float().cpu(), float(loss), grads)
    del model, out, loss
    torch.cuda.empty_cache()
    ref = {}
    for mode in ("autocast", "pure"):
        rv, rt, rl, rg = O.run_reduced_precision(sd, video, ids, mask, cfg, dev, mode)
        ref[mode] = _errors_vs_full_golden(gold, rv, rt, rl, rg)
    print(f"\n[full12, batch {pad_to}] relative L2 vs the fp32 reference golden      ours   | reference bf16-autocast | reference all-bf16")
    for k in ours:
        print(f"  {k:72s} {ours[k]:.2e} | {ref['autocast'][k]:.2e} | {ref['pure'][k]:.2e}")
    return ours, ref


def _assert_calibrated(ours, ref):
    """Features, logits matrix and the stored gradients: our deviation from the fp32 reference golden may be at
    most CALIBRATION = 1.5 x the deviation of the REFERENCE's own bf16 path (autocast: fp32 residual stream, bf16 matmul inputs)
    on the same inputs on this GPU — tighter than SURVEY.md §8c's 2x.  Measured (profiles/r02_pytest_gpu_parity_v2_fp32_residual.log):
    features 0.95x, logits 1.24x, gradients 0.93x - 1.29x.  With `residual_fp32=False` (round-1 bf16 stream) the features sit at
    2.4x and only the all-bf16 bar holds, which is why the fp32 stream is the default."""
    import os
    against = "pure" if os.environ.get("XP_RESIDUAL_BF16") == "1" else "autocast"
    for k in ours:
        if k == "loss":
            continue
        assert ours[k] <= CALIBRATION * ref[against][k] + 1e-6, (k, ours[k], ref[against][k])
    # the scalar loss is ONE sample of the logits error (the reference's own two bf16 runs differ 18x on it): bounded by the
    # larger of the reference deviations, with a floor of 2e-3
    assert ours["loss"] <= max(CALIBRATION * max(ref["pure"]["loss"], ref["autocast"]["loss"]), 2e-3), (ours["loss"], ref)


def test_full_depth_t12_full_gradients_calibrated_against_reference_bf16(dev, golden_dir):
    ours, ref = _full12_case(dev, golden_dir, pad_to=4)
    _assert_calibrated(ours, ref)


def test_bench_batch64_rows_against_reference_golden(dev, golden_dir):
    """BASELINE.json configs[1] (batch 64 x 12 frames, 12 layers): the golden pairs ride in rows 0..3 of the 64-pair batch."""
    ours, ref = _full12_case(dev, golden_dir, pad_to=64)
    _assert_calibrated(ours, ref)


def test_hidden_states_against_oracle(dev):
    """Layer-by-layer hidden states of a 2-layer model vs the oracle run on the host (seeded, not from goldens)."""
    from oracle import clipvip_oracle as O
    from xpretrain_b200.modeling import clip_vip as M
    cfg = O.ClipVipCfg(vision=O.TowerCfg(768, 12, 2, 3072), text=O.TowerCfg(512, 8, 2, 2048))
    sd = O.init_state_dict(cfg, seed=11)
    video, ids, mask = O.synthetic_batch(2, 3, 16, cfg, seed=5, ragged_text=True)
    _, vh = O.vision_tower(sd, video, cfg, return_hidden=True)
    model = _build(cfg, sd, dev)
    M._refresh_weights(model.clipmodel)
    proj, sv = M._vision_fwd(model.clipmodel, video.to(dev), save=True)
    S = sv.S
    for i, want in enumerate(vh[:-1]):
        got = sv.layers[i][0].view(2, S, 768).cpu()          # saved input of layer i == hidden state i
        assert _rel(got, want) < 8e-3, i
    xl, pend = sv.x_last                                          # fp32 residual stream + the last block's bf16 branch output
    last = xl.float() + (pend.float() if pend is not None else 0)
    assert _rel(last.view(2, S, 768).cpu(), vh[-1]) < 1e-2


def test_full_size_properties(dev):
    """BASELINE.json configs[1] shapes (12 frames, 12 layers) at a batch the test can afford: size-independent
    properties — unit-norm rows, row i of text pairs with row i of video (permutation equivariance), determinism,
    and the loss of identical towers' outputs under a row permutation."""
    from oracle import clipvip_oracle as O
    from xpretrain_b200.optimization.loss import NCELearnableTempLoss
    cfg = O.ClipVipCfg()
    sd = O.init_state_dict(cfg, seed=0)
    model = _build(cfg, sd, dev)
    B = 8
    video, ids, mask = O.synthetic_batch(B, 12, 32, cfg, seed=77)
    video, ids, mask = video.to(dev), ids.to(dev), mask.to(dev)
    with torch.no_grad():
        o1 = model(video=video, text_input_ids=ids, text_input_mask=mask)
        o2 = model(video=video, text_input_ids=ids, text_input_mask=mask)
        perm = torch.randperm(B, device=dev)
        o3 = model(video=video[perm], text_input_ids=ids[perm], text_input_mask=mask[perm])
    for k in ("vis_features", "text_features"):
        assert torch.equal(o1[k], o2[k])                                           # deterministic
        assert float((o1[k].norm(dim=-1) - 1).abs().max()) < 1e-5                 # L2-normalised rows
        assert float((o1[k][perm] - o3[k]).abs().max()) < 1e-6                    # samples are independent
    temp = model.clipmodel.logit_scale.detach()
    l1 = NCELearnableTempLoss()(o1["vis_features"], o1["text_features"], temp)
    l3 = NCELearnableTempLoss()(o3["vis_features"], o3["text_features"], temp)
    assert abs(float(l1) - float(l3)) < 1e-4 * abs(float(l1))


def test_state_dict_round_trip(dev):
    """Checkpoint compatibility (SURVEY.md §8b): keys / shapes / dtypes equal the reference CLIPModel's."""
    from oracle import clipvip_oracle as O
    cfg = O.ClipVipCfg()
    sd = O.init_state_dict(cfg, seed=0)
    model = _build(cfg, sd, dev)
    own = model.state_dict()
    assert set(own) == {"clipmodel." + k for k in sd}
    for k, v in sd.items():
        assert own["clipmodel." + k].shape == v.shape and own["clipmodel." + k].dtype == v.dtype, k


def test_image_caption_branch_and_vsc_fc_loss_against_oracle(dev):
    """The released pre-training path (VidCLIP.py:70-79 + loss.py:288-324): video/subtitle pass plus a T = 1 frame/caption
    pass through the same towers (temporal table interpolated 12 -> 1), six-term loss, backward through both passes."""
    from oracle import clipvip_oracle as O
    from xpretrain_b200.optimization.loss import build_loss_func
    cfg = O.ClipVipCfg(vision=O.TowerCfg(768, 12, 1, 3072), text=O.TowerCfg(512, 8, 1, 2048))
    sd = O.init_state_dict(cfg, seed=5)
    B, T, Lt = 4, 2, 16
    video, ids, mask = O.synthetic_batch(B, T, Lt, cfg, seed=21)
    image, cap_ids, cap_mask = O.synthetic_batch(B, 1, Lt, cfg, seed=22, ragged_text=True)
    model = _build(cfg, sd, dev)
    out = model(video=video.to(dev), text_input_ids=ids.to(dev), text_input_mask=mask.to(dev), image=image.to(dev),
                caption_ids=cap_ids.to(dev), caption_masks=cap_mask.to(dev))
    assert set(out) == {"text_features", "vis_features", "img_features", "cap_features"}
    loss_fn = build_loss_func({"loss_name": "NCELearnableTempLoss_vsc_fc"})
    loss = loss_fn(out["vis_features"], out["text_features"], out["img_features"], out["cap_features"],
                   model.clipmodel.logit_scale)
    loss.backward()
    # oracle (fp32, host): the same two passes share the weights, gradients accumulate over both
    sdo = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    o1 = O.clip_vip_forward(sdo, video, ids, mask, cfg)
    o2 = O.clip_vip_forward(sdo, image.reshape(-1, 1, *image.shape[2:]), cap_ids, cap_mask, cfg)
    want = O.nce_vsc_fc_loss(o1["vis_features"], o1["text_features"], o2["vis_features"], o2["text_features"],
                             sdo["logit_scale"])
    want.backward()
    for k, ref in (("vis_features", o1["vis_features"]), ("text_features", o1["text_features"]),
                   ("img_features", o2["vis_features"]), ("cap_features", o2["text_features"])):
        assert _rel(out[k].detach().cpu(), ref.detach()) < EMB_REL_L2, k
    assert abs(float(loss) - float(want)) < LOSS_REL * abs(float(want))
    named = dict(model.clipmodel.named_parameters())
    for k in ("vision_model.embeddings.temporal_embedding", "vision_model.encoder.layers.0.mlp.fc1.weight",
              "text_model.encoder.layers.0.self_attn.q_proj.weight", "visual_projection.weight", "text_projection.weight",
              "vision_model.embeddings.patch_embedding.weight"):
        got, ref = named[k].grad.detach().flatten().cpu(), sdo[k].grad.flatten()
        cos = float(torch.nn.functional.cosine_similarity(got, ref, dim=0))
        assert cos > GRAD_COSINE, (k, cos)
    assert abs(float(model.clipmodel.logit_scale.grad) - float(sdo["logit_scale"].grad)) < 0.05 * abs(float(sdo["logit_scale"].grad)) + 1e-3
