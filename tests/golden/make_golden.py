"""Generate the golden vectors under tests/golden/ from the REAL reference.

Runs only in the authoring container, where /root/reference (microsoft/XPretrain) is mounted:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

It imports the reference's own modules (CLIP-ViP/src/modeling/CLIP_ViP.py, src/optimization/loss.py)
unmodified, loads the oracle's deterministic synthetic weights into them, runs forward / loss /
backward in fp32 on CPU, (1) asserts that oracle/clipvip_oracle.py reproduces the reference to fp32
round-off — this is what pins the oracle — and (2) writes small .pt fixtures that
tests/test_oracle_golden.py (CPU) and tests/test_gpu_parity.py (B200) replay without the reference.
No reference source is copied; only numeric outputs are stored.
"""
import os
import sys
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = os.environ.get("XP_REFERENCE_ROOT", "/root/reference")
sys.path.insert(0, os.path.join(REF, "CLIP-ViP"))
sys.dont_write_bytecode = True

from oracle import clipvip_oracle as O  # noqa: E402


def build_reference(cfg: O.ClipVipCfg):
    from transformers.models.clip.configuration_clip import CLIPConfig
    import src.modeling.CLIP_ViP as ref

    tc = dict(vocab_size=cfg.vocab, hidden_size=cfg.text.width, intermediate_size=cfg.text.mlp,
              num_hidden_layers=cfg.text.layers, num_attention_heads=cfg.text.heads,
              max_position_embeddings=cfg.max_text_pos, hidden_act="quick_gelu")
    vc = dict(hidden_size=cfg.vision.width, intermediate_size=cfg.vision.mlp, num_hidden_layers=cfg.vision.layers,
              num_attention_heads=cfg.vision.heads, image_size=cfg.image_size, patch_size=cfg.patch,
              hidden_act="quick_gelu")
    hf = CLIPConfig(text_config=tc, vision_config=vc, projection_dim=cfg.proj_dim)
    hf.vision_additional_config = types.SimpleNamespace(type="ViP", temporal_size=cfg.temporal_size,
                                                        if_use_temporal_embed=1,
                                                        logit_scale_init_value=cfg.logit_scale_init,
                                                        add_cls_num=cfg.add_cls_num)
    return ref.CLIPModel(hf)


def rel(a, b):
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


# weight gradients kept by the full-depth case: GRAD_SAMPLES elements of each tensor, its first and last row plus a fixed,
# seeded random sample (flat indices + values, fp16 after a per-tensor max-normalisation); every bias / LayerNorm vector of
# the model is kept whole, packed the same way.  This keeps the fixture under 1 MB.
FULL_GRAD_KEYS = (
    "vision_model.encoder.layers.11.mlp.fc1.weight", "vision_model.encoder.layers.0.self_attn.q_proj.weight",
    "vision_model.encoder.layers.0.self_attn.k_proj.weight", "vision_model.encoder.layers.0.self_attn.out_proj.weight",
    "vision_model.encoder.layers.11.self_attn.out_proj.weight", "vision_model.encoder.layers.11.self_attn.v_proj.weight",
    "vision_model.embeddings.patch_embedding.weight", "vision_model.embeddings.position_embedding.weight",
    "text_model.encoder.layers.0.mlp.fc1.weight", "text_model.encoder.layers.11.self_attn.q_proj.weight",
    "visual_projection.weight", "text_projection.weight",
    "vision_model.encoder.layers.0.mlp.fc1.weight", "vision_model.encoder.layers.0.mlp.fc2.weight",
)
GRAD_SAMPLES = 4096


def _pack_f16(g):
    s = float(g.abs().max().clamp_min(1e-30))
    return {"scale": s, "data": (g / s).to(torch.float16)}


def _sample_f16(g, candidates, gen):
    """Flat indices of g drawn from `candidates` ([rows, width] of flat indices): its first and last row whole, so that a fault
    confined to an edge tile shows, plus a seeded random pick of the other rows' elements that brings the total to GRAD_SAMPLES
    (at least GRAD_SAMPLES // 4 of them).  Sorted, with g's values there packed by _pack_f16."""
    edge = torch.cat([candidates[0], candidates[-1]])
    inner = candidates[1:-1].flatten()
    n = max(GRAD_SAMPLES - edge.numel(), GRAD_SAMPLES // 4)
    pick = torch.cat([edge, inner[torch.randperm(inner.numel(), generator=gen)[:n]]]).sort().values
    return {"index": pick.to(torch.int32), **_pack_f16(g.flatten()[pick])}


def run_case(name, cfg, B, T, Lt, ragged, weight_seed, data_seed, with_hidden, full_grads=False):
    from src.optimization.loss import NCELearnableTempLoss

    sd = O.init_state_dict(cfg, seed=weight_seed)
    model = build_reference(cfg)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all("position_ids" in m for m in missing), missing
    video, ids, mask = O.synthetic_batch(B, T, Lt, cfg, seed=data_seed, ragged_text=ragged)

    out = model(input_ids=ids, attention_mask=mask, pixel_values=video, return_loss=False,
                output_hidden_states=with_hidden, return_dict=True)
    vis, txt = out["image_embeds"], out["text_embeds"]
    loss = NCELearnableTempLoss(None)(vis, txt, model.logit_scale)
    loss.backward()
    grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}

    # --- pin the oracle against the reference (fp32 round-off only) ---
    sdg = {k: (v.clone().requires_grad_(True) if v.is_floating_point() else v) for k, v in sd.items()}
    o = O.clip_vip_forward(sdg, video, ids, mask, cfg)
    oloss = O.nce_learnable_temp_loss(o["vis_features"], o["text_features"], sdg["logit_scale"])
    oloss.backward()
    e_vis, e_txt = rel(o["vis_features"].detach(), vis.detach()), rel(o["text_features"].detach(), txt.detach())
    e_loss = abs(float(oloss) - float(loss)) / abs(float(loss))
    # k_proj.bias has an analytically zero gradient (softmax is shift-invariant per query), so its
    # value is pure round-off in both implementations: compare against the tensor's natural scale.
    scale = {k: max(float(g.norm()), 1e-4 * float(sd[k].numel()) ** 0.5 * float(loss)) for k, g in grads.items()}
    errs = {k: float((sdg[k].grad - g).norm()) / scale[k] for k, g in grads.items()}
    worst_key = max(errs, key=errs.get)
    worst = errs[worst_key]
    print(f"  worst gradient key: {worst_key} ({worst:.2e}; |g|={float(grads[worst_key].norm()):.3e})")
    print(f"[{name}] oracle vs reference: vis {e_vis:.2e} txt {e_txt:.2e} loss {e_loss:.2e} worst-grad {worst:.2e}")
    assert e_vis < 2e-5 and e_txt < 2e-5 and e_loss < 1e-5 and worst < 5e-4, "oracle does not match the reference"

    gold = {
        "meta": dict(name=name, B=B, T=T, Lt=Lt, ragged=ragged, weight_seed=weight_seed, data_seed=data_seed,
                     vision_layers=cfg.vision.layers, text_layers=cfg.text.layers, torch=torch.__version__),
        "input_ids": ids, "attention_mask": mask, "video_checksum": float(video.double().sum()),
        "vis_features": vis.detach(), "text_features": txt.detach(), "loss": loss.detach(),
        "grad_norms": {k: float(g.norm()) for k, g in grads.items()},
        "grad_samples": {k: grads[k].flatten()[:256].clone() for k in grads
                         if any(s in k for s in ("logit_scale", "class_embedding", "added_cls", "temporal_embedding",
                                                 "final_layer_norm", "post_layernorm", "pre_layrnorm",
                                                 "layers.0.self_attn.q_proj.bias", "layers.0.mlp.fc1.bias",
                                                 "visual_projection", "text_projection",
                                                 "vision_model.embeddings.position_embedding"))},
    }
    if full_grads:
        gen = torch.Generator().manual_seed(2024)
        full = {k: _sample_f16(grads[k], torch.arange(grads[k].numel()).view(grads[k].shape[0], -1), gen)
                for k in FULL_GRAD_KEYS}
        tk = "text_model.embeddings.token_embedding.weight"
        rows = torch.unique(ids)
        width = grads[tk].shape[1]
        full[tk] = _sample_f16(grads[tk], rows[:, None] * width + torch.arange(width), gen)   # touched rows only
        rest = grads[tk].clone()
        rest[rows] = 0
        assert float(rest.abs().max()) == 0.0                                        # untouched rows: exactly zero
        gold["grad_full"] = full
        gold["grad_vectors"] = {k: _pack_f16(g) for k, g in grads.items() if g.dim() <= 1 or g.numel() <= 4096}
    if with_hidden:
        vh = out["vision_model_output"].hidden_states
        th = out["text_model_output"].hidden_states
        # rows 0..7 (cls, proxies, first patches) and the last 4 rows of every layer's hidden state
        gold["vision_hidden_rows"] = torch.stack([torch.cat([h[:, :8], h[:, -4:]], 1).detach() for h in vh])
        gold["text_hidden"] = torch.stack([h.detach() for h in th])
    path = os.path.join(HERE, f"{name}.pt")
    torch.save(gold, path)
    print(f"  wrote {path} ({os.path.getsize(path) / 1024:.1f} KiB)")


def loss_case():
    from src.optimization.loss import NCELearnableTempLoss

    g = torch.Generator().manual_seed(7)
    W, b, d = 4, 8, 512
    vis = [torch.nn.functional.normalize(torch.randn(b, d, generator=g), dim=-1) for _ in range(W)]
    txt = [torch.nn.functional.normalize(torch.randn(b, d, generator=g), dim=-1) for _ in range(W)]
    V = O.gather_rank_major(vis).requires_grad_(True)
    T = O.gather_rank_major(txt).requires_grad_(True)
    temp = torch.tensor(4.6, requires_grad=True)
    loss = NCELearnableTempLoss(None)(V, T, temp)
    loss.backward()
    dv, dt, dl = O.nce_closed_form_grads(V.detach(), T.detach(), temp.detach())
    assert rel(dv, V.grad) < 1e-5 and rel(dt, T.grad) < 1e-5 and abs(float(dl) - float(temp.grad)) < 1e-5
    assert abs(float(O.nce_learnable_temp_loss(V.detach(), T.detach(), temp.detach())) - float(loss)) < 1e-6
    torch.save({"world": W, "vis_per_rank": vis, "txt_per_rank": txt, "logit_scale": temp.detach(),
                "loss": loss.detach(), "d_vis": V.grad, "d_txt": T.grad, "d_logit_scale": temp.grad},
               os.path.join(HERE, "nce_loss_w4.pt"))
    print("[nce_loss_w4] closed-form gradients match autograd of the reference loss")


def vsc_fc_loss_case():
    """The released pre-training default loss (pretrain_vip_base_16.json:74-77): NCELearnableTempLoss_vsc_fc, loss.py:288-324."""
    from src.optimization.loss import NCELearnableTempLoss_vsc_fc

    g = torch.Generator().manual_seed(11)
    N, d = 24, 512
    feats = [torch.nn.functional.normalize(torch.randn(N, d, generator=g), dim=-1).requires_grad_(True) for _ in range(4)]
    temp = torch.tensor(4.6, requires_grad=True)
    loss = NCELearnableTempLoss_vsc_fc(None)(*feats, temp)
    loss.backward()
    ref_grads = [f.grad.clone() for f in feats] + [temp.grad.clone()]
    f2 = [f.detach().clone().requires_grad_(True) for f in feats]
    t2 = temp.detach().clone().requires_grad_(True)
    lo = O.nce_vsc_fc_loss(*f2, t2)
    lo.backward()
    assert abs(float(lo) - float(loss)) < 1e-5 * abs(float(loss))
    for a, b in zip([f.grad for f in f2] + [t2.grad], ref_grads):
        assert rel(a, b) < 1e-5
    torch.save({"vis": feats[0].detach(), "txt": feats[1].detach(), "img": feats[2].detach(), "cap": feats[3].detach(),
                "logit_scale": temp.detach(), "loss": loss.detach(), "d_vis": ref_grads[0], "d_txt": ref_grads[1],
                "d_img": ref_grads[2], "d_cap": ref_grads[3], "d_logit_scale": ref_grads[4]},
               os.path.join(HERE, "nce_vsc_fc_n24.pt"))
    print("[nce_vsc_fc_n24] oracle restatement matches the reference loss and its autograd gradients")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "losses":      # regenerate only the (cheap) loss fixtures
        loss_case()
        vsc_fc_loss_case()
        sys.exit(0)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    full = O.ClipVipCfg()
    if len(sys.argv) > 1 and sys.argv[1] == "full12":      # the BENCH shape: T = 12, 12 + 12 layers, ragged text, full gradients
        run_case("full12_b4_t12_ragged", full, B=4, T=12, Lt=32, ragged=True, weight_seed=3, data_seed=4321,
                 with_hidden=False, full_grads=True)
        sys.exit(0)
    # BASELINE.json configs[0]: ViT-B/16, 1 video x 4 frames, 32 tokens, batch 2, fp32 CPU (temporal interp 12 -> 4)
    run_case("cfg1_b2_t4", full, B=2, T=4, Lt=32, ragged=False, weight_seed=0, data_seed=1234, with_hidden=False)
    # reduced depth, native T=12, ragged text (EOS not last, padding mask active), hidden states kept
    small = O.ClipVipCfg(vision=O.TowerCfg(768, 12, 2, 3072), text=O.TowerCfg(512, 8, 2, 2048))
    run_case("depth2_b3_t12_ragged", small, B=3, T=12, Lt=32, ragged=True, weight_seed=1, data_seed=99,
             with_hidden=True)
    loss_case()
