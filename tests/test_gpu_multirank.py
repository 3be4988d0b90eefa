"""B200 x 2 (NCCL): the N > 1 PRODUCT path — `gather_nce_loss` (the fused embedding exchange + InfoNCE kernels) and
`OverlappedGradAverager` — against (1) the single-process run of the same kernels on the concatenated 2B batch and
(2) the oracle's closed form (oracle.nce_closed_form_grads, pinned to the reference loss's autograd).

Replaces: hvd.allgather x2 + NCELearnableTempLoss + hvd.DistributedOptimizer averaging
(CLIP-ViP/src/pretrain/run_pretrain.py:226-228,344-356,379; semantics of the gather pinned by LF-VILA/src/utils/dist.py:21-41).
The per-rank batch is 3 (not a multiple of 8) on purpose: rank 1's rows start at an offset that is not 16-byte aligned.
"""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def _build(dev, layers=1):
    from types import SimpleNamespace
    from oracle import clipvip_oracle as O
    from xpretrain_b200.modeling import VidCLIP
    from xpretrain_b200.modeling.clip_vip import ClipVipConfig, TowerConfig
    cfg = O.ClipVipCfg(vision=O.TowerCfg(768, 12, layers, 3072), text=O.TowerCfg(512, 8, layers, 2048))
    sd = O.init_state_dict(cfg, seed=2)
    add = SimpleNamespace(type="ViP", temporal_size=12, if_use_temporal_embed=1, logit_scale_init_value=4.6, add_cls_num=3)
    mc = ClipVipConfig(vision=TowerConfig(768, 12, layers, 3072), text=TowerConfig(512, 8, layers, 2048))
    model = VidCLIP(SimpleNamespace(clip_config=mc, clip_weights="", clip_vision_additional_config=add))
    model.clipmodel.load_state_dict(sd, strict=False)
    return O, cfg, model.to(dev)


def _worker(rank, world, port, b, q):
    try:
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                          LOCAL_RANK=str(rank))
        import torch.distributed as dist
        from xpretrain_b200.optimization.loss import NCELearnableTempLoss, gather_nce_loss
        from xpretrain_b200.utils import distributed as xd
        r, local, w = xd.init_from_env("nccl")
        dev = torch.device("cuda", local)
        O, cfg, model = _build(dev)
        data = [O.synthetic_batch(b, 2, 16, cfg, seed=50 + k, ragged_text=True) for k in range(world)]
        video, ids, mask = (t.to(dev) for t in data[rank])

        # ---- the data-parallel step: local forward, fused gather + loss, backward with overlapped gradient averaging
        model.clipmodel.grad_ready_hook = xd.OverlappedGradAverager()
        out = model(video=video, text_input_ids=ids, text_input_mask=mask)
        loss = gather_nce_loss(out["vis_features"], out["text_features"], model.clipmodel.logit_scale)
        loss.backward()
        torch.cuda.synchronize()
        dp_grads = {n: p.grad.detach().clone() for n, p in model.clipmodel.named_parameters()}
        # ---- the head alone on leaf features: local rows of dV / dT
        v = out["vis_features"].detach().clone().requires_grad_(True)
        t = out["text_features"].detach().clone().requires_grad_(True)
        p = model.clipmodel.logit_scale.detach().clone().requires_grad_(True)
        loss_h = gather_nce_loss(v, t, p)
        loss_h.backward()
        feats = [torch.empty(world, b, 512, device=dev) for _ in range(2)]
        dist.all_gather_into_tensor(feats[0], out["vis_features"].detach().contiguous())
        dist.all_gather_into_tensor(feats[1], out["text_features"].detach().contiguous())
        V, T = feats[0].reshape(world * b, 512).cpu(), feats[1].reshape(world * b, 512).cpu()
        dv, dt, dl = O.nce_closed_form_grads(V, T, p.detach().cpu())
        want_loss = float(O.nce_learnable_temp_loss(V, T, p.detach().cpu()))
        res = {
            "rank": rank,
            "loss": float(loss), "loss_head": float(loss_h), "oracle_loss": want_loss,
            # SyncFunction semantics: SUM over ranks of identical losses, then the local slice = W x the local rows
            "e_dv": _rel(v.grad.cpu(), world * dv[rank * b:(rank + 1) * b]),
            "e_dt": _rel(t.grad.cpu(), world * dt[rank * b:(rank + 1) * b]),
            "e_dl": abs(float(p.grad) - float(dl)) / abs(float(dl)),
        }
        if rank == 0:
            # ---- single process, the same kernels, global batch 2b: the averaged DP gradients must equal these
            _, _, ref = _build(dev)
            gv, gi, gm = (torch.cat([d[k] for d in data]).to(dev) for k in range(3))
            o2 = ref(video=gv, text_input_ids=gi, text_input_mask=gm)
            l2 = NCELearnableTempLoss()(o2["vis_features"], o2["text_features"], ref.clipmodel.logit_scale)
            l2.backward()
            torch.cuda.synchronize()
            res["single_loss"] = float(l2)
            errs = {}
            for n, p2 in ref.clipmodel.named_parameters():
                if float(p2.grad.norm()) < 1e-6:
                    continue
                errs[n] = _rel(dp_grads[n], p2.grad)
            res["worst_param"] = max(errs, key=errs.get)
            res["worst_param_err"] = errs[res["worst_param"]]
            res["median_param_err"] = sorted(errs.values())[len(errs) // 2]
        q.put(res)
        dist.barrier()
        dist.destroy_process_group()
    except Exception as e:  # noqa: BLE001
        import traceback
        q.put({"rank": rank, "error": traceback.format_exc()})
        raise


@pytest.mark.timeout(600)
@pytest.mark.parametrize("b", [3, 8])
def test_gather_nce_and_overlapped_averaging_match_single_process(b):
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs 2 B200s")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, b, q)) for r in range(2)]
    for p in procs:
        p.start()
    results = [q.get(timeout=500) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    for res in results:
        assert "error" not in res, res.get("error")
    results.sort(key=lambda r: r["rank"])
    r0, r1 = results
    print(f"[2 ranks, b={b}] loss {r0['loss']:.6f} / {r1['loss']:.6f}  single-process {r0['single_loss']:.6f}  oracle "
          f"{r0['oracle_loss']:.6f};  local dV {r0['e_dv']:.1e}/{r1['e_dv']:.1e} dT {r0['e_dt']:.1e}/{r1['e_dt']:.1e} "
          f"dscale {r0['e_dl']:.1e};  averaged parameter gradients vs single process: median {r0['median_param_err']:.1e} "
          f"worst {r0['worst_param_err']:.1e} ({r0['worst_param']})")
    assert r0["loss"] == r1["loss"]                                            # every rank computes the same scalar
    for r in results:
        assert abs(r["loss"] - r["oracle_loss"]) < 1e-4 * abs(r["oracle_loss"])  # fp32-grade logits (hi/lo split)
        assert abs(r["loss_head"] - r["loss"]) < 1e-6 * abs(r["loss"])
        assert r["e_dv"] < 1e-2 and r["e_dt"] < 1e-2 and r["e_dl"] < 1e-3       # bf16 G operand
    # features at batch b vs 2b come from different GEMM tilings: near-equal, not bit-equal
    assert abs(r0["loss"] - r0["single_loss"]) < 1e-3 * abs(r0["single_loss"])
    assert r0["median_param_err"] < 1e-2 and r0["worst_param_err"] < 5e-2
