"""End-to-end parity of the CUDA encoder path against (a) golden fixtures produced by the
unmodified reference and (b) the CPU oracle on seeded inputs, forward and backward.

Tolerances (SURVEY.md §8c; bf16 GEMM operands + fp32 residual stream vs the fp32 oracle, eval
mode, valid positions only):
  outputs   max-abs <= 6e-2, mean-abs <= 8e-3, per-token cosine >= 0.999
  gradients per-parameter relative Frobenius error <= 3e-2; attention.self.key.bias, whose exact
            gradient is identically zero (softmax is invariant to a per-query constant), is
            checked in absolute terms.
(tests/test_bench_path_gpu.py additionally holds the outputs to 1.5x the error of the oracle under
torch bf16 autocast, at the benchmark configuration.)
"""
import json

import numpy as np
import pytest
import torch

from hero_b200 import synth
from oracle import hero_oracle as orc
from tests import golden_util as gu

pytestmark = pytest.mark.gpu

OUT_ATOL, OUT_RTOL, OUT_MEAN, OUT_COS, GRAD_REL, GRAD_REL_FT = 6e-2, 0.0, 8e-3, 0.999, 3e-2, 3e-2


def _json(tmp_path, d):
    def cfg(n, v):
        c = {"attention_probs_dropout_prob": 0.1, "hidden_act": "gelu", "hidden_dropout_prob": 0.1,
             "hidden_size": d["hidden"], "initializer_range": 0.02,
             "intermediate_size": d["inter"], "max_position_embeddings": 514,
             "num_attention_heads": d["heads"], "num_hidden_layers": n, "type_vocab_size": 2}
        if v:
            c["vocab_size"] = d["vocab"]
        return c
    p = tmp_path / "m.json"
    p.write_text(json.dumps({"f_config": cfg(d["f_layers"], True),
                             "c_config": cfg(d["c_layers"], False)}))
    return str(p)


def _build(tmp_path, d, weights):
    from hero_b200.model import HierarchicalVlModel, VideoModelConfig
    m = HierarchicalVlModel(VideoModelConfig(_json(tmp_path, d)), vfeat_dim=d["vfeat_dim"],
                            max_frm_seq_len=d["max_img_len"])
    missing, unexpected = m.load_state_dict(weights, strict=False)
    assert not unexpected
    return m.cuda().eval()


def _check_out(got, ref, mask, what):
    got = got.detach().float().cpu().numpy()[mask]
    ref = np.asarray(ref)[mask]
    err = np.abs(got - ref)
    cos = (got * ref).sum(-1) / (np.linalg.norm(got, axis=-1) * np.linalg.norm(ref, axis=-1))
    viol = err - (OUT_ATOL + OUT_RTOL * np.abs(ref))
    assert viol.max() <= 0, (f"{what}: {(viol > 0).sum()} elements out of tolerance, "
                             f"max abs err {err.max():.4f}")
    assert err.mean() <= OUT_MEAN, f"{what}: mean abs err {err.mean():.5f}"
    assert cos.min() >= OUT_COS, f"{what}: min cosine {cos.min():.5f}"


def test_config1_cross_modal_layer_matches_reference_golden(tmp_path):
    fx = gu.load("xm1_config1.npz")
    d = gu.dims_of(fx)
    model = _build(tmp_path, d, gu.weights_for(fx))
    xb = synth.to_device(synth.syn_xm_1(seed=int(fx["seed_batch"])), "cuda")
    with torch.no_grad():
        seq, pooled = model.f_encoder(xb, "repr")
    _check_out(seq, fx["seq_out"], np.ones(seq.shape[:2], bool), "config-1 sequence output")
    assert np.abs(pooled.float().cpu().numpy() - fx["pooled"]).max() < 3e-2


def test_full_depth_encoder_matches_reference_golden(tmp_path):
    fx = gu.load("hier_full_small.npz")
    d = gu.dims_of(fx)
    model = _build(tmp_path, d, gu.weights_for(fx))
    vb, qb = gu.full_small_batches(fx)
    with torch.no_grad():
        clip = model(synth.to_device(vb, "cuda"), "repr")
        q = model.f_encoder(synth.to_device(qb, "cuda"), "txt")[0]
    _check_out(clip, fx["clip_out"], vb["c_attn_masks"].bool().numpy(), "clip outputs")
    _check_out(q, fx["q_seq_out"], qb["attn_masks"].bool().numpy(), "query rows")
    # padded positions are zeros in this implementation
    assert float(clip[~vb["c_attn_masks"].bool().cuda()].abs().max()) == 0.0


def _oracle_loss_and_grads(P, vb, qb, d, w1, w2):
    P = {k: v.clone().requires_grad_(True) for k, v in P.items()}
    clip = orc.hierarchical_repr(P, vb, d["f_layers"], d["c_layers"], d["heads"])
    q = orc.cross_modal_txt(P, "f_encoder.", qb, d["f_layers"], d["heads"])
    loss = (clip * w1).sum() + (q * w2).sum()
    loss.backward()
    return clip.detach(), q.detach(), {k: v.grad for k, v in P.items()}


@pytest.mark.parametrize("kind", ["ragged", "dense"])
def test_forward_backward_vs_oracle(tmp_path, kind):
    d = dict(hidden=768, inter=3072, heads=12, f_layers=2, c_layers=1, vocab=50272,
             vfeat_dim=4352, max_img_len=100)
    shapes = orc.param_shapes(f_layers=2, c_layers=1)
    P = orc.seeded_weights(shapes, seed=5)
    if kind == "ragged":
        vb, qb = synth.syn_tvr_ragged(batch_size=4, seed=99, t_range=(20, 40), s_range=(4, 8),
                                      l_range=(4, 30), q_range=(6, 20))
    else:
        vb, qb = synth.syn_tvr_dense(batch_size=2, seed=7)
    g = torch.Generator().manual_seed(1)
    w1 = torch.randn(vb["c_v_feats"].shape[0], vb["c_v_feats"].shape[1], 768, generator=g)
    w1 = w1 * vb["c_attn_masks"].unsqueeze(-1)
    w2 = torch.randn(qb["input_ids"].shape[0], qb["input_ids"].shape[1], 768, generator=g)
    w2 = w2 * qb["attn_masks"].unsqueeze(-1)
    clip_ref, q_ref, g_ref = _oracle_loss_and_grads(P, vb, qb, d, w1, w2)

    model = _build(tmp_path, d, P)
    clip = model(synth.to_device(vb, "cuda"), "repr")
    q = model.f_encoder(synth.to_device(qb, "cuda"), "txt")[0]
    _check_out(clip, clip_ref.numpy(), vb["c_attn_masks"].bool().numpy(), "clip outputs")
    _check_out(q, q_ref.numpy(), qb["attn_masks"].bool().numpy(), "query rows")
    loss = (clip * w1.cuda()).sum() + (q * w2.cuda()).sum()
    loss.backward()
    named = dict(model.named_parameters())
    bad = []
    for k, gr in g_ref.items():
        if gr is None or k.endswith("pooler.dense.weight") or k.endswith("pooler.dense.bias") \
                or "mask_embedding" in k:
            continue
        got = named[k].grad
        assert got is not None, f"no gradient for {k}"
        num = (got.float().cpu() - gr).norm().item()
        den = gr.norm().item()
        if k.endswith("attention.self.key.bias"):
            qb_norm = g_ref[k.replace("key.bias", "query.bias")].norm().item()
            assert got.float().norm().item() <= 2e-2 * qb_norm, k   # exact value is 0
            continue
        if den < 1e-6:
            assert num < 1e-3, k
            continue
        limit = GRAD_REL_FT if k.startswith("frame_transform.") else GRAD_REL
        if num / den > limit:
            bad.append((k, round(num / den, 4)))
    assert not bad, f"gradient mismatch (relative Frobenius) for {bad[:12]} ({len(bad)} total)"


def test_generic_bert_encoder_api_padded_in_out(tmp_path):
    """BertEncoder.forward(hidden (N, L, H), mask) keeps the reference signature."""
    from hero_b200.encoder import RobertaModelConfig
    from hero_b200.layers import BertEncoder
    cfg = RobertaModelConfig(10, hidden_size=768, num_hidden_layers=1, num_attention_heads=12,
                             intermediate_size=3072)
    torch.manual_seed(0)
    enc = BertEncoder(cfg)
    for p in enc.parameters():
        torch.nn.init.normal_(p, std=0.02) if p.dim() > 1 else None
    enc = enc.cuda().eval()
    P = {"layer.0." + k: v.detach().cpu() for k, v in enc.layer[0].state_dict().items()}
    g = torch.Generator().manual_seed(2)
    h = torch.randn(3, 9, 768, generator=g)
    mask = torch.tensor([[1] * 9, [1] * 4 + [0] * 5, [0, 1, 1, 0, 1, 0, 0, 0, 0]])
    ref = orc.bert_encoder(h, mask, P, "", 1, 12)
    with torch.no_grad():
        out = enc(h.cuda(), mask.cuda())[0]
    _check_out(out, ref.numpy(), mask.bool().numpy(), "generic encoder")


def test_training_mode_dropout_runs_and_is_stochastic(tmp_path):
    d = dict(hidden=768, inter=3072, heads=12, f_layers=1, c_layers=1, vocab=50272,
             vfeat_dim=4352, max_img_len=100)
    P = orc.seeded_weights(orc.param_shapes(f_layers=1, c_layers=1), seed=5)
    model = _build(tmp_path, d, P)
    vb, _ = synth.syn_tvr_ragged(batch_size=2, seed=3, t_range=(10, 20), s_range=(2, 4),
                                 l_range=(4, 10))
    vbd = synth.to_device(vb, "cuda")
    with torch.no_grad():
        ev = model(vbd, "repr")
    model.train()
    torch.manual_seed(1)
    a = model(vbd, "repr")
    a.float().pow(2).mean().backward()
    torch.manual_seed(1)
    b = model(vbd, "repr")
    torch.manual_seed(2)
    c = model(vbd, "repr")
    assert torch.isfinite(a).all()
    assert torch.equal(a, b), "same torch seed must give the same dropout masks"
    assert not torch.equal(a, c)
    assert (a - ev).abs().mean() > 1e-3
    g = model.f_encoder.encoder.layer[0].intermediate.dense.weight.grad
    assert g is not None and torch.isfinite(g).all() and g.abs().sum() > 0


def test_hot_path_never_synchronises_with_collate_side_plans(tmp_path):
    """With plans attached on the host (collate / PlanPool) forward + backward must not contain a
    single device synchronisation — a hidden `.item()` / bool(tensor) drains the launch queue
    every step. torch's sync debug mode turns any such call into an error."""
    from hero_b200.params import flat_of
    from hero_b200.plan import attach_plan
    d = dict(hidden=768, inter=3072, heads=12, f_layers=2, c_layers=1, vocab=50272,
             vfeat_dim=4352, max_img_len=100)
    P = orc.seeded_weights(orc.param_shapes(f_layers=2, c_layers=1), seed=8)
    model = _build(tmp_path, d, P).train()
    flat_of(model, torch.device("cuda")).ensure_flat_grads()
    vb, qb = synth.syn_tvr_ragged(batch_size=2, seed=9, t_range=(10, 20), s_range=(2, 4),
                                  l_range=(4, 10))
    vbd = synth.to_device(attach_plan(dict(vb)), "cuda")
    qbd = synth.to_device(attach_plan(dict(qb), kind="txt"), "cuda")
    for b in (vbd, qbd):
        b["_hero_plan"].to("cuda")
    clip, q = model.forward_repr_txt(vbd, qbd)          # warm-up (flat buffers, caches, joint plan)
    (clip.float().mean() + q.float().mean()).backward()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        clip, q = model.forward_repr_txt(vbd, qbd)
        torch.autograd.backward([clip, q], [torch.ones_like(clip), torch.ones_like(q)])
    finally:
        torch.cuda.set_sync_debug_mode("default")
    torch.cuda.synchronize()
    assert torch.isfinite(clip).all()


def test_prefetch_loader_stages_batches_with_plans():
    """hero_b200.loader.PrefetchLoader (data/loader.py:89-144): device batches in order, equal to
    the host batches, plans attached (in-process here) and uploaded; slots are recycled."""
    from hero_b200.loader import PrefetchLoader
    from hero_b200.plan import PLAN_KEY
    host = []
    for seed in range(5):
        vb, qb = synth.syn_tvr_ragged(batch_size=2, seed=20 + seed, t_range=(10, 20),
                                      s_range=(2, 4), l_range=(4, 10))
        host.append(({k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in vb.items()},
                     {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in qb.items()}))
    got = 0
    for (vbd, qbd), (vb, qb) in zip(PrefetchLoader(host, "cuda:0", depth=3), host):
        assert vbd[PLAN_KEY].dev is not None and qbd[PLAN_KEY].dev is not None
        for dev_b, host_b in ((vbd, vb), (qbd, qb)):
            for k, v in host_b.items():
                if torch.is_tensor(v):
                    assert dev_b[k].is_cuda and torch.equal(dev_b[k].cpu(), v), k
        got += 1
    assert got == 5


def test_fused_adamw_follows_reference_rule_with_param_groups():
    """FusedAdamW on the flat buffer == optim/adamw.py:80-104 per parameter, with the no-decay
    grouping of optim/misc.py:22 (names containing 'bias' / 'LayerNorm.*'), clipping folded in."""
    from hero_b200.optim import FusedAdamW
    from hero_b200.params import flat_of

    class Tiny(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.dense = torch.nn.Linear(96, 64)
            self.LayerNorm = torch.nn.LayerNorm(64)
            self.proj = torch.nn.Linear(64, 40)

    torch.manual_seed(0)
    m = Tiny().cuda()
    flat = flat_of(m, torch.device("cuda"))
    opt = FusedAdamW(flat, lr=1e-3, betas=(0.9, 0.98), eps=1e-6, weight_decay=0.01)
    ref_p = {k: p.detach().cpu().clone() for k, p in m.named_parameters()}
    ref_m = {k: torch.zeros_like(v) for k, v in ref_p.items()}
    ref_v = {k: torch.zeros_like(v) for k, v in ref_p.items()}
    g = torch.Generator().manual_seed(1)
    for step in range(1, 4):
        opt.zero_grad()
        grads = {k: torch.randn(v.shape, generator=g) * 0.1 for k, v in ref_p.items()}
        for k, p in m.named_parameters():
            p.grad.copy_(grads[k].cuda())
        total = torch.sqrt(sum((v.double() ** 2).sum() for v in grads.values())).item()
        norm = opt.clip_grad_norm_(1.0)
        assert abs(norm - total) < 1e-3 * total
        scale = min(1.0, 1.0 / (total + 1e-6))
        opt.step()
        for k in ref_p:
            wd = 0.0 if any(nd in k for nd in ("bias", "LayerNorm.bias", "LayerNorm.weight")) \
                else 0.01
            ref_p[k], ref_m[k], ref_v[k] = orc.adamw_step(ref_p[k], grads[k] * scale, ref_m[k],
                                                          ref_v[k], step, 1e-3, 0.9, 0.98, 1e-6, wd)
        for k, p in m.named_parameters():
            err = (p.detach().cpu() - ref_p[k]).abs().max().item()
            assert err < 2e-6, (k, step, err)
    # the bf16 working copy was refreshed by the optimizer kernel itself
    for k, p in m.named_parameters():
        assert torch.equal(flat.bf16(p), p.detach().to(torch.bfloat16)), k


def test_vcmr_head_on_gpu_matches_its_cpu_orchestration(tmp_path, monkeypatch):
    """hero_b200.pretrain.HeroForVcmr (VSM / VCMR head, SURVEY.md 8f rank 1) on the CUDA encoder:
    same outputs as the same module run on CPU with hero_b200.ops routed to the torch
    restatements of the kernel contracts (tests/fake_ops.py) — that CPU path is what
    tests/test_heads_cpu.py pins against the reference. Full hidden size, 1 + 1 + 1 layers."""
    from hero_b200.model import VideoModelConfig
    from hero_b200.pretrain import HeroForVcmr
    from tests import fake_ops
    d = dict(hidden=768, inter=3072, heads=12, f_layers=1, c_layers=1, vocab=50272,
             vfeat_dim=4352, max_img_len=100)
    cfg = json.load(open(_json(tmp_path, d)))
    cfg["q_config"] = dict(cfg["c_config"])
    path = tmp_path / "vcmr.json"
    path.write_text(json.dumps(cfg))
    P = orc.seeded_weights(orc.param_shapes(f_layers=1, c_layers=1), seed=12)

    def build():
        torch.manual_seed(3)               # identical random head parameters in both builds
        m = HeroForVcmr(VideoModelConfig(str(path)), vfeat_dim=4352, max_frm_seq_len=100,
                        lw_neg_ctx=8, lw_neg_q=8, lw_st_ed=0.01)
        m.load_state_dict({"v_encoder." + k: v for k, v in P.items()}, strict=False)
        return m.eval()

    vb, qb = synth.syn_tvr_ragged(batch_size=3, seed=14, t_range=(10, 16), s_range=(2, 4),
                                  l_range=(4, 10), q_range=(4, 8))
    targets = torch.tensor([[1, 3], [0, 5], [2, 2]])

    def batch(dev):
        b = synth.to_device(dict(vb), dev) if dev != "cpu" else dict(vb)
        for k, v in (("query_input_ids", qb["input_ids"]), ("query_pos_ids", qb["pos_ids"]),
                     ("query_attn_masks", qb["attn_masks"]), ("targets", targets)):
            b[k] = v.to(dev)
        return b

    gpu = build().cuda()
    with torch.no_grad():
        s_g, st_g, ed_g = gpu(batch("cuda"), "tvr", compute_loss=False)
        losses_g = gpu(batch("cuda"), "tvr", compute_loss=True)
    head_sd = {k: v.cpu() for k, v in gpu.state_dict().items()}
    fake_ops.install(monkeypatch)
    cpu = build()
    cpu.load_state_dict(head_sd)
    with torch.no_grad():
        s_c, st_c, ed_c = cpu(batch("cpu"), "tvr", compute_loss=False)
        losses_c = cpu(batch("cpu"), "tvr", compute_loss=True)
    assert s_g.shape == (3, 3) and st_g.shape == st_c.shape
    assert float((s_g.cpu() - s_c).abs().max()) < 2e-2
    valid = vb["c_attn_masks"].bool()
    for a, b in ((st_g, st_c), (ed_g, ed_c)):
        diff = (a.float().cpu() - b.float())[valid].abs().max()
        assert float(diff) <= 3e-2 * float(b.float()[valid].abs().max()) + 3e-2
    for a, b in zip(losses_g, losses_c):
        assert float((a.float().cpu() - b.float()).abs().max()) < 0.2


def test_batch_without_f_v_feats_on_gpu(tmp_path):
    """A batch that omits `f_v_feats` (the subtitle-level copies of the clip frames) gives the
    same forward as the legacy batch: the frame slots are read from `c_v_feats` through the plan."""
    d = dict(hidden=768, inter=3072, heads=12, f_layers=1, c_layers=1, vocab=50272,
             vfeat_dim=4352, max_img_len=100)
    P = orc.seeded_weights(orc.param_shapes(f_layers=1, c_layers=1), seed=15)
    model = _build(tmp_path, d, P)
    vb, qb = synth.syn_tvr_ragged(batch_size=3, seed=16, t_range=(10, 18), s_range=(2, 4),
                                  l_range=(4, 10))
    full = synth.to_device(dict(vb), "cuda")
    slim = {k: v for k, v in full.items() if k != "f_v_feats"}
    qd = synth.to_device(dict(qb), "cuda")
    with torch.no_grad():
        a = model(full, "repr")
        b = model(slim, "repr")
        a2, qa = model.forward_repr_txt(full, qd)
        b2, qb2 = model.forward_repr_txt(slim, qd)
    assert torch.equal(a, b) and torch.equal(a2, b2) and torch.equal(qa, qb2)
