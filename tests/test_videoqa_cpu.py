"""Video QA head (TVQA / How2QA, hero_b200/videoqa.py) on CPU: the query-fused plan, the module's
host orchestration with hero_b200.ops routed through tests/fake_videoqa_ops.py, the padded oracle and the
four-group optimizer, against outputs of the unmodified reference HeroForVideoQA
(tests/golden/videoqa_tiny.npz, oracle/gen_golden_videoqa.py). The CUDA kernels are checked by
tests/test_videoqa_gpu.py."""
import json
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from hero_b200 import synth
from tests import fake_videoqa_ops
from tests import golden_util as gu
from oracle import videoqa_oracle as vo

SKIP = ("num_subs", "sub_idx2frame_idx", "task", "logits", "pred_st_ed", "qa_loss",
        "temporal_loss")


def golden_batch(vx, tag):
    b = {k[2:]: torch.from_numpy(v) for k, v in vx.items()
         if k.startswith(tag + ".") and not k.startswith(tag + ".grad.") and k[2:] not in SKIP}
    b["num_subs"] = json.loads(str(vx[tag + ".num_subs"]))
    b["sub_idx2frame_idx"] = [[(s, fr) for s, fr in clip]
                              for clip in json.loads(str(vx[tag + ".sub_idx2frame_idx"]))]
    return b


def videoqa_model(tmp_path):
    from hero_b200.model import VideoModelConfig
    from hero_b200.videoqa import HeroForVideoQA
    from tests.test_orchestration_cpu import _json
    fx, vx = gu.load("hier_tiny.npz"), gu.load("videoqa_tiny.npz")
    d = gu.dims_of(fx)
    model = HeroForVideoQA(VideoModelConfig(_json(tmp_path, d)), vfeat_dim=d["vfeat_dim"],
                           max_frm_seq_len=d["max_img_len"])
    sd = {"v_encoder." + k: v for k, v in gu.weights_for(fx).items()}
    sd.update(vo.head_weights(json.loads(str(vx["state_dict_shapes"])),
                              seed=int(vx["head_seed"])))
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert not [k for k in missing if k.startswith(("qa_", "st_ed_"))]
    return model.eval(), vx, d


def oracle_params(model):
    return {k: p.detach().clone().requires_grad_(True) for k, p in model.named_parameters()}


def rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


# ------------------------------------------------------------------------------------- plan
def test_videoqa_plan_packs_frames_then_qa_tokens_row_major():
    from hero_b200.plan import PLAN_KEY, VIDEOQA_PLAN_KEY, attach_plan
    vx = gu.load("videoqa_tiny.npz")
    b = attach_plan(golden_batch(vx, "a"), kind="videoqa")
    rp, vp = b[PLAN_KEY], b[VIDEOQA_PLAN_KEY]
    cm, qm = b["c_attn_masks"].numpy(), b["qa_attn_masks"].numpy()
    rows, T = cm.shape
    assert (vp.nv, vp.nq, vp.t) == (3, 5, T) and rows == 15
    # row-major packing: row r = its valid frames, then its valid QA tokens
    tok = 0
    for r in range(rows):
        nf, nqa = int(cm[r].sum()), int(qm[r].sum())
        assert vp.seq.cu[r] == tok and vp.seq.lens[r] == nf + nqa
        assert list(vp.frame_tok.reshape(rows, T)[r, :nf]) == list(range(tok, tok + nf))
        assert (vp.frame_tok.reshape(rows, T)[r, nf:] == -1).all()
        tok += nf + nqa
    # clip tokens (CPlan order) and QA tokens cover every joint row exactly once
    both = np.concatenate([vp.c_row, vp.qa_row])
    assert np.array_equal(np.sort(both), np.arange(vp.seq.n_tok))
    assert np.array_equal(vp.c_row, vp.frame_tok[vp.frame_tok >= 0])
    qr, qc = np.nonzero(qm)
    assert np.array_equal(vp.qa_ids, b["qa_input_ids"].numpy()[qr, qc])
    assert np.array_equal(vp.qa_pos, b["qa_pos_ids"].numpy()[0, qc])
    assert np.array_equal(vp.qa_row, vp.seq.cu[qr] + cm.sum(1)[qr] + qc)
    # position-table CSR lists every QA token under its position id
    for p in range(vp.n_pos):
        assert set(vp.qa_pos_idx[vp.qa_pos_off[p]:vp.qa_pos_off[p + 1]].tolist()) == \
            set(np.nonzero(vp.qa_pos == p)[0].tolist())
    assert rp.c.seq.n_tok == vp.n_frame
    with pytest.raises(ValueError):
        from hero_b200.plan import VideoQaPlan
        VideoQaPlan(b["c_attn_masks"], b["qa_attn_masks"], b["qa_input_ids"], b["qa_pos_ids"], 4,
                    rp.c)


def test_videoqa_plan_sends_long_joint_rows_to_the_long_tiles():
    from hero_b200.plan import VIDEOQA_PLAN_KEY, attach_plan
    for T, n_long in ((60, 0), (100, 20)):
        b = attach_plan(synth.syn_tvqa(n_frames=T, vfeat_dim=16), kind="videoqa")
        vp = b[VIDEOQA_PLAN_KEY]
        assert vp.seq.max_len == T + 30 and vp.seq.n_long == n_long
        short = vp.seq.n_tiles - vp.seq.n_long
        assert (vp.seq.tile_ntok[:short] <= 128).all()
        assert (vp.seq.tile_ntok[short:] == T + 30).all()


# ------------------------------------------------------------------------------------- module
def test_videoqa_state_dict_matches_reference_and_pools_start_equal(tmp_path):
    model, vx, _ = videoqa_model(tmp_path)
    ref = json.loads(str(vx["state_dict_shapes"]))
    ours = {k: list(v.shape) for k, v in model.state_dict().items()}
    assert set(ours) == set(ref), (sorted(set(ref) - set(ours))[:5],
                                   sorted(set(ours) - set(ref))[:5])
    assert all(ours[k] == ref[k] for k in ref)
    from hero_b200.model import VideoModelConfig
    from hero_b200.videoqa import HeroForVideoQA
    from tests.test_orchestration_cpu import _json
    fresh = HeroForVideoQA(VideoModelConfig(_json(tmp_path, gu.dims_of(gu.load("hier_tiny.npz")))),
                           vfeat_dim=64, max_frm_seq_len=20)
    assert torch.equal(fresh.st_ed_pool.weight, fresh.qa_pool.weight)
    assert fresh.st_ed_pool.weight is not fresh.qa_pool.weight


def test_videoqa_oracle_matches_reference_golden(tmp_path):
    model, vx, d = videoqa_model(tmp_path)
    for tag in ("a", "b"):
        P = oracle_params(model)
        out = vo.video_qa(P, golden_batch(vx, tag), d["f_layers"], d["c_layers"], d["heads"])
        (out["qa_loss"] + 0.4 * out["temporal_loss"]).backward()
        for key in ("logits", "pred_st_ed"):
            ref = vx[f"{tag}.{key}"]
            assert np.abs(out[key].detach().numpy() - ref).max() <= 2e-5 * np.abs(ref).max(), key
        for key in ("qa_loss", "temporal_loss"):
            assert abs(out[key].item() - float(vx[f"{tag}.{key}"])) <= 2e-5 * abs(
                float(vx[f"{tag}.{key}"])), key
        for k in [k for k in vx if k.startswith(tag + ".grad.")]:
            ref, got = vx[k], P[k[len(tag) + 6:]].grad.numpy()
            # the biases after the last LayerNorm of each MLP head have a zero exact gradient
            # (softmax gradients sum to zero): absolute bound there
            assert np.linalg.norm(got - ref) <= 1e-4 * np.linalg.norm(ref) + 1e-6, k


def test_videoqa_host_orchestration_matches_reference_golden(tmp_path, monkeypatch):
    fake_videoqa_ops.install(monkeypatch)
    model, vx, _ = videoqa_model(tmp_path)
    named = dict(model.named_parameters())
    for tag in ("a", "b"):
        task = str(vx[f"{tag}.task"])
        cap = {}
        hook = model.st_ed_pred_head.register_forward_hook(
            lambda m, i, o: cap.__setitem__("pred", o.detach().clone()))
        with torch.no_grad():
            logits = model(golden_batch(vx, tag), task=task, compute_loss=False)
        hook.remove()
        ref = vx[f"{tag}.logits"]
        assert logits.shape == ref.shape
        assert np.abs(logits.numpy() - ref).max() <= 2e-2 * np.abs(ref).max()
        ref = vx[f"{tag}.pred_st_ed"]
        valid = golden_batch(vx, tag)["c_attn_masks"].view(ref.shape[0], -1, ref.shape[1])[:, 0]
        valid = valid.bool().numpy()          # padded frames: documented deviation (masked out)
        assert np.abs(cap["pred"].numpy() - ref)[valid].max() <= 2e-2 * np.abs(ref[valid]).max()
        model.zero_grad()
        qa_loss, temporal_loss = model(golden_batch(vx, tag), task=task, compute_loss=True)
        assert abs(float(qa_loss) - float(vx[f"{tag}.qa_loss"])) < 2e-2
        assert abs(float(temporal_loss) - float(vx[f"{tag}.temporal_loss"])) < 2e-2
        (qa_loss + 0.4 * temporal_loss).backward()
        # The candidates of one question differ only through their QA tokens: on this tiny model
        # their answer logits are ~0.1 apart while the bf16 activations of the fake ops move each
        # by ~1e-2, so the answer-side gradients carry up to ~15 % relative error here (the
        # oracle test above pins the arithmetic; the GPU tests pin the kernels at 3e-2 on a
        # well-conditioned loss).
        for k in [k for k in vx if k.startswith(tag + ".grad.")]:
            ref, got = vx[k], named[k[len(tag) + 6:]].grad.numpy()
            assert np.linalg.norm(got - ref) <= 0.25 * np.linalg.norm(ref) + 1e-5, k
    with pytest.raises(ValueError):
        model(golden_batch(vx, "a"), task="violin")


def test_videoqa_attached_plan_equals_plan_built_in_forward(tmp_path, monkeypatch):
    from hero_b200.plan import attach_plan
    fake_videoqa_ops.install(monkeypatch)
    model, vx, _ = videoqa_model(tmp_path)
    with torch.no_grad():
        a = model(golden_batch(vx, "b"), task="how2qa", compute_loss=False)
        b = model(attach_plan(golden_batch(vx, "b"), kind="videoqa"), task="how2qa",
                  compute_loss=False)
    assert torch.equal(a, b)


# ------------------------------------------------------------------------------------- optimizer
def _opts(lr_mul):
    return SimpleNamespace(optim="adamw", lr_mul=lr_mul, learning_rate=1e-3, betas=[0.9, 0.98],
                           weight_decay=0.01)


def test_build_optimizer_lr_mul_gives_the_reference_four_groups(tmp_path, monkeypatch):
    """optim/misc.py:14-37 with lr_mul = 10: groups in the reference's order, each covering exactly
    its parameters, and one step equal to the reference AdamW rule per group."""
    from oracle import hero_oracle as orc
    from hero_b200.optim import build_optimizer
    from hero_b200.params import is_no_decay
    fake_videoqa_ops.install(monkeypatch)
    model, _, _ = videoqa_model(tmp_path)
    opt = build_optimizer(model, _opts(10.0), device=torch.device("cpu"))
    flat = opt.flat
    assert [g["lr"] for g in opt.param_groups] == [1e-2, 1e-2, 1e-3, 1e-3]
    assert [g["weight_decay"] for g in opt.param_groups] == [0.01, 0.0, 0.01, 0.0]
    assert sum(len(g["ranges"]) for g in opt.param_groups) <= 6
    covered = {}
    for gi, g in enumerate(opt.param_groups):
        for a, b in g["ranges"]:
            for name, _, off, n in flat.entries:
                if a <= off and off + n <= b:
                    covered[name] = gi
    for name, _, _, _ in flat.entries:
        want = 2 * ("v_encoder" in name) + is_no_decay(name)
        assert covered[name] == want, name
    ranges = sorted(r for g in opt.param_groups for r in g["ranges"])
    assert ranges[0][0] == 0 and ranges[-1][1] == flat.total
    assert all(a[1] == b[0] for a, b in zip(ranges, ranges[1:]))     # disjoint, no gaps
    # one step against the reference rule
    before = {k: p.detach().clone() for k, p in model.named_parameters()}
    g = torch.Generator().manual_seed(2)
    grads = {k: torch.randn(p.shape, generator=g) * 0.01 for k, p in model.named_parameters()}
    opt.zero_grad()
    for k, p in model.named_parameters():
        p.grad.copy_(grads[k])
    opt.step()
    for k, p in model.named_parameters():
        lr = 1e-3 if "v_encoder" in k else 1e-2
        wd = 0.0 if is_no_decay(k) else 0.01
        z = torch.zeros_like(before[k])
        ref, _, _ = orc.adamw_step(before[k], grads[k], z, z.clone(), 1, lr, 0.9, 0.98, 1e-6, wd)
        assert (p.detach() - ref).abs().max() < 2e-6, k


def test_build_optimizer_without_lr_mul_keeps_two_groups(tmp_path, monkeypatch):
    from hero_b200.optim import build_optimizer
    fake_videoqa_ops.install(monkeypatch)
    model, _, _ = videoqa_model(tmp_path)
    opt = build_optimizer(model, _opts(1.0), device=torch.device("cpu"))
    split = opt.flat.no_decay_start
    assert [g["ranges"] for g in opt.param_groups] == [[(0, split)], [(split, opt.flat.total)]]
    with pytest.raises(ValueError):
        build_optimizer(model, SimpleNamespace(**dict(vars(_opts(10.0)), optim="adam")))
