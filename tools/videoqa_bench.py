"""Training-step time of the video QA head (hero_b200/videoqa.py) at SYN-TVQA (T = 60, 90-token
joint rows) and SYN-TVQA-long (T = 100, 130-token joint rows on the long-sequence attention
tiles), full HERO dimensions (6 + 3 layers, H = 768), two arms alternated in one process:

    native    HeroForVideoQA.forward: packed query-fused stage + csrc/videoqa.cu pooling
    generic   the reference head's call sequence (model/videoQA.py:61-121) over this package's
              generic module APIs: forward_repr(encode_clip=False) -> c_encoder.embeddings ->
              f_encoder._compute_txt_embeddings -> c_encoder.forward_encoder -> torch pooling

Per arm and size: ms/step (CUDA events around forward + backward [+ FusedAdamW], after warm-up),
questions/s, hero_b200 launches per step, and the output / gradient agreement between the arms
on the same batch. Prints one JSON line per size and a summary line; `--out PATH` also writes the
whole record to PATH.

    python tools/videoqa_bench.py [--steps 20] [--warmup 5] [--optimizer] [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hero_b200 import ops, synth  # noqa: E402
from hero_b200.layers import mask_logits  # noqa: E402

DIMS = dict(hidden=768, inter=3072, heads=12, f_layers=6, c_layers=3, vocab=50272,
            vfeat_dim=4352, max_img_len=100)
SIZES = {"SYN-TVQA": 60, "SYN-TVQA-long": 100}


def model_json(path, d, dropout=0.0):
    def cfg(n, v):
        c = {"attention_probs_dropout_prob": dropout, "hidden_act": "gelu",
             "hidden_dropout_prob": dropout, "hidden_size": d["hidden"],
             "initializer_range": 0.02, "intermediate_size": d["inter"],
             "max_position_embeddings": 514, "num_attention_heads": d["heads"],
             "num_hidden_layers": n, "type_vocab_size": 2}
        if v:
            c["vocab_size"] = d["vocab"]
        return c
    with open(path, "w") as f:
        json.dump({"f_config": cfg(d["f_layers"], True), "c_config": cfg(d["c_layers"], False)}, f)
    return path


def build_model(path, d=DIMS, seed=0):
    from hero_b200.model import VideoModelConfig
    from hero_b200.videoqa import HeroForVideoQA
    torch.manual_seed(seed)
    m = HeroForVideoQA(VideoModelConfig(path), vfeat_dim=d["vfeat_dim"],
                       max_frm_seq_len=d["max_img_len"])
    with torch.no_grad():       # answer / span pools apart, so the two kernels' roles differ
        m.st_ed_pool.weight.normal_(0.0, 0.05)
        m.qa_pool.weight.normal_(0.0, 0.05)
    return m


def generic_frames(model, batch):
    """(P_se, P_qa, video_masks) through the generic APIs, as model/videoQA.py:66-95 does."""
    ve = model.v_encoder
    c_attn_masks = batch["c_attn_masks"]
    frames = ve.forward_repr(batch, encode_clip=False)
    frames = ve.c_encoder.embeddings(frames, position_ids=None)
    qa = ve.f_encoder._compute_txt_embeddings(batch["qa_input_ids"], batch["qa_pos_ids"])
    fused = ve.c_encoder.forward_encoder(torch.cat((frames, qa), dim=1),
                                         torch.cat((c_attn_masks, batch["qa_attn_masks"]), dim=1))
    T = c_attn_masks.shape[1]
    nv = len(batch["targets"])
    video = fused[:, :T].reshape(nv, -1, T, fused.shape[-1])
    vmask = c_attn_masks.view(nv, -1, T).to(video.dtype)
    a_se = torch.softmax(mask_logits(model.st_ed_pool(video).squeeze(-1), vmask), dim=1)
    a_qa = torch.softmax(mask_logits(model.qa_pool(video).squeeze(-1), vmask), dim=2)
    p_se = torch.einsum("vqt,vqtd->vtd", a_se, video)
    p_qa = torch.einsum("vqt,vqtd->vqd", a_qa, video)
    return p_se, p_qa, vmask[:, 0]


def heads_and_losses(model, batch, p_se, p_qa, video_masks):
    pred = model.st_ed_pred_head(p_se)
    st_prob = mask_logits(pred[:, :, 0], video_masks)
    ed_prob = mask_logits(pred[:, :, 1], video_masks)
    logits = model.qa_pred_head(p_qa).squeeze(-1)
    ts = batch["ts_targets"]
    temporal = (F.cross_entropy(st_prob, ts[:, 0], ignore_index=-1)
                + F.cross_entropy(ed_prob, ts[:, 1], ignore_index=-1)) / 2.
    qa_loss = F.cross_entropy(logits, batch["targets"].squeeze(-1), ignore_index=-1)
    return logits, st_prob, qa_loss, temporal


def arm_step(model, batch, arm):
    fr = model.forward_frames(batch) if arm == "native" else generic_frames(model, batch)
    logits, st_prob, qa_loss, temporal = heads_and_losses(model, batch, *fr)
    (qa_loss + 0.4 * temporal).backward()
    return logits, st_prob


def make_batch(T, seed=7):
    from hero_b200.plan import attach_plan
    b = synth.syn_tvqa(n_frames=T, seed=seed)
    return synth.to_device(attach_plan(b, kind="videoqa"), "cuda")


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        out = "unknown"
    return {"gpu": name, "power_limit_and_max_sm_clock": out}


def agreement(model, batch):
    """Outputs and gradients of the two arms on one batch. The gradients come from a fixed
    weighted sum of the answer logits and the span head's output: the cross entropies' gradient
    would hinge on how close the candidates' logits are, which bf16 activations shift."""
    res = {}
    g = torch.Generator().manual_seed(0)
    for arm in ("native", "generic"):
        model.zero_grad(set_to_none=True)
        fr = model.forward_frames(batch) if arm == "native" else generic_frames(model, batch)
        logits, st, _, _ = heads_and_losses(model, batch, *fr)
        pred = model.st_ed_pred_head(fr[0])
        if "w" not in res:
            res["w"] = (torch.randn(logits.shape, generator=g).cuda(),
                        torch.randn(pred.shape, generator=g).cuda() * fr[2][..., None])
        ((logits * res["w"][0]).sum() + (pred * res["w"][1]).sum()).backward()
        res[arm] = (logits.detach().float(), st.detach().float(),
                    {n: p.grad.detach().clone() for n, p in model.named_parameters()
                     if p.grad is not None})
    (ln, sn, gn), (lg, sg, gg) = res["native"], res["generic"]
    # key.bias has an exact gradient of 0 (softmax invariance): absolute difference there
    rels, abs_zero = [], []
    for k in gg:
        if k not in gn:
            continue
        den = gg[k].norm().item()
        diff = (gn[k] - gg[k]).norm().item()
        if k.endswith("key.bias") or den < 1e-6:
            abs_zero.append(diff)
        else:
            rels.append(diff / den)
    return {"logits_max_abs": (ln - lg).abs().max().item(),
            "st_prob_valid_max_abs": (sn - sg)[sg > -1e3].abs().max().item(),
            "worst_grad_rel_fro": max(rels),
            "worst_grad_abs_fro_where_exactly_zero": max(abs_zero) if abs_zero else 0.0}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3, help="alternations of the two arms")
    ap.add_argument("--optimizer", action="store_true", help="time FusedAdamW in the step too")
    ap.add_argument("--out", default=None, help="write the JSON record here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("videoqa_bench needs a CUDA device")
    import tempfile
    from types import SimpleNamespace
    from hero_b200.optim import build_optimizer
    tmp = tempfile.mkdtemp()
    model = build_model(model_json(os.path.join(tmp, "m.json"), DIMS)).cuda().train()
    opt = build_optimizer(model, SimpleNamespace(optim="adamw", lr_mul=10.0, learning_rate=1e-5,
                                                 betas=[0.9, 0.98], weight_decay=0.01))
    out = {"dims": DIMS, "steps": args.steps, "warmup": args.warmup, "rounds": args.rounds,
           "optimizer": args.optimizer, "questions_per_step": 4, "candidates": 5,
           "optimizer_launches": sum(len(g["ranges"]) for g in opt.param_groups), **gpu_info(),
           "sizes": {}}
    for size, T in SIZES.items():
        batch = make_batch(T)
        vplan = batch["_hero_videoqa_plan"]
        rec = {"T": T, "joint_rows": vplan.seq.n_seq, "joint_tokens": vplan.seq.n_tok,
               "joint_rows_on_long_path": vplan.seq.n_long, "max_joint_len": vplan.seq.max_len,
               "agreement": agreement(model, batch), "arms": {}}
        for arm in ("native", "generic"):
            rec["arms"][arm] = {"ms_per_step": []}
        for _ in range(args.rounds):
            for arm in ("native", "generic"):
                for _ in range(args.warmup):
                    opt.zero_grad()
                    arm_step(model, batch, arm)
                torch.cuda.synchronize()
                ops.reset_launch_count()
                start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(
                    enable_timing=True)
                start.record()
                for _ in range(args.steps):
                    opt.zero_grad()
                    arm_step(model, batch, arm)
                    if args.optimizer:
                        opt.step()
                end.record()
                torch.cuda.synchronize()
                rec["arms"][arm]["ms_per_step"].append(start.elapsed_time(end) / args.steps)
                rec["arms"][arm]["hero_launches_per_step"] = ops.launch_count() / args.steps
        for arm in ("native", "generic"):
            a = rec["arms"][arm]
            a["ms_per_step_min"] = min(a["ms_per_step"])
            a["questions_per_s"] = 4 * 1000.0 / a["ms_per_step_min"]
        out["sizes"][size] = rec
        print(size, json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items() if k != "sizes"}))


if __name__ == "__main__":
    main()
