"""Generates tests/golden/videoqa_tiny.npz by running the UNMODIFIED reference HeroForVideoQA
(model/videoQA.py) on the tiny encoder of tests/golden/hier_tiny.npz, on CPU in eval mode.

Only this one file is written (the other fixtures stay byte-identical: savez stamps times). The
batches are built by the reference's own `video_qa_collate` (data/videoQA.py) from synthetic items,
and `synth.videoqa_batch` is asserted to reproduce that layout. Needs the reference sources
(HERO_REFERENCE, as oracle/gen_golden.py).

    python oracle/gen_golden_videoqa.py
"""
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hero_b200 import synth  # noqa: E402
from oracle import hero_oracle as orc  # noqa: E402
from oracle import videoqa_oracle as vo  # noqa: E402
from oracle.gen_golden import install_stubs, model_json, np_batch  # noqa: E402

TINY = dict(hidden=128, inter=256, heads=2, f_layers=2, c_layers=2, vocab=120, vfeat_dim=64,
            max_img_len=20)
GRAD_KEYS = ["v_encoder.c_encoder.embeddings.position_embeddings.weight",
             "v_encoder.c_encoder.embeddings.LayerNorm.weight",
             "v_encoder.c_encoder.embeddings.LayerNorm.bias",
             "v_encoder.c_encoder.encoder.layer.0.attention.self.query.weight",
             "v_encoder.f_encoder.embeddings.word_embeddings.weight",
             "v_encoder.f_encoder.embeddings.position_embeddings.weight",
             "v_encoder.f_encoder.embeddings.token_type_embeddings.weight",
             "v_encoder.f_encoder.embeddings.LayerNorm.weight",
             "v_encoder.f_encoder.encoder.layer.1.attention.output.LayerNorm.weight",
             "v_encoder.frame_transform.net.1.bias"]
HEAD_SEED = 123
# gradients of every head parameter except the two 256 x 128 linear_1 weights (file size)
HEAD_GRAD_SKIP = "linear_1.weight"


def questions(seed, specs, vfeat_dim, vocab):
    """specs: per question (T, sub frame lists, sub lengths, QA lengths per candidate, target, ts)."""
    gen = torch.Generator().manual_seed(seed)
    out = []
    for T, frames, lens, qa_lens, target, ts in specs:
        clip = synth.make_clip(gen, T, frames, lens, vfeat_dim=vfeat_dim, vocab=vocab)
        out.append(synth.make_qa_question(gen, clip, qa_lens, target, ts, vocab=vocab))
    return out


def reference_items(qs):
    """The items data/videoQA.py VideoQaDataset.__getitem__ returns for these questions."""
    items = []
    for i, qn in enumerate(qs):
        c = qn["clip"]
        T = c["feats"].shape[0]
        ids, feats, masks = [], [], []
        for sub, (_, fr) in zip(c["subs"], c["sub2frames"]):
            fr = [f for f in fr if f in range(T)]
            if fr:
                feats.append(torch.index_select(c["feats"], 0, torch.tensor(fr)))
                masks.append(torch.tensor([1] * (len(sub) + len(fr))))
            else:
                feats.append(torch.zeros(1, c["feats"].shape[1]))
                masks.append(torch.tensor([0] + [1] * len(sub)))
            ids.append(sub)
        video_qa, qa_ids, qa_masks = [], [], []
        for qa in qn["qas"]:
            qa_mask = torch.tensor([1] * len(qa))
            video_qa.append(([torch.cat((s, qa)) for s in ids], feats,
                             [torch.cat((m, qa_mask)) for m in masks], c["feats"],
                             torch.tensor([1] * T), len(c["subs"]), c["sub2frames"]))
            qa_ids.append(qa)
            qa_masks.append(qa_mask)
        items.append((video_qa, qa_ids, qa_masks, [f"vid{i}"],
                      [torch.LongTensor([qn["target"]])], [torch.LongTensor(list(qn["ts"]))]))
    return items


def collate(qs):
    from data.videoQA import video_qa_collate
    ref = video_qa_collate(reference_items(qs))
    mine = synth.videoqa_batch(qs)
    for k in ("f_sub_input_ids", "f_sub_pos_ids", "f_v_feats", "f_v_pos_ids", "f_attn_masks",
              "f_gather_index", "c_v_feats", "c_attn_masks", "targets", "ts_targets",
              "qa_input_ids", "qa_pos_ids", "qa_attn_masks"):
        assert torch.equal(ref[k], mine[k]), k
    assert ref["num_subs"] == mine["num_subs"]
    assert ref["sub_idx2frame_idx"] == mine["sub_idx2frame_idx"]
    return ref


def main():
    install_stubs()
    from model.model import VideoModelConfig
    from model.videoQA import HeroForVideoQA
    torch.manual_seed(0)
    d = TINY
    with tempfile.NamedTemporaryFile("w", suffix=".json", delete=False) as f:
        json.dump(model_json(d["hidden"], d["inter"], d["heads"], d["f_layers"], d["c_layers"],
                             d["vocab"]), f)
        path = f.name
    model = HeroForVideoQA(VideoModelConfig(path), vfeat_dim=d["vfeat_dim"],
                           max_frm_seq_len=d["max_img_len"])
    os.unlink(path)
    shapes = orc.param_shapes(d["hidden"], d["inter"], d["f_layers"], d["c_layers"], d["vocab"],
                              514, 2, d["vfeat_dim"], d["max_img_len"])
    W = orc.seeded_weights(shapes, seed=11, std=0.05)          # the weights of hier_tiny.npz
    missing, unexpected = model.load_state_dict({"v_encoder." + k: v for k, v in W.items()},
                                                strict=False)
    assert not unexpected, unexpected
    # head weights from a seed (st_ed_pool drawn apart from qa_pool on purpose)
    head = vo.head_weights({k: v.shape for k, v in model.state_dict().items()}, seed=HEAD_SEED)
    missing, unexpected = model.load_state_dict(head, strict=False)
    assert not unexpected and not [k for k in missing if k.startswith(vo.HEAD_PREFIXES)]
    model.eval()
    vocab = d["vocab"] - 7
    # 5 candidates (TVQA): ragged T, subtitles with and without frames, ragged QA lengths,
    # question 1 without an answer target, question 2 without a (start, end) target
    qa = questions(5, [(9, [[0, 1, 2], [3, 4], [], [6, 7, 8]], [4, 6, 3, 5], [7, 9, 6, 8, 7], 2,
                        (1, 4)),
                       (6, [[0, 1], [2, 3, 4, 5]], [5, 3], [8, 6, 9, 7, 6], -1, (0, 2)),
                       (11, [[0, 1, 2, 3], [4, 5], [6, 7, 8, 9, 10]], [3, 7, 4],
                        [6, 6, 8, 9, 7], 4, (-1, -1))], d["vfeat_dim"], vocab)
    # 4 candidates (How2QA), equal T
    hb = questions(6, [(8, [[0, 1, 2, 3], [4, 5, 6, 7]], [5, 4], [7, 8, 6, 9], 1, (2, 5)),
                       (8, [[0, 1], [2, 3, 4], [5, 6, 7]], [3, 6, 4], [9, 7, 7, 8], 3, (0, 7))],
                   d["vfeat_dim"], vocab)
    named = dict(model.named_parameters())
    out = {}
    for tag, qs, task in (("a", qa, "tvqa"), ("b", hb, "how2qa")):
        batch = collate(qs)
        cap = {}
        hook = model.st_ed_pred_head.register_forward_hook(
            lambda m, i, o: cap.__setitem__("pred_st_ed", o.detach().clone()))
        with torch.no_grad():
            logits = model(dict(batch), task=task, compute_loss=False)
        hook.remove()
        model.zero_grad()
        qa_loss, temporal_loss = model(dict(batch), task=task, compute_loss=True)
        (qa_loss + 0.4 * temporal_loss).backward()
        out.update({f"{tag}.{k}": v for k, v in np_batch(batch).items()})
        out[f"{tag}.num_subs"] = json.dumps(batch["num_subs"])
        out[f"{tag}.sub_idx2frame_idx"] = json.dumps(batch["sub_idx2frame_idx"])
        out[f"{tag}.task"] = task
        out[f"{tag}.logits"] = logits.numpy()
        out[f"{tag}.pred_st_ed"] = cap["pred_st_ed"].numpy()
        out[f"{tag}.qa_loss"] = np.float64(qa_loss.item())
        out[f"{tag}.temporal_loss"] = np.float64(temporal_loss.item())
        for k in GRAD_KEYS + [k for k in named if k.startswith(vo.HEAD_PREFIXES)
                              and not k.endswith(HEAD_GRAD_SKIP)]:
            out[f"{tag}.grad.{k}"] = named[k].grad.numpy().copy()
        print(f"videoqa {task}: logits {tuple(logits.shape)} qa_loss {qa_loss.item():.5f} "
              f"temporal_loss {temporal_loss.item():.5f}")
    np.savez_compressed(
        os.path.join(ROOT, "tests", "golden", "videoqa_tiny.npz"), **out, head_seed=HEAD_SEED,
        loss_weight_st_ed=0.4,
        state_dict_shapes=json.dumps({k: list(v.shape) for k, v in model.state_dict().items()}))


if __name__ == "__main__":
    main()
