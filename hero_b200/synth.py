"""Synthetic HERO batches in the reference's collate layout (SURVEY.md §8d).

`video_batch` restates the tensor layout produced by the reference's `video_collate`
(data/data.py:406-471) and `get_gather_index` (data/data.py:504-512) from per-clip items shaped
like `VideoFeatSubTokDataset.__getitem__` (data/data.py:346-397): per subtitle a token list that
starts with [SEP], the frames matched to it (or one all-zero dummy frame, masked), and the clip's
full frame-feature matrix. Everything is built on the host with a seeded generator; there is no
dataset I/O in this repo.
"""
import random

import torch

VFEAT_DIM = 4352      # utils/const.py:6
MAX_CLIP_LEN = 100    # utils/const.py:7 / config max_clip_len
SEP, CLS, PAD = 2, 0, 1


def make_clip(gen, n_frames, sub_frames, sub_lens, vfeat_dim=VFEAT_DIM, vocab=50265):
    """One clip item: (sub token ids, matched frame lists, clip features)."""
    feats = torch.randn(n_frames, vfeat_dim, generator=gen)
    subs = []
    for L in sub_lens:
        ids = torch.randint(3, vocab, (L,), generator=gen)
        ids[0] = SEP
        subs.append(ids)
    sub2frames = [(i, list(fr)) for i, fr in enumerate(sub_frames)]
    return {"feats": feats, "subs": subs, "sub2frames": sub2frames}


def video_batch(clips):
    """Collate clip items into the batch dict consumed by HierarchicalVlModel.forward."""
    sub_ids, sub_feats, sub_masks = [], [], []
    num_subs, sub_idx2frame_idx = [], []
    for c in clips:
        T, D = c["feats"].shape
        num_subs.append(len(c["subs"]))
        sub_idx2frame_idx.append(c["sub2frames"])
        for ids, (_, frames) in zip(c["subs"], c["sub2frames"]):
            frames = [f for f in frames if 0 <= f < T]
            if frames:
                sub_feats.append(c["feats"][torch.tensor(frames)])
                sub_masks.append(torch.ones(len(ids) + len(frames), dtype=torch.long))
            else:   # data/data.py:380-382: one dummy zero frame, masked out
                sub_feats.append(torch.zeros(1, D))
                sub_masks.append(torch.cat([torch.zeros(1, dtype=torch.long),
                                            torch.ones(len(ids), dtype=torch.long)]))
            sub_ids.append(ids)
    R = len(sub_ids)
    txt_lens = [len(i) for i in sub_ids]
    v_lens = [f.shape[0] for f in sub_feats]
    max_sl, max_vl = max(txt_lens), max(v_lens)
    out_size = max(m.numel() for m in sub_masks)
    D = clips[0]["feats"].shape[1]
    f_sub_input_ids = torch.full((R, max_sl), PAD, dtype=torch.long)
    f_v_feats = torch.zeros(R, max_vl, D)
    f_attn_masks = torch.zeros(R, out_size, dtype=torch.long)
    f_gather_index = torch.arange(out_size, dtype=torch.long).unsqueeze(0).repeat(R, 1)
    for r in range(R):
        tl, nf = txt_lens[r], v_lens[r]
        f_sub_input_ids[r, :tl] = sub_ids[r]
        f_v_feats[r, :nf] = sub_feats[r]
        f_attn_masks[r, :sub_masks[r].numel()] = sub_masks[r]
        f_gather_index[r, nf:nf + tl] = torch.arange(max_vl, max_vl + tl)
    f_sub_pos_ids = torch.arange(max_sl, dtype=torch.long).clamp(max=511).unsqueeze(0)
    f_v_pos_ids = torch.arange(max_vl, dtype=torch.long).unsqueeze(0)

    B = len(clips)
    n_frames = [c["feats"].shape[0] for c in clips]
    max_t = max(n_frames)
    c_v_feats = torch.zeros(B, max_t, D)
    c_attn_masks = torch.zeros(B, max_t, dtype=torch.long)
    for b, c in enumerate(clips):
        c_v_feats[b, :n_frames[b]] = c["feats"]
        c_attn_masks[b, :n_frames[b]] = 1
    c_pos_ids = torch.arange(max_t, dtype=torch.long).unsqueeze(0).repeat(B, 1)
    return {
        "f_sub_input_ids": f_sub_input_ids, "f_sub_pos_ids": f_sub_pos_ids,
        "f_v_feats": f_v_feats, "f_v_pos_ids": f_v_pos_ids,
        "f_attn_masks": f_attn_masks, "f_gather_index": f_gather_index,
        "c_v_feats": c_v_feats, "c_pos_ids": c_pos_ids, "c_attn_masks": c_attn_masks,
        "num_subs": num_subs, "sub_idx2frame_idx": sub_idx2frame_idx,
    }


def query_batch(gen, lens, vocab=50265):
    """Text-only rows for CrossModalTrm.forward(batch, 'txt') (data/data.py txt_input_collate)."""
    n, max_l = len(lens), max(lens)
    ids = torch.full((n, max_l), PAD, dtype=torch.long)
    masks = torch.zeros(n, max_l, dtype=torch.long)
    for i, L in enumerate(lens):
        row = torch.randint(3, vocab, (L,), generator=gen)
        row[0] = CLS
        ids[i, :L] = row
        masks[i, :L] = 1
    pos = torch.arange(max_l, dtype=torch.long).clamp(max=511).unsqueeze(0)
    return {"input_ids": ids, "pos_ids": pos, "attn_masks": masks}


def syn_tvr_dense(batch_size=32, seed=1234, n_frames=100, n_subs=20, frames_per_sub=5,
                  sub_len=20, query_len=16, vfeat_dim=VFEAT_DIM, vocab=50265):
    """SYN-TVR-dense: B clips x 100 frames, 20 subs of 5 frames + 20 tokens, 1 query of 16."""
    gen = torch.Generator().manual_seed(seed)
    clips = []
    for _ in range(batch_size):
        frames = [range(s * frames_per_sub, (s + 1) * frames_per_sub) for s in range(n_subs)]
        clips.append(make_clip(gen, n_frames, frames, [sub_len] * n_subs, vfeat_dim, vocab))
    return video_batch(clips), query_batch(gen, [query_len] * batch_size, vocab)


def syn_tvr_ragged(batch_size=32, seed=4321, vfeat_dim=VFEAT_DIM, vocab=50265, t_range=(40, 100),
                   s_range=(8, 30), l_range=(4, 40), q_range=(6, 24)):
    """SYN-TVR-ragged: variable T/S/L, ~10 % unmatched frames, ~5 % subs without frames."""
    gen = torch.Generator().manual_seed(seed)
    rnd = random.Random(seed)
    clips, qlens = [], []
    for _ in range(batch_size):
        T = rnd.randint(*t_range)
        S = rnd.randint(*s_range)
        cuts = sorted(rnd.sample(range(1, T), min(S - 1, T - 1)))
        bounds = [0] + cuts + [T]
        groups = []
        for s in range(len(bounds) - 1):
            fr = [f for f in range(bounds[s], bounds[s + 1]) if rnd.random() >= 0.10]
            if rnd.random() < 0.05:
                fr = []
            groups.append(fr)
        lens = [rnd.randint(*l_range) for _ in groups]
        clips.append(make_clip(gen, T, groups, lens, vfeat_dim, vocab))
        qlens.append(rnd.randint(*q_range))
    return video_batch(clips), query_batch(gen, qlens, vocab)


def syn_xm_1(seed=0, vfeat_dim=VFEAT_DIM, vocab=50265):
    """SYN-XM-1 (BASELINE config 1): 2 rows x (8 frames + 16 sub tokens), all valid."""
    gen = torch.Generator().manual_seed(seed)
    R, F, L = 2, 8, 16
    return {
        "f_v_feats": torch.randn(R, F, vfeat_dim, generator=gen),
        "f_sub_input_ids": torch.randint(3, 50000, (R, L), generator=gen),
        "f_sub_pos_ids": torch.arange(L).unsqueeze(0),
        "f_v_pos_ids": torch.arange(F).unsqueeze(0),
        "f_attn_masks": torch.ones(R, F + L, dtype=torch.long),
        "f_gather_index": torch.arange(F + L).unsqueeze(0).repeat(R, 1),
    }


def to_device(batch, device, non_blocking=True):
    """Tensors to `device`; python lists stay on the host (as data/loader.py:62-73 does)."""
    out = {}
    for k, v in batch.items():
        out[k] = v.to(device, non_blocking=non_blocking) if torch.is_tensor(v) else v
    return out


# --------------------------------------------------------------------------------------------
# Pretraining task batches (BASELINE config 5: pretrain.py task mix on HowTo100M-shape clips).
# Each generator restates the masking / collate logic of the reference's task dataset on top of a
# SYN-HT100M-dense video batch (T = 30 frames, 6 subtitles of 5 frames + 20 tokens; SURVEY.md §8d).
MASK_ID = 50264            # <mask> of the RoBERTa vocabulary (data/data.py:60-63)


def syn_ht100m_dense(batch_size=32, seed=2345, n_frames=30, n_subs=6, frames_per_sub=5, sub_len=20,
                     query_len=16, vfeat_dim=VFEAT_DIM):
    return syn_tvr_dense(batch_size=batch_size, seed=seed, n_frames=n_frames, n_subs=n_subs,
                         frames_per_sub=frames_per_sub, sub_len=sub_len, query_len=query_len,
                         vfeat_dim=vfeat_dim)


def syn_mlm_batch(vb, seed=0, mask_prob=0.15, vocab=50265):
    """data/mlm.py:21-58,132-175 (random_word + mlm_collate) on the subtitle rows of `vb`: 15 % of
    the subtitle tokens are selected, 80 % -> <mask>, 10 % -> random id, 10 % kept; `txt_mask_tgt`
    marks them in the [frames, text] row layout, `txt_labels` are their original ids."""
    rnd = random.Random(seed)
    ids = vb["f_sub_input_ids"].clone()
    R, L = ids.shape
    n_frames = vb["f_attn_masks"].sum(1) - (ids != PAD).sum(1)       # valid frame slots per row
    tgt = torch.zeros(vb["f_attn_masks"].shape, dtype=torch.bool)
    labels = []
    for r in range(R):
        toks = ids[r].tolist()
        valid = [j for j in range(1, L) if toks[j] != PAD]             # position 0 is [SEP]/[CLS]
        picked = [j for j in valid if rnd.random() < mask_prob] or valid[:1]
        nf = max(int(n_frames[r]), 1 if int(vb["f_attn_masks"][r, 0]) == 0 else int(n_frames[r]))
        for j in picked:
            labels.append(toks[j])
            p = rnd.random()
            if p < 0.8:
                ids[r, j] = MASK_ID
            elif p < 0.9:
                ids[r, j] = rnd.randrange(3, vocab)
            tgt[r, nf + j] = True
    return {"input_ids": ids, "position_ids": vb["f_sub_pos_ids"], "v_feat": vb["f_v_feats"],
            "attn_masks": vb["f_attn_masks"], "gather_index": vb["f_gather_index"],
            "txt_mask_tgt": tgt, "txt_labels": torch.tensor(labels, dtype=torch.long)}


def syn_mfm_batch(vb, seed=0, mask_prob=0.15):
    """data/mfm.py:19-97: 15 % of each clip's frames masked (>= 1); masked features zeroed in the
    clip-level AND the subtitle-level tensors, originals kept as regression / NCE targets."""
    rnd = random.Random(seed)
    b = {k: (v.clone() if torch.is_tensor(v) else v) for k, v in vb.items()}
    B, T, D = b["c_v_feats"].shape
    c_mask = torch.zeros(B, T, dtype=torch.bool)
    for i in range(B):
        n = int(b["c_attn_masks"][i].sum())
        m = [rnd.random() < mask_prob for _ in range(n)]
        if not any(m):
            m[rnd.randrange(n)] = True
        c_mask[i, :n] = torch.tensor(m)
    f_mask = torch.zeros(b["f_v_feats"].shape[:2], dtype=torch.bool)
    row = 0
    for i, clip in enumerate(b["sub_idx2frame_idx"]):
        for _, frames in clip:
            frames = [f for f in frames if 0 <= f < T]
            if frames:
                f_mask[row, :len(frames)] = c_mask[i, torch.tensor(frames)]
            row += 1
    b["feat_targets"] = b["c_v_feats"][c_mask].contiguous()
    b["c_v_feats"] = b["c_v_feats"].masked_fill(c_mask.unsqueeze(-1), 0)
    b["f_v_feats"] = b["f_v_feats"].masked_fill(f_mask.unsqueeze(-1), 0)
    b["c_v_masks"], b["f_v_masks"] = c_mask, f_mask
    return b


def syn_fom_batch(vb, seed=0, reorder_p=0.15):
    """data/fom.py:50-115 (random_reorder + fom_collate): 15 % of each clip's frame positions are
    shuffled among themselves; `targets` holds, at each shuffled slot, the original position
    (-1 elsewhere)."""
    rnd = random.Random(seed)
    b = dict(vb)
    B, T = vb["c_attn_masks"].shape
    orders = torch.arange(T).unsqueeze(0).repeat(B, 1)
    targets = torch.full((B, T), -1, dtype=torch.long)
    for i in range(B):
        n = int(vb["c_attn_masks"][i].sum())
        sel = [t for t in range(n) if rnd.random() < reorder_p]
        shuf = sel[:]
        rnd.shuffle(shuf)
        for pos, new in zip(sel, shuf):
            orders[i, pos] = new
            targets[i, new] = pos
    b["shuffled_orders"], b["targets"] = orders, targets
    return b


def syn_vsm_batch(vb, qb, seed=0):
    """data/vsm.py / data/vcmr.py: one query per clip with a (start, end) frame target."""
    rnd = random.Random(seed)
    b = dict(vb)
    B = vb["c_attn_masks"].shape[0]
    tg = []
    for i in range(B):
        n = int(vb["c_attn_masks"][i].sum())
        st = rnd.randrange(0, max(n - 1, 1))
        tg.append((st, min(n - 1, st + rnd.randrange(1, 5))))
    b.update(query_input_ids=qb["input_ids"], query_pos_ids=qb["pos_ids"],
             query_attn_masks=qb["attn_masks"], targets=torch.tensor(tg, dtype=torch.long))
    return b


# --------------------------------------------------------------------------------------------
# Video QA (TVQA / How2QA): data/videoQA.py. Every (question, answer candidate) pair becomes one
# clip row whose subtitles carry the QA text appended ([SEP] question [SEP] answer,
# data/videoQA.py:93-109); the QA text alone is collated as `qa_*` (txt_input_collate).
def make_qa_question(gen, clip, qa_lens, target, ts, vocab=50265):
    """One question: the clip item, one QA token row per answer candidate, the answer index and
    the (start, end) frame target (-1 entries are ignored by the losses)."""
    qas = []
    for L in qa_lens:
        ids = torch.randint(3, vocab, (L,), generator=gen)
        ids[0] = SEP
        ids[L // 3] = SEP
        qas.append(ids)
    return {"clip": clip, "qas": qas, "target": int(target), "ts": (int(ts[0]), int(ts[1]))}


def videoqa_batch(questions):
    """Collate questions into the batch dict of data/videoQA.py video_qa_collate."""
    clips, qa_ids = [], []
    for qn in questions:
        c = qn["clip"]
        for qa in qn["qas"]:
            clips.append({"feats": c["feats"], "sub2frames": c["sub2frames"],
                          "subs": [torch.cat([s, qa]) for s in c["subs"]]})
            qa_ids.append(qa)
    batch = video_batch(clips)
    n, max_l = len(qa_ids), max(len(q) for q in qa_ids)
    ids = torch.full((n, max_l), PAD, dtype=torch.long)
    masks = torch.zeros(n, max_l, dtype=torch.long)
    for i, q in enumerate(qa_ids):
        ids[i, :len(q)] = q
        masks[i, :len(q)] = 1
    batch["targets"] = torch.tensor([[qn["target"]] for qn in questions], dtype=torch.long)
    batch["ts_targets"] = torch.tensor([list(qn["ts"]) for qn in questions], dtype=torch.long)
    batch["qa_input_ids"] = ids
    batch["qa_pos_ids"] = torch.arange(max_l, dtype=torch.long).clamp(max=511).unsqueeze(0)
    batch["qa_attn_masks"] = masks
    return batch


def syn_tvqa(n_questions=4, n_cand=5, n_frames=60, seed=3456, n_subs=12, frames_per_sub=5,
             sub_len=14, qa_len=30, vfeat_dim=VFEAT_DIM, vocab=50265):
    """SYN-TVQA: 4 questions x 5 candidates, T = 60, 12 subtitles of 5 frames + 14 tokens, 30 QA
    tokens (49-token cross-modal rows, 90-token joint rows). n_frames=100 gives SYN-TVQA-long:
    130-token joint rows, all on the long-sequence attention tiles. Shapes chosen to cover both
    attention paths, not dataset statistics."""
    gen = torch.Generator().manual_seed(seed)
    rnd = random.Random(seed)
    questions = []
    for _ in range(n_questions):
        frames = [range(s * frames_per_sub, min((s + 1) * frames_per_sub, n_frames))
                  for s in range(n_subs)]
        clip = make_clip(gen, n_frames, frames, [sub_len] * n_subs, vfeat_dim, vocab)
        st = rnd.randrange(0, n_frames - 1)
        ed = min(n_frames - 1, st + rnd.randrange(1, 10))
        questions.append(make_qa_question(gen, clip, [qa_len] * n_cand,
                                          rnd.randrange(n_cand), (st, ed), vocab))
    return videoqa_batch(questions)
