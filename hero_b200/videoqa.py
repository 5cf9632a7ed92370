"""Video question answering head (TVQA with 5 answer candidates, How2QA with 4) on the hero_b200
encoder: HeroForVideoQA of the reference (model/videoQA.py), same constructor, task names, return
values and parameter names, so `train_videoQA.py` and its checkpoints keep working.

Every (question, candidate) pair is one row of the video batch: the collate appends the QA text to
each subtitle (data/videoQA.py:93-115). The pipeline runs packed end to end:

    repr_packed(encode_clip=False)          cross-modal transformer + frame merge
    -> query_fused_embed                    frames: c_encoder.embeddings; QA tokens:
                                            f_encoder.embeddings; both into one packed joint row
    -> c_encoder.encoder (layer runtime)    over [valid frames | valid QA tokens] per row
    -> videoqa_pool (csrc/videoqa.cu)       the two attention poolings, forward and backward

The MLP heads, mask_logits and the cross entropies act on Nv*T and Nv*Nq rows and stay torch.
With a plan attached at collate time (`plan.attach_plan(batch, kind="videoqa")`) a training step
reads nothing back from the device.

Known deviation: the pooled video P_se at a padded frame is 0 here; the reference averages what
its transformer left at that padded position. That row only feeds st/ed logits that mask_logits
then replaces by -1e4, so the returned logits and losses agree at every position.
"""
import copy
from collections import defaultdict

from torch import nn
from torch.nn import functional as F

from . import functional as Fn
from .layers import MLPLayer, mask_logits
from .model import HeroModel
from .plan import PLAN_KEY, VIDEOQA_PLAN_KEY, VideoQaPlan

TASKS = ("tvqa", "how2qa")


class HeroForVideoQA(HeroModel):
    def __init__(self, config, vfeat_dim, max_frm_seq_len):
        super().__init__(config, vfeat_dim, max_frm_seq_len)
        hsz = config.c_config.hidden_size
        self.qa_pool = nn.Linear(in_features=hsz, out_features=1, bias=False)
        self.qa_pred_head = MLPLayer(hsz, 1)
        # the start / end pooling starts as a copy of the answer pooling (model/videoQA.py:33)
        self.st_ed_pool = copy.deepcopy(self.qa_pool)
        self.st_ed_pred_head = MLPLayer(hsz, 2)

    def _plans(self, batch):
        plan, vplan = batch[PLAN_KEY], batch[VIDEOQA_PLAN_KEY]
        if plan is None:
            plan = self.v_encoder._plan(batch)  # reads the masks back to the host once (one sync)
        if vplan is None:
            vplan = VideoQaPlan(batch["c_attn_masks"], batch["qa_attn_masks"],
                                batch["qa_input_ids"], batch["qa_pos_ids"], len(batch["targets"]),
                                plan.c)
        return plan, vplan

    def forward_frames(self, batch):
        """Pooled video of the query-fused temporal stack: (P_se (Nv, T, H), P_qa (Nv, Nq, H),
        video_masks (Nv, T)) — model/videoQA.py:66-95 up to the prediction heads."""
        if not isinstance(batch, defaultdict):
            batch = defaultdict(lambda: None, batch)
        plan, vplan = self._plans(batch)
        ve = self.v_encoder
        g, _ = ve.repr_packed(batch, plan, encode_clip=False)
        pdev, dev = plan.to(g.device), vplan.to(g.device)
        ce, fe = ve.c_encoder, ve.f_encoder
        if vplan.n_pos > fe.embeddings.position_embeddings.num_embeddings:
            raise IndexError("a QA position id is outside the subtitle position table")
        drop = ce.encoder.dropout_state()
        cfg = {"drop": drop, "n_tok": vplan.seq.n_tok, "n_frame": vplan.n_frame,
               "n_qa": vplan.n_qa, "c_t": pdev.c_t, "c_row": dev.c_row,
               "c_pos_off": pdev.c_pos_off, "c_pos_idx": pdev.c_pos_idx,
               "qa_ids": dev.qa_ids, "qa_pos": dev.qa_pos, "qa_row": dev.qa_row,
               "qa_pos_off": dev.qa_pos_off, "qa_pos_idx": dev.qa_pos_idx,
               "pad_idx": fe.embeddings.padding_idx}
        c, f = ce.embeddings, fe.embeddings
        emb, emb32 = Fn.query_fused_embed(g, cfg, [
            c.position_embeddings.weight, c.LayerNorm.weight, c.LayerNorm.bias,
            f.word_embeddings.weight, f.position_embeddings.weight,
            f.token_type_embeddings.weight, f.LayerNorm.weight, f.LayerNorm.bias])
        y = ce.encoder.forward_packed(emb, vplan.seq.attn(dev, "j_"), drop, x_f32=emb32,
                                      out_f32=True)
        p_se, p_qa = Fn.videoqa_pool(y, dev.frame_tok, self.st_ed_pool.weight,
                                     self.qa_pool.weight, vplan.nv, vplan.nq, vplan.t)
        video_masks = batch["c_attn_masks"].view(vplan.nv, vplan.nq, vplan.t)[:, 0]
        return p_se, p_qa, video_masks.to(p_se.dtype)

    def forward(self, batch, task="tvqa", compute_loss=True):
        batch = defaultdict(lambda: None, batch)
        if task not in TASKS:
            raise ValueError(f"Unrecognized task: {task}")
        p_se, p_qa, video_masks = self.forward_frames(batch)
        wdt = self.st_ed_pred_head.linear_1.weight.dtype
        pred_st_ed = self.st_ed_pred_head(p_se.to(wdt))
        st_prob = mask_logits(pred_st_ed[:, :, 0], video_masks)
        ed_prob = mask_logits(pred_st_ed[:, :, 1], video_masks)
        logits = self.qa_pred_head(p_qa.to(wdt)).squeeze(-1)
        if not compute_loss:
            return logits
        targets = batch["targets"].squeeze(-1)
        ts_targets = batch["ts_targets"]
        st_loss = F.cross_entropy(st_prob, ts_targets[:, 0], reduction="mean", ignore_index=-1)
        ed_loss = F.cross_entropy(ed_prob, ts_targets[:, 1], reduction="mean", ignore_index=-1)
        temporal_loss = (st_loss + ed_loss) / 2.
        qa_loss = F.cross_entropy(logits, targets, reduction="mean", ignore_index=-1)
        return qa_loss, temporal_loss
