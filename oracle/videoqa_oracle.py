"""CPU oracle of the video QA head (HeroForVideoQA.forward, model/videoQA.py:61-121).
TEST INFRASTRUCTURE ONLY, like oracle/hero_oracle.py, whose padded fp32 building blocks it uses:
plain torch ops on the reference's padded layout, autograd for the backward, parameters read from
a dict keyed by the reference's state_dict names (HeroForVideoQA: `v_encoder.*` + the head).
Pinned against the unmodified reference by tests/golden/videoqa_tiny.npz.
"""
import torch
import torch.nn.functional as F

from oracle import hero_oracle as orc


def mlp_layer(P, pfx, x):
    """MLPLayer (model/layers.py:48-61): linear -> gelu -> LayerNorm(eps 1e-5) -> linear."""
    h = orc.gelu_erf(orc.linear(x, P, pfx + "linear_1"))
    h = orc.layer_norm(h, P[pfx + "LayerNorm.weight"], P[pfx + "LayerNorm.bias"], 1e-5)
    return orc.linear(h, P, pfx + "linear_2")


def mask_logits(target, mask):
    return target * mask + (1 - mask) * -1e4


def video_qa(P, batch, f_layers, c_layers, heads):
    """Returns dict(logits (Nv, Nq), pred_st_ed (Nv, T, 2), st_prob, ed_prob, frames (Nv*Nq, T, H)
    = the frame half of the query-fused stack output, qa_loss, temporal_loss)."""
    g = orc.hierarchical_repr(P, batch, f_layers, c_layers, heads, encode_clip=False,
                              pfx="v_encoder.")
    T = g.shape[1]
    ce, fe = "v_encoder.c_encoder.", "v_encoder.f_encoder.embeddings."
    frames = orc.layer_norm(g + P[ce + "embeddings.position_embeddings.weight"][:T][None],
                            P[ce + "embeddings.LayerNorm.weight"],
                            P[ce + "embeddings.LayerNorm.bias"], 1e-5)
    qa = orc.sub_embeddings(P, fe, batch["qa_input_ids"], batch["qa_pos_ids"])
    mask = torch.cat([batch["c_attn_masks"], batch["qa_attn_masks"]], dim=1)
    fused = orc.bert_encoder(torch.cat([frames, qa], dim=1), mask, P, ce + "encoder.", c_layers,
                             heads)
    video = fused[:, :T]
    nv = len(batch["targets"])
    H = video.shape[-1]
    video = video.reshape(nv, -1, T, H)
    vmask = batch["c_attn_masks"].view(nv, -1, T).to(video.dtype)
    s_se = mask_logits(video @ P["st_ed_pool.weight"][0], vmask)
    s_qa = mask_logits(video @ P["qa_pool.weight"][0], vmask)
    p_se = torch.einsum("vqt,vqtd->vtd", torch.softmax(s_se, dim=1), video)
    p_qa = torch.einsum("vqt,vqtd->vqd", torch.softmax(s_qa, dim=2), video)
    pred = mlp_layer(P, "st_ed_pred_head.", p_se)
    st_prob = mask_logits(pred[:, :, 0], vmask[:, 0])
    ed_prob = mask_logits(pred[:, :, 1], vmask[:, 0])
    logits = mlp_layer(P, "qa_pred_head.", p_qa).squeeze(-1)
    ts = batch["ts_targets"]
    temporal = (F.cross_entropy(st_prob, ts[:, 0], ignore_index=-1)
                + F.cross_entropy(ed_prob, ts[:, 1], ignore_index=-1)) / 2.
    qa_loss = F.cross_entropy(logits, batch["targets"].squeeze(-1), ignore_index=-1)
    return {"logits": logits, "pred_st_ed": pred, "st_prob": st_prob, "ed_prob": ed_prob,
            "frames": fused[:, :T], "qa_loss": qa_loss, "temporal_loss": temporal}


HEAD_PREFIXES = ("qa_pool", "qa_pred_head", "st_ed_pool", "st_ed_pred_head")


def head_weights(shapes, seed=123):
    """Seeded weights of the head parameters (names -> shapes of HeroForVideoQA's state_dict), so
    fixtures store the seed instead of the tensors. LayerNorm weights near 1, pooling vectors
    0.2-scaled, the rest 0.05-scaled; each tensor from its own generator (name order only)."""
    out = {}
    names = sorted(k for k in shapes if k.startswith(HEAD_PREFIXES))
    for i, k in enumerate(names):
        g = torch.Generator().manual_seed(seed * 1000 + i)
        r = torch.randn(tuple(shapes[k]), generator=g)
        if "LayerNorm.weight" in k:
            out[k] = 1.0 + 0.05 * r
        else:
            out[k] = r * (0.2 if "pool" in k else 0.05)
    return out
