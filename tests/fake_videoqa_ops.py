"""TEST INFRASTRUCTURE: torch restatements of the video QA pooling C-ABI (hero_videoqa_pool_fwd /
_bwd, include/hero_b200.h), on top of tests/fake_ops.py, so the video QA head's host
orchestration runs on a CPU-only box."""
import torch

from tests import fake_ops


def _videoqa_pool(y, frame_tok, w_se, w_qa, nv, nq, t):
    tok = frame_tok.long().view(nv, nq, t)
    on = tok >= 0
    x = torch.where(on[..., None], y[tok.clamp(min=0)], torch.zeros((), dtype=y.dtype))
    fill = torch.full(on.shape, -1e4, dtype=y.dtype)
    s_se = torch.where(on, x @ w_se, fill)
    s_qa = torch.where(on, x @ w_qa, fill)
    a_se, a_qa = torch.softmax(s_se, dim=1), torch.softmax(s_qa, dim=2)
    return (torch.einsum("vqt,vqtd->vtd", a_se, x), torch.einsum("vqt,vqtd->vqd", a_qa, x),
            a_se, a_qa)


def videoqa_pool_fwd(y, frame_tok, w_se, w_qa, nv, nq, t):
    return _videoqa_pool(y, frame_tok, w_se, w_qa, nv, nq, t)


def videoqa_pool_bwd(y, frame_tok, w_se, w_qa, a_se, a_qa, dp_se, dp_qa, nv, nq, t, dy, dw_se,
                     dw_qa):
    """dy is overwritten at the frame rows only; dw_se / dw_qa are accumulated."""
    with torch.enable_grad():
        yy = y.detach().requires_grad_(True)
        ws, wq = w_se.detach().requires_grad_(True), w_qa.detach().requires_grad_(True)
        p_se, p_qa, _, _ = _videoqa_pool(yy, frame_tok, ws, wq, nv, nq, t)
        gy, gws, gwq = torch.autograd.grad((p_se * dp_se).sum() + (p_qa * dp_qa).sum(),
                                           (yy, ws, wq))
    rows = frame_tok[frame_tok >= 0].long()
    dy[rows] = gy[rows]
    dw_se.add_(gws)
    dw_qa.add_(gwq)


def install(monkeypatch):
    """fake_ops.install plus the video QA pooling restatements."""
    from hero_b200 import ops
    fake_ops.install(monkeypatch)
    for name in ("videoqa_pool_fwd", "videoqa_pool_bwd"):
        monkeypatch.setattr(ops, name, globals()[name])
