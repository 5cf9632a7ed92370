"""TEST INFRASTRUCTURE: torch restatements of the C-ABI contracts (include/hero_b200.h), used to
exercise the host-side orchestration (plans, autograd chains, module plumbing) on a CPU-only box
by monkeypatching `hero_b200.ops`. Never imported by the product; dropout is not modelled
(p must be 0). bf16 rounding is applied where the kernels round, so tolerances stay honest.
"""
import math

import torch

BF16 = torch.bfloat16


def _ck_drop(drop):
    assert drop[0] == 0, "fake ops do not model dropout"


def gemm(a, b, out, *, a_mn=False, b_mn=False, m=None, n=None, k=None, bias=None, resid=None,
         aux_in=None, aux_out=None, act=0, accumulate_f32=False, drop=(0, 0, 1.0), block_n=0,
         k_splits=0, cta_pair=0, a_lo=None, b_lo=None, resid_ln=None, out_colsum=None):
    _ck_drop(drop)
    A = a.float().t() if a_mn else a.float()
    B = b.float() if b_mn else b.float().t()
    v = A @ B
    if a_lo is not None:      # split-bf16 operands: a*b + a_lo*b + a*b_lo
        A_lo = a_lo.float().t() if a_mn else a_lo.float()
        B_lo = b_lo.float() if b_mn else b_lo.float().t()
        v = v + A_lo @ B + A @ B_lo
    if bias is not None:
        v = v + bias
    if aux_out is not None:
        if act == 1:   # saved activation derivative gelu'(v)
            d = 0.5 * (1 + torch.erf(v / math.sqrt(2))) + \
                v * torch.exp(-0.5 * v * v) / math.sqrt(2 * math.pi)
            aux_out.copy_(d.to(BF16))
        else:
            aux_out.copy_(v.to(BF16))
    if act == 1:
        v = v * 0.5 * (1.0 + torch.erf(v / math.sqrt(2.0)))
    elif act == 2:
        v = torch.relu(v)
    elif act == 3:
        v = v * aux_in.float()
    if resid is not None and resid_ln is not None:
        mu, rs, ga, be = resid_ln
        v = v + (resid - mu[:, None]) * rs[:, None] * ga + be
    elif resid is not None:
        v = v + resid.float()
    if accumulate_f32:
        out.add_(v)
    elif out.dtype == torch.float32:      # fp32 store: pre-LayerNorm sums of the residual stream
        assert act == 0 and (resid is None or resid.dtype == torch.float32)
        out.copy_(v)
    else:
        assert resid is None or resid.dtype == BF16
        out.copy_(v.to(BF16))
        if out_colsum is not None:
            out_colsum.add_(out.float().sum(0))
    return out


def _gather_sum(x, n_rows, x_rows, add_tab, add_idx, add_vec):
    s = x.float()[x_rows.long()] if x_rows is not None else x.float()[:n_rows]
    if add_tab is not None:
        s = s + add_tab[add_idx.long()]
    if add_vec is not None:
        s = s + add_vec
    return s


def ln_fwd(x, gamma, beta, eps, y, *, n_rows, x_rows=None, add_tab=None, add_idx=None,
           add_vec=None, y_rows=None, mean=None, rstd=None, drop=(0, 0, 1.0), y_f32=None,
           y_lo=None):
    _ck_drop(drop)
    s = _gather_sum(x, n_rows, x_rows, add_tab, add_idx, add_vec)
    mu = s.mean(-1, keepdim=True)
    var = ((s - mu) ** 2).mean(-1, keepdim=True)
    r = torch.rsqrt(var + eps)
    out32 = (s - mu) * r * gamma + beta
    out = out32.to(BF16)
    lo = (out32 - out.float()).to(BF16)
    if y_rows is not None:
        y[y_rows.long()] = out
        if y_f32 is not None:
            y_f32[y_rows.long()] = out32
        if y_lo is not None:
            y_lo[y_rows.long()] = lo
    else:
        y[:n_rows] = out
        if y_f32 is not None:
            y_f32[:n_rows] = out32
        if y_lo is not None:
            y_lo[:n_rows] = lo
    if mean is not None:
        mean.copy_(mu.squeeze(-1))
    if rstd is not None:
        rstd.copy_(r.squeeze(-1))
    return y


def ln_bwd(dy, x, gamma, mean, rstd, *, n_rows, x_rows=None, add_tab=None, add_idx=None,
           add_vec=None, y_rows=None, drop=(0, 0, 1.0), dx=None, dx_drop=None,
           drop2=(0, 0, 1.0), d_x_tab=None, x_pad_idx=-1, d_add_tab=None, add_pad_idx=-1,
           dgamma=None, dbeta=None, dbias=None):
    _ck_drop(drop)
    _ck_drop(drop2)
    s = _gather_sum(x, n_rows, x_rows, add_tab, add_idx, add_vec)
    xh = (s - mean[:, None]) * rstd[:, None]
    d = dy.float()[y_rows.long()] if y_rows is not None else dy.float()[:n_rows]
    g = d * gamma
    c1 = g.mean(-1, keepdim=True)
    c2 = (g * xh).mean(-1, keepdim=True)
    dxv = rstd[:, None] * (g - c1 - xh * c2)
    if dgamma is not None:
        dgamma.add_((d * xh).sum(0))
    if dbeta is not None:
        dbeta.add_(d.sum(0))
    dxb = dxv.to(BF16)
    if dx is not None:
        dx.copy_(dxb)
    if dx_drop is not None:
        dx_drop.copy_(dxb)
    if dbias is not None:
        dbias.add_(dxb.float().sum(0))
    if d_x_tab is not None:
        keep = x_rows.long() != x_pad_idx
        d_x_tab.index_add_(0, x_rows.long()[keep], dxv[keep])
    if d_add_tab is not None and add_tab is not None:
        keep = add_idx.long() != add_pad_idx
        d_add_tab.index_add_(0, add_idx.long()[keep], dxv[keep])


def _attn_core(qkv, cu, heads):
    H = heads * 64
    outs = []
    cu = cu.tolist()
    for s in range(len(cu) - 1):
        blk = qkv[cu[s]:cu[s + 1]]
        n = blk.shape[0]
        q, k, v = (blk[:, i * H:(i + 1) * H].reshape(n, heads, 64).transpose(0, 1)
                   for i in range(3))
        p = torch.softmax(q @ k.transpose(1, 2) / 8.0, dim=-1)
        outs.append((p @ v).transpose(0, 1).reshape(n, H))
    return torch.cat(outs, 0) if outs else qkv.new_zeros((0, H))


def _check_att(att):
    """The tiling must cover the token stream with whole sequences: <= 128 tokens and <= 16 sequences per tile, then
    (the last n_long tiles) one whole sequence of 129..768 tokens per tile."""
    t0, tn = att["tile_tok0"].tolist(), att["tile_ntok"].tolist()
    assert len(t0) == att["n_tiles"] and sum(tn) == att["n_tok"]
    cu = att["cu"].tolist()
    bounds = set(cu)
    n_long = att.get("n_long", 0)
    n_short = len(t0) - n_long
    covered = sorted(zip(t0, tn))
    pos = 0
    for a, n in covered:
        assert a == pos and a in bounds and (a + n) in bounds
        pos += n
    starts = sorted(b for b in bounds if b < att["n_tok"])
    for a, n in zip(t0[:n_short], tn[:n_short]):
        assert 0 < n <= 128
        assert sum(1 for b in starts if a <= b < a + n) <= 16     # sequences per tile
    for a, n in zip(t0[n_short:], tn[n_short:]):
        assert 128 < n <= att.get("max_long", 0) <= 768 and cu[cu.index(a) + 1] == a + n
    lo, hi = att["seq_lo"].tolist(), att["seq_hi"].tolist()
    for s in range(len(cu) - 1):
        for t in range(cu[s], cu[s + 1]):
            assert lo[t] == cu[s] and hi[t] == cu[s + 1]


def attn_fwd(qkv, att, ctx, *, heads, head_dim=64, drop=(0, 0, 1.0), lse=None):
    _ck_drop(drop)
    assert head_dim == 64 and att["max_len"] <= 768
    _check_att(att)
    ctx.copy_(_attn_core(qkv.float(), att["cu"], heads).to(BF16))
    return ctx


def attn_bwd(qkv, att, ctx, dctx, lse, dqkv, *, heads, head_dim=64, drop=(0, 0, 1.0), dbias=None):
    _ck_drop(drop)
    with torch.enable_grad():
        q = qkv.float().detach().requires_grad_(True)
        out = _attn_core(q, att["cu"], heads)
        out.backward(dctx.float())
    dqkv.copy_(q.grad.to(BF16))
    if dbias is not None:
        dbias.add_(dqkv.float().sum(0))
    return dqkv


def cast_bf16(src, dst):
    dst.copy_(src.to(BF16))
    return dst


def gather_rows(src, idx, dst):
    i = idx.long()
    dst.copy_(torch.where((i >= 0)[:, None], src[i.clamp(min=0)], torch.zeros_like(dst)))
    return dst


def gather_sum_rows(src, off, idx, dst):
    n = off.numel() - 1
    counts = (off[1:] - off[:-1]).long()
    rows = torch.repeat_interleave(torch.arange(n), counts)
    acc = torch.zeros(n, src.shape[-1])
    acc.index_add_(0, rows, src.float()[idx.long()])
    if dst.dtype == torch.float32:
        dst.add_(acc)
    else:
        dst.copy_(acc.to(BF16))
    return dst


def colsum(x, out):
    out.add_(x.float().sum(0))
    return out


def relu_bwd(dy, pre, out):
    out.copy_(torch.where(pre.float() > 0, dy, torch.zeros_like(dy)))
    return out


def adamw_step(p, g, m, v, p_bf16, *, step_size, beta1, beta2, eps, lr_wd, grad_scale=1.0,
               clip_sumsq=None, clip_max_norm=0.0):
    if clip_sumsq is not None:
        grad_scale = grad_scale * min(1.0, clip_max_norm / (float(clip_sumsq.sqrt()) + 1e-6))
    gr = g * grad_scale
    m.mul_(beta1).add_(gr, alpha=1 - beta1)
    v.mul_(beta2).addcmul_(gr, gr, value=1 - beta2)
    p.addcdiv_(m, v.sqrt() + eps, value=-step_size)
    if lr_wd > 0:
        p.add_(p, alpha=-lr_wd)
    if p_bf16 is not None:
        p_bf16.copy_(p.to(BF16))


def sumsq(x, out):
    out.add_((x.double() ** 2).sum().float())
    return out


def bert_stack_fwd(x, layers, att, *, heads, eps, drop, save, x_f32=None):
    """Contract of `hero_bert_stack_fwd` (include/hero_b200.h) composed from the per-kernel
    restatements above; dropout thresholds must be 0. The residual stream (layer inputs as
    residuals, pre-LayerNorm sums, LayerNorm outputs as residuals) is fp32; GEMM operands bf16."""
    assert drop[0][0] == 0 and drop[1][0] == 0, "fake ops do not model dropout"
    M, H = x.shape
    saved = []
    h = x
    h32 = x.float() if x_f32 is None else x_f32
    for lw in layers:
        inter = lw.w1.shape[0]
        qkv = torch.empty(M, 3 * H, dtype=BF16)
        gemm(h, lw.wqkv, qkv, bias=lw.bqkv)
        cx = torch.empty(M, H, dtype=BF16)
        attn_fwd(qkv, att, cx, heads=heads)
        s1 = torch.empty(M, H)
        gemm(cx, lw.wo, s1, bias=lw.bo, resid=h32)
        a = torch.empty(M, H, dtype=BF16)
        a32 = torch.empty(M, H)
        mean1, rstd1 = torch.empty(M), torch.empty(M)
        ln_fwd(s1, lw.ln1_g, lw.ln1_b, eps, a, n_rows=M, mean=mean1, rstd=rstd1, y_f32=a32)
        f = torch.empty(M, inter, dtype=BF16)
        pre = torch.empty(M, inter, dtype=BF16) if save else None
        gemm(a, lw.w1, f, bias=lw.b1, act=1, aux_out=pre)
        s2 = torch.empty(M, H)
        gemm(f, lw.w2, s2, bias=lw.b2, resid=a32)
        out = torch.empty(M, H, dtype=BF16)
        out32 = torch.empty(M, H)
        mean2, rstd2 = torch.empty(M), torch.empty(M)
        ln_fwd(s2, lw.ln2_g, lw.ln2_b, eps, out, n_rows=M, mean=mean2, rstd=rstd2, y_f32=out32)
        saved.append(dict(h=h, qkv=qkv, cx=cx, s1=s1, mean1=mean1, rstd1=rstd1, a=a, pre=pre, f=f,
                          s2=s2, mean2=mean2, rstd2=rstd2, out=out))
        h, h32 = out, out32
    return h, h32, (saved if save else None)


def bert_stack_bwd(x, layers, att, saved, dout, grads, *, heads, eps, drop, need_dx=True):
    """Contract of `hero_bert_stack_bwd`: gradients are accumulated into `grads`."""
    M, H = dout.shape
    dy = dout
    for li in range(len(layers) - 1, -1, -1):
        lw, S, G = layers[li], saved[li], grads[li]
        inter = lw.w1.shape[0]
        ds2 = torch.empty(M, H, dtype=BF16)
        ln_bwd(dy, S["s2"], lw.ln2_g, S["mean2"], S["rstd2"], n_rows=M, dx=ds2,
               dgamma=G["dln2_g"], dbeta=G["dln2_b"])
        colsum(ds2, G["db2"])
        gemm(ds2, S["f"], G["dw2"], a_mn=True, b_mn=True, accumulate_f32=True)
        dpre = torch.empty(M, inter, dtype=BF16)
        gemm(ds2, lw.w2, dpre, b_mn=True, act=3, aux_in=S["pre"])
        colsum(dpre, G["db1"])
        gemm(dpre, S["a"], G["dw1"], a_mn=True, b_mn=True, accumulate_f32=True)
        da = torch.empty(M, H, dtype=BF16)
        gemm(dpre, lw.w1, da, b_mn=True, resid=ds2)
        ds1 = torch.empty(M, H, dtype=BF16)
        ln_bwd(da, S["s1"], lw.ln1_g, S["mean1"], S["rstd1"], n_rows=M, dx=ds1,
               dgamma=G["dln1_g"], dbeta=G["dln1_b"])
        colsum(ds1, G["dbo"])
        gemm(ds1, S["cx"], G["dwo"], a_mn=True, b_mn=True, accumulate_f32=True)
        dcx = torch.empty(M, H, dtype=BF16)
        gemm(ds1, lw.wo, dcx, b_mn=True)
        dqkv = torch.empty(M, 3 * H, dtype=BF16)
        attn_bwd(S["qkv"], att, S["cx"], dcx, None, dqkv, heads=heads)
        colsum(dqkv, G["dbqkv"])
        gemm(dqkv, S["h"], G["dwqkv"], a_mn=True, b_mn=True, accumulate_f32=True)
        dx = torch.empty(M, H, dtype=BF16)
        gemm(dqkv, lw.wqkv, dx, b_mn=True, resid=ds1)
        dy = dx
    return dy if need_dx else None


def l2norm_split(x, hi, lo, inv, eps=1e-5):
    nrm = x.norm(dim=-1)
    s = 1.0 / nrm.clamp(min=eps)
    xh = x * s[:, None]
    h = xh.to(BF16)
    hi[:x.shape[0]] = h
    lo[:x.shape[0]] = (xh - h.float()).to(BF16)
    inv.copy_(torch.where(nrm < eps, -s, s))


def vsm_masked_max(s, mask_u8, nq, nv, length, scores, argmax):
    v = s[:, :nv * length].reshape(nq, nv, length)
    v = torch.where(mask_u8.bool()[None], v, torch.full_like(v, -1e4))
    best, arg = v.max(dim=2)
    scores.copy_(best)
    argmax.copy_(arg.int())


def _normalize_bwd(acc, xh, inv):
    s = inv.abs()[:, None]
    proj = acc - xh * (xh * acc).sum(-1, keepdim=True)
    return torch.where((inv < 0)[:, None], acc, proj) * s


def vsm_scores_bwd(g, argmax, mask_u8, q_hi, q_lo, q_inv, c_hi, c_lo, c_inv, nq, nv, length, d,
                   dq, dctx):
    qh = q_hi.float() + q_lo.float()
    ch = (c_hi.float() + c_lo.float())[:nv * length]
    am = argmax.long()
    rows = torch.arange(nv)[None, :] * length + am                 # (nq, nv) frame rows
    live = mask_u8.reshape(-1)[rows].float() * g
    if dq is not None:
        dq.copy_(_normalize_bwd((live[:, :, None] * ch[rows]).sum(1), qh, q_inv))
    if dctx is not None:
        acc = torch.zeros(nv * length, d)
        acc.index_add_(0, rows.reshape(-1), (live[:, :, None] * qh[:, None, :]).reshape(-1, d))
        dctx.copy_(_normalize_bwd(acc, ch, c_inv).view_as(dctx))


def _conv_same(sim, w):
    k = w.numel()
    return torch.nn.functional.conv1d(sim[:, None, :], w.view(1, 1, k), padding=k // 2)[:, 0]


def vsm_span_fwd(query, ctx, mask_u8, w_st, w_ed, sim, st, ed):
    s = torch.einsum("bd,bld->bl", query, ctx)
    on = mask_u8.bool()
    sim.copy_(s)
    st.copy_(torch.where(on, _conv_same(s, w_st), torch.full_like(s, -1e4)))
    ed.copy_(torch.where(on, _conv_same(s, w_ed), torch.full_like(s, -1e4)))


def vsm_span_bwd(dst, ded, mask_u8, w_st, w_ed, sim, query, ctx, dquery, dctx, dw_st, dw_ed):
    with torch.enable_grad():
        q = query.detach().requires_grad_(True)
        c = ctx.detach().requires_grad_(True)
        ws, we = w_st.detach().requires_grad_(True), w_ed.detach().requires_grad_(True)
        s = torch.einsum("bd,bld->bl", q, c)
        on = mask_u8.bool().float()
        loss = (_conv_same(s, ws) * on * dst).sum() + (_conv_same(s, we) * on * ded).sum()
        gq, gc, gws, gwe = torch.autograd.grad(loss, (q, c, ws, we))
    dquery.copy_(gq)
    dctx.copy_(gc)
    dw_st.add_(gws)
    dw_ed.add_(gwe)


def lm_head_ce_fwd(h, emb, bias, labels, n_valid):
    logits = (h.float() @ emb.float().t() + bias)[:, :n_valid]
    lse = torch.logsumexp(logits, dim=-1)
    return lse - logits.gather(1, labels.long()[:, None])[:, 0], lse


def lm_head_ce_dlogits(h, emb, bias, labels, lse, grad, n_valid, out):
    logits = h.float() @ emb.float().t() + bias
    p = torch.exp(logits - lse[:, None])
    p[torch.arange(h.shape[0]), labels.long()] -= 1.0
    p[:, n_valid:] = 0.0
    out[:, :emb.shape[0]] = (p * grad[:, None]).to(BF16)
    return out


def install(monkeypatch):
    """Route hero_b200.ops through the torch restatements for the duration of a test."""
    from hero_b200 import ops
    for name in ("gemm", "ln_fwd", "ln_bwd", "attn_fwd", "attn_bwd", "cast_bf16", "gather_rows",
                 "gather_sum_rows", "colsum", "relu_bwd", "adamw_step", "sumsq", "bert_stack_fwd",
                 "bert_stack_bwd", "l2norm_split", "vsm_masked_max", "vsm_scores_bwd",
                 "vsm_span_fwd", "vsm_span_bwd", "lm_head_ce_fwd", "lm_head_ce_dlogits"):
        monkeypatch.setattr(ops, name, globals()[name])
