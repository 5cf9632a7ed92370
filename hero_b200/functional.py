"""Autograd glue: hand-written forward AND backward chains over the C-ABI kernels.

Each Function below replaces one stretch of the reference's module graph (and PyTorch autograd's
derivative of it) with an explicit sequence of kernel launches on packed (valid-token-only)
activations. fp32 master parameters enter the Functions only so autograd can route their
gradients; the arithmetic reads the bf16 working copies held in `ctx_w` objects.

    transformer_stack   BertEncoder.forward           model/layers.py:298-327 (A.4 in SURVEY.md)
    cross_modal_embed   _compute_img_txt_embeddings   model/encoder.py:256-285 (+ embed.py:28-117)
    frame_merge         collect_frame_outputs + frame_transform residual  model/model.py:156-212
    frame_embed         FrameEmbeddings               model/embed.py:146-161
    query_fused_embed   frame + QA embeddings of the video QA head    model/videoQA.py:68-79
    videoqa_pool        HeroForVideoQA.get_modularized_video          model/videoQA.py:36-59
    pack / unpack       padded <-> packed layouts
"""
import torch

from . import ops

BF16 = torch.bfloat16
F32 = torch.float32


# Data-parallel hook of distributed.FlatGradExchange(overlap=True): it counts transformer-stack
# forwards / backwards and is told when the cross-modal embedding backward (the last node of the
# graph) begins — at that point every gradient outside the embedding tables is final and their
# all-reduce can run beside the embedding backward.
EXCHANGE_HOOK = [None]


class DropoutState:
    """Per-forward dropout configuration: probabilities + a key stream (fwd and bwd regenerate the
    same masks from (key, element index); nothing is stored)."""

    def __init__(self, hidden_p=0.0, attn_p=0.0, training=False, base_key=None):
        self.hidden_p = hidden_p if training else 0.0
        self.attn_p = attn_p if training else 0.0
        if base_key is None and (self.hidden_p > 0 or self.attn_p > 0):
            base_key = int(torch.empty((), dtype=torch.int64).random_().item())
        self.base = base_key or 0
        self.count = 0

    def next_key(self):
        self.count += 1
        return (self.base * 2654435761 + self.count * 40503) & 0xFFFFFFFF

    def next(self, p):
        if p <= 0.0:
            return (0, 0, 1.0)
        return ops.drop_params(p, self.next_key())


def _empty(shape, like, dtype=BF16):
    return torch.empty(shape, dtype=dtype, device=like.device)


def _zeros(shape, like, dtype=F32):
    return torch.zeros(shape, dtype=dtype, device=like.device)


def _sink(p):
    """Where a parameter gradient is accumulated: straight into an existing fp32 `p.grad` (what
    autograd's AccumulateGrad would do with our result anyway — this skips the zero-fill and the
    extra add pass; with FlatParams.ensure_flat_grads every grad is a view of one flat buffer), or a
    fresh zero tensor that is handed back to autograd. Returns (target, value_for_autograd)."""
    g = p.grad
    if g is not None and g.dtype == F32 and g.is_contiguous() and not g.requires_grad:
        return g, None
    z = torch.zeros_like(p, dtype=F32)
    return z, z


def _fused_sink(ps):
    """One contiguous accumulation target covering several parameters whose existing grads are
    adjacent in memory (q/k/v weights or biases in the flat gradient buffer); else None."""
    gs = [p.grad for p in ps]
    if any(g is None or g.dtype != F32 or not g.is_contiguous() for g in gs):
        return None
    st = gs[0].untyped_storage()
    base = gs[0].data_ptr()
    off = 0
    for g in gs:
        if g.untyped_storage().data_ptr() != st.data_ptr() or g.data_ptr() != base + off * 4:
            return None
        off += g.numel()
    rows = sum(g.shape[0] for g in gs)
    out = torch.empty(0, dtype=F32, device=gs[0].device)
    out.set_(st, gs[0].storage_offset(), (rows,) + tuple(gs[0].shape[1:]))
    return out


# ---------------------------------------------------------------------------------------------
class LayerWeights:
    """bf16 working copies + fp32 vectors of one BertLayer (views into the flat buffers)."""
    __slots__ = ("wqkv", "bqkv", "wo", "bo", "ln1_g", "ln1_b", "w1", "b1", "w2", "b2", "ln2_g",
                 "ln2_b")


class _TransformerStack(torch.autograd.Function):
    """L x BertLayer on packed tokens through the native layer runtime (one C call per direction).
    args = (x, x_f32, cfg, *params) with 16 fp32 params per layer in the order
    q.w q.b k.w k.b v.w v.b o.w o.b ln1.w ln1.b i.w i.b out.w out.b ln2.w ln2.b.
    `x` (bf16) feeds the first GEMM, `x_f32` (same values, fp32; may be None) the first residual
    add: the residual stream stays fp32 through the stack. Returns the last layer's output as bf16
    (default: it feeds further bf16 kernels) or fp32 (`cfg["out_f32"]`: it is the final result)."""

    @staticmethod
    def forward(ctx, x, x_f32, cfg, *params):
        drop = cfg["drop"]
        dspec = (ops.drop_params(drop.hidden_p, 0), ops.drop_params(drop.attn_p, 0),
                 drop.next_key())
        need_grad = any(ctx.needs_input_grad)
        out, out_f32, saved = ops.bert_stack_fwd(x, cfg["layers"], cfg["att"], heads=cfg["heads"],
                                                 eps=cfg["eps"], drop=dspec, save=need_grad,
                                                 x_f32=x_f32)
        ctx.cfg, ctx.dspec, ctx.saved, ctx.params = cfg, dspec, saved, params
        ctx.x = x
        if need_grad and EXCHANGE_HOOK[0] is not None:
            EXCHANGE_HOOK[0].stack_forward()
        return out_f32 if cfg.get("out_f32") else out

    @staticmethod
    def backward(ctx, dout):
        cfg, params = ctx.cfg, ctx.params
        if dout.dtype != BF16:
            dout = dout.to(BF16)
        grads, ret = _stack_sinks(cfg, params, ctx.x.shape[1], dout.device)
        dx = ops.bert_stack_bwd(ctx.x, cfg["layers"], cfg["att"], ctx.saved,
                                dout.contiguous(), grads, heads=cfg["heads"], eps=cfg["eps"],
                                drop=ctx.dspec, need_dx=ctx.needs_input_grad[0])
        ctx.saved = None
        if EXCHANGE_HOOK[0] is not None:
            EXCHANGE_HOOK[0].stack_backward()
        return (dx, None, None) + tuple(ret)


def _stack_sinks(cfg, params, H, device):
    """Accumulation targets of a stack's 16 n parameter gradients + what to hand back to autograd.
    When every gradient already lives in an existing fp32 `.grad` (FlatParams.ensure_flat_grads)
    the targets are the same views every step: they are cached on the encoder (`cfg["cache"]`)
    and re-validated by pointer (16 n attribute reads instead of rebuilding ~30 views per layer)."""
    cache = cfg.get("cache")
    if cache is not None:
        hit = cache.get("sinks")
        if hit is not None:
            ptrs, grads = hit
            ok = True
            for p, ptr in zip(params, ptrs):
                g = p.grad
                if g is None or g.data_ptr() != ptr:
                    ok = False
                    break
            if ok:
                return grads, [None] * len(params)
    n = len(params) // 16
    ret = [None] * (16 * n)
    grads = []
    for li in range(n):
        P = params[16 * li:16 * li + 16]
        o = 16 * li
        g = {}
        g["dwqkv"] = _fused_sink([P[0], P[2], P[4]])
        if g["dwqkv"] is None:
            t = torch.zeros((3 * H, H), dtype=F32, device=device)
            g["dwqkv"] = t
            ret[o + 0], ret[o + 2], ret[o + 4] = t[:H], t[H:2 * H], t[2 * H:]
        g["dbqkv"] = _fused_sink([P[1], P[3], P[5]])
        if g["dbqkv"] is None:
            t = torch.zeros((3 * H,), dtype=F32, device=device)
            g["dbqkv"] = t
            ret[o + 1], ret[o + 3], ret[o + 5] = t[:H], t[H:2 * H], t[2 * H:]
        for name, k in (("dwo", 6), ("dbo", 7), ("dln1_g", 8), ("dln1_b", 9), ("dw1", 10),
                        ("db1", 11), ("dw2", 12), ("db2", 13), ("dln2_g", 14), ("dln2_b", 15)):
            g[name], ret[o + k] = _sink(P[k])
        grads.append(g)
    if cache is not None:
        if all(r is None for r in ret):     # everything accumulates in place: reusable
            cache["sinks"] = ([p.grad.data_ptr() for p in params], grads)
        else:
            cache.pop("sinks", None)
    return grads, ret


def transformer_stack(x, cfg, params, x_f32=None):
    return _TransformerStack.apply(x, x_f32, cfg, *params)


def _slot_table_grad(dx, off, idx, slot_pos, dtable, tok_pos):
    """dtable[pos] += sum of dx rows that used position `pos`. Rows are grouped per slot with a
    CSR gather-sum; `slot_pos` maps slot -> table row (None: fall back to a per-token index_add)."""
    if slot_pos is None:
        dtable.index_add_(0, tok_pos.long(), dx.float())
        return
    n_slot = off.numel() - 1
    dslot = torch.zeros((n_slot, dx.shape[1]), dtype=F32, device=dx.device)
    ops.gather_sum_rows(dx, off, idx, dslot)
    dtable.index_add_(0, slot_pos[:n_slot].long(), dslot)


# ---------------------------------------------------------------------------------------------
class _CrossModalEmbed(torch.autograd.Function):
    """Packed cross-modal embeddings. params order:
    word, pos, type, ln_w, ln_b, [img_lin_w, img_lin_b, img_ln_w, img_ln_b, img_pos, mask_emb,
    img_out_ln_w, img_out_ln_b]."""

    @staticmethod
    def forward(ctx, cfg, *params):
        word, pos, typ, ln_w, ln_b = params[:5]
        drop = cfg["drop"]
        n_tok, H = cfg["n_tok"], word.shape[1]
        emb = torch.empty((n_tok, H), dtype=BF16, device=word.device)
        emb32 = torch.empty((n_tok, H), dtype=F32, device=word.device)   # residual of layer 0
        type_row = typ[1]
        st = {}
        # text tokens: LN(word[id] + pos[pid] + type[1]) -> packed row  (model/embed.py:44-58)
        n_txt = cfg["n_txt"]
        if n_txt:
            st["t_mean"] = torch.empty(n_txt, device=word.device)
            st["t_rstd"] = torch.empty(n_txt, device=word.device)
            st["t_drop"] = drop.next(drop.hidden_p)
            ops.ln_fwd(word, ln_w, ln_b, 1e-5, emb, n_rows=n_txt, x_rows=cfg["txt_ids"],
                       add_tab=pos, add_idx=cfg["txt_pos"], add_vec=type_row,
                       y_rows=cfg["txt_tok"], mean=st["t_mean"], rstd=st["t_rstd"],
                       drop=st["t_drop"], y_f32=emb32)
        n_img = cfg["n_img"]
        if n_img:
            (lin_w, lin_b, iln_w, iln_b, ipos, mask_emb, oln_w, oln_b) = params[5:13]
            D = iln_w.numel()
            feats = cfg["img_feats"]                      # fp32 [R*max_vl, D]
            xn = torch.empty((n_img, D), dtype=BF16, device=word.device)
            st["i_mean"] = torch.empty(n_img, device=word.device)
            st["i_rstd"] = torch.empty(n_img, device=word.device)
            ops.ln_fwd(feats, iln_w, iln_b, 1e-5, xn, n_rows=n_img, x_rows=cfg["img_src"],
                       add_tab=mask_emb if cfg["img_mask"] is not None else None,
                       add_idx=cfg["img_mask"], mean=st["i_mean"], rstd=st["i_rstd"])
            proj = torch.empty((n_img, H), dtype=BF16, device=word.device)
            ops.gemm(xn, cfg["img_lin_w_bf16"], proj, bias=lin_b)
            st["o_mean"] = torch.empty(n_img, device=word.device)
            st["o_rstd"] = torch.empty(n_img, device=word.device)
            st["o_drop"] = drop.next(drop.hidden_p)
            ops.ln_fwd(proj, oln_w, oln_b, 1e-5, emb, n_rows=n_img, add_tab=ipos,
                       add_idx=cfg["img_k"], add_vec=type_row, y_rows=cfg["img_tok"],
                       mean=st["o_mean"], rstd=st["o_rstd"], drop=st["o_drop"], y_f32=emb32)
            st["xn"], st["proj"] = xn, proj
        ctx.cfg, ctx.st = cfg, st
        ctx.params = params      # python refs: backward accumulates into the parameters' .grad
        ctx.mark_non_differentiable(emb32)
        return emb, emb32

    @staticmethod
    def backward(ctx, demb, _demb32=None):
        if EXCHANGE_HOOK[0] is not None:
            EXCHANGE_HOOK[0].embedding_backward_begins()
        cfg, st = ctx.cfg, ctx.st
        params = ctx.params
        word, pos, typ, ln_w, ln_b = params[:5]
        demb = demb.contiguous()
        H = word.shape[1]
        dev = word.device
        grads = [None] * len(params)
        dtyp, grads[2] = _sink(typ)
        n_txt, n_img = cfg["n_txt"], cfg["n_img"]
        type_row = typ[1]
        if n_txt:
            dword, grads[0] = _sink(word)
            dpos, grads[1] = _sink(pos)
            dlnw, grads[3] = _sink(ln_w)
            dlnb, grads[4] = _sink(ln_b)
            dx = torch.empty((n_txt, H), dtype=BF16, device=dev)
            ops.ln_bwd(demb, word, ln_w, st["t_mean"], st["t_rstd"], n_rows=n_txt,
                       x_rows=cfg["txt_ids"], add_tab=pos, add_idx=cfg["txt_pos"],
                       add_vec=type_row, y_rows=cfg["txt_tok"], drop=st["t_drop"], dx=dx,
                       d_x_tab=dword, x_pad_idx=cfg["pad_idx"], dgamma=dlnw, dbeta=dlnb)
            # position rows are shared by every sequence: deterministic CSR gather-sum per
            # text slot, then slot -> position id (identity for the collate's arange ids)
            _slot_table_grad(dx, cfg["txtpos_off"], cfg["txtpos_idx"], cfg["txt_slot_pos"], dpos,
                             cfg.get("txt_pos"))
            ops.colsum(dx, dtyp[1])
        if n_img:
            (lin_w, lin_b, iln_w, iln_b, ipos, mask_emb, oln_w, oln_b) = params[5:13]
            D = iln_w.numel()
            dproj = torch.empty((n_img, H), dtype=BF16, device=dev)
            doln_w, grads[11] = _sink(oln_w)
            doln_b, grads[12] = _sink(oln_b)
            ops.ln_bwd(demb, st["proj"], oln_w, st["o_mean"], st["o_rstd"], n_rows=n_img,
                       add_tab=ipos, add_idx=cfg["img_k"], add_vec=type_row,
                       y_rows=cfg["img_tok"], drop=st["o_drop"], dx=dproj, dgamma=doln_w,
                       dbeta=doln_b)
            dipos, grads[9] = _sink(ipos)
            _slot_table_grad(dproj, cfg["imgpos_off"], cfg["imgpos_idx"], cfg["img_slot_pos"],
                             dipos, cfg.get("img_k"))
            ops.colsum(dproj, dtyp[1])
            dlin_b, grads[6] = _sink(lin_b)
            ops.colsum(dproj, dlin_b)
            dlin_w, grads[5] = _sink(lin_w)
            ops.gemm(dproj, st["xn"], dlin_w, a_mn=True, b_mn=True, accumulate_f32=True)
            # gradient wrt the normalised 4352-d features -> img_LayerNorm gamma/beta (+ mask emb)
            dxn = torch.empty((n_img, D), dtype=BF16, device=dev)
            ops.gemm(dproj, cfg["img_lin_w_bf16"], dxn, b_mn=True)
            diln_w, grads[7] = _sink(iln_w)
            diln_b, grads[8] = _sink(iln_b)
            has_mask = cfg["img_mask"] is not None
            dmask = None
            if has_mask:
                dmask, grads[10] = _sink(mask_emb)
            ops.ln_bwd(dxn, cfg["img_feats"], iln_w, st["i_mean"], st["i_rstd"], n_rows=n_img,
                       x_rows=cfg["img_src"], add_tab=mask_emb if has_mask else None,
                       add_idx=cfg["img_mask"], d_add_tab=dmask, add_pad_idx=0, dgamma=diln_w,
                       dbeta=diln_b)
        ctx.st = None
        return (None,) + tuple(grads)


def cross_modal_embed(cfg, params):
    return _CrossModalEmbed.apply(cfg, *params)


# ---------------------------------------------------------------------------------------------
class _FrameMerge(torch.autograd.Function):
    """g[c] = relu(LN_4352(c_v[c]) W^T + b) + sum_{f -> c} Hf[f]   (model/model.py:156-212).
    params: ln_w, ln_b, lin_w, lin_b."""

    @staticmethod
    def forward(ctx, hf, cfg, ln_w, ln_b, lin_w, lin_b):
        drop = cfg["drop"]
        n_c, H = cfg["n_tok"], lin_w.shape[0]
        D = ln_w.numel()
        dev = hf.device
        matched = torch.empty((n_c, H), dtype=BF16, device=dev)
        ops.gather_sum_rows(hf, cfg["fwd_off"], cfg["fwd_idx"], matched)
        xn = torch.empty((n_c, D), dtype=BF16, device=dev)
        xn_lo = torch.empty((n_c, D), dtype=BF16, device=dev)
        mean, rstd = torch.empty(n_c, device=dev), torch.empty(n_c, device=dev)
        d_in = drop.next(drop.hidden_p)   # LinearLayer: dropout sits between LN and Linear
        ops.ln_fwd(cfg["feats"], ln_w, ln_b, 1e-5, xn, n_rows=n_c, x_rows=cfg["src"], mean=mean,
                   rstd=rstd, drop=d_in, y_lo=xn_lo)
        g = torch.empty((n_c, H), dtype=BF16, device=dev)
        pre = torch.empty((n_c, H), dtype=BF16, device=dev)
        # The ReLU gate of this Linear decides, per unit, whether a whole gradient column flows:
        # with plain bf16 operands ~0.08 % of the 2.5 M pre-activations change sign against fp32,
        # which alone is a 4e-2 relative error in frame_transform's gradients. Split-bf16 operands
        # (x = hi + lo, W = hi + lo; three MMA passes into one accumulator) bring the flips to
        # ~2e-6 of the units for 2 extra passes over a 21 GFLOP GEMM (1.3 % of the step's FLOPs).
        w_hi = cfg["lin_w_bf16"]
        w_lo = (lin_w.detach() - w_hi.float()).to(BF16)
        ops.gemm(xn, w_hi, g, bias=lin_b, act=ops.ACT_RELU, resid=matched, aux_out=pre,
                 a_lo=xn_lo, b_lo=w_lo)
        ctx.cfg = cfg
        ctx.st = (xn, mean, rstd, pre, d_in)
        ctx.params = (ln_w, ln_b, lin_w, lin_b)
        return g

    @staticmethod
    def backward(ctx, dg):
        cfg = ctx.cfg
        xn, mean, rstd, pre, d_in = ctx.st
        ln_w, ln_b, lin_w, lin_b = ctx.params
        dg = dg.contiguous()
        n_c, H = dg.shape
        dev = dg.device
        # residual branch: every f token receives the gradient of the clip frames it fed
        dhf = torch.empty((cfg["n_f_tok"], H), dtype=BF16, device=dev)
        ops.gather_sum_rows(dg, cfg["bwd_off"], cfg["bwd_idx"], dhf)
        dpre = torch.empty_like(dg)
        ops.relu_bwd(dg, pre, dpre)
        dlin_b, r_lin_b = _sink(lin_b)
        ops.colsum(dpre, dlin_b)
        dlin_w, r_lin_w = _sink(lin_w)
        ops.gemm(dpre, xn, dlin_w, a_mn=True, b_mn=True, accumulate_f32=True)
        dxn = torch.empty((n_c, ln_w.numel()), dtype=BF16, device=dev)
        ops.gemm(dpre, cfg["lin_w_bf16"], dxn, b_mn=True)
        dln_w, r_ln_w = _sink(ln_w)
        dln_b, r_ln_b = _sink(ln_b)
        ops.ln_bwd(dxn, cfg["feats"], ln_w, mean, rstd, n_rows=n_c, x_rows=cfg["src"], drop=d_in,
                   dgamma=dln_w, dbeta=dln_b)
        ctx.st = None
        return dhf, None, r_ln_w, r_ln_b, r_lin_w, r_lin_b


def frame_merge(hf, cfg, params):
    return _FrameMerge.apply(hf, cfg, *params)


class _FrameEmbed(torch.autograd.Function):
    """z = dropout(LN(g + pos[t]))  (model/embed.py:146-161). params: pos, ln_w, ln_b."""

    @staticmethod
    def forward(ctx, g, cfg, pos, ln_w, ln_b):
        drop = cfg["drop"]
        n, H = g.shape
        z = torch.empty_like(g)
        z32 = torch.empty(g.shape, dtype=F32, device=g.device)    # residual of layer 0
        mean, rstd = torch.empty(n, device=g.device), torch.empty(n, device=g.device)
        d = drop.next(drop.hidden_p)
        ops.ln_fwd(g, ln_w, ln_b, 1e-5, z, n_rows=n, add_tab=pos, add_idx=cfg["t"], mean=mean,
                   rstd=rstd, drop=d, y_f32=z32)
        ctx.cfg, ctx.st = cfg, (mean, rstd, d)
        ctx.save_for_backward(g)
        ctx.params = (pos, ln_w, ln_b)
        ctx.mark_non_differentiable(z32)
        return z, z32

    @staticmethod
    def backward(ctx, dz, _dz32=None):
        cfg = ctx.cfg
        mean, rstd, d = ctx.st
        (g,) = ctx.saved_tensors
        pos, ln_w, ln_b = ctx.params
        dz = dz.contiguous()
        n, H = dz.shape
        dgx = torch.empty_like(dz)
        dln_w, r_ln_w = _sink(ln_w)
        dln_b, r_ln_b = _sink(ln_b)
        ops.ln_bwd(dz, g, ln_w, mean, rstd, n_rows=n, add_tab=pos, add_idx=cfg["t"], drop=d,
                   dx=dgx, dgamma=dln_w, dbeta=dln_b)
        dpos, r_pos = _sink(pos)
        n_slot = cfg["pos_off"].numel() - 1
        ops.gather_sum_rows(dgx, cfg["pos_off"], cfg["pos_idx"], dpos[:n_slot])
        return dgx, None, r_pos, r_ln_w, r_ln_b


def frame_embed(g, cfg, params):
    return _FrameEmbed.apply(g, cfg, *params)


class _QueryFusedEmbed(torch.autograd.Function):
    """Input of the video QA head's query-fused temporal stack (model/videoQA.py:68-79), written
    straight into the packed joint rows (plan.VideoQaPlan): frame tokens
    LN_c(g + c_pos[t]) (c_encoder.embeddings, the TemporalTrm frame embedding), QA tokens
    LN_f(word[id] + f_pos[pid] + type[1]) (f_encoder.embeddings), each followed by dropout.
    params: c_pos, c_ln_w, c_ln_b, word, f_pos, type, f_ln_w, f_ln_b. Returns the bf16 rows and
    their fp32 copy (residual of the first layer).
    The backward does not signal EXCHANGE_HOOK: the cross-modal embedding backward that runs after
    it is the last node of the graph, and the QA gradients land in f_encoder.embeddings, whose
    range is exchanged after that node anyway (params.LATE_GRAD)."""

    @staticmethod
    def forward(ctx, g, cfg, c_pos, c_ln_w, c_ln_b, word, f_pos, typ, f_ln_w, f_ln_b):
        drop = cfg["drop"]
        dev = g.device
        H = g.shape[1]
        n_c, n_qa = cfg["n_frame"], cfg["n_qa"]
        emb = torch.empty((cfg["n_tok"], H), dtype=BF16, device=dev)
        emb32 = torch.empty((cfg["n_tok"], H), dtype=F32, device=dev)
        st = {}
        st["f_mean"], st["f_rstd"] = torch.empty(n_c, device=dev), torch.empty(n_c, device=dev)
        st["f_drop"] = drop.next(drop.hidden_p)
        ops.ln_fwd(g, c_ln_w, c_ln_b, 1e-5, emb, n_rows=n_c, add_tab=c_pos, add_idx=cfg["c_t"],
                   y_rows=cfg["c_row"], mean=st["f_mean"], rstd=st["f_rstd"], drop=st["f_drop"],
                   y_f32=emb32)
        if n_qa:
            st["q_mean"] = torch.empty(n_qa, device=dev)
            st["q_rstd"] = torch.empty(n_qa, device=dev)
            st["q_drop"] = drop.next(drop.hidden_p)
            ops.ln_fwd(word, f_ln_w, f_ln_b, 1e-5, emb, n_rows=n_qa, x_rows=cfg["qa_ids"],
                       add_tab=f_pos, add_idx=cfg["qa_pos"], add_vec=typ[1], y_rows=cfg["qa_row"],
                       mean=st["q_mean"], rstd=st["q_rstd"], drop=st["q_drop"], y_f32=emb32)
        ctx.cfg, ctx.st = cfg, st
        ctx.save_for_backward(g)
        ctx.params = (c_pos, c_ln_w, c_ln_b, word, f_pos, typ, f_ln_w, f_ln_b)
        ctx.mark_non_differentiable(emb32)
        return emb, emb32

    @staticmethod
    def backward(ctx, demb, _demb32=None):
        cfg, st = ctx.cfg, ctx.st
        (g,) = ctx.saved_tensors
        c_pos, c_ln_w, c_ln_b, word, f_pos, typ, f_ln_w, f_ln_b = ctx.params
        demb = demb.contiguous()
        n_c, n_qa = cfg["n_frame"], cfg["n_qa"]
        grads = [None] * 8
        dg = torch.empty_like(g)
        dclnw, grads[1] = _sink(c_ln_w)
        dclnb, grads[2] = _sink(c_ln_b)
        ops.ln_bwd(demb, g, c_ln_w, st["f_mean"], st["f_rstd"], n_rows=n_c, add_tab=c_pos,
                   add_idx=cfg["c_t"], y_rows=cfg["c_row"], drop=st["f_drop"], dx=dg,
                   dgamma=dclnw, dbeta=dclnb)
        dcpos, grads[0] = _sink(c_pos)
        ops.gather_sum_rows(dg, cfg["c_pos_off"], cfg["c_pos_idx"],
                            dcpos[:cfg["c_pos_off"].numel() - 1])
        if n_qa:
            dword, grads[3] = _sink(word)
            dfpos, grads[4] = _sink(f_pos)
            dtyp, grads[5] = _sink(typ)
            dflnw, grads[6] = _sink(f_ln_w)
            dflnb, grads[7] = _sink(f_ln_b)
            dq = torch.empty((n_qa, g.shape[1]), dtype=BF16, device=g.device)
            # the word-table scatter-add skips the padding id, as _CrossModalEmbed does
            ops.ln_bwd(demb, word, f_ln_w, st["q_mean"], st["q_rstd"], n_rows=n_qa,
                       x_rows=cfg["qa_ids"], add_tab=f_pos, add_idx=cfg["qa_pos"],
                       add_vec=typ[1], y_rows=cfg["qa_row"], drop=st["q_drop"], dx=dq,
                       d_x_tab=dword, x_pad_idx=cfg["pad_idx"], dgamma=dflnw, dbeta=dflnb)
            ops.gather_sum_rows(dq, cfg["qa_pos_off"], cfg["qa_pos_idx"],
                                dfpos[:cfg["qa_pos_off"].numel() - 1])
            ops.colsum(dq, dtyp[1])
        ctx.st = None
        return (dg, None) + tuple(grads)


def query_fused_embed(g, cfg, params):
    return _QueryFusedEmbed.apply(g, cfg, *params)


class _VideoQaPool(torch.autograd.Function):
    """(P_se [Nv, T, H], P_qa [Nv, Nq, H]) = modularized-video pooling of the frame rows of the
    packed fp32 stack output y (model/videoQA.py:36-59; hero_b200/csrc/videoqa.cu). The gradient
    of y is zero at the QA-token rows, which the reference slices off (model/videoQA.py:82)."""

    @staticmethod
    def forward(ctx, y, frame_tok, w_se, w_qa, nv, nq, t):
        y = y.contiguous()
        ws, wq = w_se.detach().reshape(-1), w_qa.detach().reshape(-1)
        p_se, p_qa, a_se, a_qa = ops.videoqa_pool_fwd(y, frame_tok, ws, wq, nv, nq, t)
        ctx.st = (y, frame_tok, ws, wq, a_se, a_qa, (nv, nq, t))
        ctx.params = (w_se, w_qa)
        return p_se, p_qa

    @staticmethod
    def backward(ctx, dp_se, dp_qa):
        y, frame_tok, ws, wq, a_se, a_qa, (nv, nq, t) = ctx.st
        w_se, w_qa = ctx.params
        H = y.shape[1]
        dp_se = _zeros((nv, t, H), y) if dp_se is None else dp_se.float().contiguous()
        dp_qa = _zeros((nv, nq, H), y) if dp_qa is None else dp_qa.float().contiguous()
        dy = torch.zeros_like(y)
        dws, r_se = _sink(w_se)
        dwq, r_qa = _sink(w_qa)
        ops.videoqa_pool_bwd(y, frame_tok, ws, wq, a_se, a_qa, dp_se, dp_qa, nv, nq, t, dy,
                             dws.view(-1), dwq.view(-1))
        ctx.st = None
        return dy, None, r_se, r_qa, None, None, None


def videoqa_pool(y, frame_tok, w_se, w_qa, nv, nq, t):
    return _VideoQaPool.apply(y, frame_tok, w_se, w_qa, nv, nq, t)


# ---------------------------------------------------------------------------------------------
class _GatherRows(torch.autograd.Function):
    """out[i] = idx[i] >= 0 ? src[idx[i]] : 0 with the transposed gather as backward; used for
    pack (padded -> packed) and unpack (packed -> padded, zeros at padding)."""

    @staticmethod
    def forward(ctx, src, idx, inv_idx):
        out = torch.empty((idx.numel(), src.shape[1]), dtype=src.dtype, device=src.device)
        ops.gather_rows(src.contiguous(), idx, out)
        ctx.inv = inv_idx
        return out

    @staticmethod
    def backward(ctx, dout):
        dsrc = torch.empty((ctx.inv.numel(), dout.shape[1]), dtype=dout.dtype, device=dout.device)
        ops.gather_rows(dout.contiguous(), ctx.inv, dsrc)
        return dsrc, None, None


def gather_rows(src, idx, inv_idx):
    """`inv_idx[j]` = the i with idx[i] == j (or -1): both maps are injective here. bf16 or fp32
    rows (the output has the dtype of `src`)."""
    return _GatherRows.apply(src, idx, inv_idx)


# ---------------------------------------------------------------------------------------------
class _VsmVideoScores(torch.autograd.Function):
    """(Nq, Nv) = max over a clip's valid frames of the cosine of every query with every frame
    (model/pretrain.py:364-413 after the cross-rank gather): l2norm (split-bf16) -> tcgen05 GEMM
    q^ . c^ with split-bf16 operands -> masked max; backward through the arg-max frames."""

    @staticmethod
    def forward(ctx_, q, frames, mask):
        nq, d = q.shape
        nv, length, _ = frames.shape
        dev = q.device
        q = q.float().contiguous()
        c = frames.float().contiguous().view(nv * length, d)
        rows_c = (nv * length + 7) // 8 * 8          # GEMM N must be a multiple of 8
        q_hi, q_lo = _empty((nq, d), q), _empty((nq, d), q)
        c_hi = torch.zeros((rows_c, d), dtype=BF16, device=dev)
        c_lo = torch.zeros((rows_c, d), dtype=BF16, device=dev)
        q_inv = torch.empty(nq, dtype=F32, device=dev)
        c_inv = torch.empty(nv * length, dtype=F32, device=dev)
        ops.l2norm_split(q, q_hi, q_lo, q_inv)
        ops.l2norm_split(c, c_hi, c_lo, c_inv)
        s = torch.empty((nq, rows_c), dtype=F32, device=dev)
        ops.gemm(q_hi, c_hi, s, a_lo=q_lo, b_lo=c_lo)
        mask_u8 = (mask != 0).to(torch.uint8).contiguous()
        scores = torch.empty((nq, nv), dtype=F32, device=dev)
        argmax = torch.empty((nq, nv), dtype=torch.int32, device=dev)
        ops.vsm_masked_max(s, mask_u8, nq, nv, length, scores, argmax)
        ctx_.st = (q_hi, q_lo, q_inv, c_hi, c_lo, c_inv, mask_u8, argmax, (nq, nv, length, d))
        ctx_.in_dtypes = (q.dtype, frames.dtype)
        return scores

    @staticmethod
    def backward(ctx_, g):
        q_hi, q_lo, q_inv, c_hi, c_lo, c_inv, mask_u8, argmax, (nq, nv, length, d) = ctx_.st
        need_q, need_c = ctx_.needs_input_grad[0], ctx_.needs_input_grad[1]
        dq = torch.empty((nq, d), dtype=F32, device=g.device) if need_q else None
        dc = torch.empty((nv, length, d), dtype=F32, device=g.device) if need_c else None
        ops.vsm_scores_bwd(g.float().contiguous(), argmax, mask_u8, q_hi, q_lo, q_inv, c_hi, c_lo,
                           c_inv, nq, nv, length, d, dq, dc)
        return dq, dc, None


def vsm_video_scores(q, frames, mask):
    return _VsmVideoScores.apply(q, frames, mask)


class _VsmSpanLogits(torch.autograd.Function):
    """Start / end logits of each query against its own clip (model/pretrain.py:128-166, non-cross
    form): per-frame similarity + two width-K convolutions + mask_logits, one kernel each way."""

    @staticmethod
    def forward(ctx_, query, frames, mask, w_st, w_ed):
        n, length, d = frames.shape
        dev = frames.device
        query = query.float().contiguous()
        frames = frames.float().contiguous()
        ws, we = w_st.float().reshape(-1).contiguous(), w_ed.float().reshape(-1).contiguous()
        mask_u8 = (mask != 0).to(torch.uint8).contiguous()
        sim = torch.empty((n, length), dtype=F32, device=dev)
        st, ed = torch.empty_like(sim), torch.empty_like(sim)
        ops.vsm_span_fwd(query, frames, mask_u8, ws, we, sim, st, ed)
        ctx_.st = (query, frames, mask_u8, ws, we, sim)
        ctx_.w_shape = tuple(w_st.shape)
        return st, ed

    @staticmethod
    def backward(ctx_, dst, ded):
        query, frames, mask_u8, ws, we, sim = ctx_.st
        dquery, dframes = torch.empty_like(query), torch.empty_like(frames)
        dws, dwe = torch.zeros_like(ws), torch.zeros_like(we)
        ops.vsm_span_bwd(dst.float().contiguous(), ded.float().contiguous(), mask_u8, ws, we, sim,
                         query, frames, dquery, dframes, dws, dwe)
        return dquery, dframes, None, dws.view(ctx_.w_shape), dwe.view(ctx_.w_shape)


def vsm_span_logits(query, frames, mask, w_st, w_ed):
    return _VsmSpanLogits.apply(query, frames, mask, w_st, w_ed)


# ---------------------------------------------------------------------------------------------
class _LmHeadCrossEntropy(torch.autograd.Function):
    """loss[r] = cross_entropy(h[r] @ E^T + bias, label[r]) over the first n_valid vocabulary
    entries (model/layers.py:347-354 decoder + model/encoder.py:366-372), as ONE tcgen05 GEMM whose
    epilogue keeps only online-softmax partials; the backward recomputes the logits tile by tile
    and emits d logits in bf16, which feeds the tied-embedding weight gradient (fp32 accumulate
    into the embedding table's gradient), the bias gradient and d h.
    args: h (fp32/bf16 [n, H]), emb (fp32 master [V, H], tied), bias (fp32 [V]), cfg."""

    @staticmethod
    def forward(ctx, h, emb, bias, cfg):
        hb = h.to(BF16).contiguous()
        labels = cfg["labels"].to(torch.int32).contiguous()
        loss, lse = ops.lm_head_ce_fwd(hb, cfg["emb_bf16"], bias.detach(), labels, cfg["n_valid"])
        ctx.st = (hb, labels, lse)
        ctx.cfg = cfg
        ctx.params = (emb, bias)
        ctx.h_dtype = h.dtype
        return loss

    @staticmethod
    def backward(ctx, g):
        hb, labels, lse = ctx.st
        cfg = ctx.cfg
        emb, bias = ctx.params
        n, Hd = hb.shape
        V = emb.shape[0]
        ld = (V + 63) // 64 * 64
        dl_full = torch.empty((n, ld), dtype=BF16, device=hb.device)
        if ld > V:
            dl_full[:, V:].zero_()
        dl = dl_full[:, :V]
        ops.lm_head_ce_dlogits(hb, cfg["emb_bf16"], bias.detach(), labels, lse,
                               g.float().contiguous(), cfg["n_valid"], dl_full)
        demb, r_emb = _sink(emb)
        ops.gemm(dl, hb, demb, a_mn=True, b_mn=True, accumulate_f32=True)      # dE += dl^T h
        dbias, r_bias = _sink(bias)
        ops.colsum(dl, dbias)
        dh = torch.empty((n, Hd), dtype=BF16, device=hb.device)
        ops.gemm(dl, cfg["emb_bf16"], dh, b_mn=True)                             # dh = dl E
        return dh.to(ctx.h_dtype), r_emb, r_bias, None


def lm_head_cross_entropy(h, emb, bias, cfg):
    return _LmHeadCrossEntropy.apply(h, emb, bias, cfg)
