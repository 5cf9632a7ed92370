"""Tensor-level wrappers over the C-ABI: torch supplies device memory and the current stream,
the arithmetic runs in `libhero_b200.so`. No autograd here (see `functional.py`).

Every wrapper enqueues on torch's current CUDA stream, which is what the reference's
PrefetchLoader has already synchronised the inputs against (data/loader.py:135-138).
"""
import ctypes as C

import torch

from . import _lib

ACT_NONE, ACT_GELU, ACT_RELU, ACT_GELU_GRAD, ACT_CE, ACT_CE_GRAD = 0, 1, 2, 3, 4, 5

BF16 = torch.bfloat16


_LAUNCHES = 0


def _count(n=1):
    global _LAUNCHES
    _LAUNCHES += n


def reset_launch_count():
    global _LAUNCHES
    _LAUNCHES = 0


def launch_count():
    """Number of hero_b200 kernels launched since the last reset (bench.py's gpu_launches)."""
    return _LAUNCHES


def sm_count():
    """SMs the persistent kernels are sized for: the device's count."""
    return _lib.lib().hero_sm_count()


def start_gemm_profile():
    """Bracket every GEMM launch (direct or from the layer runtime) with CUDA events on the
    launching stream (bench.py roofline); implemented in the library."""
    _lib.check(_lib.lib().hero_gemm_profile_begin())


def stop_gemm_profile():
    ms, fl, n = C.c_double(), C.c_double(), C.c_int64()
    _lib.check(_lib.lib().hero_gemm_profile_end(C.byref(ms), C.byref(fl), C.byref(n)))
    return {"ms": ms.value, "flops": fl.value, "launches": n.value}


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)


def _stream():
    """Handle of torch's current CUDA stream (the raw getter skips building a Stream object:
    ~0.5 us instead of ~15 us, on a path called for every launch)."""
    if _raw_stream is not None and _raw_device is not None:
        return C.c_void_p(_raw_stream(_raw_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise _lib.HeroError("hero_b200 ops need CUDA tensors (there is no CPU fallback)")


def drop_params(p, key):
    """(threshold, key, scale) for dropout probability p; p == 0 disables."""
    if p <= 0.0:
        return 0, 0, 1.0
    thr = min(int(p * 4294967296.0), 4294967295)
    return thr, int(key) & 0xFFFFFFFF, 1.0 / (1.0 - p)


def gemm(a, b, out, *, a_mn=False, b_mn=False, m=None, n=None, k=None, bias=None, resid=None,
         aux_in=None, aux_out=None, act=ACT_NONE, accumulate_f32=False, drop=(0, 0, 1.0),
         block_n=0, k_splits=0, cta_pair=0, a_lo=None, b_lo=None, resid_ln=None,
         out_colsum=None):
    """out = epilogue(A·B) with the operand conventions of `hero_gemm_args`.

    a: [M,K] (a_mn=False) or [K,M] (a_mn=True) bf16; b: [N,K] (b_mn=False) or [K,N] (b_mn=True).
    """
    _require_cuda(a, b, out)
    assert a.dtype == BF16 and b.dtype == BF16
    if m is None:
        m = a.shape[1] if a_mn else a.shape[0]
    if k is None:
        k = a.shape[0] if a_mn else a.shape[1]
    if n is None:
        n = b.shape[1] if b_mn else b.shape[0]
    g = _lib.GemmArgs()
    g.a, g.b = _ptr(a), _ptr(b)
    g.lda, g.ldb = a.stride(0), b.stride(0)
    g.a_mn_major, g.b_mn_major = int(a_mn), int(b_mn)
    g.m, g.n, g.k = m, n, k
    g.bias = _ptr(bias)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == n
    g.resid = _ptr(resid)
    g.ld_resid = resid.stride(0) if resid is not None else 0
    g.resid_f32 = int(resid is not None and resid.dtype == torch.float32)
    g.aux_in = _ptr(aux_in)
    g.ld_aux_in = aux_in.stride(0) if aux_in is not None else 0
    g.aux_out = _ptr(aux_out)
    g.ld_aux_out = aux_out.stride(0) if aux_out is not None else 0
    g.out = _ptr(out)
    g.ld_out = out.stride(0)
    g.act = act
    g.out_f32_accumulate = int(accumulate_f32)
    # an fp32 `out` without accumulate_f32 is a plain fp32 store (pre-LayerNorm sums of the
    # residual stream); its residual, if any, is fp32 too
    g.out_f32_store = int(out.dtype == torch.float32 and not accumulate_f32)
    assert out.dtype in (torch.float32, BF16) and (out.dtype == torch.float32 or not accumulate_f32)
    g.drop_threshold, g.drop_key, g.drop_scale = drop
    g.block_n, g.k_splits, g.cta_pair = block_n, k_splits, cta_pair
    if a_lo is not None or b_lo is not None:     # split-bf16 operands: a*b + a_lo*b + a*b_lo
        assert a_lo is not None and b_lo is not None
        assert a_lo.dtype == BF16 and b_lo.dtype == BF16
        assert a_lo.shape == a.shape and a_lo.stride() == a.stride()
        assert b_lo.shape == b.shape and b_lo.stride() == b.stride()
        g.a_lo, g.b_lo = _ptr(a_lo), _ptr(b_lo)
    if resid_ln is not None:     # (mean[m], rstd[m], gamma[n], beta[n]): resid is a pre-LN fp32 sum
        assert resid is not None and resid.dtype == torch.float32
        for t in resid_ln:
            assert t.dtype == torch.float32 and t.is_contiguous()
        (g.resid_ln_mean, g.resid_ln_rstd, g.resid_ln_gamma,
         g.resid_ln_beta) = (_ptr(t) for t in resid_ln)
    if out_colsum is not None:   # f32 [n] += column sums of the stored bf16 rows
        assert out_colsum.dtype == torch.float32 and out_colsum.numel() == n and out.dtype == BF16
        g.out_colsum = _ptr(out_colsum)
    _count()
    _lib.check(_lib.lib().hero_gemm_bf16(C.byref(g), _stream()))
    return out


def _ln_args(x, gamma, beta, eps, n_rows, h, x_rows=None, add_tab=None, add_idx=None,
             add_vec=None):
    a = _lib.LnArgs()
    a.x = _ptr(x)
    a.x_is_f32 = int(x.dtype == torch.float32)
    assert x.dtype in (torch.float32, BF16)
    a.x_rows = _ptr(x_rows)
    a.add_tab, a.add_idx, a.add_vec = _ptr(add_tab), _ptr(add_idx), _ptr(add_vec)
    a.gamma, a.beta = _ptr(gamma), _ptr(beta)
    a.eps = eps
    a.n_rows, a.h = n_rows, h
    a.x_pad_idx = -1
    a.add_pad_idx = -1
    for t in (x_rows, add_idx):
        assert t is None or t.dtype == torch.int32
    for t in (add_tab, add_vec, gamma, beta):
        assert t is None or t.dtype == torch.float32
    return a


def ln_fwd(x, gamma, beta, eps, y, *, n_rows, x_rows=None, add_tab=None, add_idx=None,
           add_vec=None, y_rows=None, mean=None, rstd=None, drop=(0, 0, 1.0), y_f32=None,
           y_lo=None):
    """Fused gather + add + LayerNorm (+dropout) + scatter; see `hero_ln_args`. `y_f32`: optional
    fp32 copy of the output (same rows): the residual stream of the transformer layers."""
    _require_cuda(x, y)
    h = gamma.numel()
    a = _ln_args(x, gamma, beta, eps, n_rows, h, x_rows, add_tab, add_idx, add_vec)
    a.y, a.y_rows = _ptr(y), _ptr(y_rows)
    if y_f32 is not None:
        assert y_f32.dtype == torch.float32 and y_f32.is_contiguous() and y_f32.shape == y.shape
    a.y_f32 = _ptr(y_f32)
    if y_lo is not None:      # low half of a split-bf16 operand: bf16(y_f32 - float(bf16(y)))
        assert y_lo.dtype == BF16 and y_lo.is_contiguous() and y_lo.shape == y.shape
    a.y_lo = _ptr(y_lo)
    a.mean, a.rstd = _ptr(mean), _ptr(rstd)
    a.drop_threshold, a.drop_key, a.drop_scale = drop
    _count()
    _lib.check(_lib.lib().hero_ln_fwd(C.byref(a), _stream()))
    return y


def ln_bwd(dy, x, gamma, mean, rstd, *, n_rows, x_rows=None, add_tab=None, add_idx=None,
           add_vec=None, y_rows=None, drop=(0, 0, 1.0), dx=None, dx_drop=None,
           drop2=(0, 0, 1.0), d_x_tab=None, x_pad_idx=-1, d_add_tab=None, add_pad_idx=-1,
           dgamma=None, dbeta=None, dbias=None):
    """Backward of ln_fwd (`hero_ln_bwd`): row gradients dx / dx_drop (dropout-masked copy) and
    table scatter-adds, parameter gradients dgamma / dbeta (accumulated), and `dbias` (fp32 [h]) +=
    column sums of dx_drop (else dx) — the bias gradient of the Linear feeding this LayerNorm."""
    _require_cuda(dy, x)
    h = gamma.numel()
    a = _ln_args(x, gamma, None, 0.0, n_rows, h, x_rows, add_tab, add_idx, add_vec)
    a.y_rows = _ptr(y_rows)
    a.mean, a.rstd = _ptr(mean), _ptr(rstd)
    a.drop_threshold, a.drop_key, a.drop_scale = drop
    a.dy, a.dx, a.dx_drop = _ptr(dy), _ptr(dx), _ptr(dx_drop)
    a.drop2_threshold, a.drop2_key, a.drop2_scale = drop2
    a.d_x_tab, a.x_pad_idx = _ptr(d_x_tab), x_pad_idx
    a.d_add_tab, a.add_pad_idx = _ptr(d_add_tab), add_pad_idx
    a.dgamma, a.dbeta, a.dbias = _ptr(dgamma), _ptr(dbeta), _ptr(dbias)
    _count(int(dx is not None or dx_drop is not None or d_x_tab is not None or
               d_add_tab is not None) +
           int(dgamma is not None or dbeta is not None or dbias is not None))
    _lib.check(_lib.lib().hero_ln_bwd(C.byref(a), _stream()))


def attn_fwd(qkv, att, ctx, *, heads, head_dim=64, drop=(0, 0, 1.0), lse=None):
    """ctx = softmax(QK^T / sqrt(d)) V per (sequence, head) on packed tokens; `att` is the device
    attention plan of `SeqPlan.attn` (tiles of <= 128 tokens + per-token sequence ranges)."""
    _require_cuda(qkv, ctx)
    assert qkv.dtype == BF16 and qkv.is_contiguous() and ctx.is_contiguous()
    _count()
    _lib.check(_lib.lib().hero_attn_fwd(
        _ptr(qkv), _ptr(att["tile_tok0"]), _ptr(att["tile_ntok"]), _ptr(att["seq_lo"]),
        _ptr(att["seq_hi"]), _ptr(ctx), _ptr(lse), att["n_tok"], att["n_tiles"],
        att.get("n_long", 0), att.get("max_long", 0), heads, head_dim,
        1.0 / (head_dim ** 0.5), drop[0], drop[1], drop[2], _stream()))
    return ctx


def attn_bwd(qkv, att, ctx, dctx, lse, dqkv, *, heads, head_dim=64, drop=(0, 0, 1.0), dbias=None):
    """`dbias` (f32 [3 * heads * head_dim], optional): the column sums of dqkv are ACCUMULATED
    into it (bias gradient of the QKV projection)."""
    _require_cuda(qkv, ctx, dctx, dqkv)
    assert dctx.is_contiguous() and dqkv.is_contiguous() and ctx.is_contiguous()
    if dbias is not None:
        assert dbias.dtype == torch.float32 and dbias.numel() == dqkv.shape[1]
    _count()
    _lib.check(_lib.lib().hero_attn_bwd(
        _ptr(qkv), _ptr(att["tile_tok0"]), _ptr(att["tile_ntok"]), _ptr(att["seq_lo"]),
        _ptr(att["seq_hi"]), _ptr(ctx), _ptr(dctx), _ptr(lse), _ptr(dqkv),
        _ptr(dbias), att["n_tok"],
        att["n_tiles"], att.get("n_long", 0), att.get("max_long", 0),
        heads, head_dim, 1.0 / (head_dim ** 0.5), drop[0], drop[1], drop[2], _stream()))
    return dqkv


# kernels launched per layer by the native runtime (for bench.py's gpu_launches)
_STACK_FWD_LAUNCHES, _STACK_BWD_LAUNCHES = 7, 11   # bwd: 8 GEMM, 2 LN (one pass each), attention
_ACT_FIELDS = ("qkv", "cx", "lse", "s1", "mean1", "rstd1", "a", "a_f32", "pre", "f", "s2", "mean2",
               "rstd2", "out", "out_f32")
_GRAD_FIELDS = ("dwqkv", "dbqkv", "dwo", "dbo", "dln1_g", "dln1_b", "dw1", "db1", "dw2", "db2",
                "dln2_g", "dln2_b")


def _al(n):
    return (n + 255) // 256 * 256


def _stack_layout(M, H, inter, save):
    """Byte offsets of one layer's activations inside the workspace slot."""
    sizes = {"qkv": M * 3 * H * 2, "cx": M * H * 2, "lse": M * (H // 64) * 4 if save else 0,
             "s1": M * H * 4, "mean1": M * 4,
             "rstd1": M * 4, "a": M * H * 2, "a_f32": 0,
             "pre": M * inter * 2 if save else 0,
             "f": M * inter * 2, "s2": M * H * 4, "mean2": M * 4, "rstd2": M * 4,
             "out": M * H * 2, "out_f32": M * H * 4}
    offs, o = {}, 0
    for k in _ACT_FIELDS:
        offs[k] = o
        o += _al(sizes[k])
    return offs, o, sizes


def _stack_struct(x, layers, att, heads, eps, drop, act_ptrs, x_f32=None):
    n = len(layers)
    W = (_lib.LayerWeights * n)()
    A = (_lib.LayerActs * n)()
    for i, lw in enumerate(layers):
        w = W[i]
        w.wqkv, w.bqkv, w.wo, w.bo = (lw.wqkv.data_ptr(), lw.bqkv.data_ptr(), lw.wo.data_ptr(),
                                      lw.bo.data_ptr())
        w.ln1_g, w.ln1_b, w.w1, w.b1 = (lw.ln1_g.data_ptr(), lw.ln1_b.data_ptr(),
                                        lw.w1.data_ptr(), lw.b1.data_ptr())
        w.w2, w.b2, w.ln2_g, w.ln2_b = (lw.w2.data_ptr(), lw.b2.data_ptr(), lw.ln2_g.data_ptr(),
                                        lw.ln2_b.data_ptr())
        a = A[i]
        for name, ptr in zip(_ACT_FIELDS, act_ptrs[i]):
            setattr(a, name, ptr)
    s = _lib.StackArgs()
    s.n_layers, s.n_tok, s.hidden = n, x.shape[0], x.shape[1]
    s.inter, s.heads, s.n_tiles = layers[0].w1.shape[0], heads, att["n_tiles"]
    s.n_long, s.max_long = att.get("n_long", 0), att.get("max_long", 0)
    s.eps = eps
    s.weights, s.acts = W, A
    s.x = x.data_ptr()
    s.x_f32 = None if x_f32 is None else x_f32.data_ptr()
    s.tile_tok0, s.tile_ntok = att["tile_tok0"].data_ptr(), att["tile_ntok"].data_ptr()
    s.seq_lo, s.seq_hi = att["seq_lo"].data_ptr(), att["seq_hi"].data_ptr()
    (hthr, _, hscale), (athr, _, ascale), key = drop
    s.hidden_drop_threshold, s.attn_drop_threshold, s.drop_key = hthr, athr, key
    s.hidden_drop_scale, s.attn_drop_scale = hscale, ascale
    return s, (W, A)


def bert_stack_fwd(x, layers, att, *, heads, eps, drop, save, x_f32=None):
    """All layers of a BertEncoder forward in ONE native call (`hero_bert_stack_fwd`).

    x: packed bf16 [n_tok, H] (GEMM operand) and x_f32: the same values in fp32 (residual of
    layer 0; derived from x when omitted); layers: functional.LayerWeights per layer; att:
    attention plan; drop: ((hidden thr, _, scale), (attn thr, _, scale), base key).
    Returns (out_bf16, out_f32, saved) where `saved` is what bert_stack_bwd needs (None when save
    is False: activations then ping-pong between two workspace slots)."""
    _require_cuda(x)
    assert x.dtype == BF16 and x.is_contiguous()
    if x_f32 is None:
        x_f32 = x.float()
    assert x_f32.dtype == torch.float32 and x_f32.is_contiguous() and x_f32.shape == x.shape
    n = len(layers)
    M, H = x.shape
    inter = layers[0].w1.shape[0]
    offs, slot, sizes = _stack_layout(M, H, inter, save)
    n_slots = n if save else min(n, 2)
    ws = torch.empty(n_slots * slot, dtype=torch.uint8, device=x.device)
    base = ws.data_ptr()
    act_ptrs = []
    for i in range(n):
        b = base + (i if save else i % 2) * slot
        # a_f32 is never materialised (the FFN-down epilogue recomputes LayerNorm(s1) in fp32);
        # out_f32 only for the last layer (the stack's fp32 result)
        act_ptrs.append([None if ((k in ("pre", "lse") and not save) or k == "a_f32" or
                                  (k == "out_f32" and i != n - 1)) else b + offs[k]
                         for k in _ACT_FIELDS])
    s, keep = _stack_struct(x, layers, att, heads, eps, drop, act_ptrs, x_f32)
    _count(_STACK_FWD_LAUNCHES * n)
    _lib.check(_lib.lib().hero_bert_stack_fwd(C.byref(s), _stream()))
    base_last = ((n - 1) if save else (n - 1) % 2) * slot
    last = base_last + offs["out"]
    out = ws[last:last + M * H * 2].view(BF16).view(M, H)
    last32 = base_last + offs["out_f32"]
    out_f32 = ws[last32:last32 + M * H * 4].view(torch.float32).view(M, H)
    return out, out_f32, ((ws, act_ptrs) if save else None)


def bert_stack_bwd(x, layers, att, saved, dout, grads, *, heads, eps, drop, need_dx=True):
    """Backward of the whole stack (`hero_bert_stack_bwd`). grads: per layer a dict of fp32
    tensors (keys of hero_layer_grads) that are ACCUMULATED into. Returns dx (bf16) or None."""
    _require_cuda(x, dout)
    assert dout.dtype == BF16 and dout.is_contiguous()
    ws, act_ptrs = saved
    s, keep = _stack_struct(x, layers, att, heads, eps, drop, act_ptrs)
    n = len(layers)
    G = (_lib.LayerGrads * n)()
    for i, gr in enumerate(grads):
        for name in _GRAD_FIELDS:
            t = gr[name]
            assert t.dtype == torch.float32 and t.is_contiguous()
            setattr(G[i], name, t.data_ptr())
    s.grads = G
    s.dout = dout.data_ptr()
    dx = torch.empty((s.n_tok, s.hidden), dtype=BF16, device=dout.device) if need_dx else None
    s.dx = None if dx is None else dx.data_ptr()
    nbytes = _lib.lib().hero_bert_stack_bwd_scratch_bytes(s.n_tok, s.hidden, s.inter)
    scratch = torch.empty(nbytes, dtype=torch.uint8, device=x.device)
    s.scratch = scratch.data_ptr()
    _count(_STACK_BWD_LAUNCHES * n)
    _lib.check(_lib.lib().hero_bert_stack_bwd(C.byref(s), _stream()))
    return dx


def cast_bf16(src, dst):
    """dst (bf16, same numel) = src (fp32)."""
    _require_cuda(src, dst)
    assert src.dtype == torch.float32 and dst.dtype == BF16 and src.is_contiguous()
    assert dst.is_contiguous() and src.numel() == dst.numel()
    _count()
    _lib.check(_lib.lib().hero_cast_f32_to_bf16(_ptr(src), _ptr(dst), src.numel(), _stream()))
    return dst


def gather_rows(src, idx, dst):
    """dst[i] = idx[i] >= 0 ? src[idx[i]] : 0 over bf16 rows, or over fp32 rows (both fp32)."""
    _require_cuda(src, idx, dst)
    assert src.dtype == dst.dtype and src.dtype in (BF16, torch.float32)
    assert idx.dtype == torch.int32 and src.is_contiguous() and dst.is_contiguous()
    h = src.shape[-1]
    _count()
    fn = (_lib.lib().hero_gather_rows_f32 if src.dtype == torch.float32
          else _lib.lib().hero_gather_rows_bf16)
    _lib.check(fn(_ptr(src), _ptr(idx), _ptr(dst), idx.numel(), h, _stream()))
    return dst


def gather_sum_rows(src, off, idx, dst):
    """dst[i] = sum_{e in off[i]:off[i+1]} src[idx[e]]; dst bf16 (overwrite) or f32 (accumulate)."""
    _require_cuda(src, off, idx, dst)
    assert src.dtype == BF16 and off.dtype == torch.int32 and idx.dtype == torch.int32
    n, h = off.numel() - 1, src.shape[-1]
    fn = (_lib.lib().hero_gather_sum_rows_f32 if dst.dtype == torch.float32
          else _lib.lib().hero_gather_sum_rows_bf16)
    _count()
    _lib.check(fn(_ptr(src), _ptr(off), _ptr(idx), _ptr(dst), n, h, _stream()))
    return dst


def colsum(x, out):
    """out[n] += sum_m x[m, n]  (x bf16 2-D, out fp32)."""
    _require_cuda(x, out)
    assert x.dtype == BF16 and out.dtype == torch.float32 and x.dim() == 2
    _count()
    _lib.check(_lib.lib().hero_colsum_bf16(_ptr(x), x.stride(0), x.shape[0], x.shape[1],
                                           _ptr(out), _stream()))
    return out


def relu_bwd(dy, pre, out):
    _require_cuda(dy, pre, out)
    _count()
    _lib.check(_lib.lib().hero_relu_bwd_bf16(_ptr(dy), _ptr(pre), _ptr(out), dy.numel(),
                                             _stream()))
    return out


def adamw_step(p, g, m, v, p_bf16, *, step_size, beta1, beta2, eps, lr_wd, grad_scale=1.0,
               clip_sumsq=None, clip_max_norm=0.0):
    """`clip_sumsq`: device scalar holding sum(g^2) over ALL gradients (ops.sumsq); the kernel then
    scales g by min(1, clip_max_norm / (sqrt(sumsq) + 1e-6)) — global-norm clipping without a
    device->host read."""
    _require_cuda(p, g, m, v)
    _count()
    _lib.check(_lib.lib().hero_adamw_step(_ptr(p), _ptr(g), _ptr(m), _ptr(v), _ptr(p_bf16),
                                          p.numel(), step_size, beta1, beta2, eps, lr_wd,
                                          grad_scale, _ptr(clip_sumsq), clip_max_norm, _stream()))


def sumsq(x, out):
    _require_cuda(x, out)
    _count()
    _lib.check(_lib.lib().hero_sumsq_f32(_ptr(x), x.numel(), _ptr(out), _stream()))
    return out


# ---------------------------------------------------------------------------------------------
# VSM / moment-retrieval head (hero_b200/csrc/vsm.cu)
def l2norm_split(x, hi, lo, inv, eps=1e-5):
    """Rows of x (fp32 [R, d]) L2-normalised (F.normalize, eps clamp) into split-bf16 halves;
    inv[r] = 1 / max(|x_r|, eps) (negative where clamped). hi / lo may have more rows than x."""
    _require_cuda(x, hi, lo, inv)
    assert x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 2
    assert hi.dtype == BF16 and lo.dtype == BF16 and hi.shape[1] == x.shape[1]
    _count()
    _lib.check(_lib.lib().hero_l2norm_split_f32(_ptr(x), x.shape[0], x.shape[1], eps, _ptr(hi),
                                                _ptr(lo), _ptr(inv), _stream()))


def vsm_masked_max(s, mask_u8, nq, nv, length, scores, argmax):
    _require_cuda(s, mask_u8, scores, argmax)
    assert s.dtype == torch.float32 and mask_u8.dtype == torch.uint8 and argmax.dtype == torch.int32
    _count()
    _lib.check(_lib.lib().hero_vsm_masked_max(_ptr(s), s.stride(0), _ptr(mask_u8), nq, nv, length,
                                              _ptr(scores), _ptr(argmax), _stream()))


def vsm_scores_bwd(g, argmax, mask_u8, q_hi, q_lo, q_inv, c_hi, c_lo, c_inv, nq, nv, length, d,
                   dq, dctx):
    _require_cuda(g, argmax, mask_u8)
    assert g.dtype == torch.float32 and g.is_contiguous()
    _count(2)
    _lib.check(_lib.lib().hero_vsm_scores_bwd(_ptr(g), _ptr(argmax), _ptr(mask_u8), _ptr(q_hi),
                                              _ptr(q_lo), _ptr(q_inv), _ptr(c_hi), _ptr(c_lo),
                                              _ptr(c_inv), nq, nv, length, d, _ptr(dq), _ptr(dctx),
                                              _stream()))


def vsm_span_fwd(query, ctx, mask_u8, w_st, w_ed, sim, st, ed):
    _require_cuda(query, ctx, mask_u8, sim, st, ed)
    n, length, d = ctx.shape
    for t in (query, ctx, w_st, w_ed):
        assert t.dtype == torch.float32 and t.is_contiguous()
    _count()
    _lib.check(_lib.lib().hero_vsm_span_fwd(_ptr(query), _ptr(ctx), _ptr(mask_u8), _ptr(w_st),
                                            _ptr(w_ed), n, length, d, w_st.numel(), _ptr(sim),
                                            _ptr(st), _ptr(ed), _stream()))


def vsm_span_bwd(dst, ded, mask_u8, w_st, w_ed, sim, query, ctx, dquery, dctx, dw_st, dw_ed):
    _require_cuda(dst, ded, query, ctx)
    n, length, d = ctx.shape
    for t in (dst, ded, sim, query, ctx, w_st, w_ed):
        assert t.dtype == torch.float32 and t.is_contiguous()
    _count()
    _lib.check(_lib.lib().hero_vsm_span_bwd(_ptr(dst), _ptr(ded), _ptr(mask_u8), _ptr(w_st),
                                            _ptr(w_ed), _ptr(sim), _ptr(query), _ptr(ctx), n, length,
                                            d, w_st.numel(), _ptr(dquery), _ptr(dctx), _ptr(dw_st),
                                            _ptr(dw_ed), _stream()))


# ---------------------------------------------------------------------------------------------
# Video QA head (hero_b200/csrc/videoqa.cu)
def videoqa_pool_fwd(y, frame_tok, w_se, w_qa, nv, nq, t):
    """Modularized-video pooling (model/videoQA.py:36-59) over the frame rows of the packed fp32
    stack output y [n_joint, H]. Returns (p_se [nv, t, H], p_qa [nv, nq, H], a_se, a_qa), the a_*
    being the two softmax probability tensors [nv, nq, t] the backward needs."""
    _require_cuda(y, frame_tok, w_se, w_qa)
    for x in (y, w_se, w_qa):
        assert x.dtype == torch.float32 and x.is_contiguous()
    assert frame_tok.dtype == torch.int32 and frame_tok.numel() == nv * nq * t
    h = y.shape[1]
    s = torch.empty((4, nv, nq, t), dtype=torch.float32, device=y.device)
    p_se = torch.empty((nv, t, h), dtype=torch.float32, device=y.device)
    p_qa = torch.empty((nv, nq, h), dtype=torch.float32, device=y.device)
    _count(2)
    _lib.check(_lib.lib().hero_videoqa_pool_fwd(_ptr(y), _ptr(frame_tok), _ptr(w_se), _ptr(w_qa),
                                                nv, nq, t, h, _ptr(s[0]), _ptr(s[1]), _ptr(s[2]),
                                                _ptr(s[3]), _ptr(p_se), _ptr(p_qa), _stream()))
    return p_se, p_qa, s[2], s[3]


def videoqa_pool_bwd(y, frame_tok, w_se, w_qa, a_se, a_qa, dp_se, dp_qa, nv, nq, t, dy, dw_se,
                     dw_qa):
    """dy (fp32 [n_joint, H]) is OVERWRITTEN at the frame rows only; dw_se / dw_qa (fp32 [H]) are
    accumulated."""
    _require_cuda(y, frame_tok, dp_se, dp_qa, dy, dw_se, dw_qa)
    for x in (y, w_se, w_qa, a_se, a_qa, dp_se, dp_qa, dy, dw_se, dw_qa):
        assert x.dtype == torch.float32 and x.is_contiguous()
    da = torch.empty((2, nv, nq, t), dtype=torch.float32, device=y.device)
    _count(2)
    _lib.check(_lib.lib().hero_videoqa_pool_bwd(_ptr(y), _ptr(frame_tok), _ptr(w_se), _ptr(w_qa),
                                                _ptr(a_se), _ptr(a_qa), _ptr(dp_se), _ptr(dp_qa),
                                                nv, nq, t, y.shape[1], _ptr(da[0]), _ptr(da[1]),
                                                _ptr(dy), _ptr(dw_se), _ptr(dw_qa), _stream()))


# ---------------------------------------------------------------------------------------------
# Fused LM-head cross entropy (MLM): vocabulary logits are never materialised in fp32.
def lm_head_ce_fwd(h, emb, bias, labels, n_valid):
    """h: bf16 [n, H] (LM-head transform of the masked tokens), emb: bf16 [V, H] (tied word
    embedding), bias: fp32 [V], labels: int32 [n]. Returns (loss fp32 [n], lse fp32 [n]) of
    F.cross_entropy(h @ emb.T + bias, labels, reduction='none') over the first n_valid columns."""
    _require_cuda(h, emb, bias, labels)
    assert h.dtype == BF16 and emb.dtype == BF16 and labels.dtype == torch.int32
    n, V = h.shape[0], emb.shape[0]
    n_slabs = (V + 63) // 64
    ld = (n + 7) // 8 * 8
    partial = torch.empty((n_slabs, ld, 2), dtype=torch.float32, device=h.device)
    lab = torch.empty(n, dtype=torch.float32, device=h.device)
    g = _lib.GemmArgs()
    g.a, g.b = _ptr(h), _ptr(emb)
    g.lda, g.ldb = h.stride(0), emb.stride(0)
    g.m, g.n, g.k = n, V, h.shape[1]
    g.bias = _ptr(bias)
    g.act = ACT_CE
    g.drop_scale = 1.0
    g.ce_label, g.ce_partial, g.ce_label_logit = _ptr(labels), _ptr(partial), _ptr(lab)
    g.ce_ld_partial, g.ce_n_valid = ld, n_valid
    _count(2)
    _lib.check(_lib.lib().hero_gemm_bf16(C.byref(g), _stream()))
    loss = torch.empty(n, dtype=torch.float32, device=h.device)
    lse = torch.empty(n, dtype=torch.float32, device=h.device)
    _lib.check(_lib.lib().hero_ce_finish(_ptr(partial), ld, n_slabs, _ptr(lab), n, _ptr(loss),
                                         _ptr(lse), _stream()))
    return loss, lse


def lm_head_ce_dlogits(h, emb, bias, labels, lse, grad, n_valid, out):
    """out[:, :V] (bf16, row stride a multiple of 64) = grad[r] * (softmax(logits)[r] - onehot)."""
    _require_cuda(h, emb, out)
    n, V = h.shape[0], emb.shape[0]
    assert out.dtype == BF16 and out.stride(0) % 64 == 0 and out.shape[1] >= V
    assert lse.dtype == torch.float32 and grad.dtype == torch.float32 and grad.is_contiguous()
    g = _lib.GemmArgs()
    g.a, g.b = _ptr(h), _ptr(emb)
    g.lda, g.ldb = h.stride(0), emb.stride(0)
    g.m, g.n, g.k = n, V, h.shape[1]
    g.bias = _ptr(bias)
    g.act = ACT_CE_GRAD
    g.drop_scale = 1.0
    g.out, g.ld_out = _ptr(out), out.stride(0)
    g.ce_label, g.ce_lse, g.ce_grad, g.ce_n_valid = _ptr(labels), _ptr(lse), _ptr(grad), n_valid
    _count()
    _lib.check(_lib.lib().hero_gemm_bf16(C.byref(g), _stream()))
    return out
