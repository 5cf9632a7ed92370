"""Host-side packing plans: padded reference batch layout -> packed (valid-token-only) layout.

The reference pads every subtitle row to the batch maximum and masks padded keys with -10000
(model/layers.py:299-302); it also re-packs `[frames | pad | text | pad]` into `[frames, text,
pad]` with torch.gather (model/encoder.py:271-279, index from data/data.py:504-512) and scatters
frame outputs back to the clip timeline in a Python double loop (model/model.py:156-187). Here all
of that becomes index arithmetic done ONCE per batch on the host with numpy; the CUDA kernels then
only ever see valid tokens:

    SeqPlan   which (row, position) pairs are valid, in row-major order -> packed token ids,
              cu_seqlens for the attention kernel, maps for pack / unpack.
    FPlan     cross-modal rows: per packed token its source (frame slot or text slot).
    CPlan     clip rows + the CSR maps replacing collect_frame_outputs (forward gather-sum and its
              transpose for the backward).

Plans are pure numpy (testable without a GPU); `.to(device)` uploads the int32 index arrays in
one pinned-memory copy.
"""
import numpy as np
import torch


ATTN_TILE = 128        # tokens per tensor-core attention tile
ATTN_TILE_SEQS = 16    # sequences per tile (one K = 16 membership step of the S MMA, csrc/attention_tc.cu)
ATTN_LONG_MAX = 768    # longest sequence the long-sequence kernels take (hero_attn_fwd)


def _np(t):
    if torch.is_tensor(t):
        return t.detach().cpu().numpy()
    return np.asarray(t)


def _max_vl_of(batch):
    """Padded number of frame slots per subtitle row: from the plan inputs, the frame features, or
    (batches without f_v_feats) the (1, max_vl) frame position ids of the collate."""
    if "_max_vl" in batch:
        return int(batch["_max_vl"])
    fv = batch.get("f_v_feats") if hasattr(batch, "get") else batch["f_v_feats"]
    if fv is not None:
        return int(fv.shape[1])
    return int(batch["f_v_pos_ids"].shape[-1])


def _host_ids(t):
    """Small id tensor -> host int64 array [rows, L], or None if absent / not on the host."""
    if t is None or (torch.is_tensor(t) and t.device.type != "cpu"):
        return None
    a = np.asarray(_np(t), np.int64)
    return a.reshape(1, -1) if a.ndim == 1 else a


class DeviceIndex:
    """A bundle of int32 index arrays uploaded to the device with a single H2D copy.

    `staging(n)` (optional) returns a reusable (pinned host, device) pair of int32 buffers with at
    least n elements. Without it every upload allocates pinned memory; under load the caching host
    allocator cannot recycle blocks whose copies are still in flight and falls back to
    cudaHostAlloc — tens of milliseconds and a device synchronisation per call (measured: 30-50 ms
    holes in the step timeline). loader.BatchStager passes its per-slot buffers."""

    def __init__(self, arrays, device, staging=None):
        names = list(arrays)
        sizes = [int(arrays[n].size) for n in names]
        offs = np.concatenate([[0], np.cumsum([(s + 3) // 4 * 4 for s in sizes])]).astype(np.int64)
        total = int(offs[-1])
        if staging is not None:
            host_buf, dev_buf = staging(total)
            host, dst = host_buf[:total], dev_buf[:total]
        else:
            host = torch.empty(total, dtype=torch.int32,
                               pin_memory=torch.cuda.is_available() and device.type == "cuda")
            dst = None
        hv = host.numpy()
        for n, o, s in zip(names, offs[:-1], sizes):
            hv[o:o + s] = arrays[n].reshape(-1)
        if dst is None:
            self.flat = host.to(device, non_blocking=True)
        else:
            dst.copy_(host, non_blocking=True)
            self.flat = dst
        self._host = host  # keep pinned memory alive until the copy is consumed
        for n, o, s in zip(names, offs[:-1], sizes):
            setattr(self, n, self.flat[o:o + s])


class SeqPlan:
    """Valid positions of a padded (rows, length) mask, packed row-major."""

    def __init__(self, mask):
        mask = _np(mask) != 0
        self.rows, self.length = mask.shape
        r, c = np.nonzero(mask)                      # row-major order
        self.tok_row = r.astype(np.int32)
        self.tok_col = c.astype(np.int32)
        self.n_tok = int(r.size)
        lens = mask.sum(1).astype(np.int64)
        self.lens = lens
        self.cu = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
        self.n_seq = self.rows
        self.max_len = int(lens.max()) if lens.size else 0
        self.tok_flat = (r.astype(np.int64) * self.length + c).astype(np.int32)  # packed -> padded
        p2t = np.full(self.rows * self.length, -1, np.int32)
        p2t[self.tok_flat] = np.arange(self.n_tok, dtype=np.int32)
        self.pad_to_tok = p2t                                                    # padded -> packed
        # attention tiling: consecutive sequences packed into tiles of <= 128 tokens and <= 16
        # sequences (a sequence never straddles tiles); per token the [lo, hi) range of its own
        # sequence. Sequences
        # longer than one tile (up to ATTN_LONG_MAX tokens; the reference's position table allows
        # 514, model/encoder.py:50) become tiles of their own at the END of the list: the library
        # runs those `n_long` tiles on its long-sequence kernels (hero_attn_fwd).
        if self.max_len > ATTN_LONG_MAX:
            row = int(np.argmax(lens))
            raise ValueError(f"row {row} has {self.max_len} valid tokens; the attention kernels "
                             f"support sequences of up to {ATTN_LONG_MAX} tokens")
        self.seq_lo = np.repeat(self.cu[:-1], lens).astype(np.int32)
        self.seq_hi = np.repeat(self.cu[1:], lens).astype(np.int32)
        t0, tn, l0, ln = [], [], [], []
        start, cur, nseq = 0, 0, 0
        pos = 0
        for n in lens.tolist():
            if n == 0:
                continue
            if n > ATTN_TILE:
                if cur:
                    t0.append(start)
                    tn.append(cur)
                l0.append(pos)
                ln.append(n)
                pos += n
                start, cur, nseq = pos, 0, 0
                continue
            if cur + n > ATTN_TILE or nseq == ATTN_TILE_SEQS:
                t0.append(start)
                tn.append(cur)
                start, cur, nseq = start + cur, 0, 0
            cur += n
            nseq += 1
            pos += n
        if cur:
            t0.append(start)
            tn.append(cur)
        self.n_long = len(l0)
        self.max_long = max(ln) if ln else 0
        self.short_tok0, self.short_ntok = np.asarray(t0, np.int32), np.asarray(tn, np.int32)
        self.long_tok0, self.long_ntok = np.asarray(l0, np.int32), np.asarray(ln, np.int32)
        self.tile_tok0 = np.concatenate([self.short_tok0, self.long_tok0]).astype(np.int32)
        self.tile_ntok = np.concatenate([self.short_ntok, self.long_ntok]).astype(np.int32)
        self.n_tiles = len(t0) + len(l0)

    def arrays(self, prefix):
        return {prefix + "cu": self.cu, prefix + "tok_flat": self.tok_flat,
                prefix + "pad_to_tok": self.pad_to_tok, prefix + "seq_lo": self.seq_lo,
                prefix + "seq_hi": self.seq_hi, prefix + "tile_tok0": self.tile_tok0,
                prefix + "tile_ntok": self.tile_ntok}

    def attn(self, dev, prefix):
        """Device-side attention plan consumed by ops.attn_fwd / attn_bwd."""
        return {"cu": getattr(dev, prefix + "cu"), "seq_lo": getattr(dev, prefix + "seq_lo"),
                "seq_hi": getattr(dev, prefix + "seq_hi"),
                "tile_tok0": getattr(dev, prefix + "tile_tok0"),
                "tile_ntok": getattr(dev, prefix + "tile_ntok"), "n_tiles": self.n_tiles,
                "n_long": self.n_long, "max_long": self.max_long,
                "n_tok": self.n_tok, "n_seq": self.n_seq, "max_len": self.max_len}


def _csr(dst, src, n_dst):
    """CSR (offsets, indices) listing for each dst all its src, stable in src order."""
    dst = np.asarray(dst, np.int64)
    src = np.asarray(src, np.int32)
    order = np.argsort(dst, kind="stable")
    counts = np.bincount(dst, minlength=n_dst)
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    return off, src[order]


class FPlan:
    """Cross-modal ('repr') rows: frames + subtitle tokens per row, or text-only rows ('txt')."""

    def __init__(self, attn_mask, gather_index=None, max_vl=0, max_sl=None):
        self.seq = SeqPlan(attn_mask)
        s = self.seq
        if gather_index is None:       # text only: position j reads text slot j
            src = s.tok_col.astype(np.int64)
            max_vl = 0
            self.max_sl = s.length if max_sl is None else max_sl
        else:
            gi = _np(gather_index).astype(np.int64)
            src = gi[s.tok_row, s.tok_col]
            self.max_sl = int(max_sl)
        self.max_vl = int(max_vl)
        is_img = src < self.max_vl
        tok = np.arange(s.n_tok, dtype=np.int32)
        self.img_tok = tok[is_img]
        self.img_k = src[is_img].astype(np.int32)                       # frame slot in the row
        self.img_src = (s.tok_row[is_img].astype(np.int64) * self.max_vl
                        + src[is_img]).astype(np.int32)                 # row in f_v_feats.view(-1, D)
        self.txt_tok = tok[~is_img]
        self.txt_j = (src[~is_img] - self.max_vl).astype(np.int32)
        self.txt_src = (s.tok_row[~is_img].astype(np.int64) * self.max_sl
                        + self.txt_j).astype(np.int32)                  # index in input_ids.view(-1)
        self.n_img = int(self.img_tok.size)
        self.n_txt = int(self.txt_tok.size)

    def arrays(self, prefix="f_"):
        a = self.seq.arrays(prefix)
        a.update({prefix + "img_tok": self.img_tok, prefix + "img_k": self.img_k,
                  prefix + "img_src": self.img_src, prefix + "txt_tok": self.txt_tok,
                  prefix + "txt_j": self.txt_j, prefix + "txt_src": self.txt_src})
        for name in ("txt_ids", "txt_pos", "img_kpos"):
            v = getattr(self, name, None)
            if v is not None:
                a[prefix + name] = v
        return a

    def gather_ids(self, input_ids=None, pos_ids=None, img_pos_ids=None):
        """Per packed token: its vocabulary id, text position id and frame position id, gathered
        HERE on the host (collate side) when the id tensors are host tensors, so the forward
        does not spend ~15 small index kernels on them. All optional: what is missing is gathered
        on the device as before."""
        ids, pos, ipos = _host_ids(input_ids), _host_ids(pos_ids), _host_ids(img_pos_ids)
        self.txt_ids = self.txt_pos = self.img_kpos = None
        if ids is not None and self.n_txt:
            self.txt_ids = ids.reshape(-1)[self.txt_src].astype(np.int32)
        if pos is not None and self.n_txt:
            if pos.shape[0] == 1:
                self.txt_pos = pos[0][self.txt_j].astype(np.int32)
            elif ids is not None and pos.shape == ids.shape:
                self.txt_pos = pos.reshape(-1)[self.txt_src].astype(np.int32)
        if ipos is not None and self.n_img:
            self.img_kpos = ipos.reshape(-1)[self.img_k].astype(np.int32)


class CPlan:
    """Clip-level rows and the frame-merge maps (collect_frame_outputs as CSR gathers)."""

    def __init__(self, c_attn_mask, fplan, num_subs, sub_idx2frame_idx):
        self.seq = SeqPlan(c_attn_mask)
        s = self.seq
        B, T = s.rows, s.length
        self.c_src = s.tok_flat                       # row in c_v_feats.view(-1, D)
        self.c_t = s.tok_col                          # temporal position id
        # (clip, frame) <- (sub row, slot k): model/model.py:171-186
        rows, ks, dst = [], [], []
        start = 0
        for vid, n_sub in enumerate(num_subs):
            for sid, frames in sub_idx2frame_idx[vid]:
                n = len(frames)
                if n:
                    rows.extend([start + sid] * n)
                    ks.extend(range(n))
                    dst.extend(vid * T + int(t) for t in frames)
            start += n_sub
        rows = np.asarray(rows, np.int64)
        ks = np.asarray(ks, np.int64)
        dst = np.asarray(dst, np.int64)
        if dst.size and (dst.max() >= B * T or dst.min() < 0):
            raise IndexError("sub_idx2frame_idx refers to a frame outside the clip tensor")
        # (sub row, slot) -> row of c_v_feats.view(-1, D); -1 where the slot holds no clip frame
        self.frame_source = np.full(fplan.seq.rows * max(fplan.max_vl, 1), -1, np.int32)
        if rows.size:
            self.frame_source[rows * fplan.max_vl + ks] = dst
        f_tok = fplan.seq.pad_to_tok[rows * fplan.seq.length + ks] if rows.size else \
            np.zeros(0, np.int32)
        c_tok = s.pad_to_tok[dst] if dst.size else np.zeros(0, np.int32)
        keep = (f_tok >= 0) & (c_tok >= 0)            # masked slots carry no defined value
        f_tok, c_tok = f_tok[keep], c_tok[keep]
        self.n_pairs = int(f_tok.size)
        self.fwd_off, self.fwd_idx = _csr(c_tok, f_tok, s.n_tok)             # c token <- f tokens
        self.bwd_off, self.bwd_idx = _csr(f_tok, c_tok, fplan.seq.n_tok)     # f token <- c tokens

    def arrays(self, prefix="c_"):
        a = self.seq.arrays(prefix)
        a.update({prefix + "src": self.c_src, prefix + "t": self.c_t,
                  prefix + "fwd_off": self.fwd_off, prefix + "fwd_idx": self.fwd_idx,
                  prefix + "bwd_off": self.bwd_off, prefix + "bwd_idx": self.bwd_idx})
        return a


def table_csr(idx, n_rows):
    """CSR listing, for every embedding-table row, the packed tokens that used it (deterministic
    table gradients via gather-sum instead of contended atomics)."""
    idx = np.asarray(idx, np.int64)
    return _csr(idx, np.arange(idx.size, dtype=np.int32), n_rows)


class ReprPlan:
    """Everything HierarchicalVlModel.forward_repr needs for one batch."""

    def __init__(self, batch):
        # `plan_inputs` dicts carry the two padded lengths instead of the big tensors
        max_vl = _max_vl_of(batch)
        max_sl = batch["_max_sl"] if "_max_sl" in batch else batch["f_sub_input_ids"].shape[1]
        self.f = FPlan(batch["f_attn_masks"], batch["f_gather_index"], max_vl, max_sl)
        self.c = CPlan(batch["c_attn_masks"], self.f, batch["num_subs"],
                       batch["sub_idx2frame_idx"])
        # Every frame slot of a subtitle row is a copy of a clip frame (data/data.py:380-395 fills
        # f_v_feats with index_select(c_v_feats, frames)): row of c_v_feats.view(-1, D) behind each
        # packed frame token, so a batch may omit `f_v_feats` altogether (half the H2D bytes).
        self.f.img_src_c = self.c.frame_source[self.f.img_src] if self.f.n_img else \
            np.zeros(0, np.int32)
        # a frame slot that is valid in f_attn_masks but not listed in sub_idx2frame_idx has no
        # clip frame behind it: such a batch must ship its own f_v_feats (checked on the host, the
        # LayerNorm kernels index x_rows without a sign test)
        self.f.shared_feats_ok = self.shared_feats_ok = bool((self.f.img_src_c >= 0).all())
        self.shape_f = tuple(batch["f_attn_masks"].shape)
        self.shape_c = tuple(batch["c_attn_masks"].shape)
        # position-table CSRs for the deterministic embedding gradients
        self.f_txtpos_off, self.f_txtpos_idx = table_csr(self.f.txt_j, max(max_sl, 1))
        self.f_imgpos_off, self.f_imgpos_idx = table_csr(self.f.img_k, max(max_vl, 1))
        self.c_pos_off, self.c_pos_idx = table_csr(self.c.c_t, max(self.shape_c[1], 1))
        # subtitle position ids as the collate made them (lets JointPlan decide on the host
        # whether video and query rows share one slot -> position table)
        get = batch.get if hasattr(batch, "get") else (lambda k: None)
        self.sub_pos = _host_ids(get("f_sub_pos_ids"))
        self.f.gather_ids(get("f_sub_input_ids"), get("f_sub_pos_ids"), get("f_v_pos_ids"))
        self.dev = None

    def to(self, device, staging=None):
        if self.dev is None or self.dev.flat.device != torch.device(device):
            a = self.f.arrays("f_")
            a["f_img_src_c"] = self.f.img_src_c
            a.update(self.c.arrays("c_"))
            a.update({"f_txtpos_off": self.f_txtpos_off, "f_txtpos_idx": self.f_txtpos_idx,
                      "f_imgpos_off": self.f_imgpos_off, "f_imgpos_idx": self.f_imgpos_idx,
                      "c_pos_off": self.c_pos_off, "c_pos_idx": self.c_pos_idx})
            self.dev = DeviceIndex(a, torch.device(device), staging)
        return self.dev


class TxtPlan:
    """Text-only rows (CrossModalTrm 'txt' task, and the generic BertEncoder API)."""

    def __init__(self, attn_mask, with_embedding=True, pos_ids=None, input_ids=None):
        self.f = FPlan(attn_mask)
        self.shape = tuple(_np(attn_mask).shape)
        self.with_embedding = with_embedding
        self.pos = _host_ids(pos_ids)
        if with_embedding:
            self.f.gather_ids(input_ids, pos_ids)
        if with_embedding:
            self.pos_off, self.pos_idx = table_csr(self.f.txt_j, max(self.shape[1], 1))
        self.dev = None

    def to(self, device, staging=None):
        if self.dev is None or self.dev.flat.device != torch.device(device):
            a = self.f.arrays("f_")
            if self.with_embedding:
                a.update({"pos_off": self.pos_off, "pos_idx": self.pos_idx})
            self.dev = DeviceIndex(a, torch.device(device), staging)
        return self.dev


class JointPlan:
    """Video rows ('repr') and text-only query rows ('txt') of the SAME CrossModalTrm concatenated
    into one packed token stream, so both go through the 6 layers as one set of GEMMs (32 query
    rows x 16 tokens alone would run every GEMM at M = 512, ~10 % tensor utilisation).
    Query tokens follow the video tokens: packed index = n_video_tokens + query index."""

    def __init__(self, rplan, tplan):
        self.r, self.t = rplan, tplan
        fv, fq = rplan.f, tplan.f
        a = fv.seq.n_tok
        self.n_video_tok = a
        self.n_tok = a + fq.seq.n_tok
        self.n_txt = fv.n_txt + fq.n_txt
        self.n_img = fv.n_img
        self.max_vl, self.max_sl_v, self.max_sl_q = fv.max_vl, fv.max_sl, fq.max_sl
        sv, sq = fv.seq, fq.seq
        self.n_seq = sv.n_seq + sq.n_seq
        self.max_len = max(sv.max_len, sq.max_len)
        self.n_tiles = sv.n_tiles + sq.n_tiles
        # long-sequence tiles (rare) of both row kinds go last, after every 128-token tile
        self.n_long = sv.n_long + sq.n_long
        self.max_long = max(sv.max_long, sq.max_long)
        self.arr = {
            "j_cu": np.concatenate([sv.cu, sq.cu[1:] + a]).astype(np.int32),
            "j_seq_lo": np.concatenate([sv.seq_lo, sq.seq_lo + a]).astype(np.int32),
            "j_seq_hi": np.concatenate([sv.seq_hi, sq.seq_hi + a]).astype(np.int32),
            "j_tile_tok0": np.concatenate([sv.short_tok0, sq.short_tok0 + a, sv.long_tok0,
                                           sq.long_tok0 + a]).astype(np.int32),
            "j_tile_ntok": np.concatenate([sv.short_ntok, sq.short_ntok, sv.long_ntok,
                                           sq.long_ntok]).astype(np.int32),
            "j_txt_tok": np.concatenate([fv.txt_tok, fq.txt_tok + a]).astype(np.int32),
            "j_txt_j": np.concatenate([fv.txt_j, fq.txt_j]).astype(np.int32),
        }
        n_slot = max(fv.max_sl, fq.max_sl, 1)
        self.arr["j_txtpos_off"], self.arr["j_txtpos_idx"] = table_csr(self.arr["j_txt_j"], n_slot)
        for name in ("txt_ids", "txt_pos"):      # host-gathered ids of both row kinds, if known
            a_v, a_q = getattr(fv, name, None), getattr(fq, name, None)
            if (a_v is not None or fv.n_txt == 0) and a_q is not None:
                parts = ([a_v] if fv.n_txt else []) + [a_q]
                self.arr["j_" + name] = np.concatenate(parts).astype(np.int32)
        # Do both row kinds use the same slot -> position map (the collate's arange)? Decided here
        # on the host when the plans saw the position ids; None = unknown (the encoder then has
        # to compare the device tensors, which costs a device sync per step).
        self.same_slot_pos = None
        pv, pq = getattr(rplan, "sub_pos", None), getattr(tplan, "pos", None)
        if pv is not None and pq is not None and pv.shape[0] == 1 and pq.shape[0] == 1:
            n = min(pv.shape[1], pq.shape[1])
            self.same_slot_pos = bool(np.array_equal(pv[0, :n], pq[0, :n]))
        self.dev = None

    def to(self, device, staging=None):
        device = torch.device(device)
        if self.dev is None or self.dev.flat.device != device:
            self.dev = DeviceIndex(self.arr, device, staging)
        return self.dev

    def attn(self, dev):
        return {"cu": dev.j_cu, "seq_lo": dev.j_seq_lo, "seq_hi": dev.j_seq_hi,
                "tile_tok0": dev.j_tile_tok0, "tile_ntok": dev.j_tile_ntok,
                "n_tiles": self.n_tiles, "n_long": self.n_long, "max_long": self.max_long,
                "n_tok": self.n_tok, "n_seq": self.n_seq, "max_len": self.max_len}


class VideoQaPlan:
    """Query-fused temporal stage of the video QA head (model/videoQA.py:66-82): per (question,
    answer candidate) row r = v * Nq + q the joint sequence is the row's valid clip frames followed
    by its valid QA tokens, i.e. a SeqPlan over cat(c_attn_masks, qa_attn_masks, dim=1) (row-major
    packing). Rows over 128 tokens (T = 100 frames + 30 QA tokens) take SeqPlan's long-sequence
    tiles.
        c_row     per clip token (CPlan order): its joint row (scatter target of the frame half)
        qa_row    per QA token: its joint row; qa_ids / qa_pos: its vocabulary / position id
        frame_tok [Nv, Nq, T]: joint row of frame t of candidate q of question v, -1 if padded
    `cplan` is the CPlan of the same batch (ReprPlan.c)."""

    def __init__(self, c_attn_masks, qa_attn_masks, qa_input_ids, qa_pos_ids, n_questions, cplan):
        cm, qm = _np(c_attn_masks) != 0, _np(qa_attn_masks) != 0
        rows, T = cm.shape
        L = qm.shape[1]
        if qm.shape[0] != rows:
            raise ValueError(f"{qm.shape[0]} QA rows for {rows} clip rows")
        self.nv = int(n_questions)
        if self.nv <= 0 or rows % self.nv:
            raise ValueError(f"{rows} (question, answer) rows are not a multiple of {self.nv} "
                             "questions")
        self.nq, self.t = rows // self.nv, T
        self.seq = SeqPlan(np.concatenate([cm, qm], axis=1))
        W = T + L
        p2t = self.seq.pad_to_tok
        self.c_row = p2t[cplan.seq.tok_row.astype(np.int64) * W + cplan.seq.tok_col]
        qr, qc = np.nonzero(qm)
        self.qa_row = p2t[qr.astype(np.int64) * W + T + qc]
        self.n_qa = int(qr.size)
        self.n_frame = int(self.c_row.size)
        ids = np.asarray(_np(qa_input_ids), np.int64)     # device tensors: read back (one sync)
        pos = np.asarray(_np(qa_pos_ids), np.int64).reshape(-1, L)
        self.qa_ids = ids[qr, qc].astype(np.int32)
        self.qa_pos = (pos[0][qc] if pos.shape[0] == 1 else pos[qr, qc]).astype(np.int32)
        # position-table CSR over ids 0 .. max id (deterministic table gradient)
        self.n_pos = int(self.qa_pos.max()) + 1 if self.n_qa else 1
        self.qa_pos_off, self.qa_pos_idx = table_csr(self.qa_pos, self.n_pos)
        self.frame_tok = np.where(cm, p2t.reshape(rows, W)[:, :T], -1).astype(np.int32)
        self.dev = None

    def to(self, device, staging=None):
        device = torch.device(device)
        if self.dev is None or self.dev.flat.device != device:
            a = self.seq.arrays("j_")
            a.update({"c_row": self.c_row, "qa_row": self.qa_row, "qa_ids": self.qa_ids,
                      "qa_pos": self.qa_pos, "qa_pos_off": self.qa_pos_off,
                      "qa_pos_idx": self.qa_pos_idx, "frame_tok": self.frame_tok})
            self.dev = DeviceIndex(a, device, staging)
        return self.dev


def videoqa_plans(batch):
    """(ReprPlan, VideoQaPlan) of a video QA batch (data/videoQA.py video_qa_collate layout)."""
    rplan = ReprPlan(batch)
    vplan = VideoQaPlan(batch["c_attn_masks"], batch["qa_attn_masks"], batch["qa_input_ids"],
                        batch["qa_pos_ids"], len(batch["targets"]), rplan.c)
    return rplan, vplan


PLAN_KEY = "_hero_plan"
_REPR_KEYS = ("f_attn_masks", "f_gather_index", "c_attn_masks", "num_subs", "sub_idx2frame_idx")


def plan_inputs(batch, kind="repr"):
    """The small, picklable part of a host batch that a plan is built from (masks and index
    lists as numpy arrays; none of the feature tensors) — what is shipped to a PlanPool worker."""
    def opt(key):
        v = batch.get(key) if hasattr(batch, "get") else None
        return None if v is None else _np(v)

    if kind != "repr":
        return {"attn_masks": _np(batch["attn_masks"]), "pos_ids": opt("pos_ids"),
                "input_ids": opt("input_ids")}
    d = {k: (_np(batch[k]) if torch.is_tensor(batch[k]) else batch[k]) for k in _REPR_KEYS}
    d["f_sub_pos_ids"] = opt("f_sub_pos_ids")
    d["f_sub_input_ids"] = opt("f_sub_input_ids")
    d["f_v_pos_ids"] = opt("f_v_pos_ids")
    d["_max_vl"] = _max_vl_of(batch)
    d["_max_sl"] = int(batch["f_sub_input_ids"].shape[1])
    return d


def build_plans(repr_in, txt_in=None):
    """ReprPlan (+ TxtPlan and the JointPlan of the fused video+query pass) from `plan_inputs`
    dicts. Pure numpy: runs in collate workers / PlanPool processes."""
    rplan = ReprPlan(repr_in)
    if txt_in is None:
        return rplan, None
    tplan = TxtPlan(txt_in["attn_masks"], pos_ids=txt_in.get("pos_ids"),
                    input_ids=txt_in.get("input_ids"))
    rplan.__dict__["_joint"] = JointPlan(rplan, tplan)
    return rplan, tplan


class PlanPool:
    """Builds plans in worker processes, the way the reference builds its gather indices inside
    DataLoader collate workers (data/data.py video_collate, model/model.py:189-193) — the training
    process only uploads the finished index arrays. `submit` returns a future whose `result()` is
    (ReprPlan, TxtPlan | None); `attach(future, batch, txt_batch)` stores them in the batch dicts."""

    def __init__(self, workers=2):
        import concurrent.futures as cf
        import multiprocessing as mp
        self._ex = cf.ProcessPoolExecutor(max_workers=workers, mp_context=mp.get_context("spawn"))

    def submit(self, batch, txt_batch=None):
        return self._ex.submit(build_plans, plan_inputs(batch),
                               None if txt_batch is None else plan_inputs(txt_batch, "txt"))

    @staticmethod
    def attach(future, batch, txt_batch=None):
        rplan, tplan = future.result()
        batch[PLAN_KEY] = rplan
        if txt_batch is not None:
            txt_batch[PLAN_KEY] = tplan
        return batch, txt_batch

    def shutdown(self):
        self._ex.shutdown(wait=False, cancel_futures=True)


QUERY_PLAN_KEY = "_hero_query_plan"
VIDEOQA_PLAN_KEY = "_hero_videoqa_plan"


def attach_plan(batch, kind="repr"):
    """Collate-side hook: build the plan from HOST tensors (no device sync later) and stash it in
    the batch dict; `move_to_cuda`-style helpers leave non-tensor values alone.
    kind: 'repr' (video batch), 'txt' (query batch), or 'vsm' — a VSM / VCMR training batch that
    carries its queries as `query_input_ids / query_pos_ids / query_attn_masks` (data/vcmr.py):
    attaches the video plan, the query plan (QUERY_PLAN_KEY) and their joint plan; or 'videoqa'
    — a TVQA / How2QA batch (data/videoQA.py): the video plan and the query-fused temporal plan
    (VIDEOQA_PLAN_KEY, see VideoQaPlan).
    The plan captures the batch's token / position ids per packed token (FPlan.gather_ids): attach
    it AFTER any masking of `input_ids` (the reference masks in the dataset, before collate), and
    attach again if the ids are edited afterwards."""
    if kind == "vsm":
        rplan = ReprPlan(batch)
        tplan = TxtPlan(batch["query_attn_masks"], pos_ids=batch.get("query_pos_ids"),
                        input_ids=batch.get("query_input_ids"))
        rplan.__dict__["_joint"] = JointPlan(rplan, tplan)
        batch[PLAN_KEY], batch[QUERY_PLAN_KEY] = rplan, tplan
        return batch
    if kind == "videoqa":
        batch[PLAN_KEY], batch[VIDEOQA_PLAN_KEY] = videoqa_plans(batch)
        return batch
    if kind == "repr":
        batch[PLAN_KEY] = ReprPlan(batch)
    else:
        get = batch.get if hasattr(batch, "get") else (lambda k: None)
        batch[PLAN_KEY] = TxtPlan(batch["attn_masks"], pos_ids=get("pos_ids"),
                                  input_ids=get("input_ids"))
    return batch
