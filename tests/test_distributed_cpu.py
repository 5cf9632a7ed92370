"""World-size-2 gloo tests of the data-parallel plumbing (hero_b200/distributed.py) — the N > 1
path of bench.py minus NCCL. Semantics follow utils/distributed.py and model/pretrain.py:427-447
of the reference (Horovod allreduce = mean over ranks; allgather concatenates in rank order)."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, fn_name, ret):
    os.environ.update({"RANK": str(rank), "WORLD_SIZE": str(world), "LOCAL_RANK": str(rank),
                       "MASTER_ADDR": "127.0.0.1", "MASTER_PORT": str(port)})
    import torch.distributed as dist
    from hero_b200 import distributed as hd
    hd.init(backend="gloo")
    try:
        ret[rank] = globals()[fn_name](rank, world, hd)
    finally:
        dist.destroy_process_group()


def _run(fn_name, world=2):
    port = _free_port()
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, port, fn_name, ret), nprocs=world, join=True)
    return dict(ret)


def _allreduce_case(rank, world, hd):
    # separate tensors (coalesced path) and views of one flat buffer (in-place path)
    a = torch.full((5,), float(rank + 1))
    b = torch.arange(6, dtype=torch.float32).view(2, 3) * (rank + 1)
    hd.all_reduce_and_rescale_tensors([a, b], 1.0)
    flat = torch.arange(128 + 64, dtype=torch.float32) * (rank + 1)
    v1, v2 = flat[:100].view(10, 10), flat[128:128 + 64]
    hd.all_reduce_and_rescale_tensors([v1, v2], 2.0)
    return a.tolist(), b.flatten().tolist(), flat.tolist()


def test_all_reduce_is_mean_over_ranks_and_rescales():
    out = _run("_allreduce_case")
    for r in (0, 1):
        a, b, flat = out[r]
        assert a == [1.5] * 5
        assert b == [x * 1.5 for x in range(6)]
        assert flat == [x * 1.5 / 2.0 for x in range(192)]


def _broadcast_case(rank, world, hd):
    t1 = torch.full((4,), float(rank + 10))
    t2 = torch.full((2, 2), float(rank + 20))
    hd.broadcast_tensors([t1, t2], 0)
    objs = hd.all_gather_list({"rank": rank, "n": rank * 3})
    task = hd.any_broadcast("task_%d" % rank, 1)
    return t1.tolist(), t2.flatten().tolist(), objs, task


def test_broadcast_gather_list_and_any_broadcast():
    out = _run("_broadcast_case")
    for r in (0, 1):
        t1, t2, objs, task = out[r]
        assert t1 == [10.0] * 4 and t2 == [20.0] * 4
        assert objs == [{"rank": 0, "n": 0}, {"rank": 1, "n": 3}]
        assert task == "task_1"


def _vsm_case(rank, world, hd):
    n = 2 + rank                       # ranks contribute different row counts
    x = (torch.arange(n * 3, dtype=torch.float32).view(n, 3) + 100 * rank).requires_grad_(True)
    y = hd.vsm_allgather(x)
    w = torch.arange(y.numel(), dtype=torch.float32).view_as(y)
    (y * w).sum().backward()
    return y.detach().tolist(), x.grad.tolist()


def test_vsm_allgather_forward_concat_backward_own_slice():
    out = _run("_vsm_case")
    full = [[0, 1, 2], [3, 4, 5], [100, 101, 102], [103, 104, 105], [106, 107, 108]]
    w = torch.arange(15, dtype=torch.float32).view(5, 3)
    for r in (0, 1):
        y, g = out[r]
        assert y == [[float(v) for v in row] for row in full]
    assert out[0][1] == w[0:2].tolist()
    assert out[1][1] == w[2:5].tolist()


def test_single_process_degenerates_to_identity():
    from hero_b200 import distributed as hd
    t = torch.ones(3)
    hd.all_reduce_and_rescale_tensors([t], 2.0)
    assert t.tolist() == [0.5] * 3
    assert hd.all_gather_list(7) == [7] and hd.any_broadcast("x", 0) == "x"
    x = torch.ones(2, 2, requires_grad=True)
    assert hd.vsm_allgather(x) is x or torch.equal(hd.vsm_allgather(x), x)
    assert hd.overlapped_exchange(None, "none") is None
    with pytest.raises(ValueError):
        hd.overlapped_exchange(None, "p2p")


def _vsm_scores_case(rank, world, hd):
    """get_video_level_scores with the cross-rank gather: ranks hold clips of different padded
    lengths; every rank must obtain the scores of ALL queries against ALL clips."""
    import types
    from tests import fake_ops
    from hero_b200 import ops
    from hero_b200.pretrain import HeroForPretraining
    for name in ("gemm", "l2norm_split", "vsm_masked_max", "vsm_scores_bwd"):
        setattr(ops, name, getattr(fake_ops, name))          # CPU process: no CUDA library
    gen = torch.Generator().manual_seed(5)
    D = 16
    data = []
    for r in range(world):
        L = 5 + 2 * r
        q = torch.randn(2, D, generator=gen)
        ctx = torch.randn(2, L, D, generator=gen)
        mask = torch.ones(2, L, dtype=torch.long)
        mask[1, L - 2:] = 0
        data.append((q, ctx, mask))
    q, ctx, mask = data[rank]
    # (a) equal per-rank counts, clips padded to max_clip_len: no length / count exchange at all
    me = types.SimpleNamespace(training=True, gather_gpus=True, gather_equal_counts=True,
                               v_encoder=types.SimpleNamespace(max_clip_len=12))
    got = HeroForPretraining.get_video_level_scores(me, q, ctx, mask)
    # (b) the reference's protocol (lengths and counts exchanged)
    me_b = types.SimpleNamespace(training=True, gather_gpus=True, gather_equal_counts=False,
                                 v_encoder=types.SimpleNamespace(max_clip_len=12))
    got_b = HeroForPretraining.get_video_level_scores(me_b, q, ctx, mask)
    assert torch.allclose(got, got_b, atol=1e-6)
    # single-process reference: pad to the longest clip and concatenate in rank order
    Lmax = max(c.shape[1] for _, c, _ in data)
    qa = torch.cat([d[0] for d in data])
    ca = torch.cat([torch.nn.functional.pad(d[1], (0, 0, 0, Lmax - d[1].shape[1])) for d in data])
    ma = torch.cat([torch.nn.functional.pad(d[2], (0, Lmax - d[2].shape[1])) for d in data])
    alone = types.SimpleNamespace(training=True, gather_gpus=False, gather_equal_counts=True,
                                  v_encoder=types.SimpleNamespace(max_clip_len=12))
    want = HeroForPretraining.get_video_level_scores(alone, qa, ca, ma)
    return got.tolist(), want.tolist()


def test_vsm_video_level_scores_gather_all_ranks():
    out = _run("_vsm_scores_case")
    for r in (0, 1):
        got, want = out[r]
        assert torch.allclose(torch.tensor(got), torch.tensor(want), atol=1e-5)
        assert len(got) == 4 and len(got[0]) == 4


class _TinyModel(torch.nn.Module):
    """Parameter names shaped like the encoder's: early (stack) and late (embedding) tensors in
    both the decay and the no-decay group."""

    def __init__(self):
        super().__init__()
        self.f_encoder = torch.nn.Module()
        self.f_encoder.embeddings = torch.nn.Module()
        self.f_encoder.embeddings.word_embeddings = torch.nn.Embedding(50, 16)
        self.f_encoder.embeddings.LayerNorm = torch.nn.LayerNorm(16)
        self.f_encoder.encoder = torch.nn.Linear(16, 16)
        self.c_encoder = torch.nn.Linear(16, 8)


def _flat_exchange_case(rank, world, hd):
    from tests import fake_ops
    from hero_b200 import ops
    from hero_b200.params import flat_of, is_late_grad
    ops.cast_bf16 = fake_ops.cast_bf16          # CPU process: no CUDA library
    torch.manual_seed(0)
    model = _TinyModel()
    flat = flat_of(model, torch.device("cpu"))
    out = {}
    # layout: the embedding tensors close each group; early + late ranges tile the buffer
    ranges = sorted(flat.early_ranges() + flat.late_ranges())
    out["tiles"] = ranges[0][0] == 0 and ranges[-1][1] == flat.total and all(
        a[1] == b[0] for a, b in zip(ranges, ranges[1:]))
    late = [(off, off + n) for name, _, off, n in flat.entries if is_late_grad(name)]
    out["late_inside"] = all(any(a <= lo and hi <= b for a, b in flat.late_ranges())
                             for lo, hi in late)
    early = [(off, off + n) for name, _, off, n in flat.entries if not is_late_grad(name)]
    out["early_inside"] = all(any(a <= lo and hi <= b for a, b in flat.early_ranges())
                              for lo, hi in early)
    for wire in ("fp32", "bf16"):
        ex = hd.FlatGradExchange(flat, wire=wire, overlap=True)   # CPU: no side stream, plain path
        g = flat.ensure_flat_grads()
        base = ((torch.arange(g.numel()) % 31) - 15).float() / 16.0
        g.copy_(base * (rank + 1))
        ex.prepare()
        ex.all_reduce()
        out[wire] = bool(torch.equal(g, base * 1.5)) and ex.ranks_agree()
        out[wire + "_check"] = ex.self_check().startswith("ok")
    return out


def test_flat_grad_exchange_layout_and_mean_on_both_wires():
    out = _run("_flat_exchange_case")
    for r in (0, 1):
        assert all(out[r].values()), out[r]
