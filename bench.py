"""Headline benchmark: clips/sec, forward + backward of the HERO hierarchical encoder at
train-tvr-8gpu shapes (BASELINE.json), data-parallel over N B200s.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference          # the UNMODIFIED reference's CPU path (rank 0)

One step = one pass of the hot path over one synthetic SYN-TVR-dense batch per rank
(B = 32 clips x 100 frames x 4352-d features, 20 subtitle rows of 5 frames + 20 tokens per clip,
one 16-token query per clip; hero_finetune dims: 6 cross-modal + 3 temporal layers, H = 768):
HierarchicalVlModel 'repr' forward + CrossModalTrm 'txt' forward on the query rows (by default
through `forward_repr_txt`, which runs the query rows in the same cross-modal pass as the video
rows; `--separate-txt` issues the reference's two calls), backward of both from fixed upstream
gradients, and (N > 1) the mean all-reduce of the flat gradient buffer.
Training mode (dropout 0.1 as in config/train-tvr-8gpu.json). No optimizer step inside `value`
(the metric is fwd+bwd); BASELINE configs 2 (fwd-only) and 3 (fwd+bwd+AdamW+clip) are timed in the
same run and reported under `extra`.

`value`   whole-job clips/s with inputs (and the per-batch packing plan, a collate-side product)
          resident in HBM, CUDA-event timed, max over ranks.
`e2e`     same metric through the public module API from PINNED HOST batches: per step the packing
          plan is built from that step's masks in loader worker processes (hero_b200.plan.PlanPool;
          the reference builds its gather indices in DataLoader collate workers), the batch and the
          plan's index arrays are copied host->device on a side stream (prefetch one step ahead,
          like the reference's PrefetchLoader, data/loader.py:89-144) and a loss scalar is read
          back. The loader is primed (two plans in flight) when the timed region starts.
`gpu_reference`  the UNMODIFIED reference modules (staged in git-ignored baseline/_ref by
          baseline/stage_ref.py; apex FusedLayerNorm -> torch.nn.LayerNorm, Horovod ->
          torch.distributed shim) doing the same step on the same GPU(s) in the same run under
          torch.autocast(bfloat16): the PyTorch-GPU baseline of BASELINE.json's north star.
`cpu_baseline` / `--impl reference`  the same reference modules on the host cores (fp32); falls
          back to the oracle port (kind "port") only if baseline/_ref was not staged.
"""
import argparse
import collections
import gc
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

H, INTER, HEADS, F_LAYERS, C_LAYERS, D = 768, 3072, 12, 6, 3, 4352
METRIC = "clips/sec fwd+bwd HERO encoder (TVR 8gpu shapes)"


def model_json(path):
    def cfg(n, with_vocab):
        c = {"attention_probs_dropout_prob": 0.1, "hidden_act": "gelu", "hidden_dropout_prob": 0.1,
             "hidden_size": H, "initializer_range": 0.02, "intermediate_size": INTER,
             "max_position_embeddings": 514, "num_attention_heads": HEADS, "num_hidden_layers": n,
             "type_vocab_size": 2}
        if with_vocab:
            c["vocab_size"] = 50272
        return c
    with open(path, "w") as f:
        json.dump({"f_config": cfg(F_LAYERS, True), "c_config": cfg(C_LAYERS, False)}, f)


def algorithmic_flops_fwd(vb, qb):
    """SURVEY.md §8d counting rule: valid tokens only, GEMMs + QK^T + PV, multiply-add = 2."""
    def f_layer(n):
        return 24 * n * H * H + 4 * n * n * H
    f_lens = vb["f_attn_masks"].sum(1).tolist()
    c_lens = vb["c_attn_masks"].sum(1).tolist()
    q_lens = qb["attn_masks"].sum(1).tolist()
    n_img = sum(len(fr) for clip in vb["sub_idx2frame_idx"] for _, fr in clip)
    fl = F_LAYERS * sum(f_layer(n) for n in f_lens) + F_LAYERS * sum(f_layer(n) for n in q_lens)
    fl += C_LAYERS * sum(f_layer(n) for n in c_lens)
    fl += 2 * D * H * (n_img + sum(c_lens))
    return float(fl)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (rank 0's GPU)."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index
        self.t_marks = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def window(self, t0, t1):
        """Only samples taken between t0 and t1 (perf_counter) count as 'during the region'."""
        self.t_marks.append((t0, t1))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, r in self.rows:
            if self.t_marks and not any(a - 0.06 <= t <= b + 0.06 for a, b in self.t_marks):
                continue
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def build_pretrain_model(device, seed=0):
    """HeroForPretraining (pretrain.py task heads on the encoder) with the hero_pretrain.json
    architecture: 6 + 3 layers, q_config with 0 layers (config/hero_pretrain.json), loss weights of
    config/pretrain-tv-16gpu.json."""
    from hero_b200.model import VideoModelConfig
    from hero_b200.pretrain import HeroForPretraining
    torch.manual_seed(seed)
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "hero_pretrain.json")
        model_json(p)
        cfg = json.load(open(p))
        q = dict(cfg["c_config"], num_hidden_layers=0, vocab_size=50272)
        cfg["q_config"] = q
        json.dump(cfg, open(p, "w"))
        model = HeroForPretraining(VideoModelConfig(p), vfeat_dim=D, max_frm_seq_len=100,
                                   lw_neg_ctx=8.0, lw_neg_q=8.0, lw_st_ed=0.01, margin=0.1)
    return model.to(device).train()


def pretrain_mix(args, rank, world, device, B):
    """BASELINE config 5: the pretrain.py task mix (mlm : mfm-nce : fom : vsm = 2 : 2 : 1 : 2,
    config/pretrain-tv-16gpu.json) on synthetic HowTo100M-shape clips (30 frames, 6 subtitles of
    5 frames + 20 tokens), fwd + bwd + gradient exchange + global-norm clip + fused AdamW per step,
    device-resident batches; clips/s over one cycle of 7 steps."""
    from hero_b200 import distributed as hdist
    from hero_b200 import synth
    from hero_b200.optim import FusedAdamW
    from hero_b200.params import flat_of
    from hero_b200.plan import attach_plan
    model = build_pretrain_model(device, seed=0)
    flat = flat_of(model, device)
    hdist.broadcast_tensors([flat.flat], 0)
    flat.mark_dirty()
    gflat = flat.ensure_flat_grads()
    exchange = hdist.FlatGradExchange(flat, wire=args.dp_wire, overlap=False) if world > 1 else None
    opt = FusedAdamW(flat, lr=1e-5)
    vb, qb = synth.syn_ht100m_dense(batch_size=B, seed=2345 + rank)
    tasks = {
        "mlm": synth.syn_mlm_batch(vb, seed=1),
        "mfm-nce": synth.syn_mfm_batch(vb, seed=2),
        "fom": attach_plan(synth.syn_fom_batch(vb, seed=3)),
        "vsm": attach_plan(synth.syn_vsm_batch(vb, qb, seed=4), kind="vsm"),
    }
    tasks["mfm-nce"] = attach_plan(tasks["mfm-nce"])
    tasks = {k: synth.to_device(v, device) for k, v in tasks.items()}
    cycle = ["mlm", "mfm-nce", "vsm", "fom", "mlm", "mfm-nce", "vsm"]

    def step(i):
        task = cycle[i % len(cycle)]
        gflat.zero_()
        batch = dict(tasks[task])
        if task == "mfm-nce":      # forward_mfm overwrites c_v_feats in place (model/model.py:244)
            batch["c_v_feats"] = batch["c_v_feats"].clone()
        loss = model(batch, task, compute_loss=True)
        if isinstance(loss, tuple):
            loss = sum(l.sum() for l in loss)
        loss.float().mean().backward()
        if exchange is not None:
            exchange.all_reduce()
        opt.clip_grad_norm_device_(1.0)
        opt.step()

    for i in range(len(cycle)):
        step(i)
    n = 2 * len(cycle)
    t_ms, med, host_ms, gaps = timed_loop(step, n, device, world)
    per_task = collections.defaultdict(list)
    for i, gms in enumerate(gaps):
        per_task[cycle[i % len(cycle)]].append(gms)
    del model, opt
    torch.cuda.empty_cache()
    return {"value": round(world * B / (t_ms / n * 1e-3), 2), "unit": "clips/s",
            "ms_per_step": round(t_ms / n, 4), "steps": n,
            "ms_per_task_step": {k: round(statistics.median(v), 3) for k, v in per_task.items()},
            "host_enqueue_ms_per_step": round(host_ms, 3),
            "what": "BASELINE config 5: pretrain.py task mix mlm:mfm-nce:fom:vsm = 2:2:1:2 on "
                    "synthetic HowTo100M-shape batches (32 clips x 30 frames, 6 subtitles of 5 "
                    "frames + 20 tokens per clip), fwd+bwd"
                    + (" + gradient all-reduce" if world > 1 else "")
                    + " + clip + fused AdamW per step"}


def build_model(device, seed=0):
    from hero_b200.model import HierarchicalVlModel, VideoModelConfig
    torch.manual_seed(seed)
    with tempfile.TemporaryDirectory() as td:
        p = os.path.join(td, "hero_finetune.json")
        model_json(p)
        model = HierarchicalVlModel(VideoModelConfig(p), vfeat_dim=D, max_frm_seq_len=100)
    model.initialize()   # random init of the hero_finetune architecture (no checkpoints offline)
    return model.to(device).train()


def _max_over_ranks(x, device, world):
    t = torch.tensor([x], dtype=torch.float64, device=device)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())


HOST_FREE_MS = []     # host ms of the first <= 3 steps of the latest timed_loop (queue not yet full)


def timed_loop(step_fn, steps, device, world, sampler=None):
    """barrier + synchronize immediately before the first event, one event per step, synchronize +
    barrier after; returns (total ms = max over ranks, median per-step ms of THIS rank, host
    enqueue ms per step)."""
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    evs[0].record()
    marks = [t0]
    for i in range(steps):
        step_fn(i)
        evs[i + 1].record()
        marks.append(time.perf_counter())
    host_ms = (marks[-1] - t0) * 1e3 / max(steps, 1)
    # The first steps after the synchronize are enqueued into an empty launch queue: their host
    # time is the real cost of enqueueing a step. Later steps include launch-queue back-pressure
    # (the host runs ahead of the device until the queue is full, then waits for the GPU).
    HOST_FREE_MS[:] = [(b - a) * 1e3 for a, b in zip(marks[:3], marks[1:4])]
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    if world > 1:
        torch.distributed.barrier()
    if sampler is not None:
        sampler.window(t0, t1)
    total = evs[0].elapsed_time(evs[-1])
    gaps = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
    return _max_over_ranks(total, device, world), statistics.median(gaps), host_ms, gaps


# Per-array caps of --dump-outputs: 2 outputs x 16 MiB + 186 parameters x 128 KiB < 64 MiB
DUMP_OUTPUT_ELEMS, DUMP_GRAD_ELEMS, DUMP_MAX_BYTES = 1 << 22, 1 << 15, 64 << 20


def _dump_array(t, cap, name):
    """float32 host copy of `t`; above `cap` elements, the same `cap` positions (drawn from a
    generator seeded with the name) of the flattened tensor in every run and build."""
    t = t.detach()
    if t.numel() > cap:
        g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
        idx = torch.randint(t.numel(), (cap,), generator=g).sort().values
        t = t.flatten()[idx.to(t.device)]
    return t.float().cpu().numpy()


def dump_outputs(out_dir, outputs, model):
    """What one timed step hands its caller: the clip outputs (`clip.npy`), the query rows
    (`query.npy`) and every parameter's gradient (`grad.<parameter name>.npy`), float32."""
    import numpy as np
    arrays = {k: _dump_array(v, DUMP_OUTPUT_ELEMS, k) for k, v in outputs.items()}
    for name, p in model.named_parameters():
        if p.grad is not None:
            arrays["grad." + name] = _dump_array(p.grad, DUMP_GRAD_ELEMS, name)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs would write {total} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_ours(args):
    from hero_b200 import distributed as hdist
    from hero_b200 import ops, synth
    from hero_b200.params import flat_of
    from hero_b200.loader import BatchStager, record_plans
    from hero_b200.plan import PlanPool, attach_plan
    from hero_b200.optim import FusedAdamW

    rank, world, local_rank = hdist.init()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    model = build_model(device, seed=0)
    flat = flat_of(model, device)
    hdist.broadcast_tensors([flat.flat], 0)
    flat.mark_dirty()
    bucketer = None
    if world > 1 and args.dp_transport != "none" and not args.dp_skip_exchange:
        bucketer = hdist.overlapped_exchange(flat, transport=args.dp_transport,
                                             min_elems=args.bucket_elems,
                                             overlap_ctas=args.overlap_ctas)
    gflat = flat.ensure_flat_grads()
    exchange = None
    if world > 1 and bucketer is None and not args.dp_skip_exchange:
        exchange = hdist.FlatGradExchange(flat, wire=args.dp_wire, overlap=not args.no_dp_overlap)

    B = args.batch_size
    n_host = 3
    host = []
    for i in range(n_host):
        vb, qb = synth.syn_tvr_dense(batch_size=B, seed=1234 + rank + 1000 * i)
        for b in (vb, qb):
            for k, v in b.items():
                if torch.is_tensor(v):
                    b[k] = v.pin_memory()
        host.append((vb, qb))
    flops_fwd = algorithmic_flops_fwd(*host[0])
    g = torch.Generator().manual_seed(7)
    dclip = (torch.randn(B, 100, H, generator=g) * 1e-2).to(device)
    dq = (torch.randn(B, host[0][1]["input_ids"].shape[1], H, generator=g) * 1e-2).to(device)
    accum = max(1, args.accum)
    state = {"micro": 0, "accum": accum}

    def fwd_bwd(vb_dev, qb_dev, opt=None, clip_norm=None):
        if bucketer is not None:   # per-layer gradient exchange overlapped with backward
            bucketer.__enter__()
        if exchange is not None and (state["micro"] + 1) % state["accum"] == 0:
            exchange.prepare()     # this step's gradients are exchanged: overlap what is final early
        if args.separate_txt:      # the reference's two calls (model/pretrain.py:65-70)
            clip = model(vb_dev, "repr")
            q = model.f_encoder(qb_dev, "txt")[0]
        else:                      # same results, query rows share the video rows' GEMMs
            clip, q = model.forward_repr_txt(vb_dev, qb_dev)
        flat.wait_grads_zeroed()       # the memset of this step's gradient buffer ran beside the forward
        torch.autograd.backward([clip, q], [dclip, dq])
        state["micro"] += 1
        boundary = state["micro"] % state["accum"] == 0   # gradient_accumulation_steps (train_vcmr.py:233)
        if bucketer is not None:
            bucketer.__exit__(None, None, None)
            bucketer.finish()
        elif exchange is not None and boundary:
            exchange.all_reduce()
        if opt is not None and boundary:
            if clip_norm is not None:
                opt.clip_grad_norm_device_(clip_norm)
            opt.step()
        return clip, q

    # ------------------------------------------------------------- device-resident timing
    resident = []
    for vb, qb in host:
        vb = attach_plan(dict(vb))
        qb = attach_plan(dict(qb), kind="txt")
        resident.append((synth.to_device(vb, device), synth.to_device(qb, device)))
    torch.cuda.synchronize()
    last = {}     # outputs of the latest resident step, kept only for --dump-outputs

    def resident_step(i):
        if state["micro"] % state["accum"] == 0:
            (flat.zero_grads_async() if args.grad_zero == "async" else gflat.zero_())
        vb_dev, qb_dev = resident[i % n_host]
        clip, q = fwd_bwd(vb_dev, qb_dev)
        if args.dump_outputs:
            last["clip"], last["query"] = clip.detach(), q.detach()

    # known-answer test of the gradient exchange on this job's ranks / transport (raises on a
    # mismatch): every rank must end with the mean of the per-rank patterns, bit-identical
    allreduce_check = None
    if world > 1 and exchange is not None:
        allreduce_check = exchange.self_check()
        # and on real gradients through the overlapped path: per-rank batches differ, so the ranks
        # can only agree bit for bit afterwards if every range of the buffer was reduced
        state["micro"] = accum - 1
        gflat.zero_()
        fwd_bwd(*resident[0])
        if not exchange.ranks_agree():
            raise RuntimeError("ranks disagree on the exchanged gradients of a training step")
        allreduce_check += "; ranks bit-identical after an exchanged training step"
        state["micro"] = 0
    for i in range(args.warmup):
        resident_step(i)
    ops.reset_launch_count()
    state["micro"] = 0
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler is not None:
        sampler.start()           # forks nvidia-smi BEFORE the barrier that opens the timed region
        time.sleep(0.2)
    ms_total, ms_median, host_enqueue_ms, gaps = timed_loop(resident_step, args.steps, device,
                                                            world, sampler)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last, model)
    host_free_ms = round(statistics.median(HOST_FREE_MS), 3) if HOST_FREE_MS else None
    launches = ops.launch_count() // max(args.steps, 1)
    ms_per_step = ms_total / args.steps
    value = world * B / (ms_per_step * 1e-3)

    # ------------------------------------------------------------- GEMM-family roofline (live)
    # (the layer runtime keeps everything on one stream while GEMM launches are being timed, so
    # durations do not overlap). Runs for >= ~2 s so clocks settle where a long job runs, which is
    # what the "sustained" peak in MEASURED_PEAKS.json was measured under; both fractions reported.
    prof_steps = max(5, min(int(2000.0 / max(ms_per_step * 1.15, 1e-3)), 400))
    if args.roofline_steps > 0:      # profiler runs (ncu launch lists): a short pass is enough
        prof_steps = args.roofline_steps
    ops.start_gemm_profile()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tp0 = time.perf_counter()
    p0.record()
    for i in range(prof_steps):
        resident_step(i)
    p1.record()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.window(tp0, time.perf_counter())
    gp = ops.stop_gemm_profile()
    profiled_step_ms = p0.elapsed_time(p1) / prof_steps
    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    burst_tf = peaks.get("bf16_tflops", 1693.7)
    achieved = gp["flops"] / (gp["ms"] * 1e-3) / 1e12 if gp["ms"] > 0 else 0.0
    traffic, traffic_src = None, None
    tr_path = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tr_path):
        tj = json.load(open(tr_path))
        traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
    roofline = {"bound": "tensor", "kernel": "gemm_tcgen05_kernel (all variants)",
                "achieved": round(achieved, 1), "peak": peak_tf, "unit": "TFLOP/s",
                "frac": round(achieved / peak_tf, 4),
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (of measured); the "
                               "roofline pass runs >= 2 s" if peaks else
                               "fallback 1.4 PF/s (of fallback)",
                "frac_of_burst_peak": round(achieved / burst_tf, 4),
                "profiled_steps": prof_steps,
                "launches_per_step": gp["launches"] // prof_steps,
                "gemm_share_of_step": round(gp["ms"] / prof_steps / profiled_step_ms, 3),
                "traffic": traffic, "traffic_source": traffic_src,
                "step_algorithmic_tflops": round(3 * flops_fwd * 1e-12, 4),
                "step_frac_of_peak": round(3 * flops_fwd / (ms_per_step * 1e-3) / 1e12 / peak_tf,
                                           4)}

    # ------------------------------------------------------------- BASELINE configs 2 and 3
    extra = {}
    if not args.no_extra:
        k_extra = max(5, min(args.steps, 20))
        # config 3: fwd + bwd + global-norm clip + fused AdamW (train_vcmr.py:240-262)
        opt = FusedAdamW(flat, lr=1e-5)

        def opt_step(i):
            if state["micro"] % state["accum"] == 0:
                (flat.zero_grads_async() if args.grad_zero == "async" else gflat.zero_())
            fwd_bwd(*resident[i % n_host], opt=opt, clip_norm=1.0)
        for i in range(3):
            opt_step(i)
        t_ms, med, _, _ = timed_loop(opt_step, k_extra, device, world)
        extra["fwd_bwd_adamw"] = {
            "value": round(world * B / (t_ms / k_extra * 1e-3), 2), "unit": "clips/s",
            "ms_per_step": round(t_ms / k_extra, 4), "median_ms_per_step": round(med, 4),
            "steps": k_extra, "what": "BASELINE config 3: fwd+bwd"
            + (" + gradient all-reduce" if world > 1 else "")
            + " + global-norm clip (1.0) + fused AdamW, device-resident inputs"}
        del opt
        if world > 1 and accum == 1 and exchange is not None:
            # config 4 as the reference runs it: config/train-tvr-8gpu.json:35 accumulates two
            # micro-batches per optimizer step, so gradients are exchanged every second fwd+bwd
            # (train_vcmr.py:233-239). `value` above exchanges after EVERY micro-batch.
            state["accum"], state["micro"] = 2, 0
            for i in range(4):
                resident_step(i)
            n_micro = 2 * ((k_extra + 1) // 2)
            t_ms, med, _, _ = timed_loop(resident_step, n_micro, device, world)
            extra["accum2_schedule"] = {
                "value": round(world * B / (t_ms / n_micro * 1e-3), 2), "unit": "clips/s",
                "ms_per_micro_step": round(t_ms / n_micro, 4), "micro_steps": n_micro,
                "what": "fwd+bwd with gradient_accumulation_steps = 2 (config/train-tvr-8gpu.json:35):"
                        " one gradient all-reduce per two micro-batches of 32 clips per GPU"}
            state["accum"], state["micro"] = accum, 0
        # config 2: forward only, eval mode, no autograd graph
        model.eval()

        def fwd_only(i):
            with torch.no_grad():
                vb_dev, qb_dev = resident[i % n_host]
                model.forward_repr_txt(vb_dev, qb_dev)
        for i in range(3):
            fwd_only(i)
        t_ms, med, _, _ = timed_loop(fwd_only, k_extra, device, world)
        extra["fwd_only_eval"] = {
            "value": round(world * B / (t_ms / k_extra * 1e-3), 2), "unit": "clips/s",
            "ms_per_step": round(t_ms / k_extra, 4), "median_ms_per_step": round(med, 4),
            "steps": k_extra,
            "frac_of_peak": round(flops_fwd / (t_ms / k_extra * 1e-3) / 1e12 / peak_tf, 4),
            "what": "BASELINE config 2: full encoder forward only (eval mode, no_grad)"}
        model.train()
        flat.mark_dirty()       # the optimizer moved the weights; mirror refreshed by its kernel
        state["micro"] = 0

    # ------------------------------------------------------------- end-to-end from pinned host
    stager = BatchStager(device, depth=3)
    slim = not args.e2e_legacy_batch
    # The e2e arm ships the packed-layout batch (SURVEY §8f-2): `f_v_feats` is a row gather of
    # `c_v_feats` (data/data.py:380-395), so the batch omits it and the plan maps every frame slot
    # to its clip frame — half the host->device bytes, identical results
    # (tests/test_encoder_gpu.py::test_batch_without_f_v_feats_on_gpu). --e2e-legacy-batch ships it.
    e2e_host = []
    for vb, qb in host:
        vb2 = {k: v for k, v in vb.items() if not (slim and k == "f_v_feats")}
        e2e_host.append((vb2, qb))

    def h2d_bytes(b):
        return sum(v.numel() * v.element_size() for v in b.values() if torch.is_tensor(v))

    loader_state = {"pool": None, "mode": "loader worker processes (PlanPool, 3 workers)"}
    try:
        loader_state["pool"] = PlanPool(workers=3)
    except Exception as e:                                  # noqa: BLE001
        loader_state["mode"] = f"in-process (worker pool unavailable: {type(e).__name__})"
    plan_futs = collections.deque()

    def submit_plan(i):
        vb, qb = e2e_host[i % n_host]
        pool = loader_state["pool"]
        try:
            plan_futs.append(pool.submit(vb, qb) if pool is not None else None)
        except Exception as e:                              # noqa: BLE001
            loader_state["pool"] = None
            loader_state["mode"] = f"in-process (worker pool failed: {type(e).__name__})"
            plan_futs.append(None)

    def plans_for(fut, vb, qb):
        if fut is not None:
            try:
                return PlanPool.attach(fut, vb, qb)
            except Exception as e:                          # noqa: BLE001
                loader_state["pool"] = None
                loader_state["mode"] = f"in-process (worker pool failed: {type(e).__name__})"
        return attach_plan(vb), attach_plan(qb, kind="txt")

    stage_t = collections.defaultdict(float)

    def stage(i, total):
        t0 = time.perf_counter()
        vb, qb = e2e_host[i % n_host]
        vb, qb = plans_for(plan_futs.popleft(), dict(vb), dict(qb))
        t1 = time.perf_counter()
        if i + 2 < total:
            submit_plan(i + 2)
        t2 = time.perf_counter()
        stage_t["plan_wait"] += t1 - t0
        stage_t["plan_submit"] += t2 - t1
        (vb_dev, qb_dev), ev, slot = stager.stage(vb, qb)    # preallocated ring, side stream
        stage_t["h2d_enqueue"] += time.perf_counter() - t2
        return vb_dev, qb_dev, ev, slot

    RESULT_LAG = 2       # the scalar of step i is consumed after step i + 2 has been enqueued
    result_host = torch.zeros(RESULT_LAG + 1, dtype=torch.float32).pin_memory()

    def e2e_loop(n):
        """Every step: wait for its prefetched inputs, enqueue fwd+bwd, start the (async) D2H
        read of a result scalar, then build the NEXT batch's plan on the host and start its H2D
        copy on the side stream while the GPU computes. The scalar of step i is consumed right
        after step i+2 has been enqueued (lagged logging: with eight ranks meeting in an all-reduce
        every step, a one-step lag let any rank's host hiccup stall all of them), so the host
        never idles the GPU; all n results are read inside the timed region."""
        out, pending = 0.0, collections.deque()
        tt = collections.defaultdict(float)
        dones = []
        nxt = stage(0, n)
        for i in range(n):
            t_a = time.perf_counter()
            vb_dev, qb_dev, ev, ring_slot = nxt
            cur = torch.cuda.current_stream()
            cur.wait_event(ev)
            record_plans((vb_dev, qb_dev), cur)   # allocator safety across streams
            if state["micro"] % accum == 0:
                (flat.zero_grads_async() if args.grad_zero == "async" else gflat.zero_())
            t_b = time.perf_counter()
            clip, _ = fwd_bwd(vb_dev, qb_dev)
            t_c = time.perf_counter()
            slot = result_host[i % (RESULT_LAG + 1):i % (RESULT_LAG + 1) + 1]
            # (detach: the pinned result buffer must not become part of — and keep alive — the
            # step's autograd graph and its ~3 GB of saved activations)
            slot.copy_(clip.detach()[0, 0, :8].float().sum().reshape(1), non_blocking=True)   # D2H
            done = torch.cuda.Event(enable_timing=True)
            done.record(cur)
            dones.append(done)
            stager.release(ring_slot, cur)
            t_d = time.perf_counter()
            if i + 1 < n:
                nxt = stage(i + 1, n)                   # plan upload + H2D overlap this step's compute
            t_e = time.perf_counter()
            pending.append((done, slot))
            if len(pending) > RESULT_LAG:
                ev_done, ev_slot = pending.popleft()
                ev_done.synchronize()
                out += float(ev_slot[0])
            t_f = time.perf_counter()
            for k, v in (("record", t_b - t_a), ("fwd_bwd", t_c - t_b), ("d2h", t_d - t_c),
                         ("stage", t_e - t_d), ("sync_prev", t_f - t_e)):
                tt[k] += v
        while pending:
            ev_done, ev_slot = pending.popleft()
            ev_done.synchronize()
            out += float(ev_slot[0])
        gaps = [round(a.elapsed_time(b), 2) for a, b in zip(dones[:-1], dones[1:])]
        diag = {"stage_totals_ms": {k: round(v * 1e3, 1) for k, v in stage_t.items()},
                "device_ms_between_step_ends": gaps,
                "host_phases_ms_per_step": {k: round(v / n * 1e3, 2) for k, v in tt.items()}}
        stage_t.clear()
        return out, diag

    def prime():     # a running loader always has two batches of plans in flight
        plan_futs.clear()
        submit_plan(0)
        submit_plan(1)

    # start every loader worker (each imports torch once) before anything is timed
    if loader_state["pool"] is not None:
        try:
            for f in [loader_state["pool"].submit(*e2e_host[0]) for _ in range(6)]:
                f.result(timeout=300)
        except Exception as e:                              # noqa: BLE001
            loader_state["pool"] = None
            loader_state["mode"] = f"in-process (worker pool failed: {type(e).__name__})"
    prime()
    e2e_loop(max(5, args.warmup))
    prime()
    for f in plan_futs:
        if f is not None:
            try:
                f.result(timeout=300)
            except Exception:                               # noqa: BLE001
                pass
    # Host-side jitter protection for the timed e2e window: no cyclic GC passes (nothing in the
    # loop creates cycles that must be reclaimed within 20 steps), and the caching allocator must
    # not grow (every buffer of a step has been allocated during warm-up).
    gc.collect()
    gc.freeze()
    gc.disable()
    mem0 = torch.cuda.memory_stats(device).get("num_device_alloc", 0) if hasattr(
        torch.cuda, "memory_stats") else 0
    state["micro"] = 0
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _, diag = e2e_loop(args.steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    gc.enable()
    gc.unfreeze()
    mem1 = torch.cuda.memory_stats(device).get("num_device_alloc", 0) if hasattr(
        torch.cuda, "memory_stats") else 0
    if sampler is not None:
        sampler.window(t0, t0 + e2e_s)
    print("e2e diagnostics:", json.dumps(diag), file=sys.stderr)
    if loader_state["pool"] is not None:
        loader_state["pool"].shutdown()
    e2e_value = world * B * args.steps / _max_over_ranks(e2e_s, device, world)
    bi = h2d_bytes(e2e_host[0][0]) + h2d_bytes(e2e_host[0][1])
    e2e_gaps = diag["device_ms_between_step_ends"]
    clocks = sampler.stop() if sampler is not None else None

    # ------------------------------------------------------------- reference arms
    del resident, stager
    torch.cuda.empty_cache()
    if not args.no_extra and not args.no_pretrain_mix:
        try:
            extra["pretrain_mix"] = pretrain_mix(args, rank, world, device, B)
        except Exception as e:                              # noqa: BLE001
            extra["pretrain_mix"] = {"unavailable": f"{type(e).__name__}: {str(e)[:300]}"}
    gpu_ref = None
    if not args.no_gpu_reference:
        gpu_ref = gpu_reference(args, rank, world, device, B)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(sample_clips=args.cpu_clips, steps=2, warmup=1)

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "clips/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4),
            "median_ms_per_step": round(ms_median, 4),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": "SYN-TVR-dense: HierarchicalVlModel 'repr' + CrossModalTrm 'txt' "
                                   "fwd+bwd (hero_finetune dims 6+3 layers), per-rank 32 clips x "
                                   "100 frames x 4352-d + 640 rows x (5 frames + 20 tokens) + 32 "
                                   "queries x 16 tokens",
                       "global_batch": world * B, "per_gpu_batch": B, "parallelism": f"dp{world}",
                       "dropout": 0.1, "optimizer_in_step": False,
                       "gradient_accumulation_steps": accum,
                       "grad_zeroing": ("every step, 0.43 GB memset on a side stream beside the "
                                        "forward (FlatParams.zero_grads_async); backward waits "
                                        "for it") if args.grad_zero == "async" else
                                       "every step, in the compute stream before the forward",
                       "query_rows": "separate call" if args.separate_txt else
                       "fused into the video-row pass (forward_repr_txt)",
                       "allreduce_in_step": world > 1 and not args.dp_skip_exchange,
                       "allreduce": (("per-layer buckets during backward (GradBucketer)")
                                     if bucketer is not None else
                                     exchange.describe() if exchange is not None else "none"),
                       "allreduce_check": allreduce_check,
                       "e2e_plans": loader_state["mode"],
                       "e2e_batch": "packed (no f_v_feats: frame slots read from c_v_feats through "
                                    "the plan)" if slim else "legacy dict incl. f_v_feats",
                       "l2": "no explicit flush: per-step working set (~0.35 GB weights+grads, "
                             "~3 GB activations, 56-112 MB inputs) exceeds the 126 MB L2"},
            "clocks": clocks, "gpu_launches": launches,
            "host_enqueue_ms_per_step": round(host_enqueue_ms, 3),
            "host_enqueue_ms_queue_not_full": host_free_ms,
            "e2e": {"value": round(e2e_value, 2), "unit": "clips/s", "h2d_bytes_per_step": bi,
                    "d2h_bytes_per_step": 4,
                    "median_device_ms_between_step_ends":
                        round(statistics.median(e2e_gaps), 3) if e2e_gaps else None,
                    "max_device_ms_between_step_ends": max(e2e_gaps) if e2e_gaps else None,
                    "device_allocations_during_timed_region": int(mem1 - mem0)},
            "roofline": roofline,
            "extra": extra,
        }
        if gpu_ref is not None:
            line["gpu_reference"] = gpu_ref
            if gpu_ref.get("value"):
                line["vs_gpu_reference"] = {"value_ratio": round(value / gpu_ref["value"], 2),
                                            "e2e_ratio": round(e2e_value / gpu_ref["value"], 2)}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.destroy_process_group()


# ----------------------------------------------------------------------------- reference arms
def _ref_inputs(sample_clips, seed=1234):
    from hero_b200 import synth
    vb, qb = synth.syn_tvr_dense(batch_size=sample_clips, seed=seed)
    g = torch.Generator().manual_seed(7)
    dclip = torch.randn(sample_clips, 100, H, generator=g) * 1e-2
    dq = torch.randn(sample_clips, qb["input_ids"].shape[1], H, generator=g) * 1e-2
    return vb, qb, dclip, dq


def gpu_reference(args, rank, world, device, B):
    """The unmodified reference (baseline/_ref) doing the same step on the GPU under
    torch.autocast(bfloat16): fwd `forward_repr` + `f_encoder('txt')`, backward, and at N > 1 its
    own all_reduce_and_rescale_tensors over a torch.distributed-backed Horovod shim."""
    from baseline import ref_runner as rr
    from hero_b200 import synth
    if rr.available() is None:
        return {"unavailable": "baseline/_ref not staged (run baseline/stage_ref.py where "
                               "/root/reference exists)"}
    try:
        rr.install(dist_backed=world > 1)
        model = rr.build_model(device, seed=0, train=True)
        step = rr.make_step(model, autocast_dtype=torch.bfloat16, world=world, train=True)
        vb, qb, dclip, dq = _ref_inputs(B, seed=1234 + rank)
        vb, qb = synth.to_device(vb, device), synth.to_device(qb, device)
        dclip, dq = dclip.to(device), dq.to(device)
        k = max(3, min(args.steps, 10))
        for _ in range(3):
            step(vb, qb, dclip, dq)
        t_ms, med, host_ms, _ = timed_loop(lambda i: step(vb, qb, dclip, dq), k, device, world)
        ms = t_ms / k
        out = {"value": round(world * B / (ms * 1e-3), 2), "unit": "clips/s",
               "ms_per_step": round(ms, 3), "median_ms_per_step": round(med, 3), "steps": k,
               "host_ms_per_step": round(host_ms, 3), "dtype": "bf16 autocast (fp32 master)",
               "kind": "reference",
               "what": "unmodified reference HierarchicalVlModel (config/hero_finetune.json) "
                       "fwd+bwd" + (" + its all_reduce_and_rescale_tensors (NCCL)" if world > 1
                                    else "") + ", device-resident inputs, stock PyTorch kernels"}
        del model, step
        torch.cuda.empty_cache()
        return out
    except Exception as e:                                  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {str(e)[:200]}"}


def _pick_cpu_threads():
    """Intra-op thread count for the CPU arms: the box may expose more logical CPUs than the
    container may use (a 128-thread team on a smaller quota ran the reference 30x slower than 8
    threads), so a ~1 s calibration on encoder-shaped work picks the fastest of {8, 16, ...}."""
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    cands = sorted({n for n in (4, 8, 16, 32, 64, 96, 128) if n <= avail} | {min(avail, 128)})
    x = torch.randn(4096, 768)
    w = torch.randn(3072, 768)
    best_n, best_t = cands[0], float("inf")
    for n in cands:
        torch.set_num_threads(n)
        for rep in range(3):
            t0 = time.perf_counter()
            y = torch.nn.functional.layer_norm(torch.nn.functional.gelu(x @ w.t()), (3072,))
            y = y @ w
            dt = time.perf_counter() - t0
            if rep and dt < best_t:
                best_n, best_t = n, dt
    torch.set_num_threads(best_n)
    return best_n


def cpu_baseline(sample_clips=8, steps=2, warmup=1):
    """The reference's own CPU path (unmodified modules from baseline/_ref; oracle port if the
    reference was not staged) on all host cores: fwd+bwd on a bounded sample of the same workload
    (first `sample_clips` clips of SYN-TVR-dense)."""
    from baseline import ref_runner as rr
    n_thr = _pick_cpu_threads()        # torchrun exports OMP_NUM_THREADS=1: use the whole box
    vb, qb, dclip, dq = _ref_inputs(sample_clips)
    kind = "reference"
    if rr.available() is not None:
        rr.install(dist_backed=False)
        model = rr.build_model(torch.device("cpu"), seed=0, train=True)
        for m in model.modules():          # dropout 0 for fwd+bwd timing (SURVEY §8d protocol)
            if isinstance(m, torch.nn.Dropout):
                m.p = 0.0
        ref_step = rr.make_step(model, autocast_dtype=None, world=1, train=True)

        def step():
            ref_step(vb, qb, dclip, dq)
        what = "unmodified reference modules (baseline/_ref), fp32, torch CPU autograd"
    else:
        from oracle import hero_oracle as orc
        kind = "port"
        P = orc.seeded_weights(orc.param_shapes(), seed=0)
        P = {k: v.requires_grad_(True) for k, v in P.items()}

        def step():
            for v in P.values():
                v.grad = None
            clip = orc.hierarchical_repr(P, vb, F_LAYERS, C_LAYERS, HEADS)
            q = orc.cross_modal_txt(P, "f_encoder.", qb, F_LAYERS, HEADS)
            torch.autograd.backward([clip, q], [dclip, dq])
        what = "oracle port (fp32, torch CPU autograd)"

    t0 = time.perf_counter()
    for _ in range(warmup):
        step()
    if warmup and (time.perf_counter() - t0) / warmup * steps > 90.0:
        steps = 1                      # keep the whole bench run within minutes on a slow host
    best, t_all = float("inf"), 0.0
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        best = min(best, dt)
        t_all += dt
    return {"value": round(sample_clips / (t_all / steps), 3), "unit": "clips/s",
            "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(), "kind": kind,
            "best_value": round(sample_clips / best, 3),
            "ms_per_clip": round(1e3 * (t_all / steps) / sample_clips, 1),
            "sample": f"{what}: fwd+bwd on the first {sample_clips} clips of SYN-TVR-dense "
                      f"(same per-clip shapes as the GPU arm), {steps} timed steps after "
                      f"{warmup} warm-up"}


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host
    cores (all threads), bounded sample per step. Rank 0 alone runs; other ranks exit 0."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = max(1, min(args.steps, 3))
    warm = max(1, min(args.warmup, 1))
    cb = cpu_baseline(sample_clips=args.cpu_clips, steps=steps, warmup=warm)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "clips/s",
            "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": round(1e3 * args.cpu_clips / cb["value"], 2), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"SYN-TVR-dense sample of {args.cpu_clips} clips per step "
                                   "(same per-clip shapes as the GPU arm; clips/s is per clip, "
                                   "so the sample size does not change the unit)",
                       "parallelism": "cpu"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "clips/s", "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch-size", type=int, default=32)
    ap.add_argument("--accum", type=int, default=1,
                    help="gradient accumulation micro-steps per exchange (config/train-tvr-8gpu.json "
                         "uses 2); every micro-step counts as a step")
    ap.add_argument("--dp-wire", default="bf16", choices=("bf16", "fp32"),
                    help="N>1: dtype of the gradient all-reduce on the wire (the reference "
                         "exchanged fp16 gradients under apex O2)")
    ap.add_argument("--dp-transport", default="none", choices=("none", "p2p", "nccl", "auto"),
                    help="N>1: 'none' = chunked NCCL all-reduce of the flat gradient buffer "
                         "(default); 'p2p' / 'nccl' = GradBucketer: per-layer buckets during backward")
    ap.add_argument("--no-dp-overlap", action="store_true",
                    help="N>1: one all-reduce after backward instead of reducing the stack gradients "
                         "during the embedding backward")
    ap.add_argument("--dp-skip-exchange", action="store_true",
                    help="DIAGNOSTIC (invalid as a result): N>1 without any gradient exchange")
    ap.add_argument("--bucket-elems", type=int, default=1 << 20)
    ap.add_argument("--overlap-ctas", type=int, default=0)
    ap.add_argument("--separate-txt", action="store_true",
                    help="encode the query rows with a separate f_encoder(batch, 'txt') call")
    ap.add_argument("--e2e-legacy-batch", action="store_true",
                    help="e2e ships the legacy batch dict including f_v_feats (2x the H2D bytes)")
    ap.add_argument("--grad-zero", default="sync", choices=("async", "sync"),
                    help="zero the flat gradient buffer in the compute stream before the forward "
                         "(default) or on a side stream beside it (measured equal on B200: the "
                         "memset's CTAs delay the persistent GEMMs by what they save)")
    ap.add_argument("--no-extra", action="store_true", help="skip the config-2 / config-3 lines")
    ap.add_argument("--roofline-steps", type=int, default=0,
                    help="steps of the per-launch GEMM timing pass (0 = as many as fill ~2 s)")
    ap.add_argument("--no-pretrain-mix", action="store_true", help="skip the config-5 line")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-clips", type=int, default=8)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's outputs and parameter gradients "
                         "of the last timed step as DIR/<name>.npy (float32; arrays above a size "
                         "cap as a fixed seeded sample) to compare builds on identical inputs")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        run_ours(args)


if __name__ == "__main__":
    main()
