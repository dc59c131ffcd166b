#!/usr/bin/env python
"""Headline benchmark: users/sec for LRURec encode + full-catalogue score + top-20 (BASELINE.json metric)
on the scaled synthetic catalogue (configs[3]: 10M items, d=64, batch 4096, L=50), on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path over one batch of 4096 synthetic users per GPU: sequence preparation,
encoder, catalogue scoring fused with top-20, k-way merge + metrics.  With N > 1 the item table is
row-sharded over the ranks and the users are data-parallel (weak scaling: every rank brings its own batch
of 4096 users, the global batch is 4096*N, per-GPU scoring work is constant): one coalesced all-gather of
the user states + exclusion lists, local scoring of all 4096*N users against the rank's rows, one
all-to-all of the local top-20 lists, merge of the local users' N lists.  `--scaling strong` instead keeps
the global batch at 4096 (every rank scores the same 4096 users against 1/N of the rows).

Prints ONE JSON line (rank 0).  `--impl reference` times the CPU oracle port of the reference's path on the
host cores instead (the reference is pure Python/PyTorch and is not part of this repository).

`--dump-outputs DIR` writes what rank 0's last timed step returned (ids, scores, label_rank, metric_sums and the
user states u) as DIR/<name>.npy: floating point as float32, integers as float64.  Inputs and weights are
seeded, so two builds run with the same arguments can be compared array by array.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys
import threading
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ITEMS = 10_000_000
BATCH = 4096
MAX_LEN = 50
TOPK = 20
CPU_SAMPLE_USERS = 1024      # users per pass of the CPU arms: enough to amortise the 2.56 GB table read per pass
PARITY_USERS = 256           # users of the last timed step whose lists are re-derived independently
WORKLOAD = "c4_10m: 10M items, d=64, batch 4096, max_len 50, top-20 (BASELINE.json configs[3])"
DUMP_MAX_BYTES = 64 << 20


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """SM clock and throttle reasons of one GPU DURING the timed region (B200_PROFILING.md, the clocks line).

    NVML is read in-process (pynvml; the same counters `nvidia-smi --query-gpu=clocks.sm,...` prints) from a
    thread that only samples between activate() and stop(): the bench enqueues its K timed steps first and
    activates the sampler while the GPU works through them.  An `nvidia-smi -lms` loop running while the host
    is still launching was seen to stall the launch path (driver lock) for ~100 ms in 3 of 9 multi-GPU runs,
    and with N ranks in lock-step one stalled rank stalls all of them."""

    NAMES = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"),
             ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
             ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"),
             ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"))

    def __init__(self, index: int, period_s: float = 0.01):
        self.rows = []
        self.period = period_s
        self.active = False
        self.done = False
        self.nv = None
        self.handle = None
        self.thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            try:   # honours CUDA_VISIBLE_DEVICES: look the device up by the UUID torch reports
                uuid = "GPU-" + str(torch.cuda.get_device_properties(index).uuid)
                self.handle = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception as e:   # no NVML: the line says so instead of inventing clocks
            self.error = repr(e)

    def _read(self):
        nv = self.nv
        mhz = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
        mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
        return mhz, mask

    def start(self):
        if self.nv is None:
            return
        def loop():
            while not self.done:
                if self.active:
                    try:
                        self.rows.append((time.time(),) + self._read())
                    except Exception:
                        pass
                time.sleep(self.period)
        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    def activate(self):
        if self.nv is not None:
            try:   # one reading right away, so that even a region of a few ms has a sample
                self.rows.append((time.time(),) + self._read())
            except Exception:
                pass
        self.active = True

    def stop(self):
        self.active = False
        self.done = True
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable: " + getattr(self, "error", "?")]}
        if self.thread is not None:
            self.thread.join(timeout=1.0)
        sm = [r[1] for r in self.rows]
        reasons = set()
        for _, _, mask in self.rows:
            for name, attr in self.NAMES:
                if mask & int(getattr(self.nv, attr)):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(sm),
                "window": "timed region (NVML, sampled while the GPU executes the enqueued steps)"}


def model_args(n_items):
    return SimpleNamespace(num_items=n_items, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.2,
                           bert_attn_dropout=0.2)


def make_inputs(seed=42):
    from llamarec_b200 import synth
    return synth.make_sequences_fast(BATCH, N_ITEMS, MAX_LEN, seed=seed)


def build_product_model(device):
    from llamarec_b200 import LRURec, synth
    sd = synth.make_state_dict(1000, seed=42)                     # encoder weights (random init, reference shapes)
    table, bias = synth.make_table_bf16(N_ITEMS, seed=42, device=device)   # trunc-normal table, zero bias
    m = LRURec(model_args(N_ITEMS))
    m.load_state_dict({k: v for k, v in sd.items() if k not in ("embedding.token.weight", "model.bias")}, strict=False)
    m = m.to(device).eval()
    with torch.no_grad():
        m.embedding.token.weight.copy_(table)
        m.model.bias.copy_(bias)
    del table
    return m, sd


def cpu_oracle_run(sd, table_cpu, bias_cpu, ids, users, u=None):
    """The reference's path restated for the CPU: encode -> chunked last-position scoring with a running
    top-20 (the reference forward cannot allocate [B, L, N+1] at this size; BASELINE.md section 3).
    Returns (seconds, scores, ids).  `u` overrides the user states (parity runs on the kernel's bf16 operands)."""
    from oracle import lru_oracle as O
    sd_full = dict(sd)
    sd_full["embedding.token.weight"] = table_cpu
    sd_full["model.bias"] = bias_cpu
    x = ids[:users]                                    # (callers that pre-select users pass exactly `users` rows)
    t0 = time.perf_counter()
    with torch.no_grad():
        s, i = O.retrieve(x, sd_full, TOPK, exclude_history=True, chunk=65536, u=u)
    return time.perf_counter() - t0, s, i


def compare_lists(got_i, got_s, ref_i, ref_s, rtol=1e-5):
    """-> (identical, tie_only, wrong): per-user comparison of two sorted top-k lists; a differing list counts as
    tie_only when every position holds scores that agree within rtol (swaps / boundary replacements among ties)."""
    got_i, ref_i = got_i.long().cpu(), ref_i.long().cpu()
    got_s, ref_s = got_s.float().cpu(), ref_s.float().cpu()
    same = (got_i == ref_i).all(dim=1)
    tol = rtol * torch.clamp(ref_s.abs().amax(dim=1, keepdim=True), min=1.0)
    close = ((got_s - ref_s).abs() <= tol).all(dim=1)
    identical = int(same.sum())
    tie_only = int((~same & close).sum())
    return identical, tie_only, int(same.numel()) - identical - tie_only


def dump_outputs(out, directory):
    """Writes every tensor of one step's result as DIR/<name>.npy: floating point as float32 (float64 stays
    float64), integers as float64, which holds them exactly.  The full arrays are written: one step of this
    workload returns a few MB, far below DUMP_MAX_BYTES."""
    arrays = {}
    for name, t in out.items():
        if torch.is_tensor(t):
            t = t.detach().cpu()
            arrays[name] = t.float() if t.is_floating_point() and t.dtype != torch.float64 else t.double()
    total = sum(a.numel() * a.element_size() for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"--dump-outputs: {total} bytes exceed {DUMP_MAX_BYTES}"
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a.numpy())


def verbalizer_fraction(device, pk):
    """lrb_verbalizer_score at BASELINE configs[4]: CUDA-event time of the launch and its algorithmic bytes
    (hidden states once + the 20 label rows + the outputs, SURVEY 8d) against the measured copy bandwidth."""
    from llamarec_b200 import ManualVerbalizer, synth
    v = synth.make_verbalizer_inputs()

    class Tok:
        def encode(self, word, add_special_tokens=False):
            return [int(v["label_ids"][ord(word[-1]) - ord("A")])]
    vb = ManualVerbalizer(Tok(), classes=list(range(20)), label_words={i: chr(ord("A") + i) for i in range(20)},
                          prefix="", post_log_softmax=True)
    h, w = v["hidden"].to(device), v["lm_head"].to(device)
    for _ in range(5):
        vb.score_hidden(h, w)
    n = 50
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        vb.score_hidden(h, w)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / n * 1e3
    algo = 512 * 4096 * 2 + 20 * 4096 * 2 + 512 * 20 * 4
    return {"launches_per_step": 1, "us_per_launch": us, "algorithmic_bytes": algo, "GBps": algo / us * 1e-3,
            "frac_of_hbm_peak": algo / us * 1e-3 / pk["hbm_gbs"],
            "timing": "CUDA events around 50 back-to-back calls (includes launch latency: the kernel is latency-bound)"}


def kernel_trace(step_fn, n=4):
    """Per-kernel device times of `n` steps from a CUPTI kernel trace (torch.profiler), taken in a separate,
    untimed pass: -> {kernel name: (launches per step, mean microseconds)} or None when tracing is unavailable."""
    try:
        from torch.profiler import ProfilerActivity, profile
        step_fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n):
                step_fn()
            torch.cuda.synchronize()
        out = {}
        for e in prof.key_averages():
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = getattr(e, "cuda_time_total", 0.0)
            if e.count and t:
                out[e.key] = (e.count / n, float(t) / e.count)
        return out or None
    except Exception as ex:                                     # pragma: no cover - depends on the box
        print(f"kernel trace unavailable: {ex!r}", file=sys.stderr)
        return None


def run_reference(args, rank, world):
    if rank != 0:
        return
    from llamarec_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ids, _ = make_inputs()
    sd = synth.make_state_dict(1000, seed=42)
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    table, bias = synth.make_table_bf16(N_ITEMS, seed=42, device=dev)
    table, bias = table.cpu(), bias.cpu()
    # bounded sample: CPU_SAMPLE_USERS users per step -- a pass streams the whole 2.56 GB fp32 table whatever the
    # user count, so a small sample understates the reference (BASELINE.md: ~51 users/s at 1024 users, ~14 at 76);
    # shrunk only if warm-up + K steps would not end within ~10 minutes on this host
    probe_users = 64
    t_probe, _, _ = cpu_oracle_run(sd, table, bias, ids, probe_users)
    n_steps = args.warmup + args.steps
    budget_s = 600.0
    users = CPU_SAMPLE_USERS
    t_full_est = t_probe * max(1.0, users / probe_users) ** 0.5    # sub-linear: the table read is shared
    if t_full_est * n_steps > budget_s:
        users = max(probe_users, int(users * (budget_s / (t_full_est * n_steps)) ** 2))
    times = []
    for s in range(n_steps):
        dt, top_s, top_i = cpu_oracle_run(sd, table, bias, ids, users)
        if s >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs({"ids": top_i, "scores": top_s}, args.dump_outputs)
    total = sum(times)
    value = users * len(times) / total
    sample = (f"{users} of the {BATCH} users per step against the full 10M-item table "
              f"(fp32 oracle port, chunked 65536 items, running top-20; {cores} host threads)")
    line = {
        "impl": "reference", "metric": "users_per_sec_encode_score_top20", "value": value, "unit": "users/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "catalogue": N_ITEMS, "batch": BATCH, "max_len": MAX_LEN, "k": TOPK},
        "cpu_baseline": {"value": value, "unit": "users/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "users/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def run_product(args, rank, world, local_rank):
    import torch.distributed as dist
    from llamarec_b200.sharded import CudaBackend, ShardedRetriever, shard_range

    assert torch.cuda.is_available(), "bench.py (product arm) needs a CUDA device"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    model, sd = build_product_model(device)
    weak = world > 1 and args.scaling == "weak"
    ids_host, labels_host = make_inputs(42 + rank if weak else 42)     # weak: every rank has its own users
    ids_pinned = ids_host.pin_memory()
    ids_dev = ids_host.to(device)
    labels_dev = labels_host.to(device)
    ks = [1, 5, 10, 20]

    shard = world
    if world > 1:
        # row-shard degree S: the table is split over S ranks and replicated world/S times (S = world by
        # default: one copy of the table in the whole job, BASELINE.json configs[3])
        shard = args.shard_degree or world
        assert world % shard == 0 and (shard == world or weak), "--shard-degree must divide --gpus (weak scaling only)"
        group, grank = None, rank
        if shard != world:
            for g in range(world // shard):
                pg = dist.new_group(list(range(g * shard, (g + 1) * shard)))
                if rank // shard == g:
                    group, grank = pg, rank % shard
        retr = ShardedRetriever(CudaBackend(model, grank, shard, precision="bf16"), group=group, exchange=args.exchange)
        fn = retr.retrieve_dp if weak else retr.retrieve
        step = lambda x: fn(x, k=TOPK, exclude_history=True, labels=labels_dev, ks=ks)
        rows = shard_range(N_ITEMS + 1, grank, shard)
        local_rows = rows[1] - rows[0]
    else:
        step = lambda x: model.retrieve(x, k=TOPK, exclude_history=True, labels=labels_dev, ks=ks, precision="bf16")
        local_rows = N_ITEMS + 1

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # one sampler (rank 0's GPU) is enough
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("LRB_BENCH_NO_SAMPLER"):
        sampler.start()
    for _ in range(max(args.warmup, 3) + (5 if world > 1 else 0)):   # + first-use set-up of the exchange buffers
        step(ids_dev)
    barrier()

    # ---- device-resident timing (value) ----
    # a host-side pause longer than the launch queue's slack stalls the GPU, and with N ranks in lock-step any
    # rank's pause stalls all of them: keep the collector out of the timed regions
    import gc
    gc.collect()
    gc.disable()
    model.profile_events = []
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    # Let the host get ahead of the GPU before the timed steps start: a short spin kernel holds the stream while
    # the K steps are enqueued behind it, so they run back to back from a full launch queue.  Without it the
    # first steps are launched just in time, and a host-side pause on ANY rank (seen: one 15 ms step in a
    # 20-step run at N = 4, median 5.9 ms) stalls every rank of the lock-step exchange.  The spin is outside the
    # timed interval (marks[0] is recorded after it in stream order).
    try:
        torch.cuda._sleep(int(1.9e6 * min(100.0, 10.0 + 1.5 * args.steps)))
    except Exception:
        pass
    marks[0].record()
    for i in range(args.steps):
        out = step(ids_dev)
        marks[i + 1].record()
    sampler.activate()          # everything is enqueued: sample clocks while the GPU works through it
    barrier()
    clocks = sampler.stop()
    ms_total = marks[0].elapsed_time(marks[-1])
    step_ms = [a.elapsed_time(b) for a, b in zip(marks[:-1], marks[1:])]
    score_ms = [a.elapsed_time(b) for a, b in model.profile_events]
    model.profile_events = None
    last_main = {"ids": out["ids"].clone(), "scores": out["scores"].clone()}
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)          # before any later step reuses the result buffers

    def timed_variant(step_fn, x):
        """W warm-up + K timed steps of another step function, device-resident, same bracketing as the headline
        loop; -> (ms per step [max over ranks], scoring-call ms, the last step's lists)."""
        for _ in range(3):
            step_fn(x)
        barrier()
        model.profile_events = []
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
        try:
            torch.cuda._sleep(int(1.9e6 * min(100.0, 10.0 + 1.5 * args.steps)))
        except Exception:
            pass
        ev[0].record()
        for i in range(args.steps):
            o = step_fn(x)
            ev[i + 1].record()
        barrier()
        sc = [a.elapsed_time(b) for a, b in model.profile_events]
        model.profile_events = None
        per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
        t = torch.tensor([ev[0].elapsed_time(ev[-1]) / args.steps, statistics.mean(sc) if sc else 0.0,
                          statistics.median(per_step), max(per_step)], dtype=torch.float64, device=device)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        timed_variant.last_spread = {"ms_per_step_median": t[2].item(), "ms_per_step_max": t[3].item(),
                                     "steps_ms_this_rank": [round(v, 3) for v in per_step]}
        return t[0].item(), t[1].item(), {"ids": o["ids"].clone(), "scores": o["scores"].clone()}

    # ---- end-to-end through the public API with host buffers ----
    out_ids_host = torch.empty(BATCH, TOPK, dtype=torch.int32).pin_memory()
    out_scores_host = torch.empty(BATCH, TOPK, dtype=torch.float32).pin_memory()
    sums_host = torch.empty(len(ks), 3, dtype=torch.float32).pin_memory()
    ids_stage = torch.empty_like(ids_dev)

    def e2e_step():
        ids_stage.copy_(ids_pinned, non_blocking=True)
        o = step(ids_stage)
        out_ids_host.copy_(o["ids"], non_blocking=True)
        out_scores_host.copy_(o["scores"], non_blocking=True)
        sums_host.copy_(o["metric_sums"], non_blocking=True)

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    gc.enable()

    if os.environ.get("LRB_BENCH_PHASES") and weak:
        # developer aid: per-phase GPU times of the data-parallel step (rank 0, stderr)
        retr.phase_events = []
        for _ in range(10):
            step(ids_dev)
        barrier()
        evs, acc = retr.phase_events, {}
        retr.phase_events = None
        for (n0, e0), (n1, e1) in zip(evs[:-1], evs[1:]):
            if n1 != "begin":
                acc.setdefault(n1, []).append(e0.elapsed_time(e1))
        if rank == 0:
            print({k: round(1e3 * statistics.mean(v)) for k, v in acc.items()}, "us per phase", file=sys.stderr)

    t = torch.tensor([ms_total, e2e_s, statistics.mean(score_ms)], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_s, score_ms_mean = t.tolist()

    barrier()

    # ---- sub-records: the literal config-3 curve (4096 users IN TOTAL, strong scaling) and a non-zero bias ----
    sub = {}
    last_strong = None
    ids_strong = ids_dev
    if args.lean:
        if rank == 0:
            print(json.dumps({"lean": True, "value": (BATCH * world if weak else BATCH) * args.steps / (ms_total * 1e-3),
                              "ms_per_step": ms_total / args.steps, "kernel_ms": score_ms_mean}), flush=True)
        return
    if weak:
        ids_strong = make_inputs(42)[0].to(device)                  # the same 4096 users on every rank
        labels_strong = make_inputs(42)[1].to(device)
        strong_step = lambda x: retr.retrieve(x, k=TOPK, exclude_history=True, labels=labels_strong, ks=ks)
        ms_s, sc_s, last_strong = timed_variant(strong_step, ids_strong)
        sub["strong"] = {"value": BATCH / (ms_s * 1e-3), "unit": "users/s", "ms_per_step": ms_s, **timed_variant.last_spread,
                         "kernel_ms": sc_s, "global_batch": BATCH,
                         "what": f"the same {BATCH} users on every rank against 1/{world} of the rows each "
                                 "(batch-sharded encoder, all-gather of the states and of the local lists)"}
    # trained models never have a zero bias (the reference's own init draws it from the truncated normal,
    # model/lru.py:16-36); SURVEY 8d asks for the same step with an N(0, 0.01) bias: the folded-bias MMA runs
    g = torch.Generator(device=device).manual_seed(7)
    with torch.no_grad():
        model.model.bias.copy_(0.01 * torch.randn(N_ITEMS + 1, generator=g, device=device))
    ms_b, sc_b, last_bias = timed_variant(step, ids_dev)
    bias_spread = dict(timed_variant.last_spread)
    # (the CUPTI trace runs AFTER every timed region: tearing the profiler down right before a timed loop left one
    # 40-70 ms step in the loop that followed -- seen in the `bias` / `strong` sub-records of two runs)
    with torch.no_grad():
        saved_bias = model.model.bias.detach().clone()
        model.model.bias.zero_()
    # per-kernel device times of the headline step (zero bias): CUPTI trace, separate untimed pass; every rank runs
    # the same steps -- the multi-GPU step exchanges data -- rank 0 reports
    trace = kernel_trace(lambda: step(ids_dev))
    with torch.no_grad():
        model.model.bias.copy_(saved_bias)
    step(ids_dev)                                                  # re-prepare the bias block outside anything timed
    barrier()
    sub["bias"] = {"value": (BATCH * world if weak else BATCH) / (ms_b * 1e-3), "unit": "users/s", "ms_per_step": ms_b,
                   **bias_spread,
                   "kernel_ms": sc_b, "what": "the headline step with model.bias ~ N(0, 0.01) (folded-bias MMA active)"}

    # ---- parity of what was just timed (every rank checks users of ITS last step) ----
    # the same users scored by ONE unsharded single-GPU retrieve over the whole table: lists must be bit-identical
    # (merging exact per-shard top-K lists is exact).  At N = 1 the independent check is the CPU oracle on the
    # kernel's own bf16 operands (below, rank 0).
    n_par = min(PARITY_USERS, BATCH)
    parity = {}
    if world > 1:
        sel = torch.arange(0, BATCH, BATCH // n_par, device=device)[:n_par]
        model.set_row_shard(0, N_ITEMS + 1)
        ref_b = model.retrieve(ids_dev[sel].contiguous(), k=TOPK, exclude_history=True, precision="bf16")
        cb = compare_lists(last_bias["ids"][sel], last_bias["scores"][sel], ref_b["ids"], ref_b["scores"], rtol=0.0)
        with torch.no_grad():
            model.model.bias.zero_()
        ref_m = model.retrieve(ids_dev[sel].contiguous(), k=TOPK, exclude_history=True, precision="bf16")
        cm = compare_lists(last_main["ids"][sel], last_main["scores"][sel], ref_m["ids"], ref_m["scores"], rtol=0.0)
        cs = (0, 0, 0)
        if last_strong is not None:
            ref_s = model.retrieve(ids_strong[sel].contiguous(), k=TOPK, exclude_history=True, precision="bf16")
            cs = compare_lists(last_strong["ids"][sel], last_strong["scores"][sel], ref_s["ids"], ref_s["scores"], rtol=0.0)
        t = torch.tensor(list(cm) + list(cs) + list(cb), dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        v = [int(x) for x in t.tolist()]
        parity = {"users": n_par * world, "identical": v[0], "tie_only": v[1], "wrong": v[2],
                  "against": f"unsharded single-GPU retrieve of the same users over the whole table, {n_par} users "
                             "of the last timed step on every rank"}
        if last_strong is not None:
            sub["strong"]["parity_check"] = {"users": n_par * world, "identical": v[3], "tie_only": v[4], "wrong": v[5]}
        sub["bias"]["parity_check"] = {"users": n_par * world, "identical": v[6], "tie_only": v[7], "wrong": v[8]}

    if rank != 0:
        return
    pk = peaks()
    ms_per_step = ms_total / args.steps
    global_batch = BATCH * world if weak else BATCH
    value = global_batch * args.steps / (ms_total * 1e-3)
    e2e_value = global_batch * args.steps / e2e_s
    scored_users = BATCH * shard if weak else BATCH             # users one rank scores against its rows
    flops = 2.0 * scored_users * local_rows * 64                # algorithmic FLOPs of one rank's scoring call
    sms = torch.cuda.get_device_properties(device).multi_processor_count
    cap = (sms // 2 // 2) * 256                                 # users per scoring launch (score.cu: users_per_launch)
    score_launches = -(-scored_users // cap) if scored_users > cap else 1
    achieved = flops / (score_ms_mean * 1e-3) / 1e12
    # burst vs sustained: a timed region of K steps lasts ~0.1 s -- far from the seconds-long, power-capped regime
    # the sustained figure was measured in -- so the denominator is the BURST peak unless the region ran >= 2 s
    region_s = ms_total * 1e-3
    peak_kind = "sustained" if region_s >= 2.0 else "burst"
    peak_tf = pk["bf16_tflops_sustained"] if peak_kind == "sustained" else pk["bf16_tflops"]
    step_flops = flops
    traffic = None
    traffic_source = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            traffic = tj.get("score_topk_tc_dram_bytes_per_launch")
            traffic_source = tj.get("source")
        except (ValueError, OSError):
            traffic = None
    line = {
        "metric": "users_per_sec_encode_score_top20", "value": value, "unit": "users/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "ms_per_step_median": statistics.median(step_ms), "ms_per_step_max": max(step_ms), "higher_is_better": True,
        "scaling": "weak" if (weak or world == 1) else "strong", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "catalogue": N_ITEMS, "batch": BATCH, "batch_per_gpu": BATCH if (weak or world == 1) else BATCH // world,
                   "global_batch": global_batch, "max_len": MAX_LEN, "k": TOPK,
                   "parallelism": (f"item table row-sharded x{shard}" + (f" (replicated x{world // shard})" if shard != world else "")
                                   + f"; users data-parallel ({BATCH} per GPU); user states "
                                   f"gathered and local top-{TOPK} lists scattered to their owners by "
                                   + ("the kernels' own stores into peer memory over NVLink" if retr._peer and all(
                                       v is not None for v in retr._peer.values()) else "NCCL all-gather / all-to-all")
                                   if weak else
                                   f"item table row-sharded x{world}, same {BATCH} users on every rank, batch-sharded encoder"
                                   if world > 1 else "single GPU"),
                   "l2": "item table (1.28 GB bf16) is 10x larger than L2; no flush needed",
                   "scoring_operands": "bf16 table and user state, fp32 accumulate (tcgen05); encoder fp32"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "users/s", "h2d_bytes_per_step": ids_pinned.numel() * 8 * (world if weak else 1),
                "d2h_bytes_per_step": (BATCH * TOPK * 8 + len(ks) * 3 * 4) * (world if weak else 1)},
        # per step: prepare_sequences, 6 encoder kernels, scoring launch(es), local merge (+ final merge)
        # (+ the peer-push kernel of the data-parallel exchange; torch's barrier kernels are not counted)
        "gpu_launches": args.steps * (1 + 6 + score_launches + 1 + (1 if world > 1 else 0) + (1 if weak else 0)),
        "roofline": {"bound": "tensor", "kernel": "score_topk_tc_kernel", "achieved": achieved,
                     "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic,
                     "traffic_source": traffic_source,
                     "peak_source": f"{pk['source']} ({peak_kind} bf16: the timed region lasted {region_s:.2f} s)",
                     "frac_of_burst": achieved / pk["bf16_tflops"],
                     "frac_of_sustained": achieved / pk["bf16_tflops_sustained"],
                     "frac_step": step_flops / (ms_per_step * 1e-3) / 1e12 / peak_tf,
                     "frac_e2e": step_flops / (e2e_s / args.steps) / 1e12 / peak_tf,
                     "kernel_ms": score_ms_mean, "kernel_share_of_step": score_ms_mean / ms_per_step},
        "sub_records": sub,
    }
    # ---- secondary kernels: HBM fractions (north_star asks for scan / merge / metrics / verbalizer) ----
    if trace is not None:
        mine = {k: v for k, v in trace.items() if "lrb::" in k or k.startswith("lrb")}
        line["gpu_launches"] = int(round(sum(c for c, _ in mine.values()) * args.steps))
        line["gpu_launches_source"] = "counted: kernels of libllamarec_b200.so in a CUPTI trace of 4 steps x K"
        tok = int(model._prepare_sequences(ids_dev, all_positions=False, want_excl=False)["tok_offset"][-1].item())
        users_step = scored_users
        sec = {}
        for name, (cnt, us) in sorted(mine.items(), key=lambda kv: -kv[1][0] * kv[1][1]):
            mname = re.search(r"(\w+_kernel)", name)
            short = mname.group(1) if mname else name.split("(")[0].split("<")[0].split("::")[-1]
            rec = {"launches_per_step": cnt, "us_per_launch": us}
            if short == "lru_scan_kernel":
                # reads bu once, writes h once: 2 KB per token in the first block, 1 KB + 1 KB per user in the last
                algo = (2048.0 * tok + 1024.0 * tok + 1024.0 * BATCH) / 2.0     # mean of the two blocks' launches
                rec.update({"algorithmic_bytes": algo, "GBps": algo / us * 1e-3, "frac_of_hbm_peak": algo / us * 1e-3 / pk["hbm_gbs"]})
            elif short == "merge_metrics_kernel":
                S = 12 if world == 1 else None
                if S is not None:
                    algo = users_step * (S * TOPK * 8.0 + S * 4.0 + TOPK * 8.0 + 12.0)
                    rec.update({"algorithmic_bytes": algo, "GBps": algo / us * 1e-3, "frac_of_hbm_peak": algo / us * 1e-3 / pk["hbm_gbs"]})
            sec[short] = {**sec.get(short, {}), **rec} if short not in sec else sec[short]
        line["kernels"] = {"source": "CUPTI kernel trace (torch.profiler) of 4 steps after the timed regions; "
                                     "HBM fractions against the measured copy bandwidth", "per_kernel": sec}

    if world > 1:
        line["parity_check"] = parity
    if world == 1 and not args.skip_cpu_baseline:
        from oracle import lru_oracle as O
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        # (1) parity of the lists that were just timed: the CPU oracle on the kernel's own operands (bf16 user
        #     states and bf16 table, fp32 accumulate), PARITY_USERS users spread over the batch, with and
        #     without the bias; the encoder is checked against the oracle's fp32 encoder on the same users
        sel = torch.arange(0, BATCH, BATCH // n_par)[:n_par]
        u, u16 = model.encode(ids_dev[sel.to(device)].contiguous(), want_bf16=True)
        t16 = model._prepare()["table_bf16"].float().cpu()
        ids_sel = ids_host[sel]
        bias_cpu = model.model.bias.detach().float().cpu()
        _, rs, ri = cpu_oracle_run(sd, t16, bias_cpu, ids_sel, n_par, u=u16.float().cpu())
        cb = compare_lists(last_bias["ids"][sel.to(device)], last_bias["scores"][sel.to(device)], ri, rs)
        sub["bias"]["parity_check"] = {"users": n_par, "identical": cb[0], "tie_only": cb[1], "wrong": cb[2]}
        with torch.no_grad():
            model.model.bias.zero_()
        zero = torch.zeros(N_ITEMS + 1)
        _, rs, ri = cpu_oracle_run(sd, t16, zero, ids_sel, n_par, u=u16.float().cpu())
        cm = compare_lists(last_main["ids"][sel.to(device)], last_main["scores"][sel.to(device)], ri, rs)
        del t16
        table_cpu = model.embedding.token.weight.detach().float().cpu()
        sd_enc = dict(sd)
        sd_enc["embedding.token.weight"] = table_cpu
        enc_err = (O.encode(ids_sel, sd_enc) - u.cpu()).abs().max().item()
        del sd_enc
        line["parity_check"] = {"users": n_par, "identical": cm[0], "tie_only": cm[1], "wrong": cm[2],
                                "encoder_max_abs_err": enc_err,
                                "against": "CPU oracle (oracle/lru_oracle.py) on the kernel's bf16 operands, fp32 "
                                           "accumulate, chunked running top-20; encoder vs the oracle's fp32 encoder"}
        # (2) the reported CPU baseline: the reference's fp32 path (oracle port) on the host cores, one pass
        dt, _, _ = cpu_oracle_run(sd, table_cpu, zero, ids_host, CPU_SAMPLE_USERS)
        line["cpu_baseline"] = {
            "value": CPU_SAMPLE_USERS / dt, "unit": "users/s", "cores": cores, "kind": "port",
            "sample": f"{CPU_SAMPLE_USERS} of the {BATCH} users against the full 10M-item table, one pass "
                      f"({dt:.1f} s; fp32 oracle port of model/lru.py + chunked scoring + running top-20, "
                      f"{cores} host threads)"}
        del table_cpu
        # (3) stage-2 verbalizer kernel at BASELINE configs[4] (512 x 4096 x 32000, 20 labels): HBM fraction
        try:
            line["kernels"] = line.get("kernels") or {"per_kernel": {}}
            line["kernels"]["per_kernel"]["verbalizer_kernel"] = verbalizer_fraction(device, pk)
        except Exception as ex:                                   # pragma: no cover
            print(f"verbalizer timing skipped: {ex!r}", file=sys.stderr)
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="product", choices=["product", "reference"])
    ap.add_argument("--shard-degree", type=int, default=0,
                    help="N > 1, weak scaling: ranks per copy of the item table (default N: one copy per job)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "collective"],
                    help="N > 1, weak scaling: stores into peer memory (default when available) or NCCL collectives")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = 4096 users per GPU (default), strong = 4096 users in total")
    ap.add_argument("--lean", action="store_true",
                    help="profiling convenience (ncu): only the timed loops -- no kernel trace, sub-records, parity "
                         "checks or CPU legs")
    ap.add_argument("--skip-cpu-baseline", action="store_true",
                    help="profiling convenience: omit the ~20 s CPU oracle leg (the default run includes it)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, for comparing builds")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local_rank))
    try:
        run_product(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
