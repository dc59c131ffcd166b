#!/usr/bin/env python
"""Times the train step (`model.ce_loss(x, labels).backward()`, lrb_train_step / lrb_train_step_dropout) with dropout
off and on, alternated in one process, at the C2 (64 x 50, 12 087 rows) and C3 (2048 x 50, 11 001 rows) shapes of
synth.CONFIGS, bert_dropout = bert_attn_dropout = 0.2.  CUDA events around rounds of steps, at least 1 s of timed work
per variant; prints JSON with the device name and power limit, and writes it to --out as well if given.
Run: python tools/train_dropout_time.py [--seconds S] [--out result.json]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from llamarec_b200 import LRURec, synth  # noqa: E402


def gpu_info():
    try:   # read-only query
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = (s.strip() for s in out[0].split(","))
    except Exception as e:  # noqa: BLE001
        name, power = torch.cuda.get_device_name(0), f"unknown ({e.__class__.__name__})"
    return {"device": name, "power_limit": power}


def setup(cfg_name, p):
    cfg = synth.CONFIGS[cfg_name]
    args = SimpleNamespace(num_items=cfg.num_items, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=p,
                           bert_attn_dropout=p)
    m = LRURec(args)
    m.load_state_dict(synth.make_state_dict(cfg.num_items, seed=42))
    m = m.cuda().train()
    ids, last = synth.make_sequences(cfg, num_users=max(cfg.batch, 64), seed=42)
    ids, last = ids[:cfg.batch], last[:cfg.batch]
    lab = torch.zeros_like(ids)                   # next-item labels, 0 (ignored) at padding
    lab[:, :-1] = ids[:, 1:]
    lab[:, -1] = last.view(-1)
    lab[ids == 0] = 0
    return cfg, m, ids.cuda(), lab.cuda()


def step(m, x, y, dropout):
    m.zero_grad(set_to_none=True)
    loss = m.ce_loss(x, y, dropout=dropout)
    loss.backward()
    return loss


def time_round(m, x, y, dropout, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        step(m, x, y, dropout)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--seconds", type=float, default=1.5, help="timed seconds per variant and shape (>= 1)")
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("train_dropout_time.py needs a CUDA device")
    out = {**gpu_info(), "what": "ce_loss(x, labels[, dropout=True]).backward() with zero_grad, fp32, 2 blocks; "
                                 "dropout on: bert_dropout = bert_attn_dropout = 0.2; off/on rounds alternated",
           "configs": {}}
    torch.manual_seed(0)
    for name in ("c2_beauty", "c3_games"):
        cfg, m, x, y = setup(name, 0.2)
        loss_off = step(m, x, y, False).item()
        loss_on = step(m, x, y, True).item()
        for _ in range(3):                             # warm-up of both variants
            step(m, x, y, False)
            step(m, x, y, True)
        torch.cuda.synchronize()
        t1 = time_round(m, x, y, False, 3)             # calibrate: steps per round so that rounds cover a.seconds
        n = max(1, int(round(a.seconds * 1e3 / a.rounds / t1)))
        per = {False: [], True: []}
        for r in range(a.rounds):
            for dropout in ((False, True) if r % 2 == 0 else (True, False)):
                per[dropout].append(time_round(m, x, y, dropout, n))
        off, on = statistics.median(per[False]), statistics.median(per[True])
        out["configs"][name] = {
            "B": cfg.batch, "L": cfg.max_len, "rows": cfg.num_items + 1, "steps_per_round": n, "rounds": a.rounds,
            "timed_s_per_variant": n * a.rounds * (off + on) / 2e3,
            "step_ms_dropout_off": off, "step_ms_dropout_on": on, "overhead_pct": 100.0 * (on - off) / off,
            "rounds_ms_dropout_off": per[False], "rounds_ms_dropout_on": per[True],
            "loss_dropout_off": loss_off, "loss_dropout_on": loss_on}
        del m
        torch.cuda.empty_cache()
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
