"""Cost of top-K lists longer than 50 (DESIGN section 2.2) at the headline shape.

4096 users x 10 M items, L = 50, the benchmark's table (trunc-normal, sigma 0.02), zero bias and N(0, 0.01) bias.
Per case: ms per retrieve() call (host clock around calls that end in a device synchronise, median of --reps after
one warm-up call) for bf16 K = 20 and 50 (the streaming kernels) and K = 51 ... 1024 (the wide path); for the wide
path also the split into sample / collect+select / retry / fallback / merge from CUDA events of one more call, the
topk_path counts and the collected mean and maximum.  Then fp32 at C3's shape (2048 users x 11 001 items) at
K = 50, 100, 1024.  Prints the card's name and power limit, one JSON line per case and a markdown table; writes
nothing.

    python tools/wide_topk_time.py [--items 10000000] [--users 4096] [--reps 5]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from types import SimpleNamespace

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from llamarec_b200 import LRURec, synth  # noqa: E402


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), out


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def model(items, table, state, bias):
    args = SimpleNamespace(num_items=items, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.0,
                           bert_attn_dropout=0.0)
    with torch.device("cuda"):
        m = LRURec(args)
    m.load_state_dict(state, strict=False)
    with torch.no_grad():
        m.embedding.token.weight.copy_(table)
        m.model.bias.copy_(bias)
    return m.eval()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=10_000_000)
    ap.add_argument("--users", type=int, default=4096)
    ap.add_argument("--max-len", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wide_topk_time.py measures on the GPU; no CUDA device is visible")
    props = torch.cuda.get_device_properties(0)
    print(json.dumps({"device": props.name, "sms": props.multi_processor_count, "nvidia-smi": power_limit()}))

    sd = synth.make_state_dict(1000, seed=42)
    state = {k: v for k, v in sd.items() if k not in ("embedding.token.weight", "model.bias")}
    table, _ = synth.make_table_bf16(a.items, seed=42, device="cuda")
    ids, _ = synth.make_sequences_fast(a.users, a.items, a.max_len, seed=42)
    x = ids.cuda()
    g = torch.Generator(device="cuda").manual_seed(7)
    bias_n = torch.randn(a.items + 1, device="cuda", generator=g) * 0.01

    rows = []
    for bias_name in ("zero", "N(0,0.01)"):
        m = model(a.items, table, state, bias_n if bias_name != "zero" else torch.zeros_like(bias_n))
        u, u16 = m.encode(x, want_bf16=True)
        for k in (20, 50, 51, 100, 200, 500, 1024):
            t, res = timed(lambda: m.retrieve(x, k=k, precision="bf16", u=u, u_bf16=u16), a.reps)
            row = {"case": f"bf16 {a.users}x{a.items}", "bias": bias_name, "K": k, "ms": round(t, 3)}
            if k > 50:
                m.wide_profile_events = []
                m.retrieve(x, k=k, precision="bf16", u=u, u_bf16=u16)
                torch.cuda.synchronize()
                for name, e0, e1 in m.wide_profile_events:
                    if e1 is not None:
                        row[name + "_ms"] = round(e0.elapsed_time(e1), 3)
                m.wide_profile_events = None
                path = res["topk_path"].long()
                coll = res["topk_collected"].double()
                row["paths"] = torch.bincount(path, minlength=3).tolist()
                row["collected_mean"] = round(float(coll.mean()), 1)
                row["collected_max"] = int(coll.max())
            print(json.dumps(row), flush=True)
            rows.append(row)
        del m
        torch.cuda.empty_cache()

    # fp32 at C3's shape: the dense + select path
    c3_items, c3_users = 11_000, 2048
    sd3 = synth.make_state_dict(c3_items, seed=3, bias_std=0.01)
    with torch.device("cuda"):
        m3 = LRURec(SimpleNamespace(num_items=c3_items, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.0,
                                    bert_attn_dropout=0.0))
    m3.load_state_dict(sd3)
    m3 = m3.eval()
    ids3, _ = synth.make_sequences_fast(c3_users, c3_items, 200, seed=3)
    x3 = ids3.cuda()
    u3 = m3.encode(x3)
    for k in (50, 100, 1024):
        t, _ = timed(lambda: m3.retrieve(x3, k=k, precision="fp32", u=u3), a.reps)
        row = {"case": f"fp32 {c3_users}x{c3_items + 1}", "bias": "N(0,0.01)", "K": k, "ms": round(t, 3)}
        print(json.dumps(row), flush=True)
        rows.append(row)

    print()
    print("| case | bias | K | ms / call | sample | collect+select | retry | fallback | merge | paths 0/1/2 "
          "| collected mean / max |")
    print("|---|---|---|---|---|---|---|---|---|---|---|")
    for r in rows:
        ph = [str(r.get(n + "_ms", "")) for n in ("sample", "collect+select", "retry", "fallback", "merge")]
        paths = "/".join(map(str, r["paths"])) if "paths" in r else ""
        coll = f"{r['collected_mean']} / {r['collected_max']}" if "paths" in r else ""
        print(f"| {r['case']} | {r['bias']} | {r['K']} | {r['ms']} | " + " | ".join(ph) + f" | {paths} | {coll} |")


if __name__ == "__main__":
    main()
