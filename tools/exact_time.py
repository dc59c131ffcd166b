"""Cost of retrieve(precision="exact") against "bf16" and "fp32" at the headline shape.

4096 users x 10 M items, L = 50, K = 20 and 50; zero bias and N(0, 0.01) bias; the benchmark's table (trunc-normal,
sigma 0.02) and the same table x 10 ("trained-like").  Per case: ms per retrieve() call (host clock around calls that
end in a device synchronise, median of --reps after one warm-up call), the share of users certified by pass A, the
mean and maximum number of ids collected per user that pass A did not certify, the users sent to the fp32 path
(collect overflow), and whether the exact lists equal the fp32 ones.  Prints one JSON line per case and a markdown
table; writes nothing.

    python tools/exact_time.py [--items 10000000] [--users 4096] [--reps 5]
"""
import argparse
import json
import os
import statistics
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--items", type=int, default=10_000_000)
    ap.add_argument("--users", type=int, default=4096)
    ap.add_argument("--max-len", type=int, default=50)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("exact_time.py measures on the GPU; no CUDA device is visible")
    dev = torch.device("cuda")
    props = torch.cuda.get_device_properties(dev)
    print(json.dumps({"device": props.name, "sms": props.multi_processor_count}))

    args = SimpleNamespace(num_items=a.items, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.0,
                           bert_attn_dropout=0.0)
    sd = synth.make_state_dict(1000, seed=42)
    with torch.device("cuda"):
        m = LRURec(args)
    m.load_state_dict({k: v for k, v in sd.items() if k not in ("embedding.token.weight", "model.bias")},
                      strict=False)
    m = m.eval()
    table, _ = synth.make_table_bf16(a.items, seed=42, device="cuda")
    ids, _ = synth.make_sequences_fast(a.users, a.items, a.max_len, seed=42)
    x = ids.to(dev)
    g = torch.Generator(device="cuda").manual_seed(7)
    bias_n = torch.randn(a.items + 1, device="cuda", generator=g) * 0.01

    rows = []
    for scale in (1.0, 10.0):
        for bias_name in ("zero", "N(0,0.01)"):
            with torch.no_grad():
                m.embedding.token.weight.copy_(table * scale)
                m.model.bias.copy_(bias_n if bias_name != "zero" else torch.zeros_like(bias_n))
            m._prepare()
            for k in (20, 50):
                t16, _ = timed(lambda: m.retrieve(x, k=k, precision="bf16"), a.reps)
                tex, ex = timed(lambda: m.retrieve(x, k=k, precision="exact"), a.reps)
                t32, r32 = timed(lambda: m.retrieve(x, k=k, precision="fp32"), a.reps)
                path = ex["exact_path"].long()
                coll = ex["exact_collected"][path != 0].double()
                same = bool(torch.equal(ex["ids"], r32["ids"]) and
                            torch.equal(ex["scores"].view(torch.int32), r32["scores"].view(torch.int32)))
                row = {"table": "x%g" % scale, "bias": bias_name, "K": k, "bf16_ms": round(t16, 3),
                       "exact_ms": round(tex, 3), "fp32_ms": round(t32, 3), "exact_over_bf16": round(tex / t16, 2),
                       "certified": round(float((path == 0).float().mean()), 4),
                       "collected_mean": round(float(coll.mean()), 1) if coll.numel() else 0.0,
                       "collected_max": int(coll.max()) if coll.numel() else 0,
                       "overflow": int((path == 2).sum()), "exact_equals_fp32": same}
                print(json.dumps(row), flush=True)
                rows.append(row)
    print()
    print("| table | bias | K | bf16 ms | exact ms | fp32 ms | exact / bf16 | certified | collected mean / max "
          "| overflow | = fp32 |")
    print("|---|---|---|---|---|---|---|---|---|---|---|")
    for r in rows:
        print(f"| {r['table']} | {r['bias']} | {r['K']} | {r['bf16_ms']} | {r['exact_ms']} | {r['fp32_ms']} | "
              f"{r['exact_over_bf16']} | {r['certified']:.1%} | {r['collected_mean']} / {r['collected_max']} | "
              f"{r['overflow']} | {r['exact_equals_fp32']} |")


if __name__ == "__main__":
    main()
