import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from types import SimpleNamespace
from llamarec_b200 import LRURec, LRURetriever, synth
dev = torch.device("cuda")
cfg = synth.CONFIGS["c3_games"]
sd = synth.make_state_dict(cfg.num_items, seed=42, bias_std=0.01)
a = SimpleNamespace(num_items=cfg.num_items, bert_hidden_units=64, bert_num_blocks=2, bert_dropout=0.2, bert_attn_dropout=0.2, metric_ks=list(cfg.metric_ks), llm_negative_sample_size=19)
m = LRURec(a); m.load_state_dict(sd); m = m.to(dev).eval()
ids, labels = synth.make_sequences(cfg, num_users=2048, seed=42)
x, y = ids.to(dev), labels.to(dev)
print("tokens", int((ids > 0).sum()), "mean len", float((ids > 0).sum(1).float().mean()))
tr = LRURetriever(a, m)
fn = lambda: tr.calculate_metrics((x, y.view(-1, 1)))
for _ in range(5): fn()
torch.cuda.synchronize()
from torch.profiler import profile, ProfilerActivity
with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
    for _ in range(10): fn()
    torch.cuda.synchronize()
rows = []
for e in prof.key_averages():
    t = getattr(e, "device_time_total", 0) or 0
    if t: rows.append((t / 10, e.count / 10, e.key[:90]))
for r in sorted(rows, reverse=True)[:25]: print("%9.1f us/step  x%.1f  %s" % r)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(20): fn()
e1.record(); torch.cuda.synchronize()
print("ms per call", e0.elapsed_time(e1) / 20)
import time
t0 = time.perf_counter()
for _ in range(20): fn()
torch.cuda.synchronize()
print("wall ms per call", (time.perf_counter() - t0) / 20 * 1e3)
