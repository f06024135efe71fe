#!/usr/bin/env python3
"""BASELINE configs[4] shape on one GPU: ChatCompletion bodies with Zipf(1.2) sizes 1–64 KB through the host-buffer translate call.
Shows what size-class bucketing buys: the resident part times one launch in the largest class against one launch per size
class over a document map (the host-buffer call always buckets).  One JSON line."""
import argparse, json, os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import _workload as W
import _oracle as O
import aigw_b200 as A
from aigw_b200 import capi

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=200_000)
ap.add_argument("--steps", type=int, default=4)
ap.add_argument("--warmup", type=int, default=3)
ap.add_argument("--schema", default="aws-bedrock")
a = ap.parse_args()
rng = np.random.default_rng(5)
k = np.arange(1, 65); p = k ** -1.2; p /= p.sum()
kb = rng.choice(k, size=a.n, p=p)
pools = {}
for t in sorted(set(int(x) for x in kb)):
    cnt = int((kb == t).sum()); m = min(cnt, 512)
    arena, offs, lens = W.chat_corpus(5, 0, m, target=min(t * 1024, 62000), jitter=max(16, t * 16))
    pools[t] = [bytes(arena[int(offs[i]):int(offs[i]) + int(lens[i])]) for i in range(m)]
cur = {t: 0 for t in pools}
bodies = []
for t in kb:
    t = int(t); bodies.append(pools[t][cur[t] % len(pools[t])]); cur[t] += 1
arena, offs, lens = capi.pack_bodies(bodies)
ctx = A.Context(0)
pin, pp = ctx.host_array(len(arena) + 64); pin[: len(arena)] = arena
cfg = capi.Context.cfg(a.schema)
o2 = offs[: len(bodies)].copy()
for _ in range(a.warmup): res, out, st = ctx.chat_translate_host(cfg, pin, o2, lens)
t0 = time.perf_counter()
for _ in range(a.steps): res, out, st = ctx.chat_translate_host(cfg, pin, o2, lens)
wall = (time.perf_counter() - t0) / a.steps
ok = int((res["status"] == 0).sum())
# sampled parity
for i in range(0, a.n, max(1, a.n // 300)):
    t = O.chat_translate(a.schema, bodies[i])
    assert int(res[i]["status"]) == t.status, (i, int(res[i]["status"]), int(res[i]["reason"]), t.status)
    if t.status == 0:
        o = int(res[i]["out_off"]) + int(res[i]["path_len"])
        assert bytes(out[o:o + int(res[i]["body_len"])]) == t.body
nbytes = int(lens.astype(np.int64).sum()); obytes = int(res["body_len"].astype(np.int64).sum())
# device-resident A/B: one launch in the largest class vs one launch per size class over a document map
n = len(bodies)
out_cap = 2 * len(arena) + 600 * n
d_b = ctx.dalloc(len(arena) + 64); d_o = ctx.dalloc(o2.nbytes); d_l = ctx.dalloc(lens.nbytes); d_out = ctx.dalloc(out_cap); d_r = ctx.dalloc(n * 32); d_u = ctx.dalloc(64); d_m = ctx.dalloc(n * 4)
ctx.h2d(d_b, arena); ctx.h2d(d_o, o2); ctx.h2d(d_l, lens)
CLS = [2048, 5120, 9216, 17408, 33792, 65536]
cls = np.searchsorted(np.array(CLS), lens, side="left")
order = np.argsort(cls, kind="stable").astype(np.uint32); ctx.h2d(d_m, order)
starts = np.concatenate([[0], np.cumsum(np.bincount(cls, minlength=6))])
def single():
    ctx.memset(d_u, 0, 8); return ctx.chat_translate_device(cfg, d_b, d_o, d_l, n, int(lens.max()), d_out, out_cap, d_r, d_u)
def bucketed():
    ctx.memset(d_u, 0, 8); t = 0.0
    for k in range(6):
        c = int(starts[k + 1] - starts[k])
        if c: t += ctx.chat_translate_device_mapped(cfg, d_b, d_o, d_l, d_m, int(starts[k]), c, CLS[k], d_out, out_cap, d_r, d_u)
    return t
for f in (single, bucketed): f(); f()
ms_single = float(np.mean([single() for _ in range(a.steps)])); ms_bucket = float(np.mean([bucketed() for _ in range(a.steps)]))
rres = np.zeros(n, dtype=A.DocResult); ctx.d2h(rres, d_r)
assert (rres["status"] == res["status"]).all() and (rres["body_len"] == res["body_len"]).all()
print(json.dumps({"metric": "extproc bodies/sec, Zipf(1.2) 1-64 KB ChatCompletion translate, host buffers", "value": a.n / wall, "unit": "bodies/s", "ms_per_step": wall * 1e3,
                  "config": {"workload": f"configs[4] shape on one GPU: {a.n} bodies, sizes clamp(1 KB x Zipf(1.2), 1 KB, 64 KB), mean {nbytes // a.n} B, schema {a.schema}",
                             "accepted": ok, "declined_or_error": a.n - ok},
                  "gb_per_s_in_plus_out": (nbytes + obytes) / wall / 1e9,
                  "resident": {"single_class_ms": ms_single, "bucketed_ms": ms_bucket, "single_class_bodies_per_s": n / ms_single * 1e3, "bucketed_bodies_per_s": n / ms_bucket * 1e3,
                               "bucketed_gb_per_s": (nbytes + obytes) / ms_bucket / 1e6, "docs_per_class": [int(x) for x in np.bincount(cls, minlength=6)]}, "kernel_ms": st["kernel_ms"], "gpu_launches": st["gpu_launches"], "h2d_bytes": st["h2d_bytes"], "d2h_bytes": st["d2h_bytes"]}))
