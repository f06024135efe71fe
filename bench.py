#!/usr/bin/env python3
"""bench.py — BASELINE.json's metric.  `--config` selects the BASELINE config (default 2, the one the metric is quoted on):

  1  128 OpenAI ChatCompletion bodies (2 KB, 4 messages): passthrough translate + usage count, per-call latency shape
  2  1 M OpenAI→AWS Bedrock Converse body translate, 4 KB bodies, per GPU                      (headline; the driver's run)
  4  SSE streamed response parse through the per-chunk stream ABI: streams x 256 chunks x 80 B, usage extract
  5  mixed-provider fan-out: OpenAI / Gemini / Anthropic / Bedrock translate, Zipf(1.2) body size 1-64 KB, requests routed to
     a device by hash64(request-id) % n_gpus
  (3, embeddings + BPE count, is not built: the line says so.)

One step = one pass of the hot path over a batch of synthetic bodies.  Printed (rank 0, one JSON line):
  value      units/s, whole job, inputs already resident in HBM (device API; CUDA-event time)
  e2e        the same through the host-buffer C-ABI call; the timed region includes the multi-threaded copy of the bodies
             into the library's pinned arena, H2D, kernels, D2H and the copy of the produced bytes out of the pinned arena
  roofline   HBM roofline of the translate pass: algorithmic bytes (input + output) ÷ CUDA-event duration vs MEASURED_PEAKS.json
  cpu_baseline  the oracle (CPU restatement of the reference Go path) on this box's host cores, bounded sample, rank 0 / N=1
--impl reference times the CPU restatement alone on the same config (the reference is Go; no Go toolchain exists in the image).
--dump-outputs DIR (config 2) writes what the device pass returned in its last timed step, a fixed seeded sample, as DIR/*.npy
(float32 / float64, under 64 MB): with the same arguments the inputs are the same, so two builds can be compared output for output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (no __pycache__ of the modules it imports)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "extproc bodies/sec, 4 KB ChatCompletion translate (OpenAI→AWS Bedrock Converse)"
SEED = 2
WORKLOAD2 = "configs[1]: OpenAI→AWS Bedrock Converse translate, 4 KB bodies (4096±32 B, 4–8 messages, 10% tool use), seed 2"


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    """DRAM read+write bytes per body of the three stages, from the committed ncu --set full capture of this round
    (profiles/r02_traffic.json, written by tools/ncu_traffic.py from gpurun_out/*.ncu-rep); None when absent."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return None


def batcher_block():
    """The per-request path under concurrency: tools/batcher_load.cpp (C++ threads standing in for goroutines behind cgo) drives
    aigw_batcher_translate with the bodies of the workload; callers, req/s and latency percentiles per setting."""
    try:
        import _workload as W
        with tempfile.TemporaryDirectory() as tmp:   # the tree may be read-only and fixed names under /tmp may belong to another user
            exe, bodies_f, offs_f = (os.path.join(tmp, f) for f in ("aigw_batcher_load", "bodies.bin", "offs.u64"))
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tools", "batcher_load.cpp"), "-L", os.path.join(ROOT, "aigw_b200"),
                                   "-laigw_b200", "-Wl,-rpath," + os.path.join(ROOT, "aigw_b200"), "-lpthread", "-o", exe])
            ar, of, le = W.chat_corpus(2, 0, 8000)
            packed = b"".join(bytes(ar[int(of[i]):int(of[i]) + int(le[i])]) for i in range(8000))
            po = np.zeros(8001, dtype=np.uint64); np.cumsum(le[:8000], out=po[1:])
            open(bodies_f, "wb").write(packed); open(offs_f, "wb").write(po.tobytes())
            rows = []
            for threads, reqs, mb, win in ((1, 2000, 1, 0), (64, 1000, 64, 20), (256, 800, 256, 40), (512, 600, 512, 50)):
                out = subprocess.check_output([exe, bodies_f, offs_f, "8000", str(threads), str(reqs), str(mb), str(win)], timeout=120).decode()
                d = json.loads(out.strip().split("\n")[-1])
                rows.append({"callers": threads, "max_batch": mb, "window_us": win, "req_per_s": d["requests_per_s"], "p50_us": d["p50_us"], "p99_us": d["p99_us"], "mean_batch": d["mean_batch"],
                             "ok": d["ok"], "declined": d["declined"], "failed": d["failed"]})
            return {"tool": "tools/batcher_load.cpp (closed loop: every caller submits its next request when the previous one returns)", "rows": rows}
    except Exception as e:  # the bench line must not depend on a side tool
        return {"error": str(e)[:200]}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        busy = sorted(sm)[len(sm) // 2:] if sm else []  # upper half ≈ samples under load
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def host_cores():
    """threads the CPU legs may really use: the scheduler affinity mask, further limited by a cgroup CPU quota when one is set"""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q = open("/sys/fs/cgroup/cpu.max").read().split()
        if q[0] != "max":
            n = max(1, min(n, int(float(q[0]) / float(q[1]) + 0.5)))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read()); period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = max(1, min(n, int(quota / period + 0.5)))
        except Exception:
            pass
    return n


def build_checker():
    """oracle + workload generator only (the reference arm must not map the product library)"""
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
    import _workload as W
    W.lib()


def cpu_oracle_rate(schema, arena, offs, n_sample, threads):
    import _oracle as O
    status = np.zeros(n_sample, dtype=np.int32); olen = np.zeros(n_sample, dtype=np.uint32); tot = C.c_uint64(0)
    sec = O.lib().oracle_chat_translate_batch(schema, arena.ctypes.data, offs.ctypes.data, n_sample, 0, threads, status.ctypes.data, olen.ctypes.data, C.byref(tot))
    return n_sample / sec, status


def config2_dict(n):
    return {"workload": WORKLOAD2, "bodies_per_gpu_per_step": n, "sharding": "hash(request-id)→device, no collective"}


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(a, ncpu):
    """the reference's own CPU implementation of the path.  It is Go and cannot be built here, so the restatement (oracle, kind
    "port") is timed with every usable host thread on a bounded sample of the SAME workload (config and metric identical)."""
    import _workload as W
    build_checker()
    n = a.bodies
    sample = min(n, a.cpu_sample)
    arena, offs, lens = W.chat_corpus(SEED, 0, sample, threads=ncpu)
    times = []
    for s in range(a.warmup + a.steps):
        rate, status = cpu_oracle_rate(1, arena, offs, sample, ncpu)
        assert (status == 0).all()
        if s >= a.warmup:
            times.append(sample / rate)
    val = sample * a.steps / float(np.sum(times))
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": "bodies/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                      "ms_per_step": 1e3 * n / val, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                      "config": config2_dict(n),
                      "cpu_baseline": {"value": val, "unit": "bodies/s", "cores": ncpu, "kind": "port",
                                       "sample": f"first {sample} bodies of the {n}-body step per timed step x {a.steps} steps, {ncpu} threads; ms_per_step is extrapolated to the full step"},
                      "e2e": {"value": val, "unit": "bodies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------------------ config 2 (headline)
def escaped_corpus(arena, offs, lens, count):
    """accept-rate corpus: the first `count` workload bodies, every tenth re-serialised the way ASCII-only JSON encoders write them
    (non-ASCII characters as \\uXXXX, slashes escaped in half of those)"""
    out = []
    for i in range(count):
        b = bytes(arena[int(offs[i]):int(offs[i]) + int(lens[i])])
        if i % 10 == 0:
            b = json.dumps(json.loads(b), ensure_ascii=True, separators=(",", ":")).encode()
            if i % 20 == 0:
                b = b.replace(b"/", b"\\/")
        out.append(b)
    return out


DUMP_ROWS = 65536          # result rows written by --dump-outputs (as float64: 5 MB)
DUMP_OUT_BYTES = 8 << 20   # output bytes written by --dump-outputs (as float32: 32 MB)
DUMP_FIELDS = ("status", "reason", "body_len", "path_len", "model_off", "model_len", "body_kind", "flags", "in_len")


def dump_outputs(out_dir, ctx, res, d_out):
    """--dump-outputs: what the last timed step of the device pass returned, on a fixed seeded sample of the bodies, so that two builds
    can be compared output for output.  sample_index: the sampled bodies; result_<field>: their result rows (out_off is left out: where
    a record lands in the output arena depends on the order the blocks claim space); output_bytes: the path + body bytes of the first
    len(output_len) sampled bodies back to back, output_len[i] of them for the i-th (0 unless its status is OK)."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(res)
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, DUMP_ROWS), replace=False))
    rows = res[idx]
    np.save(os.path.join(out_dir, "sample_index.npy"), idx.astype(np.float64))
    for f in DUMP_FIELDS:
        np.save(os.path.join(out_dir, f"result_{f}.npy"), rows[f].astype(np.float64))
    rec = np.where(rows["status"] == 0, rows["path_len"].astype(np.int64) + rows["body_len"].astype(np.int64), 0)
    m = int(np.searchsorted(np.cumsum(rec), DUMP_OUT_BYTES, side="right"))
    out = np.zeros(int(rec[:m].sum()), dtype=np.uint8); o = 0
    for r, l in zip(rows[:m], rec[:m]):
        if l:
            ctx.d2h(out[o:o + l], d_out + int(r["out_off"]))
            o += int(l)
    np.save(os.path.join(out_dir, "output_len.npy"), rec[:m].astype(np.float64))
    np.save(os.path.join(out_dir, "output_bytes.npy"), out.astype(np.float32))


def run_config2(a, rank, world, local, ncpu):
    import _oracle as O
    import _workload as W
    import __graft_entry__ as entry
    entry.build()
    import aigw_b200 as A
    from aigw_b200 import capi
    node = A.load_library().aigw_bind_numa(local)      # this rank's threads and pinned arenas stay on the GPU's NUMA node
    ncpu_local = host_cores()
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    ctx = A.Context(local)
    n = a.bodies
    # ---- synthetic shard for this rank (the bodies a shim would hold in Go memory) and the pinned arena the library reads
    lens = W.chat_lens(SEED, rank * n, n, threads=ncpu_local)
    offs = W.chat_offsets(lens)
    in_bytes = int(offs[-1]) + 16
    src = np.full(in_bytes, 0x20, dtype=np.uint8)
    W.chat_fill(SEED, rank * n, n, src, offs, lens, threads=ncpu_local)
    arena, arena_ptr = ctx.host_array(in_bytes)
    arena[:] = src
    max_len = int(lens.max())
    cfg = ctx.cfg("aws-bedrock")

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload, all host threads and 1 thread
    cpu = None
    if rank == 0 and world == 1:
        r1, _ = cpu_oracle_rate(1, src, offs, max(2000, min(a.cpu_sample // 8, 50_000)), 1)
        rN = max(cpu_oracle_rate(1, src, offs, min(n, a.cpu_sample), ncpu)[0] for _ in range(2))
        cpu = {"value": rN, "unit": "bodies/s", "cores": ncpu, "kind": "port", "sample": f"first {min(n, a.cpu_sample)} bodies of the workload, {ncpu} threads (1 thread: {r1:.0f} bodies/s)",
               "p50_us_per_body_1thread": 1e6 / r1}

    # ---- device-resident pass ("value")
    d_in = ctx.dalloc(in_bytes); d_off = ctx.dalloc(offs.nbytes); d_len = ctx.dalloc(lens.nbytes)
    out_cap = int(in_bytes * 1.25) + n * 64 + 4096
    d_out = ctx.dalloc(out_cap); d_res = ctx.dalloc(n * 32); d_used = ctx.dalloc(8)
    ctx.h2d(d_in, arena); ctx.h2d(d_off, offs); ctx.h2d(d_len, lens)

    def barrier():
        ctx.sync()
        if dist is not None:
            dist.barrier()
        ctx.sync()

    for _ in range(a.warmup):
        ctx.memset(d_used, 0, 8)
        ctx.chat_translate_device(cfg, d_in, d_off, d_len, n, max_len, d_out, out_cap, d_res, d_used)
    sampler = ClockSampler(local); sampler.start()
    barrier()
    t0 = time.perf_counter(); kms = []; dev_launches = 0
    for _ in range(a.steps):
        ctx.memset(d_used, 0, 8)
        kms.append(ctx.chat_translate_device(cfg, d_in, d_off, d_len, n, max_len, d_out, out_cap, d_res, d_used))
        dev_launches += ctx.chat_last_profile()["launches"]
    barrier()
    wall = time.perf_counter() - t0
    dev_s = float(np.sum(kms)) / 1e3
    res = np.zeros(n, dtype=A.DocResult); ctx.d2h(res, d_res)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, ctx, res, d_out)
    n_ok = int((res["status"] == A.AIGW_OK).sum())
    out_bytes = int(res["body_len"].astype(np.uint64).sum() + res["path_len"].astype(np.uint64).sum())
    alg_bytes = int(lens.astype(np.uint64).sum()) + out_bytes  # SURVEY.md §8d: bytes_in + bytes_out per body
    # per-stage times: one extra pass outside the timed region with stage events (the stages already run back to back on one stream)
    ctx.chat_set_profile(True); ctx.memset(d_used, 0, 8)
    serial_ms = ctx.chat_translate_device(cfg, d_in, d_off, d_len, n, max_len, d_out, out_cap, d_res, d_used)
    pr = ctx.chat_last_profile(); stage = [pr["index_ms"], pr["walk_ms"], pr["emit_ms"]]
    ctx.chat_set_profile(False)
    for p in (d_in, d_off, d_len, d_out, d_res, d_used):
        ctx.dfree(p)

    # ---- end to end through the host-buffer C-ABI call, copies into and out of the pinned arenas included
    e2e = None; p50 = None; launches = dev_launches; checked = 0; accept = None; batcher = None
    if not a.skip_e2e:
        WL = W.lib()
        # The copies in and out model the shim's goroutines.  Default: one call over the whole step (copy in, call, copy out).  With
        # --e2e-lanes L --e2e-parts P the step is cut into P sub-batches dealt to L host threads, each with its own context on this GPU
        # (one device call in flight per context), so that one lane copies while the other waits on the GPU — measured slower than the
        # single call (sub-batches lose the call's internal H2D / kernel / D2H overlap; see DESIGN.md §4.6).  Either way every byte goes
        # arena <- caller memory, H2D, kernels, D2H, caller memory <- arena inside the timed region.
        import threading
        parts = max(1, a.e2e_parts); lanes = max(1, min(a.e2e_lanes, parts))
        pb = [int(round(k * n / parts)) for k in range(parts + 1)]
        sink_off = [int(offs[pb[k]]) + int(offs[pb[k]]) // 8 + k * (1 << 16) for k in range(parts)]   # room for 1.12x the input bytes of every part
        sink = np.empty(int(in_bytes * 1.13) + (parts + 1) * (1 << 16), dtype=np.uint8)
        lane_ctx = [ctx] + [A.Context(local) for _ in range(lanes - 1)]
        part_res = [None] * parts; part_st = [None] * parts; part_samples = [None] * parts
        def run_part(c, k, threads, sample=False):
            b, e = pb[k], pb[k + 1]
            lo = int(offs[b]); hi = int(offs[e - 1]) + int(lens[e - 1])
            WL.wl_memcpy_mt(C.c_void_p(arena.ctypes.data + lo), C.c_void_p(src.ctypes.data + lo), C.c_uint64(hi - lo), C.c_int(threads))
            r2, o2, st = c.chat_translate_host(cfg, arena, offs[b:e], lens[b:e])
            nout = min(int(st["d2h_bytes"]), len(o2), (sink_off[k + 1] if k + 1 < parts else len(sink)) - sink_off[k])     # the bytes the call produced, copied to caller memory
            WL.wl_memcpy_mt(C.c_void_p(sink.ctypes.data + sink_off[k]), C.c_void_p(o2.ctypes.data), C.c_uint64(nout), C.c_int(threads))
            part_st[k] = st
            if sample:   # last timed step only: the result table and 1 % of the records of this call, taken before the next call on the context reuses them
                part_res[k] = np.array(r2)
                idx = np.arange(-(-b // 100) * 100, e, 100) - b
                fo = r2["out_off"][idx].astype(np.int64); fl = r2["path_len"][idx].astype(np.int64) + r2["body_len"][idx].astype(np.int64)
                part_samples[k] = [(int(b + j), bytes(o2[int(a0):int(a0 + l0)])) for j, a0, l0 in zip(idx, fo, fl)]
        def e2e_step(nl, sample=False):
            if nl == 1:
                for k in range(parts):
                    run_part(ctx, k, ncpu_local, sample)
                return
            th = [threading.Thread(target=lambda l=l: [run_part(lane_ctx[l], k, ncpu_local, sample) for k in range(l, parts, nl)]) for l in range(nl)]
            for t in th: t.start()
            for t in th: t.join()
        for _ in range(max(1, min(a.warmup, 2))):
            e2e_step(lanes)
        barrier()
        t1 = time.perf_counter(); e_launch = 0
        for step in range(a.steps):
            e2e_step(lanes, sample=(step == a.steps - 1))
            e_launch += sum(st["gpu_launches"] for st in part_st)
        barrier()
        e_wall = time.perf_counter() - t1
        r2 = np.concatenate(part_res)
        assert int((r2["status"] == A.AIGW_OK).sum()) == n_ok
        e2e = {"wall_s": e_wall, "h2d": sum(st["h2d_bytes"] for st in part_st), "d2h": sum(st["d2h_bytes"] for st in part_st), "launches_per_step": e_launch // a.steps,
               "lanes": lanes, "parts": parts}
        launches += e_launch
        if lanes > 1:   # the strictly serial variant, for the record (two steps)
            e2e_step(1); barrier(); t2 = time.perf_counter(); e2e_step(1); e2e_step(1); barrier()
            e2e["serial_wall_per_step"] = (time.perf_counter() - t2) / 2
        for c in lane_ctx[1:]:
            c.close()
        # ---- parity of the timed outputs: 1 % of the bodies of the last step against the oracle, byte for byte
        if rank == 0:
            for k in range(parts):
                for i, rec in part_samples[k]:
                    t = O.chat_translate("aws-bedrock", bytes(arena[int(offs[i]):int(offs[i]) + int(lens[i])]))
                    pl = len(t.path.encode())
                    assert t.status == 0 and rec[pl:] == t.body and rec[:pl].decode() == t.path, i
                    checked += 1
            # ---- accept rate on real-world spellings (VERDICT r1: report it next to the number)
            esc = escaped_corpus(arena, offs, lens, min(n, 20_000))
            got = ctx.chat_translate(cfg, esc)
            ok = sum(1 for g in got if g["status"] == A.AIGW_OK)
            for k in range(0, len(esc), 10):
                t = O.chat_translate("aws-bedrock", esc[k])
                if got[k]["status"] == A.AIGW_OK:
                    assert t.status == 0 and got[k]["body"] == t.body, k
            div = [W.diverse_body(s) for s in range(4000)]
            gd = ctx.chat_translate(cfg, div)
            accept = {"workload": n_ok / n, "escaped_corpus": ok / len(esc), "escaped_share_of_corpus": 0.1,
                      "diverse_corpus_ok_or_reference_error": sum(1 for g in gd if g["status"] != A.AIGW_DECLINED) / len(div)}
        # p50 added latency: one 4 KB body, submit → complete, timed around the C-ABI call itself (the arguments are built once:
        # the wrapper's numpy views are not part of what a cgo caller pays)
        one_a, one_o, one_l = arena[: int(offs[1]) + 16], offs[:2].copy(), lens[:1].copy()
        from aigw_b200.capi import _BatchOut
        bo = _BatchOut(); fn = ctx.L.aigw_chat_translate_host
        args = (ctx.h, C.byref(cfg), one_a.ctypes.data, one_o.ctypes.data, one_l.ctypes.data, 1, C.byref(bo))
        lat = []
        for k in range(400):
            t = time.perf_counter(); rc = fn(*args); lat.append(time.perf_counter() - t)
            assert rc == 0
        p50 = float(np.median(lat[100:])) * 1e6
        if rank == 0:
            batcher = batcher_block()
    clocks = sampler.stop()

    # ---- reduce over ranks: MAX time, SUM bodies
    tot_bodies = n * world
    dev_s_max, wall_max, e_wall_max = dev_s, wall, (e2e["wall_s"] if e2e else 0.0)
    if dist is not None:
        import torch
        t = torch.tensor([dev_s, wall, e_wall_max], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_s_max, wall_max, e_wall_max = [float(x) for x in t.tolist()]
    if rank == 0:
        peak, peak_src = hbm_peak()
        step_s = dev_s_max / a.steps
        achieved = alg_bytes / (dev_s / a.steps) / 1e9
        tr = ncu_traffic()
        cfgd = config2_dict(n)
        detail = {}
        detail.update({"mean_in_bytes": float(lens.mean()), "mean_out_bytes": out_bytes / max(1, n_ok), "accepted": n_ok, "declined": n - n_ok,
                     "l2": f"inputs larger than L2 ({in_bytes / 1e6:.0f} MB in + {out_bytes / 1e6:.0f} MB out per step vs 126 MB L2)",
                     "wall_ms_per_step_incl_launch": wall_max / a.steps * 1e3, "numa_node": node, "host_threads": ncpu_local})
        line = {"metric": METRIC, "value": tot_bodies / step_s, "unit": "bodies/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": cfgd, "config_detail": detail,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": (tr["bytes_per_body"] * n) if tr else None, "peak_source": peak_src,
                             "traffic_source": (tr["source"] if tr else "no ncu capture committed for this round"),
                             "kernel": "chat_index_kernel + chat_walk_kernel + chat_emit_kernel (the three stages of one translate pass)",
                             "algorithmic_bytes_per_step": alg_bytes, "avg_step_ms": dev_s / a.steps * 1e3,
                             "stage_ms_profiled_pass": {"index": stage[0], "walk": stage[1], "emit": stage[2], "sum": serial_ms},
                             "launches_per_step": dev_launches // max(1, a.steps)},
                "gpu_launches": launches, "clocks": clocks}
        if e2e:
            line["e2e"] = {"value": tot_bodies * a.steps / e_wall_max, "unit": "bodies/s", "h2d_bytes_per_step": int(e2e["h2d"]), "d2h_bytes_per_step": int(e2e["d2h"]),
                           "launches_per_step": e2e["launches_per_step"], "pcie_gbs_each_way": [e2e["h2d"] * a.steps / e_wall_max / 1e9, e2e["d2h"] * a.steps / e_wall_max / 1e9],
                           "includes": "multi-threaded copy of the bodies into the pinned arena, H2D, kernels, D2H, copy of the produced bytes out of the pinned arena",
                           "calls_in_flight": e2e["lanes"], "sub_batches_per_step": e2e["parts"],
                           "serial_value": (tot_bodies / e2e["serial_wall_per_step"] if e2e.get("serial_wall_per_step") and world == 1 else None),
                           "outputs_checked_vs_oracle": checked}
            line["p50_added_us"] = p50
            if batcher:
                line["batcher"] = batcher
            if accept:
                line["accept_rate"] = accept
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    ctx.host_free(arena_ptr)
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ config 1
def run_config1(a, local, ncpu):
    """128 bodies x 2 KB, passthrough translate + response usage: the reference's own CPU-runnable case; latency shape"""
    import _workload as W
    import __graft_entry__ as entry
    entry.build()
    import aigw_b200 as A
    ctx = A.Context(local)
    arena, offs, lens = W.chat_corpus(1, 0, 128, target=2048, jitter=16)
    pin, pp = ctx.host_array(len(arena)); pin[:] = arena
    cfg = ctx.cfg("openai", cost_configured=True)
    resp = [b'{"id":"x","object":"chat.completion","model":"gpt-4o-mini","choices":[{"index":0,"message":{"role":"assistant","content":"ok"},"finish_reason":"stop"}],"usage":{"prompt_tokens":%d,"completion_tokens":%d,"total_tokens":%d}}' % (i, 2 * i, 3 * i) for i in range(128)]
    from aigw_b200 import capi
    ra, ro, rl = capi.pack_bodies(resp)
    lat = []
    for k in range(a.warmup + a.steps):
        t = time.perf_counter()
        res, out, st = ctx.chat_translate_host(cfg, pin, offs[:128].copy(), lens)
        ru = ctx.response_usage_host(ra, ro, rl)
        dt = time.perf_counter() - t
        if k >= a.warmup:
            lat.append(dt)
    assert (res["status"] == 0).all()
    r1, _ = cpu_oracle_rate(0, arena, offs, 128, 1)
    med = float(np.median(lat))
    print(json.dumps({"metric": "extproc bodies/sec, 2 KB ChatCompletion passthrough translate + usage count (128-body call)", "value": 128 / med, "unit": "bodies/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup,
                      "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                      "config": {"workload": "configs[0]: 128 OpenAI ChatCompletion bodies, 2 KB, 4 messages, passthrough + response usage, host buffers", "calls_timed": len(lat)},
                      "e2e": {"value": 128 / med, "unit": "bodies/s", "h2d_bytes_per_step": int(st["h2d_bytes"]), "d2h_bytes_per_step": int(st["d2h_bytes"])},
                      "p50_call_us": med * 1e6, "cpu_baseline": {"value": r1, "unit": "bodies/s", "cores": 1, "kind": "port", "sample": "the same 128 bodies, 1 thread"}}))
    ctx.host_free(pp); ctx.close()


# ------------------------------------------------------------------------------------------------ config 3
def run_config3(a, rank, world, local, ncpu):
    """/v1/embeddings requests of 1024 inputs x 64 characters (68.7 KB of JSON each): EmbeddingsEndpointSpec.ParseBody + the BPE token
    count of every input, one call (aigw_embeddings_count_*): request scan kernel -> text table -> BPE count kernel reading the inputs in
    place from the request bytes -> per-request sums."""
    import _oracle as O
    import __graft_entry__ as entry
    entry.build()
    import aigw_b200 as A
    from aigw_b200 import capi
    A.load_library().aigw_bind_numa(local)
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    ctx = A.Context(local)
    vocab = json.load(open(os.path.join(ROOT, "tests", "golden", "bpe_vocab.json")))
    bpe = ctx.bpe_load(vocab["byte_to_id"], vocab["merges"])
    nreq = a.requests; per = 1024; tl = 64
    # Zipf-distributed words (seed 3 + rank) so the merges are exercised; one 16 MiB base text, every input reads its own window
    r = np.random.default_rng(3 + rank)
    alpha = np.frombuffer(b"etaoinshrdlcumwfgypbvkjxqz", dtype=np.uint8)
    nw = 6000; wl = r.integers(1, 12, nw)
    words = [bytes(alpha[r.integers(0, r.integers(6, 27), int(l))]) for l in wl]
    ids = np.minimum(r.zipf(1.05, 3_000_000) - 1, nw - 1)
    base = np.frombuffer(b" ".join(words[i] for i in ids)[: 16 << 20], dtype=np.uint8)
    nt = nreq * per
    tbytes = nt * tl
    texts = np.empty(tbytes, dtype=np.uint8)
    reps = (tbytes + len(base) - 1) // len(base)
    for k in range(reps):
        lo = k * len(base); hi = min(tbytes, lo + len(base))
        texts[lo:hi] = np.roll(base, 7919 * k)[: hi - lo]
    # the requests: {"model":"text-embedding-3-small","input":["<64 chars>", ... x 1024]}, 16-byte aligned starts in one pinned arena
    head = b'{"model":"text-embedding-3-small","input":['
    H = len(head); blen = H + per * (tl + 3) - 1 + 2
    stride = (blen + 15) // 16 * 16
    nbytes = nreq * stride
    arena, ap = ctx.host_array(nbytes + 64)
    arena[:] = 0x20
    bodies2d = arena[:nbytes].reshape(nreq, stride)
    bodies2d[:, :H] = np.frombuffer(head, dtype=np.uint8)
    cells = bodies2d[:, H:H + per * (tl + 3)].reshape(nreq, per, tl + 3)
    cells[:, :, 0] = ord('"'); cells[:, :, 1:1 + tl] = texts.reshape(nreq, per, tl); cells[:, :, 1 + tl] = ord('"'); cells[:, :, 2 + tl] = ord(',')
    bodies2d[:, blen - 2] = ord(']'); bodies2d[:, blen - 1] = ord('}')
    offs = (np.arange(nreq, dtype=np.uint64) * stride); lens = np.full(nreq, blen, dtype=np.uint32)
    assert blen > 65536 and json.loads(bytes(bodies2d[0, :blen]))["input"][per - 1] == bytes(texts[(per - 1) * tl: per * tl]).decode()
    d_body = ctx.dalloc(nbytes + 64); d_off = ctx.dalloc(nreq * 8); d_len = ctx.dalloc(nreq * 4); d_res = ctx.dalloc(nreq * 32)
    ctx.h2d(d_body, arena[:nbytes]); ctx.h2d(d_off, offs); ctx.h2d(d_len, lens)
    sampler = ClockSampler(local); sampler.start()
    for _ in range(a.warmup):
        ctx.embeddings_count_device(bpe, d_body, d_off, d_len, nreq, blen, nbytes, d_res)
    barrier = (lambda: (dist.barrier(), None)) if dist is not None else (lambda: None)
    barrier(); ctx.sync()
    stage = np.zeros(4); t0 = time.perf_counter()
    for _ in range(a.steps):
        stage += np.asarray(ctx.embeddings_count_device(bpe, d_body, d_off, d_len, nreq, blen, nbytes, d_res))
    ctx.sync(); barrier()
    wall = time.perf_counter() - t0
    res = np.zeros(nreq, dtype=capi.EmbCountResult); ctx.d2h(res, d_res)
    assert (res["status"] == 0).all() and (res["n_inputs"] == per).all() and (res["declined_inputs"] == 0).all()
    # parity of the timed outputs: every 64th request against the CPU restatement (ParseBody + count of every input)
    orc = O.Bpe(vocab)
    sel = np.arange(0, nreq, 64)
    exp_tok, exp_n, _ = orc.embeddings_count_batch(arena, offs[sel].copy(), lens[sel].copy(), threads=ncpu)
    assert np.array_equal(exp_tok, res["tokens"][sel]) and (exp_n == per).all()
    checked = len(sel)
    # end to end: host request bytes -> H2D -> scan + count + sum -> D2H of the 32-byte result rows
    e2e_wall = None; st = None
    if not a.skip_e2e:
        ctx.embeddings_count_host(bpe, arena, offs, lens)
        barrier(); t1 = time.perf_counter()
        for _ in range(a.steps):
            r2, st = ctx.embeddings_count_host(bpe, arena, offs, lens)
        barrier(); e2e_wall = time.perf_counter() - t1
        assert np.array_equal(r2["tokens"], res["tokens"])
    clocks = sampler.stop()
    step_s = stage[3] / 1e3 / a.steps
    if dist is not None:
        import torch
        t = torch.tensor([step_s, e2e_wall or 0.0], dtype=torch.float64, device=f"cuda:{local}"); dist.all_reduce(t, op=dist.ReduceOp.MAX); step_s, e2e_wall = float(t[0]), (float(t[1]) if e2e_wall else None)
    cpu = None
    if rank == 0 and world == 1:
        ns = min(nreq, 8 * ncpu, 512)
        _, _, sec = orc.embeddings_count_batch(arena, offs[:ns].copy(), lens[:ns].copy(), threads=ncpu)
        n1 = max(1, ns // 16)
        _, _, sec1 = orc.embeddings_count_batch(arena, offs[:n1].copy(), lens[:n1].copy(), threads=1)
        cpu = {"value": ns / sec, "unit": "requests/s", "cores": ncpu, "kind": "port", "sample": f"first {ns} requests of the wave (JSON decode + BPE count of every input), {ncpu} threads (1 thread: {n1 / sec1:.1f} requests/s)"}
    if rank == 0:
        peak, peak_src = hbm_peak()
        alg = nreq * (blen + 4 * per)          # SURVEY 8d: bytes_in + 4 B per input
        scan_s = stage[0] / 1e3 / a.steps
        line = {"metric": "embeddings requests/sec with BPE token count (1024 inputs x 64 chars per request)", "value": nreq * world / step_s, "unit": "requests/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/u16", "data": "synthetic",
                "config": {"workload": f"configs[2]: {nreq} /v1/embeddings requests per GPU per step, each a {blen}-byte JSON body with 1024 inputs x 64 characters (Zipf words, seed 3): ParseBody (request scan) + BPE count of every input "
                                       f"(vocabulary of {vocab['vocab_size']}, tests/golden/bpe_vocab.json) + per-request sums",
                           "inputs_per_step": nt, "l2": f"requests larger than L2 ({nbytes / 1e6:.0f} MB per step vs 126 MB)", "mean_tokens_per_request": float(res["tokens"].mean()),
                           "requests_checked_vs_cpu_restatement": checked, "wall_ms_per_step": wall / a.steps * 1e3},
                "stage_ms_per_step": {"emb_scan_kernel": stage[0] / a.steps, "bpe_count_kernel": stage[1] / a.steps, "emb_sum_kernel": stage[2] / a.steps, "whole_call_incl_readback": stage[3] / a.steps},
                "roofline": {"bound": "hbm", "achieved": alg / step_s / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / step_s / 1e9 / peak, "traffic": None, "peak_source": peak_src, "kernel": "emb_scan_kernel + bpe_count_kernel",
                             "algorithmic_bytes_per_step": alg, "scan_kernel_alone": {"achieved": nreq * blen / scan_s / 1e9, "frac": nreq * blen / scan_s / 1e9 / peak},
                             "note": "algorithmic bytes = request bytes + 4 B per input (SURVEY 8d); the scan streams the request once, the count kernel re-reads the inputs and is bound by its per-lane merge loops (shared-memory table lookups), not by HBM"},
                "gpu_launches": (a.steps + a.warmup) * 3, "clocks": clocks}
        if e2e_wall:
            line["e2e"] = {"value": nreq * world * a.steps / e2e_wall, "unit": "requests/s", "h2d_bytes_per_step": int(st["h2d_bytes"]), "d2h_bytes_per_step": int(st["d2h_bytes"])}
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    ctx.host_free(ap); ctx.bpe_free(bpe); ctx.close()
    if dist is not None: dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ config 4
def run_config4(a, rank, world, local, ncpu):
    """streams x 256 chunks x 80 B through aigw_stream_chunks (one ResponseBody call per stream per round), OpenAI usage extract"""
    import _oracle as O
    import _workload as W
    import __graft_entry__ as entry
    entry.build()
    import aigw_b200 as A
    A.load_library().aigw_bind_numa(local)
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    ctx = A.Context(local)
    ns, chunks = a.streams, 256
    buf, coff, cfirst = W.sse_corpus(4, rank * ns, ns, chunks=chunks)
    nbytes = int(coff[-1])
    lens_all = (coff[1:] - coff[:-1]).astype(np.uint32)
    first_chunk = cfirst[:-1].astype(np.int64)
    from aigw_b200.capi import ChunkResult
    # the chunk bytes live in a pinned arena from aigw_host_alloc (where the shim copies them as they arrive) and the result table is
    # pinned too: the kernels read the chunks in place and the results come back with one DMA
    pinned_buf, pbp = ctx.host_array(len(buf) + 64); pinned_buf[: len(buf)] = buf; buf = pinned_buf
    res_raw, rbp = ctx.host_array(ns * ChunkResult.itemsize); res_buf = res_raw.view(ChunkResult)
    # the (offset, length) tables of every round, built before the timed region: a shim receives them with the chunks
    rounds_idx = first_chunk[None, :] + np.arange(chunks, dtype=np.int64)[:, None]
    off_rounds = np.ascontiguousarray(coff[rounds_idx]); len_rounds = np.ascontiguousarray(lens_all[rounds_idx]); del rounds_idx
    def one_pass(check):
        hs = np.array(ctx.stream_open("openai", b"gpt-4o-mini", n=ns), dtype=np.uint64)
        last = None
        for r in range(chunks):
            res, arena = ctx.stream_chunks_soa(hs, buf, off_rounds[r], len_rounds[r], res=res_buf)
            if check and r >= chunks - 3:
                m = res["mask"] != 0
                if last is None: last = np.zeros(ns, dtype=res.dtype)
                last[m] = res[m]
        ctx.stream_close(hs)
        return last
    for _ in range(max(1, a.warmup // 3)):
        one_pass(False)
    ctx.sync()
    if dist is not None: dist.barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        last = one_pass(True)
    ctx.sync()
    if dist is not None: dist.barrier()
    wall = time.perf_counter() - t0
    # parity on a sample: the usage of the final calls equals the oracle's replay
    nsamp = min(ns, 2000)
    outu = np.zeros(nsamp, dtype=np.dtype([(k, "<u4") for k in ("input", "output", "total", "cached", "cache_creation", "reasoning", "mask")]))
    sec = O.lib().oracle_sse_batch(buf.ctypes.data, coff.ctypes.data, cfirst.ctypes.data, nsamp, ncpu, outu.ctypes.data)
    assert (last["input"][:nsamp] == outu["input"]).all() and (last["total"][:nsamp] == outu["total"]).all()
    wall_max = wall
    if dist is not None:
        import torch
        t = torch.tensor([wall], dtype=torch.float64, device=f"cuda:{local}"); dist.all_reduce(t, op=dist.ReduceOp.MAX); wall_max = float(t.item())
    if rank == 0:
        val = ns * chunks * world * a.steps / wall_max
        print(json.dumps({"metric": "SSE chunks/sec through the per-chunk stream ABI, OpenAI usage extract", "value": val, "unit": "chunks/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                          "ms_per_step": wall_max / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                          "config": {"workload": f"configs[3]: {ns} streams/GPU x {chunks} chunk calls x ~80 B, 20% ragged chunking, seed 4; every round is one aigw_stream_chunks_soa call over all streams, chunk bytes in a pinned arena (read in place by the kernels)",
                                     "bytes_per_gpu": nbytes},
                          "e2e": {"value": val, "unit": "chunks/s", "h2d_bytes_per_step": nbytes + ns * chunks * 32, "d2h_bytes_per_step": ns * chunks * 64},
                          "cpu_baseline": {"value": nsamp * chunks / sec, "unit": "chunks/s", "cores": ncpu, "kind": "port", "sample": f"{nsamp} streams replayed chunk by chunk, {ncpu} threads"}}))
    ctx.close()
    if dist is not None: dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ config 5
def run_config5(a, rank, world, local, ncpu):
    """mixed-provider fan-out: every request has an id; device = hash64(id) % n_gpus (aigw_b200/shard.py); each rank translates the
    requests that hash to it, grouped by backend schema (one host-buffer call per backend)"""
    import _oracle as O
    import _workload as W
    import __graft_entry__ as entry
    entry.build()
    import aigw_b200 as A
    from aigw_b200 import capi, shard
    A.load_library().aigw_bind_numa(local)
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
    ctx = A.Context(local)
    total = a.bodies * world
    rng = np.random.default_rng(5 + rank)
    k = np.arange(1, 65); p = k ** -1.2; p /= p.sum()
    # request ids 0..total-1; this rank owns the ids whose hash64 lands on it (aigw_b200/shard.py, FNV-1a 64 as the cgo shim would)
    ids = np.arange(total, dtype=np.uint64)
    dev = shard.devices_for_requests(ids, world)
    owner = dev[:: max(1, total // 65536)]
    mine = ids[dev == rank]
    assert shard.device_for_request(int(mine[0]).to_bytes(8, "little"), world) == rank   # the scalar and the vectorised hash agree
    kb = rng.choice(k, size=len(mine), p=p)
    backend = rng.integers(0, 4, size=len(mine))
    names = ["openai", "gcp-vertexai", "gcp-anthropicai", "aws-bedrock"]
    pools = {}
    for t in sorted(set(int(x) for x in kb)):
        m = min(int((kb == t).sum()), 256)
        arena, offs, lens = W.chat_corpus(5, 0, m, target=min(t * 1024, 62000), jitter=max(16, t * 16))
        pools[t] = [bytes(arena[int(offs[i]):int(offs[i]) + int(lens[i])]) for i in range(m)]
    groups = []
    for bi, name in enumerate(names):
        sel = np.nonzero(backend == bi)[0]
        bodies = [pools[int(kb[j])][int(j) % len(pools[int(kb[j])])] for j in sel]
        arena, offs, lens = capi.pack_bodies(bodies)
        pin, pp = ctx.host_array(len(arena) + 64); pin[: len(arena)] = arena
        groups.append((name, ctx.cfg(name), pin, offs[: len(bodies)].copy(), lens, bodies))
    def step():
        acc = 0
        for name, cfg, pin, offs, lens, bodies in groups:
            res, out, st = ctx.chat_translate_host(cfg, pin, offs, lens)
            acc += int((res["status"] == 0).sum())
        return acc, None
    for _ in range(a.warmup):
        step()
    ctx.sync()
    if dist is not None: dist.barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        acc, outs = step()
    ctx.sync()
    if dist is not None: dist.barrier()
    wall = time.perf_counter() - t0
    # sampled parity per backend (a host call's views are valid until the next call on the context: check right after each)
    for name, cfg, pin, offs, lens, bodies in groups:
        res, out, st = ctx.chat_translate_host(cfg, pin, offs, lens)
        for i in range(0, len(bodies), max(1, len(bodies) // 100)):
            t = O.chat_translate(name, bodies[i], prefix="" if "anthropic" in name else "v1")
            if int(res[i]["status"]) == 0:
                o = int(res[i]["out_off"]) + int(res[i]["path_len"])
                got = bytes(out[o:o + int(res[i]["body_len"])])
                assert t.status == 0 and got == (t.body if t.body_kind == 1 else b""), (name, i, t.status, len(got), len(t.body))
    wall_max = wall; acc_all = acc
    if dist is not None:
        import torch
        t = torch.tensor([wall, -float(acc)], dtype=torch.float64, device=f"cuda:{local}"); dist.all_reduce(t, op=dist.ReduceOp.MAX); wall_max = float(t[0].item())
        t2 = torch.tensor([float(acc)], dtype=torch.float64, device=f"cuda:{local}"); dist.all_reduce(t2, op=dist.ReduceOp.SUM); acc_all = int(t2.item())
    if rank == 0:
        nb = sum(len(g[5]) for g in groups)
        mean_in = float(np.mean([len(b) for g in groups for b in g[5][:2000]]))
        print(json.dumps({"metric": "extproc bodies/sec, mixed-provider translate (OpenAI / Gemini / Anthropic / Bedrock), Zipf 1-64 KB", "value": total * a.steps / wall_max, "unit": "bodies/s", "n_gpus": world,
                          "steps": a.steps, "warmup": a.warmup, "ms_per_step": wall_max / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                          "config": {"workload": "configs[4]: 4-target mix, body size clamp(1 KB x Zipf(1.2), 1 KB, 64 KB), seed 5, device = hash64(request-id) % n_gpus", "bodies_rank0_per_step": nb, "bodies_total_per_step": total,
                                     "mean_in_bytes": mean_in, "accepted_share": acc_all / total, "hash_balance_sample": np.bincount(owner, minlength=world).tolist()},
                          "e2e": {"value": total * a.steps / wall_max, "unit": "bodies/s", "h2d_bytes_per_step": int(sum(int(g[4].sum()) for g in groups)), "d2h_bytes_per_step": None}}))
    ctx.close()
    if dist is not None: dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 5; config 1, where a step is one call and the line reports the median: 100)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5])
    ap.add_argument("--bodies", type=int, default=int(os.environ.get("AIGW_BENCH_BODIES", 0)), help="bodies per GPU per step (config 2: 1,000,000; config 5: 1,250,000)")
    ap.add_argument("--streams", type=int, default=100_000, help="config 4: streams per GPU")
    ap.add_argument("--requests", type=int, default=4096, help="config 3: embeddings requests (1024 inputs each) per GPU per step")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=400_000)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--e2e-lanes", type=int, default=1, help="config 2 e2e: host threads (each with its own context) keeping a call in flight; measured: 2 lanes x 8 sub-batches 4.81 M bodies/s vs 5.23 M for one call over the whole step (the call's own H2D / kernel / D2H pipeline is what counts)")
    ap.add_argument("--e2e-parts", type=int, default=1, help="config 2 e2e: sub-batches per step, dealt to the lanes round robin")
    ap.add_argument("--dump-outputs", metavar="DIR", help="config 2: write what the last timed step of the device pass returned (a fixed sample) to DIR/*.npy")
    a = ap.parse_args()
    if a.steps is None:
        a.steps = 100 if a.config == 1 and a.impl == "b200" else 5
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.config != 2):
        ap.error("--dump-outputs is written by the device pass of config 2")
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1)); local = int(os.environ.get("LOCAL_RANK", 0))
    ncpu = host_cores()
    if a.bodies <= 0:
        a.bodies = 1_250_000 if a.config == 5 else 1_000_000
    if a.impl == "reference":
        if rank == 0:
            run_reference(a, ncpu)
        return
    if a.config == 1:
        if rank == 0: run_config1(a, local, ncpu)
    elif a.config == 2:
        run_config2(a, rank, world, local, ncpu)
    elif a.config == 3:
        run_config3(a, rank, world, local, ncpu)
    elif a.config == 4:
        run_config4(a, rank, world, local, ncpu)
    else:
        run_config5(a, rank, world, local, ncpu)


if __name__ == "__main__":
    main()
