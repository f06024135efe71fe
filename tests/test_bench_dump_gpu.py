"""bench.py --dump-outputs: what the timed device pass returned in its last step, as float arrays within 64 MB; two runs with the same
arguments write the same outputs, the sample is a proper subset of the bodies when there are more of them than result rows dumped, and
the dumped records are the oracle's translation of the sampled bodies."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import _oracle as O
import _workload as W

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMP_ROWS = 65536   # bench.py DUMP_ROWS
FIELDS = ("status", "reason", "body_len", "path_len", "model_off", "model_len", "body_kind", "flags", "in_len")   # bench.py DUMP_FIELDS
BODIES = 100_000    # more than DUMP_ROWS: the dump samples


def _run(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--bodies", str(BODIES), "--cpu-sample", "2000",
                        "--skip-e2e", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.strip().split("\n") if l.startswith("{")][-1])
    assert line["steps"] == 3 and line["warmup"] == 1
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
def test_dump_outputs_are_reproducible_and_match_the_oracle(tmp_path):
    a = _run(tmp_path / "a")
    b = _run(tmp_path / "b")
    assert sorted(a) == sorted(["sample_index", "output_len", "output_bytes"] + [f"result_{f}" for f in FIELDS])
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
    # the sample: DUMP_ROWS distinct bodies in increasing order, spread over the whole batch
    idx = a["sample_index"].astype(np.int64)
    assert len(idx) == DUMP_ROWS and (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < BODIES
    assert idx[-1] > BODIES * 9 // 10 and len(np.setdiff1d(np.arange(DUMP_ROWS), idx)) > 0
    for k in ("result_model_len", "result_body_kind", "result_flags"):
        assert len(a[k]) == len(idx), k
    # every sampled row: status, input and output length as the oracle has them
    arena, offs, lens = W.chat_corpus(2, 0, BODIES)
    st = np.zeros(BODIES, np.int32); olen = np.zeros(BODIES, np.uint32); tot = C.c_uint64(0)
    O.lib().oracle_chat_translate_batch(1, arena.ctypes.data, offs.ctypes.data, BODIES, 0, 8, st.ctypes.data, olen.ctypes.data, C.byref(tot))
    assert (a["result_status"] == st[idx]).all() and (st[idx] == 0).all()
    assert (a["result_in_len"] == lens[idx]).all() and (a["result_body_len"] == olen[idx]).all()
    # the dumped bytes: path + body of the first sampled bodies, byte for byte
    raw = a["output_bytes"].astype(np.uint8).tobytes()
    out_len = a["output_len"].astype(np.int64)
    assert 0 < len(out_len) and out_len.sum() == len(raw)
    o = 0
    for j, l in enumerate(out_len):
        i = int(idx[j])
        t = O.chat_translate("aws-bedrock", bytes(arena[int(offs[i]):int(offs[i]) + int(lens[i])]))
        pl = int(a["result_path_len"][j])
        assert l == pl + len(t.body) and raw[o:o + pl].decode() == t.path and raw[o + pl:o + l] == t.body, i
        o += int(l)
