"""f-5 suffix tree: device time of b200sa_suffix_tree_dev from SA + LCP already in HBM.

For 100 MB of gen.dna and of gen.english: SA + LCP built once on the device, then the
tree is timed with CUDA events around each call (warm-up, then the median of the timed
calls) and, in one extra call with the library's phase events on, split into phases
(ANSV, head compaction, sort, base scan, node kernels).  The CPU baseline is the C
restatement of the reference's serial insertion (tests/cpp/tree_oracle.c) on a 10 MB
prefix, given the SA + LCP; the device tree of that prefix is checked against it.
The card's name and power limit are read in the same run.  Writes one JSON file.

    python tools/tree_bench.py [--n 100000000] [--steps 10] [--warmup 3] [--out profiles/r03_tree_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from suffix_b200 import SuffixTable, _lib, gen  # noqa: E402
from tests import tree_model as tm  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def device_tree(kind, n, steps, warmup):
    text = getattr(gen, kind)(n)
    dev = torch.device("cuda:0")
    ctx = _lib.Context(0)
    stream = torch.cuda.Stream(device=dev)
    d_text = torch.from_numpy(text).to(dev)
    d_sa = torch.empty(n, dtype=torch.int32, device=dev)
    d_lcp = torch.empty(n, dtype=torch.int32, device=dev)
    ctx.build_lcp_dev(d_text.data_ptr(), n, d_sa.data_ptr(), d_lcp.data_ptr(), stream.cuda_stream)
    out = {f: torch.empty(2 * n, dtype=torch.int32, device=dev) for f in _lib.TREE_FIELDS}
    ptrs = {f: t.data_ptr() for f, t in out.items()}
    torch.cuda.synchronize()
    times, nodes = [], 0
    for it in range(warmup + steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        nodes = ctx.suffix_tree_dev(d_text.data_ptr(), n, d_sa.data_ptr(), d_lcp.data_ptr(), ptrs, stream.cuda_stream)
        e1.record(stream)
        stream.synchronize()
        if it >= warmup:
            times.append(e0.elapsed_time(e1))
    ctx.set_timing(True)
    ctx.suffix_tree_dev(d_text.data_ptr(), n, d_sa.data_ptr(), d_lcp.data_ptr(), ptrs, stream.cuda_stream)
    stream.synchronize()
    phases = {k: round(v, 3) for k, v in ctx.phase_times()}
    st = ctx.stats()
    ctx.close()
    return {"text": "gen.%s(%d)" % (kind, n), "n": n, "nodes": nodes, "steps": steps, "warmup": warmup,
            "median_ms": round(float(np.median(times)), 3), "min_ms": round(min(times), 3),
            "max_ms": round(max(times), 3), "phases_ms": phases, "kernel_launches": st["kernel_launches"],
            "workspace_bytes": st["workspace_bytes"],
            "note": "output arrays (6 x 2n u32) and SA + LCP in HBM; 100 MB inputs exceed the 126 MB L2 "
                    "together with the outputs"}


def cpu_baseline(n):
    text = gen.dna(n).tobytes()
    st = SuffixTable(text)
    sa, lcp = np.asarray(st.table()), np.asarray(st.lcp_lens())
    t0 = time.perf_counter()
    want = tm.oracle_tree(text, sa, lcp)
    sec = time.perf_counter() - t0
    ctx = _lib.default_context(0)
    _, got = ctx.suffix_tree(np.frombuffer(text, dtype=np.uint8), sa)
    agree = all(np.array_equal(got[f], want[f]) for f in tm.FIELDS)
    return {"label": "CPU baseline: C restatement of the reference's serial insertion (to_suffix_tree), "
                     "1 core, given SA + LCP, gen.dna %d-byte prefix" % n,
            "n": n, "seconds": round(sec, 3), "ms_per_100MB_linear_extrapolation": round(sec * 1e3 * 1e8 / n, 1),
            "device_tree_equals_oracle": bool(agree)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--cpu-n", type=int, default=10_000_000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_tree_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tree_bench needs a CUDA device")
    res = {"card": card(), "device": [device_tree(k, a.n, a.steps, a.warmup) for k in ("dna", "english")],
           "cpu": cpu_baseline(a.cpu_n)}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
