"""Cost of the suffix-array check in front of the linear LCP path (phase "lcp_sorted").

Stand-alone b200sa_lcp_dev on the device-resident true SA of a 100 MB text that takes the linear
path (English: 8-bit alphabet above 32 MiB): CUDA events around each call (warm-up, then the median
of the timed calls) and the library's phase events in the same calls, so the check's share is the
median of its phase.  Then one call on the same table with two adjacent ranks swapped (the
uncapped per-pair compare), checked against the oracle.  The card's name and power limit are read
in the same run.  Writes one JSON file.

    python tools/lcp_check_bench.py [--n 100000000] [--kind english] [--steps 10] [--warmup 3] [--out profiles/r04_lcp_check.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle import oracle  # noqa: E402
from suffix_b200 import _lib, gen  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    name, power, clock = (q.stdout.strip().split(", ") + ["?", "?", "?"])[:3]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name(0)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=100_000_000)
    ap.add_argument("--kind", default="english")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_lcp_check.json"))
    a = ap.parse_args()
    text = getattr(gen, a.kind)(a.n)
    n = len(text)
    dev = torch.device("cuda:0")
    ctx = _lib.Context(0)
    stream = torch.cuda.Stream(device=dev)
    d_text = torch.from_numpy(text).to(dev)
    d_sa = torch.empty(n, dtype=torch.int32, device=dev)
    d_lcp = torch.empty(n, dtype=torch.int32, device=dev)
    ctx.build_lcp_dev(d_text.data_ptr(), n, d_sa.data_ptr(), d_lcp.data_ptr(), stream.cuda_stream)
    stream.synchronize()
    want_true = d_lcp.clone()
    ctx.set_timing(True)
    totals, phases = [], {}
    for it in range(a.warmup + a.steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.lcp_dev(d_text.data_ptr(), n, d_sa.data_ptr(), d_lcp.data_ptr(), stream.cuda_stream)
        e1.record(stream)
        stream.synchronize()
        if it >= a.warmup:
            totals.append(e0.elapsed_time(e1))
            for k, v in ctx.phase_times():
                phases.setdefault(k, []).append(v)
    assert torch.equal(d_lcp, want_true), "stand-alone LCP differs from the fused one"
    med = {k: float(np.median(v)) for k, v in phases.items()}
    # the same table with ranks n/2, n/2+1 swapped: the uncapped per-pair compare
    sw = d_sa.clone()
    r = n // 2
    sw[r], sw[r + 1] = d_sa[r + 1].item(), d_sa[r].item()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    ctx.lcp_dev(d_text.data_ptr(), n, sw.data_ptr(), d_lcp.data_ptr(), stream.cuda_stream)
    e1.record(stream)
    stream.synchronize()
    swapped_ms = e0.elapsed_time(e1)
    swapped_phases = [k for k, _ in ctx.phase_times()]
    tab = sw.cpu().numpy().view(np.uint32)
    ok = bool(np.array_equal(d_lcp.cpu().numpy().view(np.uint32), oracle.lcp_quadratic(text, tab)))
    out = {"card": card(), "kind": a.kind, "n": n, "steps": a.steps,
           "lcp_dev_true_sa_ms_median": float(np.median(totals)),
           "phases_ms_median": {k: round(v, 3) for k, v in med.items()},
           "check_ms_median": round(med.get("lcp_sorted", float("nan")), 3),
           "swapped_table_ms": round(swapped_ms, 3), "swapped_table_phases": swapped_phases,
           "swapped_table_matches_oracle": ok}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    assert ok


if __name__ == "__main__":
    main()
