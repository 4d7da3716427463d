#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

metric : MB/s of input text indexed (SuffixTable::new + lcp_lens, i.e. SA + LCP
         build); MB = 1e6 bytes.
N = 1  : configs[1] -- 100 MB synthetic DNA (sigma=4), generator G_dna of
         SURVEY.md Appendix C; one "step" = one full SA + LCP build.
N > 1  : the induce recursion is single-device by north_star, so ranks index
         independent 100 MB texts (replicas, no data-path collective):
         "scaling": "weak".

value  : device-resident (text already in HBM, SA/LCP left in HBM), CUDA events
         on the launching stream, max over ranks.
e2e    : the same step through the host-buffer C-ABI (b200sa_build_lcp) with
         pinned HOST buffers: H2D of the text and D2H of SA+LCP inside the
         timed region.
roofline / cpu_baseline / clocks: see DESIGN.md "Measurement".

--impl reference: the reference's own CPU algorithm.  The reference is Rust and
cannot be compiled in this image, so this arm times the oracle port
(oracle/sais_oracle.c: restated sais() + lcp_lens()) on one host core (the
reference is single-threaded), each step on a bounded prefix of the workload.

--dump-outputs DIR: after the timed steps, writes the SA and LCP arrays of the last
device-resident step (rank 0) as DIR/sa.npy and DIR/lcp.npy (float64, exact for
u32 values).  Above DUMP_ENTRIES entries both arrays are sampled at the same
seeded set of indices.  The input text is seeded too, so two builds of the project
run with the same arguments can be compared entry for entry.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: no bytecode caches written into it

from suffix_b200 import gen  # noqa: E402

N_TEXT = 100_000_000
METRIC = "MB/s input text indexed (SA+LCP build)"
UNIT = "MB/s"
WORKLOAD = "100 MB synthetic DNA (sigma=4) SA-IS build + LCP, G_dna seed 0x5AFE5EED0000D7A4"
DUMP_ENTRIES = 3_000_000                # per dumped array: 2 x 3e6 float64 = 48 MB, under a 64 MB budget
DUMP_SEED = 0x5AFE5EED0000D0D0


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """Samples SM clocks and throttle reasons of one GPU through NVML every few
    milliseconds on a thread; only samples taken inside a marked window count."""
    REASONS = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.samples = []          # (t, sm_mhz, reasons_bitmask)
        self.windows = []
        self.stop_flag = False
        self.ok = False
        self.thr = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical order; honour CUDA_VISIBLE_DEVICES if it is a plain index list
            idx = self.gpu
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except Exception:
                    idx = self.gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
            self.thr = threading.Thread(target=self._loop, daemon=True)
            self.thr.start()
        except Exception:
            self.ok = False

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((time.perf_counter(), mhz, rs))
            except Exception:
                pass
            time.sleep(0.004)

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thr.join(timeout=2)
        inside = [(m, r) for (t, m, r) in self.samples if any(a <= t <= b for a, b in self.windows)]
        reasons = set()
        for _, r in inside:
            for nm, bit in self.REASONS.items():
                if r & bit:
                    reasons.add(nm)
        return {"sm_mhz": statistics.median([m for m, _ in inside]) if inside else None,
                "sm_max_mhz": self.max_mhz, "samples": len(inside), "reasons": sorted(reasons),
                "how": "NVML polled every ~4 ms during the timed regions (device-resident and e2e loops)"}


def _dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def _oracle_time(text_np, with_lcp=True):
    from oracle import oracle          # CPU baseline leg: the one place bench.py executes oracle/
    t0 = time.perf_counter()
    sa = oracle.sais(text_np)
    lcp = oracle.lcp_lens(text_np, sa) if with_lcp else None
    return time.perf_counter() - t0, sa, lcp


def _pin_to_cpu(k, of=1):
    """Pins the calling thread to one host core (best effort); the `of` replicas are spread
    evenly over the cores the process may use, so that they do not share a core or crowd one
    memory controller."""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        stride = max(1, len(cpus) // max(1, of))
        os.sched_setaffinity(threading.get_native_id(), {cpus[(k * stride) % len(cpus)]})
    except Exception:
        pass


def run_reference(args):
    """The reference's own CPU algorithm on the SAME config as the GPU arm: every
    timed step indexes all N_TEXT bytes of the workload (SA + LCP).  The reference
    is single-threaded, so one replica uses one core; at --gpus N (weak scaling:
    N independent 100 MB texts) rank 0 runs N replicas concurrently on N pinned
    cores, mirroring the GPU arm's N replicas.  Warm-up steps run on a 4 MB
    prefix (a CPU run has no clocks or JIT to warm; only the allocator and page
    cache), so that the arm fits the driver's per-N time limit."""
    rank, world, _ = _dist_env()
    if rank != 0:
        return 0
    steps, warm = args.steps, args.warmup
    n = args.n
    reps = max(1, args.gpus)
    texts = [gen.dna(n, seed=gen.SEED_DNA + r) for r in range(reps)]
    for _ in range(warm):
        _oracle_time(texts[0][:4_000_000])

    def one_step():
        if reps == 1:
            dt, _sa, _l = _oracle_time(texts[0])
            return dt
        t0 = time.perf_counter()

        def work(r):
            _pin_to_cpu(r, reps)
            _oracle_time(texts[r])
        th = [threading.Thread(target=work, args=(r,)) for r in range(reps)]
        [x.start() for x in th]
        [x.join() for x in th]
        return time.perf_counter() - t0

    ts = [one_step() for _ in range(steps)]
    total = sum(ts)
    val = n * reps * steps / 1e6 / total
    sample = ("all %d bytes of the workload per step and replica (oracle port of sais()+lcp_lens(); the reference is "
              "single-threaded: %d replica(s) on %d pinned core(s)); warm-up steps on a 4 MB prefix" % (n, reps, reps))
    out = {
        "impl": "reference", "metric": METRIC, "value": round(val, 3), "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": round(total / steps * 1e3, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": _config(n, reps),
        "cpu_baseline": {"value": round(val, 3), "unit": UNIT, "cores": reps, "kind": "port", "sample": sample,
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": round(val, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    _emit(json.dumps(out))
    return 0


def _dump_outputs(out_dir, arrays):
    """Writes each named u32 array as out_dir/<name>.npy in float64.  Arrays longer than
    DUMP_ENTRIES are all sampled at the same sorted, seeded indices (fixed for a given n)."""
    os.makedirs(out_dir, exist_ok=True)
    n = len(next(iter(arrays.values())))
    idx = None
    if n > DUMP_ENTRIES:
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n, DUMP_ENTRIES, replace=False))
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), (a if idx is None else a[idx]).astype(np.float64))


def _config(n, world):
    """The `config` object shared verbatim by both arms (same-config check)."""
    return {"workload": WORKLOAD if n == N_TEXT else "%d-byte G_dna text" % n, "n_bytes_per_gpu": n,
            "parallelism": "replicas x%d (independent texts, no collective)" % world,
            "l2": "inputs larger than L2 (text 100 MB + SA 400 MB + LCP 400 MB per step)",
            "timing": "GPU arm: CUDA events on the launching stream, max over ranks; reference arm: host clock"}


def _sharded_record(args, ctx, dist, rank, world, dev):
    """BASELINE configs[4]: world x shard_bytes of G_dna as ONE text, one contiguous shard per GPU;
    type classification + LMS-suffix sort (b200sa_shard_lms_sort: NCCL all-gathers of the summaries,
    one all-to-all of (key, position) pairs over NVLink).  Device time, max over ranks."""
    import torch
    from suffix_b200 import sharded
    nb = args.shard_bytes
    text = gen.dna(nb, seed=gen.SEED_DNA + rank)           # SURVEY 8d config 5: seed + shard id
    shard = torch.from_numpy(text).to(dev)
    sharded.ensure_comm(ctx, dist)
    cap = nb // 2 + 4096
    gpos = torch.empty(cap, dtype=torch.int64, device=dev)
    names = torch.empty(cap, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream()
    st = None
    times = []
    for it in range(3):                                    # 1 warm-up + 2 timed
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        st = ctx.shard_lms_sort(shard.data_ptr(), nb, gpos.data_ptr(), names.data_ptr(), cap, stream.cuda_stream)
        e1.record(stream)
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    phases = dict(ctx.phase_times())
    k = int(st["recv_count"])
    # local sanity: positions of this slice that lie in this rank's own shard are ordered by their windows
    g = gpos[:k]
    mine = g[(g >= st["lo"]) & (g < st["lo"] + nb - 64)][:200000].cpu().numpy() - st["lo"]
    tb = text.tobytes()
    kc = int(st["kc"])
    ok = all(tb[int(a):int(a) + kc] <= tb[int(b):int(b) + kc] for a, b in zip(mine[:-1], mine[1:]))
    nm = names[:k]
    ok = ok and bool(((nm[1:] - nm[:-1]) >= 0).all().item()) if k > 1 else ok
    t = torch.tensor([min(times[1:]), st["bytes_sent"], float(k), 1.0 if ok else 0.0], dtype=torch.float64, device=dev)
    tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    tmin = t.clone(); dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
    ms = float(tmax[0].item())
    total = nb * world
    del gpos, names, shard
    torch.cuda.empty_cache()
    return {"workload": "BASELINE configs[4]: %d x %d B of G_dna as ONE text, type-classify + LMS-suffix sort sharded over "
                        "%d GPUs (b200sa_shard_lms_sort, NCCL inside the library)" % (world, nb, world),
            "n_bytes_total": total, "ms_per_step": round(ms, 3),
            "GBps_aggregate": round(total / 1e9 / (ms / 1e3), 2), "GBps_per_gpu": round(nb / 1e9 / (ms / 1e3), 2),
            "m_total": int(st["m_total"]), "slice_sum": int(tsum[2].item()), "window_chars": kc,
            "ties_total": int(st["ties_total"]), "nvlink_bytes_per_step": int(tsum[1].item()),
            "checks_ok": bool(tmin[3].item() == 1.0) and int(tsum[2].item()) == int(st["m_total"]),
            "phase_ms_rank0": {k2: round(v, 3) for k2, v in phases.items()},
            "timing": "CUDA events on the launching stream around the collective call, max over ranks, best of 2 after 1 warm-up"}


def _bind_to_gpu_numa(local):
    """Binds this rank to the cores of its GPU's NUMA node before the pinned host buffers are
    allocated (first touch then places them on that node): at N = 8 every rank moves 0.9 GB per
    step over PCIe, and buffers on the far socket cost bandwidth (round 1: e2e efficiency 0.855)."""
    try:
        import pynvml
        pynvml.nvmlInit()
        idx = local
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                idx = int(vis.split(",")[local])
            except Exception:
                idx = local
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        path = "/sys/bus/pci/devices/%s/numa_node" % bus.lower()[-12:]
        node = int(open(path).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"numa_node": node, "cpus": len(cpus)}
    except Exception:
        return None
    return None


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from suffix_b200 import _lib

    rank, world, local = _dist_env()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = _bind_to_gpu_numa(local)
    n = args.n
    steps, warm = args.steps, args.warmup

    # independent text per rank (replicas): seed + rank
    text = gen.dna(n, seed=gen.SEED_DNA + rank)
    ctx = _lib.Context(local)
    ctx.set_timing(True)
    stream = torch.cuda.current_stream()
    sptr = stream.cuda_stream

    d_text = torch.from_numpy(text).to(dev)
    d_sa = torch.empty(n, dtype=torch.int32, device=dev)
    d_lcp = torch.empty(n, dtype=torch.int32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_dev():
        ctx.build_lcp_dev(d_text.data_ptr(), n, d_sa.data_ptr(), d_lcp.data_ptr(), sptr)
        ph = ctx.phase_times()
        launches = ctx.stats()["kernel_launches"]
        return ph, [], launches

    # ---------------- device-resident timing (`value`)
    for _ in range(warm):
        step_dev()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    phase_acc, launches = {}, 0
    tw0 = time.perf_counter()
    ev0.record(stream)
    for _ in range(steps):
        ph, ph2, l = step_dev()
        launches += l
        for k, v in ph + ph2:
            phase_acc.setdefault(k, []).append(v)
    ev1.record(stream)
    barrier()
    sampler.window(tw0, time.perf_counter())
    ms_dev = ev0.elapsed_time(ev1)
    stats = ctx.stats()
    # SA-only share from the library's own phase events (same timed region)
    sa_ms = sum(sum(v) for k, v in phase_acc.items() if not k.startswith("lcp")) / steps

    # ---------------- end-to-end through the host-buffer C-ABI (`e2e`)
    h_text = torch.from_numpy(text).pin_memory()
    h_sa = torch.empty(n, dtype=torch.int32).pin_memory()
    h_lcp = torch.empty(n, dtype=torch.int32).pin_memory()
    L = _lib.lib()

    def step_host():
        rc = L.b200sa_build_lcp(ctx._h, h_text.data_ptr(), n, h_sa.data_ptr(), h_lcp.data_ptr())
        if rc != 0:
            raise RuntimeError(L.b200sa_last_error(ctx._h).decode())

    for _ in range(min(warm, 3)):
        step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_host()                       # synchronous: returns with SA/LCP in host memory
    barrier()
    ms_e2e = (time.perf_counter() - t0) * 1e3
    sampler.window(t0, time.perf_counter())
    clocks = sampler.stop() if rank == 0 else None
    e2e_result_check = int(h_lcp[0].item()) + int(h_sa[0].item() >= 0)   # touch the result

    # ---------------- N > 1: ONE text sharded over the GPUs (BASELINE config 5; SURVEY 8e):
    # classification + LMS-suffix sort of N x shard_bytes of G_dna with NCCL inside the library
    sharded_rec = None
    if world > 1 and not args.no_sharded:
        sharded_rec = _sharded_record(args, ctx, dist, rank, world, dev)

    # ---------------- max over ranks
    if world > 1:
        tt = torch.tensor([ms_dev, ms_e2e], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_dev, ms_e2e = float(tt[0].item()), float(tt[1].item())
        lt = torch.tensor([launches], dtype=torch.int64, device=dev)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt.item())

    if rank == 0:
        peak, peak_src = _peaks()
        total_bytes = n * world
        value = total_bytes * steps / 1e6 / (ms_dev / 1e3)
        e2e = total_bytes * steps / 1e6 / (ms_e2e / 1e3)
        # ---- roofline of the dominant kernel: the persistent induce passes (2 launches per build on the direct
        # path, 4 on the robust path)
        m = stats["m"]
        nL = n / 2.0
        # SURVEY.md Appendix D, level 0 (w = 1 byte): L pass 4n+(w+1)(m+nL)+4nL, S pass 4n+(w+1)n+4nS
        bytes_L = 4 * n + 2 * (m + nL) + 4 * nL
        bytes_S = 4 * n + 2 * n + 4 * (n - nL)
        ind = {k: statistics.mean(v) for k, v in phase_acc.items() if k.startswith("induce")}
        ind_ms = statistics.mean(ind.values()) if ind else None
        alg = (bytes_L + bytes_S) / 2.0
        achieved = alg / 1e9 / (ind_ms / 1e3) if ind_ms else None
        traffic, traffic_src = None, None
        ncu_p = os.path.join(ROOT, "profiles", "ncu_summary.json")
        if os.path.exists(ncu_p):
            try:
                rec = json.load(open(ncu_p)).get("k_induce", {})
                traffic, traffic_src = rec.get("dram_bytes_per_launch"), rec.get("source")
            except Exception:
                traffic = None
        phase_ms = {k: round(statistics.mean(v), 3) for k, v in phase_acc.items()}
        dom_share = (sum(ind.values()) / (ms_dev / steps)) if ind else None
        # per-phase achieved GB/s against the same peak (SURVEY.md Appendix D bytes, level 0, w = 1; the
        # LMS sort has no App. D row: 4 one-sweep passes x (8 B in + 8 B out) x m + the digit-histogram read)
        appd = {"classify": 2 * n, "lms_sort": 4 * 16 * m + 4 * m, "lms_groups": 8 * m, "lms_group": 9 * m,
                "induce1_L": bytes_L, "induce1_S": bytes_S,
                "induce2_L": bytes_L, "induce2_S": bytes_S, "compact_lms": 4 * n + n / 8 + 4 * m,
                "name": 8 * n + 4 * m, "unrename": 16 * m, "lcp_direct": 8 * n, "lcp_phi": 8 * n, "lcp_plcp": 12 * n,
                "lcp_gather": 12 * n}
        phases_roof = {}
        for k, b in appd.items():
            if k in phase_ms and phase_ms[k] > 0:
                g = b / 1e9 / (phase_ms[k] / 1e3)
                phases_roof[k] = {"GBps": round(g, 1), "frac": round(g / peak, 4)}
        n_ind = len(ind)
        roof = {"bound": "hbm", "kernel": "induce pass kernels (k_induce6<L|S> on 2-bit text; mean of the %d persistent launches per build)" % n_ind,
                "achieved": round(achieved, 1) if achieved else None, "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4) if achieved else None, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": int(alg),
                "kernel_ms_per_launch": round(ind_ms, 4) if ind_ms else None,
                "share_of_step": round(dom_share, 3) if dom_share else None,
                "pipeline_bytes_per_input_byte_compulsory": 14, "phases": phases_roof}
        # ---- CPU baseline (oracle port) on the SAME n bytes, rank 0, N=1 only; the SA and LCP the
        # device-resident loop just built are compared with the oracle's bit for bit
        cpu = None
        if world == 1 and not args.no_cpu:
            dt, sa_cpu, lcp_cpu = _oracle_time(text)
            cpu = {"value": round(n / 1e6 / dt, 3), "unit": UNIT, "cores": 1, "kind": "port",
                   "sample": "all %d bytes of the workload (one step), oracle port of sais()+lcp_lens(), 1 thread of %d host cores"
                             % (n, os.cpu_count() or 0), "seconds": round(dt, 2)}
            sa_gpu = d_sa.cpu().numpy().view(np.uint32)
            lcp_gpu = d_lcp.cpu().numpy().view(np.uint32)
            cpu["gpu_matches_oracle"] = bool(np.array_equal(sa_gpu, sa_cpu) and np.array_equal(lcp_gpu, lcp_cpu))
            cpu["gpu_matches_oracle_e2e"] = bool(np.array_equal(h_sa.numpy().view(np.uint32), sa_cpu) and
                                                 np.array_equal(h_lcp.numpy().view(np.uint32), lcp_cpu))
            cpu["compared"] = "SA and LCP, all %d entries each, device-resident result and host-API result" % n
        if args.dump_outputs:           # d_sa / d_lcp still hold the last device-resident step's result
            _dump_outputs(args.dump_outputs, {"sa": d_sa.cpu().numpy().view(np.uint32),
                                              "lcp": d_lcp.cpu().numpy().view(np.uint32)})
        out = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": warm, "ms_per_step": round(ms_dev / steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": _config(n, world),
            "e2e": {"value": round(e2e, 2), "unit": UNIT, "h2d_bytes_per_step": n, "d2h_bytes_per_step": 8 * n,
                    "ms_per_step": round(ms_e2e / steps, 3), "api": "b200sa_build_lcp (pinned host buffers)",
                    "host_binding_rank0": numa,
                    "result_touch": e2e_result_check},
            "gpu_launches": launches,
            "sa_only": {"value": round(n * world / 1e6 / (sa_ms / 1e3), 2), "unit": UNIT, "ms_per_step": round(sa_ms, 3)},
            "phase_ms": phase_ms,
            "levels": {"n": n, "m": stats["m"], "names": stats["names"], "doubling_rounds": stats["doubling_rounds"]},
            "roofline": roof, "cpu_baseline": cpu, "clocks": clocks,
        }
        if sharded_rec is not None:
            out["sharded"] = sharded_rec
        _emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()
    return 0


_REAL_STDOUT = None


def _emit(line: str):
    """The contract is ONE JSON line on stdout: everything else any library prints
    (NCCL banners etc.) is diverted to stderr by main(); this writes to the real stdout."""
    data = (line + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(line + "\n")
        sys.stdout.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)                       # fd 1 -> stderr for the duration of the run
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=N_TEXT, help="text bytes per GPU (default: the 100 MB config)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-sharded", action="store_true", help="N > 1: skip the sharded config-5 record")
    ap.add_argument("--shard-bytes", type=int, default=1_000_000_000, help="N > 1: bytes per GPU of the sharded text")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's SA and LCP (rank 0; sampled, see DUMP_ENTRIES) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; it does not apply to --impl reference")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


if __name__ == "__main__":
    sys.exit(main())
