#!/usr/bin/env python3
"""bench.py -- throughput of LaTok's tokenization hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload tweets|mixed|docs|chars1b] [--impl reference]
                    [--dump-outputs DIR]

One step = one pass of the hot path (split mask + token spans + CSR offsets) over one batch of
synthetic text.  Top-level line: BASELINE config #2, 1 M tweet-sized strings per GPU (seed 20240601).

Reported on ONE JSON line (rank 0):
  value          input UTF-8 GB/s over all GPUs, text already resident in HBM (device-pointer C-ABI entry)
  e2e            same metric through the host-buffer C-ABI call: pinned host text -> H2D -> kernels -> D2H results,
                 double-buffered INSIDE the library (pipeline depth 2, one engine, one host thread); `modes` holds
                 the same loop for spans only (what tokenize() needs) and for compact 16-bit spans
  roofline       algorithmic bytes (B + C + 8T + 16(S+1) [+ 25T], SURVEY.md 8d) / CUDA-event time of the tokenize kernel
  other_configs  (N=1, default workload) the same measurements for config #4 (mixed Unicode, classification on) and
                 config #3 (long documents, >= 3 GB of unique text)
  config5_strong the ONE 1 B-character batch of config #5 cut into byte-balanced string ranges, one per rank:
                 ms per pass, and the same batch on one GPU in the same run (speed-up)
  python_dropin  (N=1) the Python drop-in: C-side packing of list[str], tokenize_batch, tokenize_packed().to_arrow()
  cpu_baseline   the compiled reference (oracle/_ref) on all host cores over a bounded sample (rank 0, N=1)
--dump-outputs DIR writes the arrays the last timed step of the top-level measurement returned (rank 0) to DIR/*.npy,
so that two builds can be compared output for output on the same seeded inputs (see dump_outputs).
N > 1 is launched by torchrun (one rank per GPU); ranks hold different batches (weak scaling), there is
no data-path collective; the span-count exchange is one all_gather of an int64 per rank.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(1, str(ROOT / "tests"))       # synth.py (bench / test data generators) lives with the tests

DOC_BLOCK = 3000                                # documents per generator task (one seed each)
WORKLOADS = {
    "tweets": dict(desc="config#2: 1M synthetic tweet-sized strings (~140 chars, ASCII-heavy), seed 20240601", n=1_000_000),
    "mixed": dict(desc="config#4: 1M mixed-Unicode strings (~160 chars), token classification on, seed 20240603", n=1_000_000),
    "docs": dict(desc="config#3: 48 000 long documents of 64 KB (3.2 GB of unique text: 16 blocks of 3 000 documents, seeds "
                      "20240602+1000k; ~1 % with >= 32 KB space-free runs, ~2 % with multi-mark chunks)", n=16 * DOC_BLOCK),
    # strong scaling: ONE batch of ~1e9 characters, cut into byte-balanced ranges of whole strings, one range per rank
    "chars1b": dict(desc="config#5: 1B-character batch of config-#2 text (7.1M strings, seeds 20240605+) sharded by "
                         "byte-balanced string ranges", n=7_100_000),
}
CPU_SAMPLE_STRINGS = {"tweets": 200_000, "mixed": 200_000, "docs": 200, "chars1b": 200_000}


# ------------------------------------------------------------------------------------------ synthetic data
def _gen_task(task):
    import synth
    kind, n, seed = task
    if kind == "tweets":
        return synth.tweets(n, seed)
    if kind == "mixed":
        return synth.mixed_unicode(n, seed)
    return synth.long_docs(n, 65536, seed)


def batch_tasks(workload: str, n: int, seed_shift: int):
    """Generator tasks (kind, strings, seed) whose results, concatenated, are one batch of `workload`."""
    if workload == "chars1b":
        out, k = [], 0
        while n > 0:
            m = min(n, 1_000_000)
            out.append(("tweets", m, 20240605 + k)); n -= m; k += 1
        return out
    if workload == "tweets":
        return [("tweets", n, 20240601 + seed_shift)]
    if workload == "mixed":
        return [("mixed", n, 20240603 + seed_shift)]
    out, k = [], 0
    while n > 0:
        m = min(n, DOC_BLOCK)
        out.append(("docs", m, 20240602 + seed_shift + 1000 * k)); n -= m; k += 1
    return out


def concat_batches(parts):
    if len(parts) == 1:
        return parts[0]
    bufs, offs, base = [], [np.zeros(1, dtype=np.int64)], 0
    for b, o in parts:
        bufs.append(b); offs.append(o[1:] + base); base += len(b)
    return np.concatenate(bufs), np.concatenate(offs)


def generate(requests, procs=None):
    """requests: {name: [task, ...]} -> {name: (buf, offsets)}.  The generators are single-threaded NumPy (10-30 s
    per task); all tasks of the run are spread over a fork pool -- before CUDA is initialised in this process."""
    import multiprocessing as mp
    flat = [(name, i, t) for name, ts in requests.items() for i, t in enumerate(ts)]
    if not flat:
        return {}
    procs = max(1, min(procs or (os.cpu_count() or 1), len(flat)))
    order = sorted(range(len(flat)), key=lambda j: -flat[j][2][1] * (20 if flat[j][2][0] == "docs" else 1))
    if procs == 1:
        res = [_gen_task(flat[j][2]) for j in order]
    else:
        with mp.get_context("fork").Pool(procs) as pool:
            res = pool.map(_gen_task, [flat[j][2] for j in order], chunksize=1)
    got = {}
    for j, r in zip(order, res):
        got[(flat[j][0], flat[j][1])] = r
    return {name: concat_batches([got[(name, i)] for i in range(len(ts))]) for name, ts in requests.items()}


def make_batch(workload: str, n: int, seed_shift: int):
    return generate({"b": batch_tasks(workload, n, seed_shift)})["b"]


# ------------------------------------------------------------------------------------------ CPU arm
_W = {}


def _cpu_init(kind, shard_strings, shard_packed):
    _W["kind"] = kind
    if kind == "reference":
        from oracle import ref_driver
        ref_driver.ext()
        _W["ref"] = ref_driver
        _W["strings"] = shard_strings
    else:
        from oracle import oracle
        oracle.lib()
        _W["oracle"] = oracle
        _W["packed"] = shard_packed


def _cpu_step(_):
    if _W["kind"] == "reference":
        f = _W["ref"].split_positions   # np.nonzero(gen_split_mask(_gen_parse_matrix(t)))[0]
        n = 0
        for t in _W["strings"]:
            if t:
                n += len(f(t))
        return n
    buf, off = _W["packed"]
    return int(_W["oracle"].tokenize_batch_utf8(buf, off, feats=False)["n_tokens"])


class CpuArm:
    """The reference's CPU path on the host cores: one worker process per core, each holding a
    shard of the sample; a step = every worker runs its shard once."""

    def __init__(self, buf, off, n_sample, cores=None):
        import multiprocessing as mp
        import synth
        from oracle import ref_driver
        self.kind = "reference" if ref_driver.available() else "port"
        self.cores = cores or os.cpu_count() or 1
        n_sample = min(n_sample, len(off) - 1)
        self.n_strings = n_sample
        self.n_bytes = int(off[n_sample])
        bounds = np.linspace(0, n_sample, self.cores + 1).astype(np.int64)
        ctx = mp.get_context("fork")
        self.pools = []
        for w in range(self.cores):
            a, b = int(bounds[w]), int(bounds[w + 1])
            strings = synth.to_strings(buf, off, a, b) if self.kind == "reference" else None
            packed = (np.ascontiguousarray(buf[off[a]:off[b]]), (off[a:b + 1] - off[a]).copy())
            self.pools.append(ctx.Pool(1, initializer=_cpu_init, initargs=(self.kind, strings, packed)))
        self.sample = (f"first {n_sample} strings ({self.n_bytes / 1e6:.1f} MB) of the workload; call = "
                       + ("np.nonzero(gen_split_mask(_gen_parse_matrix(t)))[0] per string on the compiled reference latok.c"
                          if self.kind == "reference" else "oracle C restatement, batch call, utf-8 in"))

    def step(self):
        t0 = time.perf_counter()
        res = [p.apply_async(_cpu_step, (0,)) for p in self.pools]
        for r in res:
            r.get()
        return time.perf_counter() - t0

    def close(self):
        for p in self.pools:
            p.terminate()


def run_reference(args, rank, world):
    if rank != 0:
        return 0
    wl = args.workload
    n_sample = CPU_SAMPLE_STRINGS[wl]
    buf, off = make_batch("tweets" if wl == "chars1b" else wl, n_sample, 4 if wl == "chars1b" else 0)
    arm = CpuArm(buf, off, n_sample)
    for _ in range(args.warmup):
        arm.step()
    t = sum(arm.step() for _ in range(args.steps))
    arm.close()
    gbs = arm.n_bytes * args.steps / t / 1e9
    line = {
        "impl": "reference", "metric": "tokenized_text_throughput", "value": gbs, "unit": "GB/s",
        "strings_per_s": arm.n_strings * args.steps / t,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOADS[wl]["desc"], "step": "bounded sample: " + arm.sample},
        "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": arm.cores, "kind": arm.kind, "sample": arm.sample},
        "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
    def __init__(self, device_index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz, self.stop_flag, self.ok = [], set(), None, False, False
        self.paused = False             # set while the host works and the GPU idles (--dump-outputs)
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            if self.paused:
                time.sleep(0.004)
                continue
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.004)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def bind_near_gpu(device_index):
    """Keep this rank's threads (and therefore its first-touched pinned buffers) on the NUMA node of its GPU."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(device_index)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"numa_node": node, "bound": False}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "bound": bool(cpus), "cpus": len(cpus)}
    except Exception as exc:
        return {"numa_node": None, "bound": False, "why": repr(exc)[:80]}


# ------------------------------------------------------------------------------------------ GPU arm
def pinned_array(lib, nbytes, dtype):
    p = C.c_void_p()
    from latok_b200 import _lib
    _lib.check(lib.latok_b200_host_alloc(C.byref(p), max(nbytes, 16)))
    arr = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(nbytes, 16),))
    return arr[:nbytes].view(dtype), p


class Ctx:
    """What every measurement needs: the library, the rank's engine, torch / dist handles."""

    def __init__(self, lib, eng, torch, dist, rank, world, local_rank):
        self.lib, self.eng, self.torch, self.dist = lib, eng, torch, dist
        self.rank, self.world, self.local_rank = rank, world, local_rank

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, xs):
        if self.world == 1:
            return [float(x) for x in xs]
        t = self.torch.tensor(list(xs), device="cuda", dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]


def load_peak():
    peaks_file = ROOT / "MEASURED_PEAKS.json"
    if peaks_file.exists():
        return float(json.load(open(peaks_file))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_ARRAYS = ("splits", "char_offsets", "spans", "tok_offsets", "tok_feats")
DUMP_BYTES_PER_ARRAY = 12 << 20                 # five arrays at most: 60 MB in all


def dump_outputs(r, out_dir, seed=0):
    """Writes the arrays of the BatchResult `r` as out_dir/<name>.npy: int8 arrays as float32, wider integers as
    float64 (every value exact).  An array larger than DUMP_BYTES_PER_ARRAY keeps a sample of its rows, in order,
    drawn with a fixed seed from its length alone: two builds that agree on the sizes dump the same rows."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name in DUMP_ARRAYS:
        a = getattr(r, name)
        if a is None:
            continue
        dtype = np.dtype(np.float32 if a.dtype.itemsize == 1 else np.float64)
        keep = DUMP_BYTES_PER_ARRAY // (dtype.itemsize * int(np.prod(a.shape[1:], dtype=np.int64)))
        if len(a) > keep:
            a = a[np.sort(np.random.default_rng(seed).choice(len(a), keep, replace=False))]
        np.save(out_dir / f"{name}.npy", a.astype(dtype))


def measure_resident(cx: Ctx, host, what, steps, warmup, classify, wl_key, sample_clocks=True, dump_dir=None):
    """Device-resident pass: `host` = list of (buf, offsets) batches of this rank, rotated; returns the fields of a
    bench record (value, ms_per_step, roofline, clocks, ...) plus the per-batch stats.  `dump_dir`: rank 0 writes the
    results of the last timed step there (dump_outputs)."""
    from latok_b200 import _lib
    torch, eng, lib = cx.torch, cx.eng, cx.lib
    R = len(host)
    dev = [(torch.from_numpy(b).cuda(), torch.from_numpy(o).cuda()) for b, o in host]

    def run_resident(i):
        b, o = dev[i % R]
        eng.submit_device(b.data_ptr(), o.data_ptr(), o.numel() - 1, b.numel(), what)

    stats = []                          # sizes per batch (also sizes the span buffers of both sets: no re-runs later)
    for i in range(2 * R):
        run_resident(i)
        c, t = eng.sizes()
        if i < R:
            stats.append((len(host[i][0]), c, t, len(host[i][1]) - 1))
    for i in range(max(warmup, 3)):
        run_resident(i)
    eng.sizes()
    sampler = ClockSampler(cx.local_rank) if sample_clocks else None
    if sampler:
        sampler.start()
    launches0 = eng.launch_count()
    cx.barrier()
    eng.timer_begin()
    for i in range(steps):
        run_resident(i)
    elapsed_ms = eng.timer_end()
    cx.barrier()
    launches = eng.launch_count() - launches0
    if dump_dir and cx.rank == 0:
        # before the launches below replace the last timed step's results; the clocks of the idle GPU meanwhile are
        # not the clocks of the workload
        if sampler:
            sampler.paused = True
        dump_outputs(eng.fetch(), dump_dir)
        if sampler:
            sampler.paused = False
    # per-launch duration of the dominant kernel, measured live (CUDA events around the tokenize kernel on the
    # stream it is launched on), one step at a time after the timed region
    kernel_ms = []
    for i in range(min(steps, 50)):
        run_resident(i)
        eng.sizes()
        ms, w = C.c_float(0), C.c_int64(0)
        _lib.check(lib.latok_b200_last_stats(eng._h, C.byref(ms), C.byref(w)))
        kernel_ms.append(ms.value)
    if sampler:                         # keep the GPU under the same load until the clock sampler has enough samples
        t_end = time.time() + 1.0
        while len(sampler.samples) < 40 and time.time() < t_end:
            run_resident(0)
            eng.sizes()
        sampler.stop_flag = True
        sampler.join()
    elapsed_ms = cx.max_over_ranks(elapsed_ms)
    total_bytes, total_strings = cx.sum_over_ranks([sum(stats[i % R][0] for i in range(steps)),
                                                    sum(stats[i % R][3] for i in range(steps))])
    peak, peak_src = load_peak()
    alg = float(np.mean([b + c + 8 * t + 16 * (s + 1) + (25 * t if classify else 0) for b, c, t, s in stats]))
    k_ms = float(np.mean(kernel_ms)) if kernel_ms else float("nan")
    achieved = alg / (k_ms * 1e-3) / 1e9
    traffic, traffic_note, traffic_ratio = None, None, None
    tf = ROOT / "profiles" / "traffic.json"
    if tf.exists():
        try:
            rec = json.load(open(tf)).get(wl_key)
            if isinstance(rec, dict):
                traffic, traffic_note, traffic_ratio = rec.get("dram_bytes"), rec.get("note"), rec.get("ratio")
        except Exception:
            pass
    rec = {
        "value": total_bytes / (elapsed_ms * 1e-3) / 1e9, "unit": "GB/s",
        "strings_per_s": total_strings / (elapsed_ms * 1e-3),
        "steps": steps, "ms_per_step": elapsed_ms / steps,
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_over_algorithmic": traffic_ratio, "traffic_note": traffic_note,
                     "kernel": "latok::v5::tokenize5_kernel<kFeats>" if classify else "latok::v5::tokenize5_kernel",
                     "kernel_ms": k_ms, "algorithmic_bytes_per_launch": alg, "peak_source": peak_src,
                     "frac_of_nominal_8TBs": achieved / 8000.0},
        "sizes": {"strings_per_gpu": int(np.mean([s[3] for s in stats])), "bytes_per_step_per_gpu": int(np.mean([s[0] for s in stats])),
                  "chars_per_step_per_gpu": int(np.mean([s[1] for s in stats])),
                  "tokens_per_step_per_gpu": int(np.mean([s[2] for s in stats])), "resident_batches": R},
    }
    if sampler:
        rec["clocks"] = sampler.summary()
    del dev
    return rec, stats


def measure_e2e(cx: Ctx, hb, ho, stat, what, steps):
    """End to end through the host-buffer C-ABI calls, ONE engine and ONE host thread: pinned host text in, pinned
    host arrays out, pipeline depth 2 inside the library -- submit(i+1) (H2D + kernels) is enqueued before fetch(i)
    (D2H) blocks, so the two directions of PCIe and the kernels overlap.  Returns (seconds, h2d, d2h bytes / step)."""
    from latok_b200 import _lib
    from latok_b200.engine import SPLITS, SPANS, FEATS, SPANS16
    lib, eng = cx.lib, cx.eng
    B0, C0, T0, S0 = stat
    keep = []

    def pin(nbytes, dtype):
        a, p = pinned_array(lib, nbytes, dtype)
        keep.append(p)
        return a
    ins = []
    for _ in range(2):                  # the caller alternates two pinned input buffers, like a reader would
        pb, po = pin(len(hb), np.uint8), pin(8 * len(ho), np.int64)
        pb[:] = hb
        po[:] = ho
        ins.append((pb, po))
    outs = []
    for _ in range(2):
        outs.append(dict(
            splits=pin(C0, np.int8) if what & SPLITS else None,
            spans=pin((4 if what & SPANS16 else 8) * T0, np.uint8) if what & (SPANS | SPANS16) else None,
            coff=pin(8 * (S0 + 1), np.int64), toff=pin(8 * (S0 + 1), np.int64),
            feats=pin(25 * T0, np.int8) if what & FEATS else None))

    def ptr(a):
        return None if a is None else a.ctypes.data

    def submit(i):
        pb, po = ins[i & 1]
        _lib.check(lib.latok_b200_submit(eng._h, pb.ctypes.data, po.ctypes.data, S0, what))

    def fetch(i):
        o = outs[i & 1]
        _lib.check(lib.latok_b200_fetch(eng._h, C0, T0, S0, ptr(o["splits"]), ptr(o["coff"]), ptr(o["spans"]), ptr(o["toff"]),
                                        ptr(o["feats"]), None))
        _lib.check(lib.latok_b200_release(eng._h))

    def loop(n):
        submit(0)
        for i in range(n):
            if i + 1 < n:
                submit(i + 1)
            fetch(i)

    _lib.check(lib.latok_b200_set_pipeline_depth(eng._h, 2))
    try:
        loop(3)
        cx.barrier()
        t0 = time.perf_counter()
        loop(steps)
        cx.torch.cuda.synchronize()
        dt = time.perf_counter() - t0
    finally:
        _lib.check(lib.latok_b200_set_pipeline_depth(eng._h, 1))
    dt = cx.max_over_ranks(dt)
    # the two output sets hold the same batch: cheap end-to-end sanity check of the pipelined path
    assert np.array_equal(outs[0]["toff"], outs[1]["toff"]) and int(outs[0]["toff"][-1]) == T0
    if outs[0]["spans"] is not None:
        assert np.array_equal(outs[0]["spans"], outs[1]["spans"])
    h2d = B0 + 8 * (S0 + 1)
    d2h = ((C0 if what & SPLITS else 0) + ((4 if what & SPANS16 else 8) * T0 if what & (SPANS | SPANS16) else 0)
           + 16 * (S0 + 1) + 64 + (25 * T0 if what & FEATS else 0))
    for p in keep:
        lib.latok_b200_host_free(p)
    return dt, int(h2d), int(d2h)


def e2e_record(cx: Ctx, hb, ho, stat, what, steps, modes=True):
    from latok_b200.engine import SPLITS, SPANS, SPANS16
    B0, S0 = stat[0], stat[3]
    dt, h2d, d2h = measure_e2e(cx, hb, ho, stat, what, steps)
    rec = {"value": cx.world * B0 * steps / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "steps": steps, "strings_per_s": cx.world * S0 * steps / dt, "ms_per_step": 1e3 * dt / steps,
           "mode": "in-library double buffering: ONE engine, ONE host thread, pipeline depth 2 (submit(i+1) before fetch(i)); "
                   "pinned host buffers; outputs = int8 split mask + int32 spans + int64 CSR offsets"
                   + (" + int8[T,25] token feature sums" if what & 4 else "")}
    if modes:
        rec["modes"] = {}
        for name, w, note in (("spans", SPANS, "int32 spans + CSR offsets: what tokenize() / tokenize_batch() need"),
                              ("spans16", SPANS16, "uint16 spans (LATOK_B200_SPANS16: every string < 65 536 characters) + CSR offsets")):
            w |= what & 4
            dt2, h2, d2 = measure_e2e(cx, hb, ho, stat, w, steps)
            rec["modes"][name] = {"value": cx.world * B0 * steps / dt2 / 1e9, "unit": "GB/s", "h2d_bytes_per_step": h2,
                                  "d2h_bytes_per_step": d2, "ms_per_step": 1e3 * dt2 / steps, "outputs": note}
    return rec


def python_dropin(cx: Ctx, hb, ho, n=200_000):
    """The Python drop-in on list[str] (rank 0, N=1): C-side packing, tokenize_batch (token strings, like the reference's
    generator), tokenize_packed().to_arrow() (no Python string per token); the reference's own list(tokenize(t)) on the
    same strings, one core."""
    import synth
    from latok_b200.core import default_tokenizer as dt
    from latok_b200.engine import pack_strings
    n = min(n, len(ho) - 1)
    texts = synth.to_strings(hb, ho, 0, n)
    nb = int(ho[n])
    out = {"strings": n, "bytes": nb}
    pack_strings(texts)
    t0 = time.perf_counter(); buf, off = pack_strings(texts); t = time.perf_counter() - t0
    out["pack_strings_per_s"] = n / t
    out["pack_gbs"] = nb / t / 1e9
    dt.tokenize_batch(texts[:1000], engine=cx.eng)
    t0 = time.perf_counter(); toks = dt.tokenize_batch(texts, engine=cx.eng); t = time.perf_counter() - t0
    out["tokenize_batch_strings_per_s"] = n / t
    dt.tokenize_packed(buf, off, engine=cx.eng).to_arrow()
    t0 = time.perf_counter(); dt.tokenize_packed(*pack_strings(texts), engine=cx.eng).to_arrow(); t = time.perf_counter() - t0
    out["pack_plus_tokenize_packed_to_arrow_strings_per_s"] = n / t
    out["tokens"] = int(sum(len(x) for x in toks))
    try:
        from oracle import ref_driver
        if ref_driver.available():
            m = min(n, 20_000)
            t0 = time.perf_counter()
            ref = [list(ref_driver.tokenize(s)) for s in texts[:m]]
            t = time.perf_counter() - t0
            out["reference_list_tokenize_strings_per_s_one_core"] = m / t
            out["tokens_match_reference"] = bool(ref == toks[:m])
    except Exception as exc:
        out["reference"] = repr(exc)[:100]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed steps of the top-level measurement, on every workload (docs: each step is one pass over "
                         "3.2 GB of text); up to 50 more follow, one at a time, for the per-launch kernel time")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="tweets", choices=list(WORKLOADS))
    ap.add_argument("--strings", type=int, default=0, help="override strings per GPU -- chars1b: of the whole batch -- (smaller = NOT the named config)")
    ap.add_argument("--resident-batches", type=int, default=3)
    ap.add_argument("--e2e-steps", type=int, default=60)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="skip other_configs / config5_strong / python_dropin")
    ap.add_argument("--strong-strings", type=int, default=0, help="override the size of the config-#5 batch (NOT the named config)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step to DIR/<name>.npy "
                    "(float32 / float64; arrays over 12 MB as a seeded sample of their rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference leg returns token counts only")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if args.warmup < 3:
        args.warmup = 3
    if world == 1 and args.gpus > 1:
        print(json.dumps({"error": "launch N>1 with torch.distributed.run (one rank per GPU)"}))
        return 2
    numa = bind_near_gpu(local_rank)

    wl = args.workload
    n_strings = args.strings or WORKLOADS[wl]["n"]
    strong_top = wl == "chars1b"
    full = wl == "tweets" and not args.no_others and not args.strings
    R = 1 if wl in ("docs", "chars1b") else max(1, args.resident_batches)

    # ---- all synthetic text of the run, generated by a pool of processes before CUDA is touched --------------
    t_gen = time.time()
    req = {}
    if strong_top:
        req["strong"] = batch_tasks("chars1b", n_strings, 0)
    else:
        for r in range(R):
            req[f"top{r}"] = batch_tasks(wl, n_strings, 1000 * rank + r)
    if full:
        req["strong"] = batch_tasks("chars1b", args.strong_strings or WORKLOADS["chars1b"]["n"], 0)
        if world == 1:
            req["mixed"] = batch_tasks("mixed", WORKLOADS["mixed"]["n"], 0)
            req["docs"] = batch_tasks("docs", WORKLOADS["docs"]["n"], 0)
    data = generate(req, procs=max(1, (os.cpu_count() or 1) // max(1, min(world, 8))))
    t_gen = time.time() - t_gen

    import torch
    import torch.distributed as dist
    from latok_b200 import _lib
    from latok_b200.engine import Engine, SPLITS, SPANS, FEATS
    from latok_b200.sharding import shard_ranges, slice_shard

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = _lib.load()
    eng = Engine(local_rank)
    cx = Ctx(lib, eng, torch, dist, rank, world, local_rank)

    def strong_shard(fb, fo):
        s0, s1 = shard_ranges(fo, world)[rank]
        b, o = slice_shard(fb, fo, s0, s1)
        return np.ascontiguousarray(b), np.ascontiguousarray(o)

    classify = wl == "mixed"          # config #4 is quoted with token classification (per-token feature sums) enabled
    what = SPLITS | SPANS | (FEATS if classify else 0)
    if strong_top:
        host = [strong_shard(*data.pop("strong"))]
    else:
        host = [data.pop(f"top{r}") for r in range(R)]
    steps = args.steps
    top, stats = measure_resident(cx, host, what, steps, args.warmup, classify, wl if not args.strings else "",
                                  dump_dir=args.dump_outputs)
    if world > 1:
        # the path's only cross-GPU datum: per-rank token counts, to rebase global token offsets
        counts = torch.zeros(world, device="cuda", dtype=torch.int64)
        dist.all_gather_into_tensor(counts, torch.tensor([stats[0][2]], device="cuda", dtype=torch.int64))
    e2e_steps = args.e2e_steps if wl != "docs" else min(args.e2e_steps, 8)
    e2e = e2e_record(cx, host[0][0], host[0][1], stats[0], what, e2e_steps)

    line = {
        "metric": "tokenized_text_throughput", "value": top["value"], "unit": "GB/s",
        "strings_per_s": top["strings_per_s"],
        "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": top["ms_per_step"],
        "higher_is_better": True, "scaling": "strong" if strong_top else "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOADS[wl]["desc"] + (f" [OVERRIDE strings={args.strings}]" if args.strings else ""),
                   **top["sizes"],
                   "outputs": "int8 split mask + int32 spans + int64 CSR offsets" + (" + int8[T,25] token feature sums" if classify else ""),
                   "l2_hygiene": f"{R} distinct resident batch(es) rotated; per-step footprint "
                                 f"{top['roofline']['algorithmic_bytes_per_launch'] / 1e6:.0f} MB > 126 MB L2",
                   "sharding": ("one rank per GPU on its byte-balanced range of whole strings of the ONE batch, no data-path "
                                "collective, one all-gather of the per-rank token counts" if strong_top else
                                "one rank per GPU, independent batches, no data-path collective"),
                   "data_generation_s": round(t_gen, 1), "numa": numa},
        "e2e": e2e,
        "gpu_launches": top["gpu_launches"],
        "roofline": top["roofline"],
        "clocks": top["clocks"],
    }
    host_top = host[0]
    del host

    # ---- config #5: the ONE 1B-character batch, strong scaling ------------------------------------------------
    if full:
        fb, fo = data.pop("strong")
        sb, so = strong_shard(fb, fo)
        srec, sstats = measure_resident(cx, [(sb, so)], SPLITS | SPANS, 20, 3, False, "", sample_clocks=False)
        ms_shard = srec["ms_per_step"]
        c5 = {"workload": WORKLOADS["chars1b"]["desc"] + (f" [OVERRIDE strings={args.strong_strings}]" if args.strong_strings else ""),
              "batch_bytes": int(len(fb)), "batch_strings": int(len(fo) - 1), "n_gpus": world,
              "ms_per_pass": ms_shard, "value": len(fb) / (ms_shard * 1e-3) / 1e9, "unit": "GB/s",
              "strings_per_s": (len(fo) - 1) / (ms_shard * 1e-3),
              "rank0_range": {"bytes": int(len(sb)), "strings": int(len(so) - 1), "kernel_ms": srec["roofline"]["kernel_ms"],
                              "roofline_frac": srec["roofline"]["frac"]},
              "timing": "20 passes after 3 warm-ups, CUDA events, max over ranks; a rank's range is far larger than the 126 MB L2"}
        if world > 1:
            # the same batch on ONE GPU, in the same run (every rank runs it alone; max over ranks)
            one, _ = measure_resident(cx, [(fb, fo)], SPLITS | SPANS, 10, 3, False, "", sample_clocks=False)
            c5["ms_per_pass_one_gpu"] = one["ms_per_step"]
            c5["speedup_vs_one_gpu"] = one["ms_per_step"] / ms_shard
        else:
            c5["roofline"] = srec["roofline"]
        se2e = e2e_record(cx, sb, so, sstats[0], SPLITS | SPANS, 10, modes=False)
        c5["e2e"] = {k: se2e[k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "steps", "ms_per_step")}
        c5["e2e"]["value"] = len(fb) / (se2e["ms_per_step"] * 1e-3) / 1e9       # whole batch / time of the slowest rank's range
        line["config5_strong"] = c5
        del fb, fo, sb, so

    # ---- configs #4 and #3 on one GPU ---------------------------------------------------------------------------
    if full and world == 1:
        others = {}
        for name, w2, st, est in (("mixed", SPLITS | SPANS | FEATS, 50, 30), ("docs", SPLITS | SPANS, 20, 6)):
            hb2, ho2 = data.pop(name)
            rec, st2 = measure_resident(cx, [(hb2, ho2)], w2, st, 3, name == "mixed", name)
            rec["workload"] = WORKLOADS[name]["desc"]
            rec["e2e"] = e2e_record(cx, hb2, ho2, st2[0], w2, est, modes=False)
            if name == "mixed":          # the same corpus without classification (split mask + spans only), kernel only
                rec2, _ = measure_resident(cx, [(hb2, ho2)], SPLITS | SPANS, st, 3, False, "mixed_noclass", sample_clocks=False)
                rec["without_classification"] = {"ms_per_step": rec2["ms_per_step"], "value": rec2["value"],
                                                 "roofline": rec2["roofline"]}
            others[name] = rec
            del hb2, ho2
        line["other_configs"] = others
        try:
            line["python_dropin"] = python_dropin(cx, host_top[0], host_top[1])
        except Exception as exc:
            line["python_dropin"] = {"error": repr(exc)[:200]}

    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            arm = CpuArm(host_top[0], host_top[1], CPU_SAMPLE_STRINGS[wl])
            arm.step()
            t = sum(arm.step() for _ in range(3))
            arm.close()
            line["cpu_baseline"] = {"value": arm.n_bytes * 3 / t / 1e9, "unit": "GB/s", "cores": arm.cores,
                                    "kind": arm.kind, "sample": arm.sample,
                                    "strings_per_s": arm.n_strings * 3 / t}
        except Exception as exc:  # the baseline must never take the GPU number down with it
            line["cpu_baseline"] = {"value": None, "unit": "GB/s", "cores": 0, "kind": "unavailable", "sample": repr(exc)}
    if rank == 0:
        print(json.dumps(line))
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
