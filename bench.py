#!/usr/bin/env python
"""bench.py -- compress MB/s at -9 (BASELINE.json metric), one JSON line on rank 0.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload text|random|period1000|aab|runs|mixed]
                  [--mb 1000] [--level 9] [--engines-per-gpu 2] [--no-c4] [--sweep] [--dump-outputs DIR]

A "step" is one pass of the whole compression path (RLE1+CRC -> BWT -> MTF/RLE2 -> Huffman -> stream)
over one synthetic input of --mb MB per GPU (default: the 1 GB Zipf text of SURVEY.md 8(d) C2, BASELINE.json
configs[1]); at N GPUs the input is ONE stream of N x --mb MB, sharded by block over the GPUs (weak scaling).

  value  MB/s of input, input resident in HBM when the timed region starts (bz2b200_multi_compress with device
         pointers), output delivered to pinned host memory
  e2e    the same metric through BZ2_bzBuffToBuffCompress with pinned HOST buffers (H2D + D2H inside)
  roofline      dominant stage (BWT) and whole pass against the measured HBM copy bandwidth (one engine alone)
  cpu_baseline  the reference's own CPU path (oracle/_ref) on a bounded sample, single thread
  parity_checked_bytes   bytes of the timed output compared equal with the reference's stream of a prefix
  c4     secondary line: SURVEY 8(d) C4, 16 GB mixed, strong-scaled over the N GPUs

--dump-outputs DIR writes what the last timed step handed its caller (see dump_outputs) as .npy files, so that two
builds run with the same arguments, hence on the same seeded input, can be compared output for output.

The work is driven through the C API of libbz2_b200.so by ONE process: under torchrun (N > 1) rank 0 drives all N
GPUs (csrc/multi.cu: windows round-robin over the engines, two host integers chain them, no collective on the data
path) while the other ranks generate their part of the input, hand it to rank 0 over NCCL, and then only take part
in the barriers.  With --impl reference the reference CPU implementation (oracle/_ref) is timed on the host's
physical cores, one process per core, each on its slice of the full workload.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402


def make_input(workload, n, rank=0):
    import support as S
    seed = S.TEXT_SEED + rank
    if workload == "text":
        return S.gen_text(n, seed=seed)
    if workload == "random":
        return S.gen_random(n, seed=2 + rank)
    if workload == "period1000":
        return S.gen_period1000(n)
    if workload == "aab":
        return S.gen_tile(n, b"aab")
    if workload == "runs":
        return S.gen_runs(n, seed=3 + rank)
    if workload == "mixed":
        return S.gen_c4(n, seg=64 << 20)
    raise SystemExit(f"unknown workload {workload}")


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line) through NVML,
    at a rate that adapts to what a query costs: a query takes the driver's lock, and on some boxes spawning
    nvidia-smi (or polling NVML every few ms) stretched the timed step by 10 % to 4x."""

    def __init__(self, index, count=1, mode=None):
        self.rows = []
        self.stop = False
        self.index = index
        self.count = count            # GPUs index .. index+count-1 are sampled
        self.how = "nvml"
        self.query_ms = []
        # proc (default): a small helper process polls NVML (0.02 ms per query, no effect on the step).  thread: a sampler
        # thread in this process -- its queries sometimes waited 20-290 ms behind the process's own CUDA calls and stalled
        # one timed step in three at N = 2 (9.1 instead of 11.3 GB/s).  inline: the timed loop polls between steps.
        self.mode = mode or os.environ.get("BENCH_CLOCKS", "proc")
        self.th = threading.Thread(target=self.run, daemon=True)
        self.proc = None
        self._nv = None

    def _run_nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        hs = []
        for k in range(self.index, self.index + self.count):
            idx = k
            if vis:
                try:
                    idx = int(vis.split(",")[k])
                except Exception:  # noqa: BLE001
                    pass
            hs.append(nv.nvmlDeviceGetHandleByIndex(idx))
        mx = [nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM) for h in hs]
        bits = [(nv.nvmlClocksEventReasonHwSlowdown, 0), (nv.nvmlClocksEventReasonHwThermalSlowdown, 1),
                (nv.nvmlClocksEventReasonSwThermalSlowdown, 2), (nv.nvmlClocksEventReasonSwPowerCap, 3)]
        self.ready.set()
        while not self.stop:
            t0 = time.perf_counter()
            for h, m in zip(hs, mx):
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                row = [str(sm), str(m)] + ["Not Active"] * 4
                for bit, k in bits:
                    if r & bit:
                        row[2 + k] = "Active"
                self.rows.append(row)
            dt = time.perf_counter() - t0
            self.query_ms.append(dt * 1e3)
            time.sleep(max(0.1, 30.0 * dt))     # keep the sampler under ~3 % of the wall clock

    def _run_smi(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            time.sleep(1.0)

    def run(self):
        try:
            self._run_nvml()
        except Exception:  # noqa: BLE001
            self.how = "nvidia-smi"
            self.ready.set()
            self._run_smi()

    def _handles(self):
        import pynvml as nv
        nv.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        hs = []
        for k in range(self.index, self.index + self.count):
            idx = k
            if vis:
                try:
                    idx = int(vis.split(",")[k])
                except Exception:  # noqa: BLE001
                    pass
            hs.append(nv.nvmlDeviceGetHandleByIndex(idx))
        return nv, hs

    def poll(self):
        """inline mode: one sample, taken by the caller's thread between two steps of the timed region"""
        if self.mode != "inline" or self._nv is None:
            return
        nv, hs, mx = self._nv
        t0 = time.perf_counter()
        for h, m in zip(hs, mx):
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            row = [str(sm), str(m)] + ["Not Active"] * 4
            for bit, k in ((nv.nvmlClocksEventReasonHwSlowdown, 0), (nv.nvmlClocksEventReasonHwThermalSlowdown, 1),
                           (nv.nvmlClocksEventReasonSwThermalSlowdown, 2), (nv.nvmlClocksEventReasonSwPowerCap, 3)):
                if r & bit:
                    row[2 + k] = "Active"
            self.rows.append(row)
        self.query_ms.append((time.perf_counter() - t0) * 1e3)

    def __enter__(self):
        if self.mode == "inline":
            try:
                nv, hs = self._handles()
                self._nv = (nv, hs, [nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM) for h in hs])
                self.how = "nvml, sampled by the timing thread between steps"
                return self
            except Exception:  # noqa: BLE001
                self.mode = "thread"
        if self.mode == "proc":
            code = ("import sys,time,pynvml as nv\nnv.nvmlInit()\nh=nv.nvmlDeviceGetHandleByIndex(int(sys.argv[1]))\n"
                    "m=nv.nvmlDeviceGetMaxClockInfo(h,nv.NVML_CLOCK_SM)\nprint('ready',flush=True)\n"
                    "while True:\n t=time.perf_counter()\n s=nv.nvmlDeviceGetClockInfo(h,nv.NVML_CLOCK_SM)\n"
                    " r=nv.nvmlDeviceGetCurrentClocksEventReasons(h)\n d=(time.perf_counter()-t)*1e3\n"
                    " print(s,m,r,d,flush=True)\n time.sleep(max(0.1,30*d/1e3))\n")
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.index
            if vis:
                try:
                    idx = int(vis.split(",")[self.index])
                except Exception:  # noqa: BLE001
                    pass
            try:
                self.proc = subprocess.Popen([sys.executable, "-c", code, str(idx)], stdout=subprocess.PIPE,
                                             stderr=subprocess.DEVNULL, text=True)
                if self.proc.stdout.readline().strip() != "ready":      # NVML did not come up in the helper
                    raise RuntimeError("clock helper failed")
                self.how = "nvml, helper process"
                return self
            except Exception:  # noqa: BLE001
                if self.proc is not None:
                    self.proc.kill()
                self.proc = None
                self.mode = "thread"
        self.ready = threading.Event()
        self.th.start()
        self.ready.wait(timeout=10)          # NVML initialisation stays outside the timed region
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.proc is not None:
            self.proc.terminate()
            try:
                out, _ = self.proc.communicate(timeout=5)
            except Exception:  # noqa: BLE001
                out = ""
            for ln in out.splitlines():
                f = ln.split()
                if len(f) == 4:
                    r = int(f[2])
                    self.rows.append([f[0], f[1]] + ["Active" if r & b else "Not Active" for b in (0x8, 0x40, 0x20, 0x4)])
                    self.query_ms.append(float(f[3]))
            return
        if self.mode == "inline":
            return
        self.th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = max(int(r[1]) for r in self.rows if r[1].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[2 + k].lower().startswith("active") for r in self.rows if len(r) > 2 + k)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.rows),
                "source": self.how, "query_ms": round(sorted(self.query_ms)[len(self.query_ms) // 2], 3) if self.query_ms else None}


def physical_cores():
    try:
        import psutil
        c = psutil.cpu_count(logical=False)
        if c:
            return int(c)
    except Exception:  # noqa: BLE001
        pass
    return os.cpu_count() or 1


_REF_JOB = {}


def _ref_slice(t):
    """one worker process of the reference arm: compress slice t of the workload with the reference library"""
    import support as S
    data, per, level, use_ref = _REF_JOB["data"], _REF_JOB["per"], _REF_JOB["level"], _REF_JOB["use_ref"]
    sl = data[t * per:(t + 1) * per]
    out = np.empty(int(per * 1.02) + 70000, np.uint8)
    if use_ref:
        n = C.c_uint(out.size)
        rc = S.ref().BZ2_bzBuffToBuffCompress(S._p(out), C.byref(n), S._p(sl), sl.size, level, 0, 0)
        assert rc == 0
        return n.value
    return S.oracle().orc_compress(S._p(sl), sl.size, level, 1, None, S._p(out), out.size)


def cpu_reference_rate(data, level, procs, keep_output=False):
    """Reference CPU path on `procs` host cores: `procs` independent processes (threads of one process when procs == 1),
    each compressing its own contiguous slice as its own stream (pbzip2-style, BASELINE.md 3).
    Returns (MB/s, kind, sample description, output of slice 0 or None)."""
    import support as S
    use_ref = S.have_ref()
    per = data.size // procs
    out0 = None
    t0 = time.perf_counter()
    if procs == 1:
        lib = S.ref() if use_ref else S.oracle()
        out = np.empty(int(per * 1.02) + 70000, np.uint8)
        if use_ref:
            n = C.c_uint(out.size)
            rc = lib.BZ2_bzBuffToBuffCompress(S._p(out), C.byref(n), S._p(data), per, level, 0, 0)
            assert rc == 0
            nout = n.value
        else:
            nout = lib.orc_compress(S._p(data), per, level, 1, None, S._p(out), out.size)
        if keep_output:
            out0 = out[:nout]
    else:
        import multiprocessing as mp
        _REF_JOB.update(data=data, per=per, level=level, use_ref=use_ref)
        with mp.get_context("fork").Pool(procs) as pool:
            t0 = time.perf_counter()                # the pool is up: time the compression only
            pool.map(_ref_slice, range(procs), chunksize=1)
            dt = time.perf_counter() - t0
        kind = "reference" if use_ref else "port"
        return per * procs / dt / 1e6, kind, (f"{per * procs} B of the workload as {procs} independent slices, one process per physical "
                                              f"core, -{level}, one pass, {dt:.1f} s"), None
    dt = time.perf_counter() - t0
    kind = "reference" if use_ref else "port"
    return per / dt / 1e6, kind, f"{per} B prefix of the workload as one stream on one core, -{level}, one pass, {dt:.1f} s", out0


def merge_clocks(per_gpu):
    """One clocks object for the node: the lowest per-GPU median SM clock, every throttle reason any GPU reported."""
    ok = [c for c in per_gpu if c and c.get("sm_mhz") is not None]
    if not ok:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
    reasons = sorted({r for c in ok for r in c.get("reasons", [])})
    return {"sm_mhz": min(c["sm_mhz"] for c in ok), "sm_max_mhz": max(c["sm_max_mhz"] for c in ok), "reasons": reasons,
            "samples": sum(c.get("samples", 0) for c in ok), "source": ok[0].get("source"),
            "query_ms": max((c.get("query_ms") or 0.0) for c in ok), "per_gpu_sm_mhz": [c["sm_mhz"] for c in ok]}


class Samplers:
    """one clock sampler per GPU of the job"""

    def __init__(self, n):
        self.s = [ClockSampler(g) for g in range(n)]

    def __enter__(self):
        for x in self.s:
            x.__enter__()
        return self

    def __exit__(self, *a):
        for x in self.s:
            x.__exit__(*a)

    def summary(self):
        return merge_clocks([x.summary() for x in self.s]) if len(self.s) > 1 else self.s[0].summary()


DUMP_SAMPLE = 4 << 20          # stream bytes kept by --dump-outputs: 16 MB of float32 values + 32 MB of float64 positions


def dump_outputs(path, stream, st):
    """The .bz2 stream of the last timed step and the counts the C API returned with it.
      stream_bytes.npy  float32, the stream's bytes at the positions in stream_index.npy (all of them up to DUMP_SAMPLE
                        bytes, else a sample drawn with a fixed seed)
      stream_index.npy  float64, those positions, ascending
      stream_stats.npy  float64 [in_bytes, out_bytes, n_blocks, combined_crc, sum_nblock, sum_nmtf, n_power_blocks, out_bits]"""
    os.makedirs(path, exist_ok=True)
    n = stream.size
    idx = np.arange(n) if n <= DUMP_SAMPLE else np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))
    np.save(os.path.join(path, "stream_bytes.npy"), stream[idx].astype(np.float32))
    np.save(os.path.join(path, "stream_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(path, "stream_stats.npy"), np.array([st.in_bytes, st.out_bytes, st.n_blocks, st.combined_crc, st.sum_nblock,
                                                              st.sum_nmtf, st.n_power_blocks, st.out_bits], np.float64))


def equal_prefix(a, b):
    n = min(a.size, b.size)
    ne = np.nonzero(a[:n] != b[:n])[0]
    return int(ne[0]) if ne.size else n


class Job:
    """One workload on the N GPUs of this box, driven by this process through the C API."""

    def __init__(self, torch, B, world, level, engines_per_gpu, data):
        self.torch, self.B, self.world, self.level = torch, B, world, level
        self.n = int(data.numel())
        # engines in GPU-major round-robin order: consecutive windows sit on different GPUs
        self.devices = [g for _ in range(engines_per_gpu) for g in range(world)]
        self.multi = B.Multi(self.devices, level=level)
        self.h_in = data                                       # pinned uint8 tensor
        self.cap = self.multi.out_cap(self.n)
        self.h_out = torch.empty(self.cap, dtype=torch.uint8).pin_memory()
        self.copies = None
        self.out_len = 0
        self.span_ms = 0.0

    def make_resident(self):
        if self.copies is None:
            self.copies = [self.h_in.to(f"cuda:{g}", non_blocking=True) for g in range(self.world)]
            self.sync()
        return [self.copies[g].data_ptr() for g in self.devices]

    def drop_resident(self):
        self.copies = None
        self.torch.cuda.empty_cache()

    def sync(self):
        for g in range(self.world):
            self.torch.cuda.synchronize(g)

    def step_resident(self, ptrs):
        self.out_len = self.multi.compress_ptr(None, self.n, self.h_out.data_ptr(), self.cap, d_srcs=ptrs)
        self.span_ms += self.multi.stats.ms_span          # the job as timed ON the devices (CUDA events, max over engines)
        return self.multi.stats

    def step_host(self):
        """end to end: BZ2_bzBuffToBuffCompress (32-bit lengths) while the input is below 4 GiB, else the function it calls"""
        if self.n < 0xFFFFFFFF and self.cap <= 0xFFFFFFFF:
            dlen = C.c_uint(self.cap)
            rc = self.B.load().BZ2_bzBuffToBuffCompress(self.h_out.data_ptr(), C.byref(dlen), self.h_in.data_ptr(), self.n, self.level, 0, 0)
            assert rc == 0, rc
            self.out_len = dlen.value
            return "BZ2_bzBuffToBuffCompress, pinned host buffers, BZ2_B200_DEVICES=" + os.environ.get("BZ2_B200_DEVICES", "")
        self.out_len = self.multi.compress_ptr(self.h_in.data_ptr(), self.n, self.h_out.data_ptr(), self.cap)
        return ("bz2b200_multi_compress with host pointers (what BZ2_bzBuffToBuffCompress calls; its 32-bit lengths stop at 4 GiB), "
                "pinned host buffers")

    def timed(self, fn, steps, barrier):
        barrier()
        t0 = time.perf_counter()
        last = None
        for _ in range(steps):
            last = fn()
        self.sync()
        dt = time.perf_counter() - t0
        barrier()
        return dt, last

    def close(self):
        self.multi.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="text")
    ap.add_argument("--mb", type=int, default=1000)
    ap.add_argument("--level", type=int, default=9)
    ap.add_argument("--engines-per-gpu", type=int, default=int(os.environ.get("BENCH_ENGINES_PER_GPU", "2")))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-c4", action="store_true")
    ap.add_argument("--c4-gb", type=float, default=16.0)
    ap.add_argument("--sweep", action="store_true", help="C5: -1..-9 on --sweep-gb GB of text, outputs decoded by oracle/_ref/bzip2_ref")
    ap.add_argument("--sweep-gb", type=float, default=4.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output stream and counts as .npy files to DIR")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n = args.mb * 1_000_000
    metric = "compress MB/s at -9 (1/2/4/8 B200) vs host libbz2; byte-exact .bz2 output"
    config = {"workload": f"{args.mb} MB synthetic {args.workload} per GPU (SURVEY 8d; xorshift64* seeded), blockSize100k={args.level}; "
                          f"ONE stream of {world} x {args.mb} MB sharded by block over the GPUs",
              "l2": "input (>= 1 GB) exceeds the 126 MB L2; no flush needed",
              "level": args.level, "bytes_per_gpu": n}

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        procs = physical_cores()
        data = make_input(args.workload, n)
        vals = []
        info = None
        for it in range(args.warmup + args.steps):
            v, kind, sample, _ = cpu_reference_rate(data, args.level, procs)
            if it >= args.warmup:
                vals.append(v)
            info = (kind, sample)
        v = sum(vals) / len(vals)
        config = dict(config)
        config["workload"] = (f"{args.mb} MB synthetic {args.workload} (SURVEY 8d), blockSize100k={args.level}; the full workload cut into "
                              f"{procs} contiguous slices, one reference process per physical core (BASELINE.md 3)")
        line = {"impl": "reference", "metric": metric, "value": round(v, 2), "unit": "MB/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(n / (v * 1e6) * 1e3, 2),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": config,
                "cpu_baseline": {"value": round(v, 2), "unit": "MB/s", "cores": procs, "logical_cpus": os.cpu_count(), "kind": info[0], "sample": info[1]},
                "e2e": {"value": round(v, 2), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm (GPU)
    import torch
    import bzip2_b200 as B
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = ctl = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
        ctl = dist.new_group(backend="gloo")             # barriers of the timed regions: host side, no kernel parked on the GPUs

    def barrier():
        if dist is not None:
            dist.barrier(group=ctl)
        torch.cuda.synchronize()

    # every rank generates its own --mb MB part in parallel; rank 0 receives them over NCCL and owns the whole stream
    part = make_input(args.workload, n, rank)
    if world > 1:
        d_part = torch.from_numpy(part).to(dev)
        parts = [torch.empty_like(d_part) for _ in range(world)] if rank == 0 else None
        dist.gather(d_part, parts, dst=0)
        torch.cuda.synchronize()
        if rank != 0:
            del d_part
            torch.cuda.empty_cache()
            # idle ranks: take part in rank 0's barriers until it says stop
            flag = torch.ones(1, dtype=torch.int64)
            while True:
                dist.broadcast(flag, src=0, group=ctl)
                if int(flag.item()) == 0:
                    break
                dist.barrier(group=ctl)
            dist.destroy_process_group()
            return 0
        h_in = torch.empty(n * world, dtype=torch.uint8).pin_memory()
        for r in range(world):
            h_in[r * n:(r + 1) * n].copy_(parts[r])
        del parts, d_part
        torch.cuda.empty_cache()
    else:
        h_in = torch.from_numpy(part).pin_memory()
    total = n * world

    def job_barrier():
        """barrier + synchronize on both sides of a timed region (the idle ranks sit in the same barrier)"""
        if dist is not None:
            dist.broadcast(torch.ones(1, dtype=torch.int64), src=0, group=ctl)
            dist.barrier(group=ctl)
        for g in range(world):
            torch.cuda.synchronize(g)

    devlist = ",".join(str(g) for _ in range(args.engines_per_gpu) for g in range(world))
    if len(devlist.split(",")) > 1:
        os.environ["BZ2_B200_DEVICES"] = devlist         # device list of the libbz2 entry points
    else:
        os.environ.pop("BZ2_B200_DEVICES", None)
        os.environ["BZ2_B200_DEVICE"] = "0"

    if args.sweep:
        rc = sweep(args, torch, B, world, job_barrier, metric)
        if dist is not None:
            dist.broadcast(torch.zeros(1, dtype=torch.int64), src=0, group=ctl)
            dist.destroy_process_group()
        return rc

    job = Job(torch, B, world, args.level, args.engines_per_gpu, h_in)
    ptrs = job.make_resident()
    for _ in range(args.warmup):
        st = job.step_resident(ptrs)
    with Samplers(world) as clk:
        job.span_ms = 0.0
        dt, st = job.timed(lambda: job.step_resident(ptrs), args.steps, job_barrier)
    device_ms_per_step = job.span_ms / args.steps
    ms_per_step = dt / args.steps * 1e3
    value = total / (ms_per_step * 1e-3) / 1e6
    out_len = job.out_len
    launches = int(st.kernel_launches) * args.steps
    out_resident = job.h_out[:out_len].numpy().copy()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out_resident, st)
    job.drop_resident()

    e2e = None
    if not args.no_e2e:
        api = None
        for _ in range(max(1, args.warmup)):
            api = job.step_host()
        dt_e, api = job.timed(job.step_host, args.steps, job_barrier)
        e2e = {"value": round(total * args.steps / dt_e / 1e6, 2), "unit": "MB/s", "h2d_bytes_per_step": total,
               "d2h_bytes_per_step": int(job.out_len), "api": api}
        out_host = job.h_out[:job.out_len].numpy()
        assert job.out_len == out_len and np.array_equal(out_host, out_resident), "host and resident paths disagree"
    job.close()

    # one engine alone on GPU 0 (no second window in flight): the stage times the roofline is quoted on
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    d0 = h_in[:n].to("cuda:0")
    cap0 = (n + n // 50 + 24576 * (n // (100000 * args.level - 19) + 2) + 1024 + 255) & ~255
    d_out0 = torch.empty(cap0, dtype=torch.uint8, device="cuda:0")
    eng = B.Engine(level=args.level, device=0)
    solo_steps = max(1, min(3, args.steps))
    stage_ms = np.zeros(5)
    for it in range(2 + solo_steps):
        eng.compress_device(d0.data_ptr(), n, d_out0.data_ptr(), cap0)
        if it >= 2:
            s1 = eng.stats
            stage_ms += np.array([s1.ms_total, s1.ms_s1, s1.ms_s2, s1.ms_s3, s1.ms_s4])
    stage_ms /= solo_steps
    s1 = eng.stats
    eng.close()
    del d0, d_out0
    rho = s1.sum_nblock / max(1, s1.in_bytes)
    mu = s1.sum_nmtf / max(1, s1.sum_nblock)
    c = s1.out_bytes / max(1, s1.in_bytes)
    A = 1 + 4 * rho + 12 * rho * mu + 3 * c              # SURVEY 8(d): algorithmic bytes per input byte, whole pass
    s2_bytes = 2 * rho * n                               # BWT stage: read the block once, write the last column once
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        if args.workload == "text" and args.level == 9:
            traffic = int(tr["per_input_byte"]["S2"]["dram_bytes"] * n)
    except Exception:  # noqa: BLE001
        pass
    roof = {"bound": "hbm",
            "kernel": "S2 BWT kernel family (k_kgram*, k_refine_*, k_resolve_periodic, k_rep_*, k_bwt_out), one engine alone on GPU 0, "
                      f"{n // 1_000_000} MB of the workload per launch set of ~10 windows, timed live by CUDA events around the stage on the launching stream "
                      "(profiles/r02_launch_summary.md)",
            "algorithmic_bytes": int(s2_bytes), "algorithmic_rule": "2*rho bytes per input byte: read the block once, write the last column once (SURVEY 8d)",
            "achieved": round(s2_bytes / (stage_ms[2] * 1e-3) / 1e9, 3), "peak": peak, "unit": "GB/s",
            "frac": round(s2_bytes / (stage_ms[2] * 1e-3) / 1e9 / peak, 6), "traffic": traffic,
            "traffic_source": "ncu dram__bytes of the committed launch list (profiles/r02_traffic.json), scaled to this step; not measured in this run",
            "peak_source": peak_src,
            "whole_pass": {"A_bytes_per_input_byte": round(A, 3), "rho": round(rho, 4), "mu": round(mu, 4), "c": round(c, 4),
                           "achieved_one_engine": round(A * n / (stage_ms[0] * 1e-3) / 1e9, 3),
                           "frac_one_engine": round(A * n / (stage_ms[0] * 1e-3) / 1e9 / peak, 6),
                           "achieved_job_per_gpu": round(A * total / world / (ms_per_step * 1e-3) / 1e9, 3),
                           "frac_job_per_gpu": round(A * total / world / (ms_per_step * 1e-3) / 1e9 / peak, 6)},
            "stage_ms": {"s1_rle_crc": round(float(stage_ms[1]), 3), "s2_bwt": round(float(stage_ms[2]), 3),
                         "s3_mtf": round(float(stage_ms[3]), 3), "s4_huffman_pack": round(float(stage_ms[4]), 3),
                         "sum_events": round(float(stage_ms[0]), 3)}}

    cpu = None
    parity = None
    if not args.no_cpu:
        sample = h_in[:min(total, 200_000_000)].numpy()
        v, kind, desc, ref_out = cpu_reference_rate(sample, args.level, 1, keep_output=True)
        cpu = {"value": round(v, 2), "unit": "MB/s", "cores": 1, "kind": kind, "sample": desc}
        if ref_out is not None and kind == "reference":
            # the reference's stream of the prefix equals ours up to its last (cut-short) block
            eq = equal_prefix(out_resident, ref_out)
            slack = 1_300_000 if sample.size < total else 0
            assert eq >= ref_out.size - slack, f"timed output differs from the reference's stream at byte {eq}"
            parity = {"parity_checked_bytes": eq, "of_reference_stream_bytes": int(ref_out.size),
                      "how": f"leading bytes of the timed {total} B job's output equal to the reference's (oracle/_ref) stream of the first "
                             f"{sample.size} B; the reference's last block is cut short by the prefix, so the streams part inside it"}

    c4 = None
    if not args.no_c4 and args.workload == "text" and args.level == 9:
        c4 = c4_leg(args, torch, B, world, job_barrier)

    line = {"metric": metric, "value": round(value, 2), "unit": "MB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config, "clocks": clk.summary(),
            "e2e": e2e, "gpu_launches": launches, "roofline": roof, "cpu_baseline": cpu,
            "out_bytes": int(out_len), "blocks": int(st.n_blocks), "bwt_rounds": int(st.bwt_rounds),
            "engines": {"per_gpu": args.engines_per_gpu, "devices": devlist,
                        "driver": "one process (rank 0) drives every GPU through bz2b200_multi_* / BZ2_bzBuffToBuffCompress; other ranks idle"},
            "device_ms_per_step": round(device_ms_per_step, 3),
            "timing": "ms_per_step / value: host clock around the K synchronous C calls, bracketed by barrier + cudaDeviceSynchronize of every GPU; "
                      "device_ms_per_step: the same K jobs timed on the devices -- CUDA events on every engine's own stream at the start of a job and after "
                      "its last copy, max over the engines of all GPUs (events recorded on torch's stream would not see the engines' streams); "
                      "the host clock is the larger of the two and is the one reported"}
    if parity:
        line.update(parity)
    if c4:
        line["c4"] = c4
    print(json.dumps(line))
    if dist is not None:
        dist.broadcast(torch.zeros(1, dtype=torch.int64), src=0, group=ctl)
        dist.destroy_process_group()
    return 0


def c4_leg(args, torch, B, world, job_barrier):
    """SURVEY 8(d) C4: 16 GB of 64 MiB segments text / real binary / random, -9, ONE stream strong-scaled over the GPUs."""
    import support as S
    nbytes = int(args.c4_gb * 1e9)
    t0 = time.perf_counter()
    h_in = torch.from_numpy(S.gen_c4(nbytes, seg=64 << 20)).pin_memory()
    gen_s = time.perf_counter() - t0
    job = Job(torch, B, world, 9, args.engines_per_gpu, h_in)
    steps = max(1, min(2, args.steps))
    ptrs = job.make_resident()
    job.step_resident(ptrs)
    dt, st = job.timed(lambda: job.step_resident(ptrs), steps, job_barrier)
    out_len = job.out_len
    sha = None
    job.drop_resident()
    job.step_host()
    dt_e, api = job.timed(job.step_host, steps, job_barrier)
    assert job.out_len == out_len
    import hashlib
    sha = hashlib.sha256(job.h_out[:out_len].numpy()).hexdigest()
    job.close()
    return {"workload": f"{args.c4_gb:g} GB mixed (64 MiB segments cycling text / sample1.ref||sample2.ref tiled / random), -9, ONE stream, "
                        f"strong-scaled: {args.c4_gb / world:g} GB per GPU", "scaling": "strong",
            "value": round(nbytes * steps / dt / 1e6, 2), "unit": "MB/s", "ms_per_step": round(dt / steps * 1e3, 2), "steps": steps, "warmup": 1,
            "e2e": {"value": round(nbytes * steps / dt_e / 1e6, 2), "unit": "MB/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": int(out_len), "api": api},
            "out_bytes": int(out_len), "sha256": sha, "blocks": int(st.n_blocks), "bwt_rounds": int(st.bwt_rounds), "generate_s": round(gen_s, 1)}


def sweep(args, torch, B, world, job_barrier, metric):
    """SURVEY 8(d) C5: blockSize100k sweep -1..-9 on 4 GB of text over the N GPUs; every output is piped through the
    reference decoder (oracle/_ref/bzip2_ref -dc) and must reproduce the input (sha256)."""
    import hashlib
    import support as S
    nbytes = int(args.sweep_gb * 1e9)
    data = S.gen_text(nbytes)
    want = hashlib.sha256(data).hexdigest()
    h_in = torch.from_numpy(data).pin_memory()
    ref_cli = os.path.join(ROOT, "oracle", "_ref", "bzip2_ref")
    rows, procs = [], []
    for level in range(1, 10):
        job = Job(torch, B, world, level, args.engines_per_gpu, h_in)
        job.step_host()
        dt, api = job.timed(job.step_host, 1, job_barrier)
        out = job.h_out[:job.out_len].numpy().tobytes()
        job.close()
        row = {"level": level, "e2e_MBps": round(nbytes / dt / 1e6, 1), "out_bytes": len(out), "sha256_out": hashlib.sha256(out).hexdigest()}
        if os.path.exists(ref_cli):
            path = f"/dev/shm/bz2b200_sweep_{os.getpid()}_{level}.bz2"
            with open(path, "wb") as f:
                f.write(out)
            p = subprocess.Popen(f"{ref_cli} -dc {path} | sha256sum", shell=True, stdout=subprocess.PIPE, text=True)
            procs.append((row, p, path))
        rows.append(row)
    for row, p, path in procs:
        got = p.communicate()[0].split()[0]
        row["decoded_by_reference_bzip2_equals_input"] = (got == want)
        os.unlink(path)
    ok = all(r.get("decoded_by_reference_bzip2_equals_input", False) for r in rows) if procs else None
    print(json.dumps({"metric": metric, "mode": "C5 level sweep", "n_gpus": world, "input_bytes": nbytes, "unit": "MB/s",
                      "data": "synthetic", "roundtrip_all_levels_ok": ok, "levels": rows,
                      "api": "BZ2_bzBuffToBuffCompress / bz2b200_multi_compress, pinned host buffers, one step per level after one warm-up"}))
    return 0 if ok in (True, None) else 1


if __name__ == "__main__":
    sys.exit(main())
