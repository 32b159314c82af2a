#!/usr/bin/env python
"""bench_batch.py -- many small inputs: one bz2b200_compress_batch_device call against a loop of compress_device calls.

  python tools/bench_batch.py [--mb 256] [--sizes 4096,65536,900000,4194304] [--workloads text,random] [--level 9]
                              [--reps 3] [--loop-items 1000] [--max-items 4096]

For every (item size, workload) configuration about --mb MB of input is resident in HBM as items of that size.  Both
arms run on the same engine from bz2b200_engine_create_batch, are warmed up, and alternate --reps times:
  (a) loop   one bz2b200_compress_device call per item, each into its own region of a device buffer;
  (b) batch  one bz2b200_compress_batch_device call over all items, streams back to back.
A loop over tens of thousands of 4 KiB items would take minutes, so arm (a) covers at most --loop-items items and its
rate is per item timed; both arms report MB/s and items/s of the items they compressed.  The loop's streams are
compared byte for byte with the batch's streams of the same items.  One JSON line per configuration, with the card's
name and power limit read in the same process.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:            # the name is still reported; the limit is then unknown
        pl = "unknown"
    return name, pl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--mb", type=int, default=256)
    ap.add_argument("--sizes", default="4096,65536,900000,4194304")
    ap.add_argument("--workloads", default="text,random")
    ap.add_argument("--level", type=int, default=9)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--loop-items", type=int, default=1000)
    ap.add_argument("--max-items", type=int, default=4096)
    a = ap.parse_args()

    import torch
    import support as S
    import bzip2_b200 as B
    if not torch.cuda.is_available():
        raise SystemExit("bench_batch.py needs a CUDA device")
    name, power = card()
    e = B.Engine(level=a.level, max_items=a.max_items)
    lib = e.lib
    gens = {"text": S.gen_text, "random": S.gen_random}
    for wl in a.workloads.split(","):
        for size in map(int, a.sizes.split(",")):
            n_items = max(1, (a.mb << 20) // size)
            data = gens[wl](n_items * size, seed=S.TEXT_SEED if wl == "text" else 2)
            offs = np.arange(n_items + 1, dtype=np.uint64) * np.uint64(size)
            d_src = torch.from_numpy(data).cuda()
            cap = n_items * B.compress_bound(a.level, size)
            d_dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
            # loop arm: each call gets a 4-byte aligned region that meets compress_device's own bound
            n_loop = min(n_items, a.loop_items)
            need = size + size // 64 + (size // (100000 * a.level - 19) + 2) * 24576 + 64
            need = (need + 255) & ~255
            d_loop = torch.empty(n_loop * need, dtype=torch.uint8, device="cuda")
            import ctypes as C
            lens = [0] * n_loop

            def run_loop():
                launches = 0
                st = B.Stats()
                out_len = C.c_size_t(0)
                for k in range(n_loop):
                    rc = lib.bz2b200_compress_device(e.h, d_src.data_ptr() + k * size, size, d_loop.data_ptr() + k * need,
                                                     need, C.byref(out_len), 0, C.byref(st))
                    if rc:
                        raise SystemExit(f"compress_device rc={rc}: {lib.bz2b200_last_error().decode()}")
                    lens[k] = out_len.value
                    launches += st.kernel_launches
                torch.cuda.synchronize()
                return launches

            def run_batch():
                out = e.compress_batch_device(d_src.data_ptr(), offs, d_dst.data_ptr(), cap)
                torch.cuda.synchronize()
                return out, e.stats.kernel_launches, e.stats.n_windows

            run_loop(); run_batch()                                    # warm-up of both arms
            t_loop, t_batch = [], []
            for _ in range(a.reps):
                t0 = time.perf_counter(); loop_launches = run_loop(); t_loop.append(time.perf_counter() - t0)
                t0 = time.perf_counter(); out_offs, b_launches, windows = run_batch(); t_batch.append(time.perf_counter() - t0)
            # identical bytes: every looped item's stream equals the batch stream of that item
            hb = d_dst[: int(out_offs[n_loop])].cpu().numpy()
            hl = d_loop.cpu().numpy()
            for k in range(n_loop):
                s = hb[int(out_offs[k]):int(out_offs[k + 1])]
                assert lens[k] == s.size and np.array_equal(hl[k * need:k * need + lens[k]], s), f"item {k} differs"
            ml, mb_ = statistics.median(t_loop), statistics.median(t_batch)
            print(json.dumps({
                "bench": "batch", "workload": wl, "level": a.level, "item_bytes": size, "items": n_items,
                "loop_items": n_loop, "batch_MBps": round(n_items * size / mb_ / 1e6, 1),
                "loop_MBps": round(n_loop * size / ml / 1e6, 1),
                "batch_items_per_s": round(n_items / mb_, 1), "loop_items_per_s": round(n_loop / ml, 1),
                "speedup": round((n_items / mb_) / (n_loop / ml), 3),
                "batch_s": [round(x, 4) for x in t_batch], "loop_s": [round(x, 4) for x in t_loop],
                "launches_per_item_batch": round(b_launches / n_items, 2),
                "launches_per_item_loop": round(loop_launches / n_loop, 2),
                "windows": windows, "ratio": round(int(out_offs[-1]) / (n_items * size), 4),
                "identical": True, "gpu": name, "power_limit": power,
            }), flush=True)
            del d_src, d_dst, d_loop
            torch.cuda.empty_cache()
    e.close()


if __name__ == "__main__":
    main()
