#!/usr/bin/env python
"""Per-tile timeline of one radix pass (diagnostic build: `make -C megahit_b200/csrc timeline`).

    MHB_LIB=megahit_b200/libmhb_timeline.so python scripts/sort_timeline.py [n_records] [words] [rows.npy]

Prints, for one pass over n random records: duration of every phase of a tile (us: median / p90 / max), the
look-back depth and re-poll statistics, the stagger between consecutive tile starts, and how many tiles were in each
phase at the moment a tile started its look-back.  With rows.npy, also saves a sample of the per-tile rows there
(rows x 16 uint64)."""
import ctypes as C
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("MHB_LIB", os.path.join(ROOT, "megahit_b200", "libmhb_timeline.so"))
from megahit_b200 import dev, lib  # noqa: E402

n = int(float(sys.argv[1])) if len(sys.argv) > 1 else 1_230_000_000
words = int(sys.argv[2]) if len(sys.argv) > 2 else 2
L = lib.load()
assert hasattr(L, "mhb_debug_set_sort_timeline"), "not the timeline build (MHB_LIB)"
g = torch.Generator(device="cuda")
g.manual_seed(3)
a = torch.randint(-2**31, 2**31 - 1, (n * words + 4,), generator=g, device="cuda", dtype=torch.int32)
b = torch.empty_like(a)
rows = n // 2048 + 2
tl = torch.zeros(rows * 16, dtype=torch.int64, device="cuda")
L.mhb_debug_set_sort_timeline.argtypes = [C.c_void_p, C.c_ulonglong]
sort_byte = 4 * words - 3
for rep in range(2):
    tl.zero_()
    lib._check(L.mhb_debug_set_sort_timeline(C.c_void_p(tl.data_ptr()), rows))
    dev.sort_records(a, b, n, words, [sort_byte])
    torch.cuda.synchronize()
ms = lib.sort_pass_ms(0)[0]
t = tl.cpu().numpy().view(np.uint64).reshape(rows, 16)
t = t[t[:, 2] > 0]
t = t[np.argsort(t[:, 0])]
print(f"words {words}: {len(t)} tiles, pass {ms[0]:.3f} ms "
      f"({2 * n * words * 4 / (ms[0] * 1e-3) / 1e9:.0f} GB/s)")
mhz = torch.cuda.get_device_properties(0).clock_rate / 1e3 if hasattr(torch.cuda.get_device_properties(0), "clock_rate") else 1965.0
names = ["loads arrived", "early publish", "rank (B1)", "warp bases (B3)", "reorder", "look-back", "B4 passed", "scatter (B5)"]
v = t[:, 3:11].astype(np.float64) / mhz  # us since the tile's start
prev = np.zeros(len(t))
print("phase                 median    p90     max   (us, duration of the phase for thread 0 of the CTA)")
for i, nm in enumerate(names):
    d = v[:, i] - prev
    print(f"  {nm:18s} {np.median(d):7.2f} {np.percentile(d, 90):7.2f} {d.max():7.2f}")
    prev = v[:, i]
print(f"  whole tile         {np.median(v[:, 7]):7.2f} {np.percentile(v[:, 7], 90):7.2f} {v[:, 7].max():7.2f}")
dm, ds, sm, ss = (t[:, 11 + i].astype(np.float64) for i in range(4))
print(f"look-back descriptors examined per digit thread: mean {np.mean(ds) / 256:.2f}, max over threads: median "
      f"{np.median(dm):.0f} p90 {np.percentile(dm, 90):.0f} max {dm.max():.0f}")
print(f"re-polls of unpublished descriptors: mean per thread {np.mean(ss) / 256:.2f}, max over threads: median "
      f"{np.median(sm):.0f} p90 {np.percentile(sm, 90):.0f} max {sm.max():.0f}")
start = t[:, 2].astype(np.float64)  # globaltimer ns
gap = np.diff(start)
print(f"stagger between consecutive tile starts: median {np.median(gap):.0f} ns, mean {gap.mean():.0f} ns, "
      f"p10 {np.percentile(gap, 10):.0f} p90 {np.percentile(gap, 90):.0f}")
# how far back is the nearest tile that has finished its look-back when a tile starts its own?
lb_start = start + v[:, 4] * 1e3
lb_end = start + v[:, 5] * 1e3
idx = np.arange(len(t))
sample = idx[:: max(1, len(t) // 2000)][5:]
depth_needed = []
for i in sample:
    j = i - 1
    while j >= 0 and lb_end[j] > lb_start[i]:
        j -= 1
    depth_needed.append(i - j)
print(f"distance to the nearest predecessor whose look-back had finished when a tile began its own: median "
      f"{np.median(depth_needed):.0f}, p90 {np.percentile(depth_needed, 90):.0f}")
if len(sys.argv) > 3:
    np.save(sys.argv[3], t[:: max(1, len(t) // 20000)])
