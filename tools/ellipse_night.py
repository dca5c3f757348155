"""`--center ellipse` on the bench night: 100 tables x 1e5 rows (30 % FAINT), every channel
distorted by imperfect quadrature detectors (synthetic.make_table(quadrature=True)), resident
in HBM, one gppd_process_tables_f32_dev batch per step.  Measures, in one process:

  * the night's time, ellipse mode and `--center empirical` (the circle it generalises),
    steps alternated, CUDA events on the launching stream;
  * the per-pass split of each mode (gppd_pass_times, steps of their own);
  * k_ellipse_apply and k_repack_arrays: kernel time (torch.profiler, a run of its own), the
    bytes each must move (apply: TIME + VOLT in, t + 40 complex128 out = 324 + 648 B per row;
    repack: 40 complex128 in, 80 float32 out = 640 + 320 B per row) and their rate as a
    fraction of the HBM rate measured here by a device-to-device copy;
  * the card's name and power limit.

    python tools/ellipse_night.py [out.json] [tables] [rows] [steps]

Ten distinct tables (7 bright, 3 FAINT) are generated and uploaded 10 times each (generating
100 takes a minute of NumPy time and changes nothing on the device)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import gppd_b200 as gp                      # noqa: E402
import oracle                               # noqa: E402
from conftest import make_case              # noqa: E402
from gppd_b200 import _lib                  # noqa: E402

out_path = sys.argv[1] if len(sys.argv) > 1 else None
F = int(sys.argv[2]) if len(sys.argv) > 2 else 100
N = int(sys.argv[3]) if len(sys.argv) > 3 else 100_000
STEPS = int(sys.argv[4]) if len(sys.argv) > 4 else 5

L, h = _lib.lib(), gp.default_handle()
dev = torch.device("cuda", h.device)
distinct = []
for k in range(10):
    faint = k in (3, 6, 9)
    tab = make_case(gp.synthetic, N, k=k, faint=faint, ora=oracle)
    tab["volt"] = gp.synthetic.make_table(N, k=k, faint=faint, state=tab["state"], quadrature=True)["volt"]
    distinct.append(tab)
tabs = [distinct[i % 10] for i in range(F)]
fss = [None if tb["faintstates"] is None else
       gp.FaintStates(tb["faintstates"].timer1, tb["faintstates"].timer2, 1.0, 2.0) for tb in tabs]
time_us = [torch.from_numpy(tb["time_us"]).to(dev) for tb in tabs]
volt = [torch.from_numpy(tb["volt"]).to(dev) for tb in tabs]
vout = [torch.empty((N, 80), dtype=torch.float32, device=dev) for _ in tabs]
params = [torch.empty((32, 6), dtype=torch.float64, device=dev) for _ in tabs]
chi2 = [torch.empty(32, dtype=torch.float64, device=dev) for _ in tabs]
vp = lambda ts: (C.c_void_p * F)(*[t.data_ptr() for t in ts])
i64 = lambda v: (C.c_int64 * F)(*v)
dpp = lambda arrs: (_lib._dp * F)(*[C.cast(None, _lib._dp) if a is None else a.ctypes.data_as(_lib._dp) for a in arrs])
args = dict(n=i64([N] * F), time=vp(time_us), mjd=(C.c_double * F)(*[tb["mjd"] for tb in tabs]), volt=vp(volt),
            t1=dpp([f.timer1 if f else None for f in fss]), n1=i64([f.timer1.size if f else 0 for f in fss]),
            t2=dpp([f.timer2 if f else None for f in fss]), n2=i64([f.timer2.size if f else 0 for f in fss]),
            out=vp(vout), par=vp(params), chi=vp(chi2))
stream = torch.cuda.Stream(device=dev)
opts = {"ellipse": gp.api._options(ellipse=True), "empirical": gp.api._options(empirical=True)}


def step(mode):
    a = args
    _lib.check(L.gppd_process_tables_f32_dev(
        h.raw, 0, C.c_void_p(stream.cuda_stream), F, a["n"], None, a["time"], a["mjd"], a["volt"], None,
        a["t1"], a["n1"], a["t2"], a["n2"], C.byref(opts[mode]), a["out"], a["par"], a["chi"], None, None))


def timed(mode):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    step(mode)
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1)


for mode in opts:                     # warm-up: modules, scratch, tensor maps
    for _ in range(2):
        timed(mode)
ms = {m: [] for m in opts}
for _ in range(STEPS):                # alternated
    for mode in opts:
        ms[mode].append(timed(mode))

passes = {}
h.enable_timing(True)
for mode in opts:
    h.pass_times(reset=True)
    for _ in range(STEPS):
        timed(mode)
    passes[mode] = {k: round(v[0] / STEPS, 4) for k, v in h.pass_times(reset=True).items()}
h.enable_timing(False)

# kernel times of the two streaming transposes (a profiled run of its own)
from torch.profiler import ProfilerActivity, profile   # noqa: E402
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(STEPS):
        timed("ellipse")
kern = {}
for ev in prof.key_averages():
    for name in ("k_ellipse_apply", "k_repack_arrays", "k_circle_seg", "k_ellipse_solve"):
        if name in ev.key:
            kern.setdefault(name, [0.0, 0])
            kern[name][0] += ev.device_time_total / 1e3      # us -> ms
            kern[name][1] += ev.count

# HBM rate: a 4 GiB device-to-device copy
a = torch.empty(4 << 30, dtype=torch.uint8, device=dev)
b = torch.empty_like(a)
b.copy_(a)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10):
    b.copy_(a)
e1.record()
e1.synchronize()
hbm = 2 * 10 * a.numel() / (e0.elapsed_time(e1) * 1e-3)
del a, b

rows = F * N
bytes_per_row = {"k_ellipse_apply": 324 + 648, "k_repack_arrays": 640 + 320}
transposes = {}
for name, bpr in bytes_per_row.items():
    if name in kern:
        t = kern[name][0] / kern[name][1]                       # ms per launch (one launch per step)
        rate = rows * bpr / (t * 1e-3)
        transposes[name] = dict(ms=round(t, 4), bytes_per_row=bpr, bytes_per_s=rate,
                                fraction_of_measured_hbm=round(rate / hbm, 3))
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                      "-i", str(h.device)], capture_output=True, text=True).stdout.strip()
res = dict(workload=f"{F} tables x {N} rows (30 % FAINT, quadrature=True), resident, gppd_process_tables_f32_dev, "
                    "whole-table fits",
           gpu=smi, steps=STEPS,
           night_ms={m: dict(median=float(np.median(v)), min=float(np.min(v)), all=[round(x, 4) for x in v])
                     for m, v in ms.items()},
           pass_ms_per_step=passes,
           kernels_ms_per_step={k: round(v[0] / STEPS, 4) for k, v in kern.items()},
           measured_hbm_bytes_per_s=hbm, streaming_transposes=transposes,
           note="pass times are summed per pass (ellipse: moments, solve and apply under basis, the repack under "
                "demod); kernel times from torch.profiler in a separate profiled run; HBM rate = 2 x bytes of a 4 GiB "
                "device-to-device copy over its time")
line = json.dumps(res)
print(line)
if out_path:
    with open(out_path, "w") as fh:
        fh.write(json.dumps(res, indent=1) + "\n")
