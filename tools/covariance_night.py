"""GPPD_COVARIANCE on the bench night: 100 tables x 1e5 rows (30 % FAINT), given centres,
resident in HBM, one gppd_process_tables_f32_dev batch per step.  Measures, in one process:

  * the night's time without and with the flag, each with split chains on and off, steps
    alternated, CUDA events on the launching stream;
  * the covariance pass on its own: k_cov_seg and k_cov_final kernel time (torch.profiler, a
    run of its own), the bytes k_cov_seg must move per row (VOLT 320 + basis 16 + state 1 =
    337 B) and its FP64 rate, counted as 80 FP64 operations per diode-sample (the model, its
    sincos and the 21 entries of H; an FMA counts as one operation);
  * the card's name and power limit.

    python tools/covariance_night.py [out.json] [tables] [rows] [steps]

Ten distinct tables (7 bright, 3 FAINT) are generated and uploaded 10 times each."""
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
distinct = [make_case(gp.synthetic, N, k=k, faint=k in (3, 6, 9), ora=oracle) for k in range(10)]
tabs = [distinct[i % 10] for i in range(F)]
fss = [None if tb["faintstates"] is None else
       gp.FaintStates(tb["faintstates"].timer1, tb["faintstates"].timer2, 1.0, 2.0) for tb in tabs]
time_us = [torch.from_numpy(tb["time_us"]).to(dev) for tb in tabs]
volt = [torch.from_numpy(tb["volt"]).to(dev) for tb in tabs]
vout = [torch.empty((N, 80), dtype=torch.float32, device=dev) for _ in tabs]
params = [torch.empty((32, 6), dtype=torch.float64, device=dev) for _ in tabs]
chi2 = [torch.empty(32, dtype=torch.float64, device=dev) for _ in tabs]
offsets = torch.from_numpy(gp.synthetic.stefan_centres().view(np.float64).copy()).to(dev)
vp = lambda ts: (C.c_void_p * F)(*[t.data_ptr() for t in ts])
i64 = lambda v: (C.c_int64 * F)(*v)
dpp = lambda arrs: (_lib._dp * F)(*[C.cast(None, _lib._dp) if a is None else a.ctypes.data_as(_lib._dp) for a in arrs])
args = dict(n=i64([N] * F), time=vp(time_us), mjd=(C.c_double * F)(*[tb["mjd"] for tb in tabs]), volt=vp(volt),
            t1=dpp([f.timer1 if f else None for f in fss]), n1=i64([f.timer1.size if f else 0 for f in fss]),
            t2=dpp([f.timer2 if f else None for f in fss]), n2=i64([f.timer2.size if f else 0 for f in fss]),
            out=vp(vout), par=vp(params), chi=vp(chi2))
stream = torch.cuda.Stream(device=dev)
opts = {"plain": gp.api._options(), "covariance": gp.api._options(covariance=True)}
modes = [(m, split) for m in opts for split in (True, False)]


def step(mode):
    a = args
    _lib.check(L.gppd_process_tables_f32_dev(
        h.raw, 0, C.c_void_p(stream.cuda_stream), F, a["n"], None, a["time"], a["mjd"], a["volt"],
        C.c_void_p(offsets.data_ptr()), a["t1"], a["n1"], a["t2"], a["n2"], C.byref(opts[mode]), a["out"], a["par"],
        a["chi"], None, None))


def timed(mode, split):
    h.set_split_chains(split)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    step(mode)
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1)


for m, split in modes:                # warm-up: modules, scratch, tensor maps
    for _ in range(2):
        timed(m, split)
ms = {f"{m} split={int(s)}": [] for m, s in modes}
launches = {}
for _ in range(STEPS):                # alternated
    for m, split in modes:
        l0 = h.launches
        ms[f"{m} split={int(split)}"].append(timed(m, split))
        launches[f"{m} split={int(split)}"] = h.launches - l0

from torch.profiler import ProfilerActivity, profile   # noqa: E402
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(STEPS):
        timed("covariance", False)
kern = {}
for ev in prof.key_averages():
    for name in ("k_cov_seg", "k_cov_final"):
        if name in ev.key:
            kern.setdefault(name, [0.0, 0])
            kern[name][0] += ev.device_time_total / 1e3      # us -> ms
            kern[name][1] += ev.count
h.set_split_chains(True)

rows = F * N
seg = {}
if "k_cov_seg" in kern:
    t = kern["k_cov_seg"][0] / kern["k_cov_seg"][1]
    seg = dict(ms=round(t, 4), bytes_per_row=337, bytes_per_s=rows * 337 / (t * 1e-3),
               fp64_ops_per_diode_sample=80, fp64_ops_per_s=rows * 32 * 80 / (t * 1e-3))
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                      "-i", str(h.device)], capture_output=True, text=True).stdout.strip()
res = dict(workload=f"{F} tables x {N} rows (30 % FAINT), given centres, resident, gppd_process_tables_f32_dev, "
                    "whole-table fits",
           gpu=smi, steps=STEPS,
           night_ms={k: dict(median=float(np.median(v)), min=float(np.min(v)), all=[round(x, 4) for x in v])
                     for k, v in ms.items()},
           launches_per_step=launches,
           kernels_ms_per_step={k: round(v[0] / STEPS, 4) for k, v in kern.items()},
           k_cov_seg=seg,
           note="night times with CUDA events around one batch, the four variants alternated; kernel times from "
                "torch.profiler in a separate profiled run (flag on, one launch sequence); bytes and FP64 operations "
                "counted from shapes as stated in the tool's docstring")
line = json.dumps(res)
print(line)
if out_path:
    with open(out_path, "w") as fh:
        fh.write(json.dumps(res, indent=1) + "\n")
