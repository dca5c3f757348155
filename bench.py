#!/usr/bin/env python
"""bench.py -- diode-samples demodulated per second (BASELINE.json metric).

Workload (BASELINE.json configs[2]): a synthetic GRAVITY+ night of 100 METROLOGY
tables of 1e5 rows each (70 bright / 30 FAINT, whole-file fits, `--center stefan`)
per GPU; one *step* = one pass of the hot path over the whole night.  Weak
scaling: every rank demodulates its own night (files are independent, no
collective on the data path; SURVEY.md section 8e).

  value : whole-job diode-samples/s with all inputs resident in HBM
          (C ABI gppd_process_table_f32_dev on the bench's CUDA streams, timed
          with CUDA events on those streams, max over ranks)
  e2e   : same metric through gppd_submit_table_f32 / gppd_wait with HOST
          (pinned) buffers: H2D of TIME+VOLT and D2H of VOLT+params inside the
          timed region
  roofline     : the dominant pass (by CUDA-event time inside the timed region)
                 against the measured HBM copy bandwidth (MEASURED_PEAKS.json)
  cpu_baseline : the CPU oracle (restated reference algorithm, 8 threads like the
                 reference's Threads.@threads over the 8 diode groups) on a
                 bounded sample of the same night, on this box's host cores

`--impl reference` times that CPU restatement alone (the reference is Julia and
cannot run in this image; see DESIGN.md).

Other BASELINE.json configurations (not the headline; same JSON contract):
  --config stress  configs[3]: one exposure of 1e8 rows x 40 complex128 channels generated
                   on the device at the demodulateall boundary (a real table cannot hold it:
                   TIME is int32 microseconds), (i) 100 s windows, time blocks -> ranks,
                   (ii) ONE global fit per diode, the 8 (telescope, side) groups -> ranks
                   (gppd_options.group_mask); strong scaling, no data-path collective.
  --config sweep   configs[4]: F = 1e3 ... 1e7 (1e8 in chunks) independent fits of 512 rows,
                   bright / centres given and FAINT / centres fitted; fits/s against the HBM
                   and FP64 rooflines.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark writes nothing into the tree it runs from

ALG_BYTES_PER_ROW = 644.0          # TIME 4 B + VOLT 320 B in, VOLT 320 B out (SURVEY.md 8d)
DIODES = 32
METRIC = "diode-samples demodulated/sec"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gppd", choices=["gppd", "reference"])
    ap.add_argument("--files", type=int, default=100)
    ap.add_argument("--rows", type=int, default=100_000)
    ap.add_argument("--streams", type=int, default=5)
    ap.add_argument("--cpu-files", type=int, default=12, help="files in the CPU-baseline sample")
    ap.add_argument("--window-rows", type=int, default=0,
                    help="fit windows of this many rows instead of whole tables (reference --window); "
                         "an exploration switch, the headline workload is whole-file")
    ap.add_argument("--chains", type=int, default=1,
                    help="exploration: split the resident night into this many concurrent launch sequences")
    ap.add_argument("--config", default="night", choices=["night", "stress", "sweep"])
    ap.add_argument("--stress-rows", type=int, default=100_000_000)
    ap.add_argument("--sweep-max", type=float, default=1e7, help="largest F of the sweep (1e8: in chunks of 1e6)")
    ap.add_argument("--fp32", action="store_true",
                    help="night only: the OPTIONAL reduced-precision harmonic sums (GPPD_FP32); a separate "
                         "measurement, never the headline (which is FP64)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="night only: after the timed steps, write what the last one returned (rank 0's "
                         "tables) as .npy files in DIR, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.impl != "gppd" or args.config != "night"):
        ap.error("--dump-outputs writes the outputs of the night (--impl gppd --config night)")
    return args


# --------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons DURING the timed regions, polled through NVML
    every ~2 ms (nvidia-smi's loop mode is too coarse for a region of tens of ms)."""

    def __init__(self, index):
        self.index, self.rows, self.th, self.stop_flag = index, [], None, False
        self.nv = None

    def start(self):
        if self.index is None:       # ranks other than 0 do not poll (the line reports rank 0's clocks;
            return                   # eight processes polling NVML every 2 ms contend in the driver)
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                ut = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                self.rows.append((sm, rs, ut))
            except Exception:
                pass
            time.sleep(0.002)

    def stop(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"], "samples": 0}
        self.stop_flag = True
        self.th.join(timeout=2)
        nv = self.nv
        try:
            mx = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception:
            mx = None
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        reasons = sorted(k for k, bit in names.items() if any(r[1] & bit for r in self.rows))
        sm = [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx,
                "reasons": reasons, "samples": len(sm),
                "how": "NVML polled every ~2 ms during the resident and end-to-end timed regions"}


def pin_to_gpu_numa_node(index):
    """Run this rank on the CPUs next to its GPU, so that the pinned staging buffers
    of the end-to-end path are allocated on the GPU's own NUMA node."""
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(index))
        return True
    except Exception:
        return False


class quiet_stdout:
    """NCCL prints its version banner on stdout; keep stdout to the one JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)


# --------------------------------------------------------------------------
def night_config(F, N):
    """`config` of the night workload: the same object in the GPU arm and in the reference arm."""
    return {"workload": "night of %d METROLOGY tables x %d rows per GPU (70%% bright / 30%% FAINT), "
                        "whole-file fits, --center stefan (BASELINE.json configs[2])" % (F, N),
            "tables_per_gpu": F, "rows_per_table": N, "diodes": DIODES,
            "cache": "inputs (%.1f GB per step) larger than L2" % (F * N * 324 / 1e9),
            "sharding": "files -> ranks, no data-path collective"}


def night_plan(nfiles):
    """70 % bright, 30 % FAINT, interleaved deterministically."""
    return [(k % 10) in (3, 6, 9) for k in range(nfiles)]


def generate_night(torch, gp, dev, nfiles, nrows, rank, plan=None, faint_repeat=60):
    """Synthetic night on the GPU (same model as gppd_b200.synthetic.make_table):
    returns time_us [F, N] int32, volt [F, N, 80] float32, mjd list, FaintStates list.
    plan: which tables are FAINT (default: night_plan)."""
    centres = torch.tensor(gp.synthetic.stefan_centres().view(np.float64).reshape(40, 2),
                           device=dev)
    time_us = torch.empty((nfiles, nrows), dtype=torch.int32, device=dev)
    volt = torch.empty((nfiles, nrows, 80), dtype=torch.float32, device=dev)
    faint = night_plan(nfiles) if plan is None else list(plan)
    mjds, fss = [], []
    base = (2000 * torch.arange(nrows, device=dev, dtype=torch.int64))
    for k in range(nfiles):
        kk = rank * nfiles + k
        mjd = 59949.0 + kk / 100.0
        g = torch.Generator(device=dev)
        g.manual_seed(20230105 + kk)
        jit = torch.randint(-1, 2, (nrows,), generator=g, device=dev)
        jit[0] = 0
        tu = (base + jit).to(torch.int32)
        time_us[k] = tu
        t = tu.to(torch.float64) * 1e-6 + 86400.0 * mjd
        pscale = torch.ones(nrows, dtype=torch.float64, device=dev)
        fs = None
        if faint[k]:
            hdr = gp.synthetic.faint_header(mjd, repeat=faint_repeat)
            fs = gp.buildfaintparameters(hdr)
            st = torch.from_numpy(gp.buildstates(fs, t.cpu().numpy())).to(dev)
            pscale = torch.where(st == 3, 3.0, torch.where(st == 1, 0.2, 1.0)).to(torch.float64)
        wt = 6.283185 * t
        for grp in range(8):
            # the random walk is summed on the host: a floating-point cumsum on the GPU is not
            # bitwise reproducible, and every run must see the same night
            walk = 0.02 * torch.randn(nrows, generator=g, device=dev, dtype=torch.float64)
            phi_fc = torch.cumsum(walk.cpu(), 0).to(dev)
            phi_fc = phi_fc + float(torch.rand(1, generator=g, device=dev)) * 6.28 - 3.14
            efc = torch.polar(torch.ones_like(phi_fc), phi_fc)
            fcch = 32 + grp
            fc = torch.complex(centres[fcch, 0], centres[fcch, 1]) + 0.3 * efc
            fc = fc + 0.002 * torch.complex(torch.randn(nrows, generator=g, device=dev, dtype=torch.float64),
                                            torch.randn(nrows, generator=g, device=dev, dtype=torch.float64))
            volt[k, :, 2 * fcch] = fc.real.float()
            volt[k, :, 2 * fcch + 1] = fc.imag.float()
            par = torch.rand(16, generator=g, device=dev, dtype=torch.float64).cpu().numpy()
            for dio in range(4):
                ch = 4 * grp + dio
                amp = 0.05 + 0.45 * par[4 * dio]
                arg_a = -np.pi + 2 * np.pi * par[4 * dio + 1]
                b = 0.3 + 2.2 * par[4 * dio + 2]
                phi = -np.pi + 2 * np.pi * par[4 * dio + 3]
                a = amp * np.exp(1j * arg_a)
                mod = torch.polar(torch.ones_like(wt), b * torch.sin(wt + phi))
                noise = 0.02 * amp * torch.complex(
                    torch.randn(nrows, generator=g, device=dev, dtype=torch.float64),
                    torch.randn(nrows, generator=g, device=dev, dtype=torch.float64))
                d = torch.complex(centres[ch, 0], centres[ch, 1]) + complex(a) * pscale * efc * mod + noise
                volt[k, :, 2 * ch] = d.real.float()
                volt[k, :, 2 * ch + 1] = d.imag.float()
        mjds.append(mjd)
        fss.append(fs)
    return time_us, volt, mjds, fss


def cpu_reference_files(oracle, files, cores):
    """The restated reference algorithm (oracle) on host copies of `files`
    = [(time_us, volt, mjd, FaintStates|None)].  Returns seconds."""
    off = None
    import gppd_b200 as gp
    off = gp.synthetic.stefan_centres()
    t0 = time.perf_counter()
    for tu, v, mjd, fs in files:
        ofs = None if fs is None else oracle.FaintStates(fs.timer1, fs.timer2, 1.0, 2.0)
        oracle.processmetrology(tu, v, mjd, offsets=off, faintparam=ofs, nthreads=cores)
    return time.perf_counter() - t0


DUMP_ROWS = 131_072     # demodulated VOLT rows kept by --dump-outputs (40 MB) ...
DUMP_FITS = 262_144     # ... and fits (14 MB of params and chi2): less than 64 MB in all


def dump_outputs(path, out, params, chi2):
    """--dump-outputs: what the resident path returned, as .npy files in `path`:
    volt_out [R, 80] float32 (demodulated VOLT rows in table, row order), params [M, 6] and
    chi2 [M] float64 (fits in table, window, diode order).  Beyond DUMP_ROWS rows or
    DUMP_FITS fits, a fixed, seeded sample of them is kept, in that order."""
    import torch
    os.makedirs(path, exist_ok=True)

    def keep(a, cap, seed):
        a = a.reshape(a.shape[0] * a.shape[1], -1)
        if a.shape[0] > cap:
            pick = np.sort(np.random.default_rng(seed).choice(a.shape[0], cap, replace=False))
            a = a[torch.from_numpy(pick).to(a.device)]
        return a.cpu().numpy()

    np.save(os.path.join(path, "volt_out.npy"), keep(out, DUMP_ROWS, 0))
    np.save(os.path.join(path, "params.npy"), keep(params, DUMP_FITS, 1))
    np.save(os.path.join(path, "chi2.npy"), keep(chi2, DUMP_FITS, 1)[:, 0])


# --------------------------------------------------------------------------
def main():
    args = parse()
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        return reference_arm(args, rank, world)
    if args.config == "stress":
        return stress_config(args, rank, world, local)
    if args.config == "sweep":
        return sweep_config(args, rank, world, local)

    import ctypes as C
    import gppd_b200 as gp
    from gppd_b200 import _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: libgppd has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_pinned = pin_to_gpu_numa_node(local)
    if world > 1:
        with quiet_stdout():
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()          # creates the communicator (and prints NCCL's banner) now
            torch.cuda.synchronize()
    h = gp.Handle(local)
    L = _lib.lib()
    F, N, S = args.files, args.rows, max(1, min(args.streams, h.num_slots - 1))
    faint = night_plan(F)
    time_us, volt, mjds, fss = generate_night(torch, gp, dev, F, N, rank)
    out = torch.empty_like(volt)
    W = args.window_rows if 0 < args.window_rows < N else 0
    NW = (N + W - 1) // W if W else 1          # windows (jobs) per table
    if W:
        args.no_e2e = True
    params = torch.empty((F, NW * 32, 6), dtype=torch.float64, device=dev)
    chi2 = torch.empty((F, NW * 32), dtype=torch.float64, device=dev)
    info = torch.zeros((F, NW * 32, 4), dtype=torch.int32, device=dev)
    offsets = torch.tensor(gp.synthetic.stefan_centres().view(np.float64), device=dev)
    opt = gp.api._options(fp32=args.fp32)
    torch.cuda.synchronize()

    def p(tensor):
        return C.c_void_p(tensor.data_ptr())

    def dptr(a):
        return None if a is None else a.ctypes.data_as(_lib._dp)

    # one batched launch sequence for the whole night (gppd_process_tables_f32_dev)
    i64 = lambda v: (C.c_int64 * F)(*v)
    vp = lambda ts: (C.c_void_p * F)(*[t.data_ptr() for t in ts])
    dpp = lambda arrs: (_lib._dp * F)(*[C.cast(None, _lib._dp) if a is None else a.ctypes.data_as(_lib._dp) for a in arrs])
    b_n = i64([N] * F)
    b_w = i64([W] * F) if W else None
    b_mjd = (C.c_double * F)(*mjds)
    b_time, b_volt, b_out = vp([time_us[k] for k in range(F)]), vp([volt[k] for k in range(F)]), vp([out[k] for k in range(F)])
    b_par, b_chi, b_info = vp([params[k] for k in range(F)]), vp([chi2[k] for k in range(F)]), vp([info[k] for k in range(F)])
    b_t1 = dpp([fs.timer1 if fs else None for fs in fss])
    b_t2 = dpp([fs.timer2 if fs else None for fs in fss])
    b_n1 = i64([fs.timer1.size if fs else 0 for fs in fss])
    b_n2 = i64([fs.timer2.size if fs else 0 for fs in fss])

    bench_stream = torch.cuda.Stream(device=dev)   # a real (non-NULL) stream: events see it

    NCH = max(1, min(args.chains, h.num_slots, F))
    chain_streams = [torch.cuda.Stream(device=dev) for _ in range(NCH)] if NCH > 1 else []

    def sub(arr, idx, typ):
        return None if arr is None else (typ * len(idx))(*[arr[i] for i in idx])

    chains = []
    for c in range(NCH):
        idx = list(range(c, F, NCH))
        chains.append(dict(n=len(idx), b_n=sub(b_n, idx, C.c_int64), b_w=sub(b_w, idx, C.c_int64),
                           b_time=sub(b_time, idx, C.c_void_p), b_mjd=sub(b_mjd, idx, C.c_double),
                           b_volt=sub(b_volt, idx, C.c_void_p), b_t1=sub(b_t1, idx, _lib._dp),
                           b_n1=sub(b_n1, idx, C.c_int64), b_t2=sub(b_t2, idx, _lib._dp),
                           b_n2=sub(b_n2, idx, C.c_int64), b_out=sub(b_out, idx, C.c_void_p),
                           b_par=sub(b_par, idx, C.c_void_p), b_chi=sub(b_chi, idx, C.c_void_p),
                           b_info=sub(b_info, idx, C.c_void_p)))

    def step_resident():
        if NCH == 1:
            _lib.check(L.gppd_process_tables_f32_dev(
                h.raw, 0, C.c_void_p(bench_stream.cuda_stream), F, b_n, b_w, b_time, b_mjd, b_volt, p(offsets),
                b_t1, b_n1, b_t2, b_n2, C.byref(opt), b_out, b_par, b_chi, b_info, None))
            return
        fork = torch.cuda.Event()
        fork.record(bench_stream)
        for c, ch in enumerate(chains):
            st = chain_streams[c]
            st.wait_event(fork)
            _lib.check(L.gppd_process_tables_f32_dev(
                h.raw, c, C.c_void_p(st.cuda_stream), ch["n"], ch["b_n"], ch["b_w"], ch["b_time"],
                ch["b_mjd"], ch["b_volt"], p(offsets), ch["b_t1"], ch["b_n1"], ch["b_t2"], ch["b_n2"],
                C.byref(opt), ch["b_out"], ch["b_par"], ch["b_chi"], ch["b_info"], None))
            ev = torch.cuda.Event()
            ev.record(st)
            bench_stream.wait_event(ev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- value: inputs resident in HBM ---------------------------------
    for _ in range(args.warmup):
        step_resident()
    barrier()
    h.enable_timing(True)
    h.pass_times(reset=True)
    launches0 = h.launches
    clocks = ClockSampler(local if rank == 0 else None)
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(bench_stream)
    for _ in range(args.steps):
        step_resident()
    e1.record(bench_stream)
    barrier()
    elapsed_ms = e0.elapsed_time(e1)
    passes_overlapped = h.pass_times(reset=True)
    h.enable_timing(False)
    launches = h.launches - launches0
    if args.dump_outputs and rank == 0:     # before the regions below overwrite the buffers
        dump_outputs(args.dump_outputs, out, params, chi2)
    # ---- per-pass kernel times: a second region of the same K steps with ONE launch
    # sequence per batch.  In the throughput region above the FAINT and the bright tables
    # run as two concurrent chains (gppd_set_split_chains, default on), whose kernels
    # share the SMs and stretch each other's event-timed durations; the roofline of a
    # kernel needs its own duration.
    split_default = os.environ.get("GPPD_SPLIT_CHAINS", "1")[:1] != "0"
    passes = passes_overlapped
    if split_default:
        h.set_split_chains(False)
        step_resident()
        barrier()
        h.enable_timing(True)
        h.pass_times(reset=True)
        for _ in range(args.steps):
            step_resident()
        barrier()
        passes = h.pass_times(reset=True)
        h.enable_timing(False)
        h.set_split_chains(True)
    tmax = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_per_step = float(tmax.item()) / args.steps
    units_per_step = F * N * DIODES * world
    value = units_per_step / (ms_per_step * 1e-3)
    nfev_mean = float(info[:, :, 0].double().mean().item())

    # ---- e2e: host buffers through the C ABI ----------------------------
    e2e = None
    if not args.no_e2e:
        h_time = torch.empty((F, N), dtype=torch.int32).pin_memory()
        h_volt = torch.empty((F, N, 80), dtype=torch.float32).pin_memory()
        h_out = torch.empty((F, N, 80), dtype=torch.float32).pin_memory()
        h_par = torch.empty((F, 32, 6), dtype=torch.float64).pin_memory()
        h_chi = torch.empty((F, 32), dtype=torch.float64).pin_memory()
        h_time.copy_(time_us); h_volt.copy_(volt)
        torch.cuda.synchronize()
        offs_h = gp.synthetic.stefan_centres()

        def hp(t, typ):
            return C.cast(C.c_void_p(t.data_ptr()), typ)

        def step_e2e():
            for k in range(F):
                fs = fss[k]
                _lib.check(L.gppd_submit_table_f32(
                    h.raw, 1 + k % S, N, hp(h_time[k], _lib._i32p), mjds[k], hp(h_volt[k], _lib._fp),
                    dptr(offs_h.view(np.float64)), dptr(fs.timer1) if fs else None,
                    fs.timer1.size if fs else 0, dptr(fs.timer2) if fs else None,
                    fs.timer2.size if fs else 0, 0.0, C.byref(opt), hp(h_out[k], _lib._fp),
                    hp(h_par[k], _lib._dp), hp(h_chi[k], _lib._dp), None, None))
            for s in range(S):
                _lib.check(L.gppd_wait(h.raw, 1 + s))

        for _ in range(max(1, args.warmup - 1)):
            step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        tm = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        e2e_val = units_per_step * args.steps / float(tm.item())
        # result check of the e2e path against the resident path (same fits)
        same = bool(torch.equal(h_par.to(dev), params))
        e2e = {"value": e2e_val, "unit": "diode-samples/s",
               "h2d_bytes_per_step": int(F * (N * 4 + N * 320)),
               "d2h_bytes_per_step": int(F * (N * 320 + 32 * 7 * 8)),
               "timing": "host wall clock around the K steps, device-synchronised, max over ranks",
               "matches_resident_path": same}

    clk = clocks.stop()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant pass ----------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    dom = max((k for k in passes if passes[k][1] > 0), key=lambda k: passes[k][0])
    dom_ms, dom_n = passes[dom]
    avg_ms = dom_ms / dom_n
    alg_bytes_per_launch = ALG_BYTES_PER_ROW * N * F      # one launch covers the whole night
    achieved = alg_bytes_per_launch / (avg_ms * 1e-3) / 1e9
    fp64_peak = h.fp64_peak_tflops()
    # algorithmic FP64 work of the harmonic pass: the contraction C[48 x 8] += E^T V,
    # i.e. per (row, diode) 24 harmonics x 4 FMA (DESIGN.md section 5); the recurrences
    # that generate E and the producers' arithmetic are overhead, not counted
    harm_flops_per_launch = F * N * 32 * (24 * 4) * 2.0
    harm_ms, harm_n = passes["harmonics"]
    fp64 = {"kernel": "harmonics",
            "achieved_tflops": harm_flops_per_launch / (harm_ms / max(harm_n, 1) * 1e-3) / 1e12 if harm_n else None,
            "peak_tflops": fp64_peak,
            "peak_source": "FP64 micro-benchmark in this run (better of DFMA and mma.sync.m8n8k4.f64)",
            "objective_calls_per_fit": nfev_mean}
    fp64["frac"] = fp64["achieved_tflops"] / fp64_peak if (fp64_peak and fp64["achieved_tflops"]) else None
    # which kernel computed the harmonic sums: the int8 tensor-core kernel takes every dense
    # table (GPPD_HARMONICS=dmma forces the FP64 DMMA kernel, csrc/harm_tc_kernels.cu)
    tensor_mode = os.environ.get("GPPD_HARMONICS", "")[:1] != "d"
    tensor = None
    if tensor_mode and harm_n:
        # issued int8 work: per 32 rows four MMAs of M = 128, K = 32, N = 144 + 144 + 240 + 192
        ops = F * N / 32.0 * 128 * 720 * 32 * 2
        i8_peak = 2.0 * float(peaks.get("bf16_tflops", 2250.0))
        tensor = {"kernel": "harmonics", "instruction": "tcgen05.mma kind::i8 (48-bit fixed point, 6 x 6 byte digits)",
                  "achieved_tops": ops / (harm_ms / harm_n * 1e-3) / 1e12, "peak_tops": i8_peak,
                  "peak_source": "2 x the dense bf16 figure of MEASURED_PEAKS.json (int8 runs at twice the bf16 rate)"
                                 if "bf16_tflops" in peaks else "nominal 4.5 POPS (B200_PROFILING.md fallback)",
                  "fp64_equivalent_tflops": fp64["achieved_tflops"]}
        tensor["frac"] = tensor["achieved_tops"] / i8_peak
        fp64["note"] = ("harmonic sums ran on the int8 tensor cores: achieved_tflops is the FP64 work they "
                        "replace (192 flop per diode-sample), not FP64 instructions issued")
    traffic = None   # DRAM bytes per launch of the dominant pass, from the committed ncu capture
    try:
        tname = "r2_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r2_traffic.json")) else "r1_traffic.json"
        tj = json.load(open(os.path.join(ROOT, "profiles", tname)))
        if tj["workload"] == {"tables": F, "rows": N} and not W:
            traffic = tj["bytes_per_launch"].get(dom)
    except Exception:
        pass
    # the whole step against the HBM roofline (algorithmic bytes / ms_per_step), and every
    # HBM-bound pass against the bytes IT has to move (the contract's `achieved` credits the
    # dominant pass with the whole pipeline's 644 B/row)
    nfaint_tab = sum(1 for f in faint if f)
    own_bytes = {"harmonics": 340.0 * N * F,                      # TIME-less: VOLT 320 + basis 16 (+ state)
                 "demod": (320.0 + 16.0 + 320.0) * N * F,          # VOLT + basis in, VOLT out
                 "stats": 257.0 * N * nfaint_tab,                  # 256 B of diode columns + state, FAINT tables
                 "basis": 20.0 * N * F}                            # TIME in, basis out
    per_pass = {}
    for k, b in own_bytes.items():
        if passes.get(k, (0, 0))[1]:
            ms_k = passes[k][0] / passes[k][1]
            per_pass[k] = {"own_bytes_per_launch": b, "avg_launch_ms": ms_k,
                           "gbs": b / (ms_k * 1e-3) / 1e9, "frac": b / (ms_k * 1e-3) / 1e9 / hbm_peak}
    step_roofline = {"algorithmic_bytes_per_step": alg_bytes_per_launch, "ms_per_step": ms_per_step / 1.0,
                     "achieved": alg_bytes_per_launch / (ms_per_step * 1e-3) / 1e9,
                     "frac": alg_bytes_per_launch / (ms_per_step * 1e-3) / 1e9 / hbm_peak,
                     "note": "whole step (all passes, FAINT and bright chains overlapped) on this rank's night; "
                             "the fit needs all rows before any row can be demodulated, so a table is read "
                             "at least twice (2 x 324 + 320 B/row = 1.5 x the algorithmic bytes) unless it "
                             "stays in L2"}
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm_peak,
                "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes_per_launch,
                "avg_launch_ms": avg_ms, "launches_timed": dom_n,
                "pass_ms_per_step": {k: v[0] / args.steps for k, v in passes.items() if v[1]},
                "pass_timing": ("second region of the same %d steps in this run with one launch sequence per "
                                "batch (gppd_set_split_chains(0)): in the throughput region the FAINT and the "
                                "bright chain run concurrently and stretch each other's kernel durations"
                                % args.steps) if split_default else "throughput region",
                "pass_ms_per_step_overlapped": {k: v[0] / args.steps for k, v in passes_overlapped.items() if v[1]},
                "step": step_roofline, "per_pass_own_bytes": per_pass,
                "fp64": fp64, "tensor": tensor,
                "harmonics_kernel": "k_harm_tc (int8 tensor cores)" if tensor_mode else "k_harm_ws (FP64 DMMA)",
                "note": ("one launch of each pass covers the whole night; the harmonic pass does 192 FP64-equivalent "
                         "flop per diode-sample against 20 B: on the FP64 units (k_harm_ws) it is bound by them; "
                         "as exact fixed-point int8 MMAs (k_harm_tc) it is bound by the producers' issue rate "
                         "(digit extraction), see DESIGN.md section 5; the demod pass is the HBM-bound one")}

    # ---- CPU baseline on a bounded sample -------------------------------
    cpu = None
    if not args.no_cpu:
        import oracle
        oracle.build()
        cores = min(8, os.cpu_count() or 1)
        nf = min(args.cpu_files, F)
        files = [(time_us[k].cpu().numpy(), volt[k].cpu().numpy(), mjds[k], fss[k]) for k in range(nf)]
        secs = cpu_reference_files(oracle, files, cores)
        cpu = {"value": nf * N * DIODES / secs, "unit": "diode-samples/s", "cores": cores,
               "kind": "port",
               "sample": "first %d tables of the night (%d rows each), whole-file fits, %.1f s" % (nf, N, secs)}

    line = {
        "metric": METRIC, "value": value, "unit": "diode-samples/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64" if not args.fp32 else "f64 fit and demodulation on float32-class harmonic sums (GPPD_FP32, optional)",
        "data": "synthetic",
        "config": night_config(F, N),
        "run_details": {"e2e_slots": S, "window_rows": W or None, "rank_pinned_to_gpu_numa_node": numa_pinned},
        "e2e": e2e, "gpu_launches": int(launches), "clocks": clk,
        "roofline": roofline, "cpu_baseline": cpu,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------
# shared by the stress and sweep configurations
def _setup(local, world):
    import torch
    import torch.distributed as dist
    import gppd_b200 as gp
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: libgppd has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pin_to_gpu_numa_node(local)
    if world > 1:
        with quiet_stdout():
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
    return torch, dist, gp, dev


def _peaks():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def _max_over_ranks(torch, dist, dev, world, ms):
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


STRESS_DT = 0.002                       # 500 Hz
STRESS_T0 = 86400.0 * 59949.0           # absolute seconds, like times of :139
STRESS_WINDOW_S = 100.0


def stress_truth(ch):
    """generating parameters of diode channel ch (deterministic)"""
    rng = np.random.default_rng(7700 + ch)
    amp = rng.uniform(0.05, 0.5)
    return dict(a=amp * np.exp(1j * rng.uniform(-np.pi, np.pi)), amp=amp, b=rng.uniform(0.3, 2.5),
                phi=rng.uniform(-np.pi, np.pi))


def stress_generate(torch, dev, row0, nrows, groups, data, tvec):
    """rows row0 .. row0 + nrows of the exposure for the given groups, written into
    data [40][nrows] (complex128) and tvec [nrows] (float64 absolute seconds); same model
    as gppd_b200.synthetic (centred channels: the demodulateall boundary)."""
    CH = 4_000_000
    for lo in range(0, nrows, CH):
        hi = min(lo + CH, nrows)
        i = torch.arange(row0 + lo, row0 + hi, device=dev, dtype=torch.float64)
        rel = i * STRESS_DT
        t = rel + STRESS_T0
        tvec[lo:hi] = t
        wt = 6.283185 * t
        g = torch.Generator(device=dev)
        for grp in groups:
            g.manual_seed(1_000_003 * grp + (row0 + lo) // 1000)
            phi_fc = 0.8 * torch.sin(0.05 * rel) + 0.5 * torch.sin(0.013 * rel + grp)
            efc = torch.polar(torch.ones_like(phi_fc), phi_fc)
            nz = torch.randn((2, hi - lo), generator=g, device=dev, dtype=torch.float64)
            data[32 + grp, lo:hi] = 0.3 * efc + 0.002 * torch.complex(nz[0], nz[1])
            for dio in range(4):
                ch = 4 * grp + dio
                tr = stress_truth(ch)
                mod = torch.polar(torch.ones_like(wt), tr["b"] * torch.sin(wt + tr["phi"]))
                nz = torch.randn((2, hi - lo), generator=g, device=dev, dtype=torch.float64)
                data[ch, lo:hi] = complex(tr["a"]) * efc * mod + (0.02 * tr["amp"]) * torch.complex(nz[0], nz[1])
                del mod, nz
            del phi_fc, efc
        del i, rel, t, wt


def stress_config(args, rank, world, local):
    """BASELINE.json configs[3]: long-exposure stress at the demodulateall boundary."""
    import ctypes as C
    torch, dist, gp, dev = _setup(local, world)
    from gppd_b200 import _lib, sharding
    h = gp.Handle(local)
    L = _lib.lib()
    n = int(args.stress_rows)
    free_b, total_b = torch.cuda.mem_get_info(dev)
    stream = torch.cuda.Stream(device=dev)
    clocks = ClockSampler(local if rank == 0 else None)
    clocks.start()
    p = lambda x: C.c_void_p(x.data_ptr())
    launches0 = h.launches
    hbm_peak, peak_src = _peaks()
    wrows = int(np.rint(STRESS_WINDOW_S / ((STRESS_T0 + STRESS_DT) - STRESS_T0)))   # :192 -> 50 004
    nwin = (n + wrows - 1) // wrows

    def timed(fn):
        for _ in range(max(1, args.warmup)):
            fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return _max_over_ranks(torch, dist, dev, world, e0.elapsed_time(e1)) / args.steps

    variants = {}
    # ---- (i) 100 s windows, contiguous time blocks -> ranks --------------------------
    wlo, whi = sharding.partition_windows(nwin, rank, world)
    r0, r1 = wlo * wrows, min(whi * wrows, n)
    nr = r1 - r0
    need = nr * (40 * 16 * 2 + 8 + 16) + (2 << 30)
    if need > free_b:
        raise SystemExit("stress: %d rows need %.0f GB on this rank, %.0f GB free; use --stress-rows"
                         % (n, need / 1e9, free_b / 1e9))
    nw_r = whi - wlo
    if nr >= 2:
        tv = torch.empty(nr, dtype=torch.float64, device=dev)
        data = torch.empty((40, nr), dtype=torch.complex128, device=dev)
        out = torch.empty((40, nr), dtype=torch.complex128, device=dev)
        par = torch.zeros((nw_r * 32, 6), dtype=torch.float64, device=dev)
        chi = torch.zeros(nw_r * 32, dtype=torch.float64, device=dev)
        info = torch.zeros((nw_r * 32, 4), dtype=torch.int32, device=dev)
        stress_generate(torch, dev, r0, nr, range(8), data, tv)
        torch.cuda.synchronize()
        opt = gp.api._options()
        stream.wait_stream(torch.cuda.current_stream(dev))

        def step_w():
            _lib.check(L.gppd_demodulate_f64_dev(h.raw, 0, C.c_void_p(stream.cuda_stream), nr, wrows, p(tv),
                                                 p(data), None, C.byref(opt), p(out), p(par), p(chi), p(info)))
        ms_w = timed(step_w)
        truth_b = torch.tensor([stress_truth(c)["b"] for c in range(32)], device=dev)
        full = par.view(nw_r, 32, 6)[: max(1, nw_r - 1)] if nw_r > 1 else par.view(nw_r, 32, 6)
        berr_w = float((full[:, :, 4] - truth_b[None, :]).abs().max().item())
        nfev_w = float(info[:, 0].double().mean().item())
        del tv, data, out, par, chi, info
        torch.cuda.empty_cache()
    else:
        ms_w = timed(lambda: None)
        berr_w, nfev_w = 0.0, 0.0
    variants["windows_100s"] = {
        "ms_per_step": ms_w, "value": n * DIODES / (ms_w * 1e-3), "windows": nwin, "rows_per_window": wrows,
        "fits": nwin * 32, "sharding": "contiguous time blocks (window ranges) -> ranks, host-side gather",
        "max_abs_b_error_vs_generating": berr_w, "objective_calls_per_fit": nfev_w,
        "hbm_frac_of_boundary_bytes": n * 1288.0 / world / (ms_w * 1e-3) / 1e9 / hbm_peak}

    # ---- (ii) ONE global fit per diode, the 8 groups -> ranks ------------------------
    mask = sharding.partition_groups(rank, world)
    groups = sharding.mask_groups(mask)
    tv = torch.empty(n, dtype=torch.float64, device=dev)
    data = torch.empty((40, n), dtype=torch.complex128, device=dev)   # only this rank's channels are filled
    out = torch.empty((40, n), dtype=torch.complex128, device=dev)
    par = torch.zeros((32, 6), dtype=torch.float64, device=dev)
    chi = torch.zeros(32, dtype=torch.float64, device=dev)
    info = torch.zeros((32, 4), dtype=torch.int32, device=dev)
    stress_generate(torch, dev, 0, n, groups, data, tv)
    torch.cuda.synchronize()
    opt = gp.api._options(groups=mask)
    stream.wait_stream(torch.cuda.current_stream(dev))

    def step_g():
        _lib.check(L.gppd_demodulate_f64_dev(h.raw, 0, C.c_void_p(stream.cuda_stream), n, 0, p(tv), p(data),
                                             None, C.byref(opt), p(out), p(par), p(chi), p(info)))
    h.enable_timing(True)
    h.pass_times(reset=True)
    ms_g = timed(step_g)
    passes = h.pass_times(reset=True)
    h.enable_timing(False)
    # final host-side gather: parameters of every rank's groups (the demodulated columns stay
    # on the GPU that owns the group)
    mine = [c for c in sharding.mask_channels(mask) if c < 32]
    allpar = par.clone()
    if world > 1:
        dist.all_reduce(allpar, op=dist.ReduceOp.SUM)       # untouched entries are zero
    truth_b = torch.tensor([stress_truth(c)["b"] for c in range(32)], device=dev)
    berr_g = float((allpar[:, 4] - truth_b).abs().max().item())
    amp_ok = float(((allpar[:, 2] ** 2 + allpar[:, 3] ** 2).sqrt() -
                    torch.tensor([stress_truth(c)["amp"] for c in range(32)], device=dev)).abs().max().item())
    nfev_g = float(info[mine][:, 0].double().mean().item())
    rot = float(((out[mine[0]].abs() - data[mine[0]].abs()).abs().max() / data[mine[0]].abs().max()).item())
    steps_timed = args.steps + max(1, args.warmup)
    variants["global_fit"] = {
        "ms_per_step": ms_g, "value": n * DIODES / (ms_g * 1e-3), "fits": 32,
        "sharding": "8 (telescope, side) groups -> ranks via gppd_options.group_mask, host-side gather",
        "groups_per_rank": len(groups), "max_abs_b_error_vs_generating": berr_g,
        "max_abs_amplitude_error_vs_generating": amp_ok, "objective_calls_per_fit": nfev_g,
        "max_rel_modulus_change_of_output": rot,
        "pass_ms_per_step_rank0": {k: v[0] / steps_timed for k, v in passes.items() if v[1]},
        "hbm_frac_of_boundary_bytes": n * 1288.0 / world / (ms_g * 1e-3) / 1e9 / hbm_peak}
    clk = clocks.stop()
    launches = h.launches - launches0
    if rank == 0:
        dom = max(passes, key=lambda k: passes[k][0])
        dom_ms = passes[dom][0] / max(passes[dom][1], 1)
        alg = n * 1288.0 / world
        line = {
            "metric": METRIC, "value": variants["global_fit"]["value"], "unit": "diode-samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(1, args.warmup),
            "ms_per_step": ms_g, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "long-exposure stress: ONE exposure of %d rows x 40 complex128 channels at the "
                                   "demodulateall boundary, generated on the device (BASELINE.json configs[3]); "
                                   "value = the single global fit, variants = both modes" % n,
                       "rows": n, "diodes": DIODES, "boundary_bytes_per_row": 1288,
                       "cache": "inputs (%.0f GB per rank) larger than L2" % (n * 648.0 / world / 1e9),
                       "device_memory_gb": total_b / 1e9},
            "variants": variants,
            "e2e": None, "e2e_note": "the exposure exists on the device only (64 GB of complex128 per direction "
                                     "at 1e8 rows; a METROLOGY table cannot hold it: TIME is int32 microseconds)",
            "gpu_launches": int(launches), "clocks": clk,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": alg / (dom_ms * 1e-3) / 1e9, "peak": hbm_peak,
                         "unit": "GB/s", "frac": alg / (dom_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                         "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
                         "avg_launch_ms": dom_ms,
                         "note": "global-fit variant on rank 0; algorithmic bytes = the rank's share of the "
                                 "1 288 B/row of the complex128 boundary (t 8 + data 640 in, 640 out)"},
            "cpu_baseline": None,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------
SWEEP_W = 512                      # rows per fit window (about one modulation period)
SWEEP_TAB_WIN = 1954               # windows per table: 1 000 448 rows < the int32 TIME range
SWEEP_CHUNK_TABLES = 16            # one chunk = 16 tables = 1 000 448 fits


def sweep_config(args, rank, world, local):
    """BASELINE.json configs[4]: batched-fit sweep, F independent fits of 512 rows each at the
    METROLOGY-table boundary (the window loop of src/GPPupilDemodulation.jl:204-225)."""
    import ctypes as C
    torch, dist, gp, dev = _setup(local, world)
    from gppd_b200 import _lib
    h = gp.Handle(local)
    L = _lib.lib()
    hbm_peak, peak_src = _peaks()
    fp64_peak = h.fp64_peak_tflops()
    T, NW = SWEEP_CHUNK_TABLES, SWEEP_TAB_WIN
    N = NW * SWEEP_W
    clocks = ClockSampler(local if rank == 0 else None)
    clocks.start()
    launches0 = h.launches
    stream = torch.cuda.Stream(device=dev)
    centres = gp.synthetic.stefan_centres()
    results = {}
    for variant in ("bright_nooffsets", "faint_withoffsets"):
        faint = variant.startswith("faint")
        # one chunk of tables, generated like the night (70/30 mix replaced by all-bright / all-FAINT)
        time_us, volt, mjds, fss = generate_night(torch, gp, dev, T, N, rank, plan=[faint] * T,
                                                  faint_repeat=680)     # switching over the whole table
        out = torch.empty_like(volt)
        params = torch.empty((T, NW * 32, 6), dtype=torch.float64, device=dev)
        chi2 = torch.empty((T, NW * 32), dtype=torch.float64, device=dev)
        info = torch.zeros((T, NW * 32, 4), dtype=torch.int32, device=dev)
        offsets = None if faint else torch.tensor(centres.view(np.float64), device=dev)
        opt = gp.api._options()
        torch.cuda.synchronize()
        stream.wait_stream(torch.cuda.current_stream(dev))

        def launch(nwin_total):
            """one launch sequence over the first nwin_total windows of the chunk"""
            nt = (nwin_total + NW - 1) // NW
            rows = [min(NW, nwin_total - k * NW) * SWEEP_W for k in range(nt)]
            i64 = lambda v: (C.c_int64 * nt)(*v)
            vp = lambda ts: (C.c_void_p * nt)(*[t.data_ptr() for t in ts])
            dpp = lambda arrs: (_lib._dp * nt)(*[C.cast(None, _lib._dp) if a is None else a.ctypes.data_as(_lib._dp)
                                                 for a in arrs])
            keep = (i64(rows), i64([SWEEP_W] * nt), vp([time_us[k] for k in range(nt)]), (C.c_double * nt)(*mjds[:nt]),
                    vp([volt[k] for k in range(nt)]),
                    dpp([fss[k].timer1 if faint else None for k in range(nt)]),
                    i64([fss[k].timer1.size if faint else 0 for k in range(nt)]),
                    dpp([fss[k].timer2 if faint else None for k in range(nt)]),
                    i64([fss[k].timer2.size if faint else 0 for k in range(nt)]),
                    vp([out[k] for k in range(nt)]), vp([params[k] for k in range(nt)]),
                    vp([chi2[k] for k in range(nt)]), vp([info[k] for k in range(nt)]))

            def go():
                _lib.check(L.gppd_process_tables_f32_dev(
                    h.raw, 0, C.c_void_p(stream.cuda_stream), nt, keep[0], keep[1], keep[2], keep[3], keep[4],
                    None if offsets is None else C.c_void_p(offsets.data_ptr()), keep[5], keep[6], keep[7],
                    keep[8], C.byref(opt), keep[9], keep[10], keep[11], keep[12], None))
            return go, keep

        curve = []
        F = 1000
        while F <= args.sweep_max * 1.0001:
            nwin_total = int(np.ceil(F / 32.0))
            chunk_win = min(nwin_total, T * NW)
            reps = int(np.ceil(nwin_total / float(chunk_win)))      # > 1 only beyond one chunk
            go, keep = launch(chunk_win)
            fits = chunk_win * 32 * reps
            go()
            torch.cuda.synchronize()
            h.enable_timing(True)
            h.pass_times(reset=True)
            k_steps = max(1, min(args.steps, 3 if fits >= 1_000_000 else args.steps))
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(k_steps):
                for _ in range(reps):
                    go()
            e1.record(stream)
            torch.cuda.synchronize()
            ms = _max_over_ranks(torch, dist, dev, world, e0.elapsed_time(e1)) / k_steps
            passes = h.pass_times(reset=True)
            h.enable_timing(False)
            rows_done = fits // 32 * SWEEP_W
            nf = info[: (chunk_win + NW - 1) // NW].reshape(-1, 4)[: chunk_win * 32]
            curve.append({
                "fits": fits, "chunks": reps, "ms": ms, "fits_per_s": fits * world / (ms * 1e-3),
                "diode_samples_per_s": fits * world * SWEEP_W / (ms * 1e-3),
                "hbm_frac": rows_done * ALG_BYTES_PER_ROW / (ms * 1e-3) / 1e9 / hbm_peak,
                "fp64_equivalent_tflops": fits * SWEEP_W * 192.0 / (ms * 1e-3) / 1e12,
                "fp64_frac": fits * SWEEP_W * 192.0 / (ms * 1e-3) / 1e12 / fp64_peak if fp64_peak else None,
                "objective_calls_per_fit": float(nf[:, 0].double().mean().item()),
                "fallback_fits": int((nf[:, 2] == 1).sum().item()),
                "pass_ms": {k: v[0] / k_steps for k, v in passes.items() if v[1]}})
            F *= 10
        results[variant] = curve
        del time_us, volt, out, params, chi2, info
        torch.cuda.empty_cache()
    clk = clocks.stop()
    launches = h.launches - launches0
    if rank == 0:
        top = results["bright_nooffsets"][-1]
        dom = max(top["pass_ms"], key=lambda k: top["pass_ms"][k])
        line = {
            "metric": METRIC, "value": top["diode_samples_per_s"], "unit": "diode-samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": 1, "ms_per_step": top["ms"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "batched-fit sweep: F independent fits of %d rows (BASELINE.json configs[4]), "
                                   "METROLOGY-table boundary, window mode; value = largest F, bright" % SWEEP_W,
                       "rows_per_fit": SWEEP_W, "chunk_fits": T * NW * 32,
                       "cache": "one chunk = %.1f GB of input, larger than L2" % (T * N * 324 / 1e9),
                       "replicas": "every rank runs the same sweep on its own data"},
            "sweep": results, "e2e": None,
            "e2e_note": "device-resident sweep of the fit throughput; the end-to-end number is the night's",
            "gpu_launches": int(launches), "clocks": clk,
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": top["hbm_frac"] * hbm_peak, "peak": hbm_peak,
                         "unit": "GB/s", "frac": top["hbm_frac"], "traffic": None, "peak_source": peak_src,
                         "fp64_peak_tflops": fp64_peak,
                         "note": "whole-step figure at the largest F (644 algorithmic bytes per row); per-F "
                                 "curves with pass times under `sweep`"},
            "cpu_baseline": None,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def reference_arm(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle restatement; the
    Julia package cannot run here) on this box's host cores, same night, each
    step a bounded sample of it."""
    if rank != 0:
        return
    import gppd_b200 as gp
    import oracle
    oracle.build()
    cores = min(8, os.cpu_count() or 1)
    F, N = args.files, args.rows
    # a bounded sample of the night that keeps its mix: tables 0..9 of the plan are 7 bright and
    # 3 FAINT (k % 10 in (3, 6, 9)), exactly the night's 70 / 30
    nf = max(1, min(10, F))      # tables per step
    faint = night_plan(F)
    files = []
    for k in range(nf):
        tab = gp.synthetic.make_table(N, k=k, jitter=True)
        fs = None
        if faint[k]:
            hdr = gp.synthetic.faint_header(tab["mjd"])
            fs = oracle.buildfaintparameters(hdr)
            t = oracle.make_times(tab["time_us"], tab["mjd"])
            st = oracle.buildstates(fs, t)
            tab = gp.synthetic.make_table(N, k=k, jitter=True, faint=True, state=st)
        files.append((tab["time_us"], tab["volt"], tab["mjd"], fs))
    for _ in range(min(args.warmup, 1)):
        cpu_reference_files(oracle, files[:1], cores)
    # one table per step, cycling through the sample: K = 20 steps run every table twice, so the
    # aggregate keeps the night's mix and the whole run stays within a minute or two
    t0 = time.perf_counter()
    done = []
    for i in range(args.steps):
        cpu_reference_files(oracle, [files[i % nf]], cores)
        done.append(i % nf)
    dt = time.perf_counter() - t0
    value = N * DIODES * args.steps / dt
    nfaint = sum(1 for k in done if faint[k])
    sample = ("one table of %d rows per step, cycling through tables 0..%d of the %d-table night "
              "(7 bright + 3 FAINT per 10: the night's mix); the %d steps timed %d bright + %d FAINT tables, "
              "whole-file fits" % (N, nf - 1, F, args.steps, args.steps - nfaint, nfaint))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "diode-samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": night_config(F, N),
        "reference_sample": sample,
        "cpu_baseline": {"value": value, "unit": "diode-samples/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "diode-samples/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "note": "restated CPU reference algorithm (oracle/): the Julia package and its NEWUOA "
                "dependency cannot be installed in this image",
    }))


if __name__ == "__main__":
    main()
