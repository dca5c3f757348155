"""Command-line front end with the reference's flags (``main``,
src/GPPupilDemodulation.jl:257-426) and a night-level scheduler on top of the C ABI.

    python -m gppd_b200.cli [-s SUFFIX] [-o] [-f] [-r] [-v] [-k] [-c CENTER]
                            [-w WINDOW] [-d DIR] INPUT...

Same gating as the reference: a file is processed when its primary header has
``ESO INS PMC1 MODULATE = T`` and ``ESO INS MET MODE`` is not ``OFF``; ``FAINT`` mode
builds the laser on/off timers from the ``ESO INS ANLO3`` keywords unless
``--nofaint``.  The output is a copy of the input file with the ``METROLOGY`` table
and its header replaced, written to ``DIR/<name><SUFFIX>.fits``.

What differs is the execution: files are not processed one after the other but
pipelined over the handle's slots -- while one file's records are on the GPU the next
one is being read and uploaded and the previous one written -- and with several GPUs
(``RANK`` / ``WORLD_SIZE`` from torchrun, or ``--rank/--world``) every rank takes every
WORLD_SIZE-th file; there is no communication between ranks.  The METROLOGY records
travel as raw FITS bytes: byte swapping, de-interleaving, the fit, the demodulation and
the re-packing all happen on the device.  For plain ``.fits`` files Python never touches a
record: it reads the headers, decides (gating), and hands the file to the library's
native ingest (``gppd_file_submit`` / ``gppd_file_wait`` / ``gppd_file_write``: reader
threads fill pinned buffers straight from the file, writer threads assemble the output);
after the fit it only formats the new METROLOGY header.  Compressed files (``.fits.gz``,
``fits.Z``) are decompressed here and go through ``gppd_submit_fits_rows``.
"""
from __future__ import annotations

import argparse
import ctypes as C
import logging
import os
import sys
import time

import numpy as np

from . import _lib, fits
from .sharding import partition_files
from .api import (_options, buildfaintparameters, demodulation_keys, ellipse_keys, ellipses,
                  read_stefan_file, window_columns)

SUFFIXES = (".fits", ".fits.gz", "fits.Z")      # src/GPPupilDemodulation.jl:14
log = logging.getLogger("GPPupilDemodulation")


def build_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(prog="GPPupilDemodulation",
                                description="Simple tool to demodulate Gravity metrology table.")
    p.add_argument("--version", action="version", version="0.1")
    p.add_argument("--suffix", "-s", default="",
                   help="Store the demodulated metrology in the INPUT.SUFFIX.fits file")
    p.add_argument("--onlyhigh", "-o", action="store_true",
                   help="Demodulate metrology using parameters estimated only on HIGH and NORMAL")
    p.add_argument("--nofaint", "-f", action="store_true",
                   help="Do no use the faint mode state to demodulate")
    p.add_argument("--recursive", "-r", action="store_true", help="Recursively explore entire directories.")
    p.add_argument("--verbose", "-v", action="store_true", help="Verbose mode")
    p.add_argument("--keepraw", "-k", action="store_true", help="keep raw")
    p.add_argument("--center", "-c", default="stefan",
                   help="center voltages: stefan (default) | empirical | uncentered | fit | ellipse "
                        "(offset and ellipse correction of each channel, fitted per file)")
    p.add_argument("--window", "-w", type=float, default=0.0,
                   help="Compute demodulation on non overlapping window of WINDOW second")
    p.add_argument("--dir", "-d", default=os.getcwd(), help="output folder")
    p.add_argument("--rank", type=int, default=int(os.environ.get("RANK", "0")), help=argparse.SUPPRESS)
    p.add_argument("--world", type=int, default=int(os.environ.get("WORLD_SIZE", "1")), help=argparse.SUPPRESS)
    p.add_argument("--device", type=int, default=int(os.environ.get("LOCAL_RANK", "0")), help=argparse.SUPPRESS)
    p.add_argument("--no-native", dest="no_native", action="store_true", help=argparse.SUPPRESS)
    p.add_argument("INPUT", nargs="*", default=["."],
                   help="List of all TARGET to process. In conjunction with -r TARGET can contain directories.")
    return p


class _Job:
    """One file in flight on one pipeline slot."""

    def __init__(self, filename, outname, hdus, imet, faintparam, mjd, layout, window, keepraw,
                 native=False):
        self.filename, self.outname, self.hdus, self.imet = filename, outname, hdus, imet
        self.native = native               # plain file: records read / written by the library
        self.faintparam, self.mjd, self.window, self.keepraw = faintparam, mjd, window, keepraw
        self.row_bytes, self.n, self.cols = layout
        self.tstart = time.time()


def _plan_file(filename, args, folder):
    """Header gating of one file (reference :358-392).  Returns a _Job or None."""
    if not os.path.isfile(filename) or not filename.endswith(SUFFIXES):
        return None
    native = filename.endswith(".fits") and not getattr(args, "no_native", False)
    hdus = fits.scan_fits(filename) if native else fits.read_fits(filename)
    prim = hdus[0].header
    if "ESO INS PMC1 MODULATE" not in prim:
        log.info("no ESO INS PMC1 MODULATE keyword in %s", filename)
        return None
    if not prim["ESO INS PMC1 MODULATE"]:
        log.info("ESO INS PMC1 MODULATE set to false in %s", filename)
        return None
    log.info("Processing %s", filename)
    metmod = prim.get("ESO INS MET MODE", "ON")
    log.info("%s use %s metrology mode", filename, metmod)
    if metmod == "OFF":
        return None
    faintparam = None
    if metmod == "FAINT":
        if not args.nofaint:
            faintparam = buildfaintparameters(prim)
        else:
            log.info("FAINT mode deactivated")
    mjd = float(prim["MJD-OBS"])
    imet = next((i for i, h in enumerate(hdus) if h.is_bintable and h.name == "METROLOGY"), None)
    if imet is None:
        raise KeyError(f"{filename}: no METROLOGY table")
    layout = fits.bintable_layout(hdus[imet].header)
    for col, width in (("TIME", 4), ("VOLT", 320)):
        if col not in layout[2] or fits.tform_bytes(layout[2][col][1]) != width:
            raise ValueError(f"{filename}: METROLOGY column {col} missing or of unexpected width")
    fname = os.path.basename(filename).split(".fits")[0]
    outname = os.path.join(folder, fname + args.suffix + ".fits")
    return _Job(filename, outname, hdus, imet, faintparam, mjd, layout,
                args.window if args.window != 0.0 else None, args.keepraw, native=native)


class NightScheduler:
    """Files -> pipeline slots of one handle (one GPU)."""

    def __init__(self, handle, offsets, onlyhigh, method="auto"):
        self.h, self.L = handle, _lib.lib()
        self.empirical = offsets is True       # --center empirical: centres fitted on the device
        # --center ellipse: one ellipse per channel fitted and applied on the device
        self.ellipse = isinstance(offsets, str) and offsets == "ellipse"
        self.offsets = (None if (offsets is None or self.empirical or self.ellipse)
                        else np.ascontiguousarray(offsets, dtype=np.complex128))
        self.onlyhigh, self.method = onlyhigh, method
        self.nslots = handle.num_slots
        self.busy = [None] * self.nslots       # (job, buffers) per slot
        self.pinned = [dict() for _ in range(self.nslots)]
        self.keep = [None] * self.nslots       # per-row columns a pending native write still reads

    def _pinned(self, slot, key, nbytes):
        """A pinned staging buffer of the slot, grown on demand."""
        cur = self.pinned[slot].get(key)
        if cur is None or cur[1] < nbytes:
            if cur is not None:
                _lib.check(self.L.gppd_free_pinned(self.h.raw, cur[0]))
            p = C.c_void_p()
            cap = int(nbytes * 1.25) + 4096
            _lib.check(self.L.gppd_alloc_pinned(self.h.raw, cap, C.byref(p)))
            cur = (p, cap)
            self.pinned[slot][key] = cur
        return np.ctypeslib.as_array(C.cast(cur[0], C.POINTER(C.c_uint8)), shape=(cur[1],))[:nbytes]

    def _first_times(self, job):
        """TIME of the first two records (for the --window arithmetic, :192)."""
        rb, toff = job.row_bytes, job.cols["TIME"][0]
        met = job.hdus[job.imet]
        if job.native:
            with open(job.filename, "rb") as fh:
                fh.seek(met.data_offset)
                head = fh.read(2 * rb)
        else:
            head = bytes(met.data[:2 * rb])
        return np.array([int.from_bytes(head[k * rb + toff:k * rb + toff + 4], "big", signed=True)
                         for k in range(2)], dtype=np.int32)

    def submit(self, slot, job: _Job):
        n, rb = job.n, job.row_bytes
        rb_out = rb + (256 if job.keepraw else 0)
        wrows, nwin = n, 1
        if job.window is not None:
            t01 = self._first_times(job)
            w, k = C.c_int64(0), C.c_int64(0)
            _lib.check(self.L.gppd_table_windows(2, _lib.ptr(t01, _lib._i32p), job.mjd, float(job.window),
                                                 C.byref(w), C.byref(k)))
            wrows = w.value
            nwin = (n + wrows - 1) // wrows
        o = _options(onlyhigh=self.onlyhigh, keepraw=job.keepraw, method=self.method,
                     empirical=self.empirical, ellipse=self.ellipse)
        fp = job.faintparam
        t1 = fp.timer1 if fp is not None else None
        t2 = fp.timer2 if fp is not None else None
        off = None if self.offsets is None else self.offsets.view(np.float64)
        if job.native:
            # the library reads the records itself, straight into its pinned staging buffers
            met = job.hdus[job.imet]
            _lib.check(self.L.gppd_file_submit(
                self.h.raw, slot, os.fsencode(job.filename), met.data_offset, n, rb, job.cols["TIME"][0],
                job.cols["VOLT"][0], job.mjd, _lib.ptr(off), _lib.ptr(t1), 0 if t1 is None else t1.size,
                _lib.ptr(t2), 0 if t2 is None else t2.size, float(job.window or 0.0), C.byref(o)))
            self.busy[slot] = (job, dict(wrows=wrows, nwin=nwin, rb_out=rb_out, keep=(o, off, t1, t2)))
            return
        src = np.frombuffer(job.hdus[job.imet].data, dtype=np.uint8, count=n * rb)
        rows = self._pinned(slot, "rows", n * rb)
        rows[:] = src
        rows_out = self._pinned(slot, "rows_out", n * rb_out)
        # the small results in pinned memory too: a download into pageable memory would make
        # the submit call wait for the whole file
        params = self._pinned(slot, "params", nwin * 32 * 6 * 8).view(np.float64).reshape(nwin * 32, 6)
        chi2 = self._pinned(slot, "chi2", nwin * 32 * 8).view(np.float64)
        state = self._pinned(slot, "state", n).view(np.int8) if job.faintparam is not None else None
        _lib.check(self.L.gppd_submit_fits_rows(
            self.h.raw, slot, n, rows.ctypes.data_as(C.c_void_p), rb, job.cols["TIME"][0],
            job.cols["VOLT"][0], job.mjd, _lib.ptr(off), _lib.ptr(t1), 0 if t1 is None else t1.size,
            _lib.ptr(t2), 0 if t2 is None else t2.size, float(job.window or 0.0), C.byref(o),
            rows_out.ctypes.data_as(C.c_void_p), _lib.ptr(params), _lib.ptr(chi2), None,
            _lib.ptr(state, _lib._i8p)))
        self.busy[slot] = (job, dict(rows_out=rows_out, params=params, chi2=chi2, state=state,
                                     wrows=wrows, nwin=nwin, rb_out=rb_out, keep=(o, off, t1, t2)))

    def finish(self, slot):
        """Wait for the slot's file, take its records out of the slot's pinned buffer and hand
        the assembling and writing of the output file to the writer threads (reference
        :406-412); returns a future of the output name."""
        job, b = self.busy[slot]
        self.busy[slot] = None
        if job.native:
            return self._finish_native(slot, job, b)
        _lib.check(self.L.gppd_wait(self.h.raw, slot))
        b["ell"] = self._ellipses(slot)
        # the slot's staging buffers are reused by the next file: take the results out
        b = dict(b, rows_out=b["rows_out"].copy(), params=b["params"].copy(), chi2=b["chi2"].copy(),
                 state=None if b["state"] is None else b["state"].copy())
        return self.writers.submit(self._write, job, b)

    def _ellipses(self, slot):
        """The (40, 6) maps of the slot's last file (--center ellipse), else None."""
        return ellipses(self.h, slot, 1)[0][0] if self.ellipse else None

    def _table_edits(self, job, b, n):
        """(header keys, new columns, extra per-row bytes or None) of the output table
        (reference :174-189 whole-file keys, :209-249 window-mode columns)."""
        fitoffsets = self.offsets is None and not self.empirical and not self.ellipse
        keys, newcols, extra = [], [], None
        if self.ellipse:                    # the transform applied to VOLT, both modes
            keys += list(ellipse_keys(b["ell"]).items())
        if job.window is None:
            keys += list(demodulation_keys(b["params"], fitoffsets).items())
        else:
            cols = window_columns(b["params"], n, b["wrows"], b["nwin"], fitoffsets)
            parts = []
            for name in ("ABSA", "ARGA", "B", "PHI", "X0", "Y0"):
                if name in cols:
                    parts.append(cols[name].astype(">f4").view(np.uint8).reshape(n, 128))
                    newcols.append((name, "32E", None))
            if b["state"] is not None:      # Int8 column: FITS 'B' with TZERO = -128
                parts.append((b["state"].astype(np.int16) + 128).astype(np.uint8).reshape(n, 1))
                newcols.append(("STATE", "1B", None))
            extra = np.ascontiguousarray(np.concatenate(parts, axis=1))
        keys.append(("PROCSOFT", "GPPupilDemodulation.jl"))
        return keys, newcols, extra

    def _finish_native(self, slot, job, b):
        """Wait for the fit, format the new METROLOGY header and hand the writing of the
        output file (FITScopy!, src/FitsUtils.jl:95-156) to the library's writer threads."""
        n, nwin = job.n, b["nwin"]
        b["params"] = np.empty((nwin * 32, 6))
        b["chi2"] = np.empty(nwin * 32)
        b["state"] = np.empty(n, dtype=np.int8) if job.faintparam is not None else None
        _lib.check(self.L.gppd_file_wait(self.h.raw, slot, _lib.ptr(b["params"]), _lib.ptr(b["chi2"]), None,
                                         _lib.ptr(b["state"], _lib._i8p)))
        b["ell"] = self._ellipses(slot)
        keys, newcols, extra = self._table_edits(job, b, n)
        met = job.hdus[job.imet]
        rb_new = b["rb_out"] + (0 if extra is None else extra.shape[1])
        cards = fits.replace_bintable_cards(met, rb_new, n, {"VOLT": "144E"} if job.keepraw else None,
                                            newcols, keys)
        if b["state"] is not None and job.window is not None:
            i = next(int(v) for k, v in map(fits.parse_card, cards) if k == "TFIELDS")
            cards += [fits.format_card(f"TSCAL{i}", 1), fits.format_card(f"TZERO{i}", -128)]
        head = fits.header_bytes(cards)
        size = os.path.getsize(job.filename)
        tail = met.data_offset + met.data_padded
        segs = (_lib.FileSegment * 4)()
        segs[0].kind, segs[0].offset, segs[0].length = _lib.SEG_COPY, 0, met.hdr_offset
        segs[1].kind, segs[1].length = _lib.SEG_BYTES, len(head)
        segs[1].bytes = C.cast(C.c_char_p(head), C.c_void_p)
        segs[2].kind = _lib.SEG_RECORDS
        segs[3].kind, segs[3].offset, segs[3].length = _lib.SEG_COPY, tail, max(0, size - tail)
        _lib.check(self.L.gppd_file_write(
            self.h.raw, slot, os.fsencode(job.outname), segs, 4,
            None if extra is None else extra.ctypes.data_as(C.c_void_p), 0 if extra is None else extra.shape[1]))
        self.keep[slot] = extra             # must stay valid until the slot's next submit / the drain
        log.info("%s processed in %.3f s", job.filename, time.time() - job.tstart)
        log.info(" %s written", job.outname)
        return job.outname

    def _write(self, job, b):
        n = job.n
        records = b["rows_out"].reshape(n, b["rb_out"])
        keys, newcols, extra = self._table_edits(job, b, n)
        if extra is not None:
            records = np.concatenate([records, extra], axis=1)
        met = job.hdus[job.imet]
        new = fits.replace_bintable(met, records,
                                    tform_changes={"VOLT": "144E"} if job.keepraw else None,
                                    new_columns=newcols, new_keys=keys)
        if b["state"] is not None and job.window is not None:
            i = int(new.header["TFIELDS"])
            new.cards += [fits.format_card(f"TSCAL{i}", 1), fits.format_card(f"TZERO{i}", -128)]
        hdus = list(job.hdus)
        hdus[job.imet] = new
        fits.write_fits(job.outname, hdus)
        log.info("%s processed in %.3f s", job.filename, time.time() - job.tstart)
        log.info(" %s written", job.outname)
        return job.outname

    def run(self, jobs):
        """Pipeline the jobs over the slots -- reader threads plan (read and gate) the next
        files, the GPU works on up to `nslots` files, writer threads assemble and write the
        finished ones; returns the output names in input order."""
        from concurrent.futures import ThreadPoolExecutor
        # Slot k is in one of two halves of the ring: up to `depth` files are on the GPU (read,
        # uploaded, fitted, downloaded) while the `depth` files before them are being written.
        # A slot is only re-submitted `depth` files after its write was requested, so that
        # gppd_file_submit (which waits for the slot's previous output file) does not stall.
        done, depth = [], max(1, self.nslots // 2)
        with ThreadPoolExecutor(max_workers=3) as self.writers:
            i = 0
            self.t_plan = self.t_finish = self.t_submit = 0.0     # where the main thread's time goes
            t0 = time.perf_counter()
            for job in jobs:
                t1 = time.perf_counter()
                if i >= depth:
                    done.append(self.finish((i - depth) % self.nslots))
                t2 = time.perf_counter()
                self.submit(i % self.nslots, job)
                t3 = time.perf_counter()
                self.t_plan += t1 - t0
                self.t_finish += t2 - t1
                self.t_submit += t3 - t2
                t0 = t3
                i += 1
            for k in range(max(0, i - depth), i):
                done.append(self.finish(k % self.nslots))
            names = [f if isinstance(f, str) else f.result() for f in done]
        _lib.check(self.L.gppd_file_drain(self.h.raw))      # the library's writer threads are done
        self.keep = [None] * self.nslots
        return names


def main(argv=None) -> int:
    args = build_parser().parse_args(argv)
    logging.basicConfig(level=logging.INFO if args.verbose else logging.WARNING,
                        format="[ Info: %(message)s", stream=sys.stderr)
    files = []
    for arg in args.INPUT:              # reference :324-331
        if os.path.isdir(arg) and args.recursive:
            for root, _, names in os.walk(arg):
                files += [os.path.join(root, f) for f in sorted(names)]
        else:
            files.append(arg)
    folder = args.dir
    if not folder.startswith("/"):
        folder = os.path.join(os.getcwd(), folder)
    os.makedirs(folder, exist_ok=True)   # (the reference creates relative folders only)
    if args.center == "stefan":          # reference :346-354
        offsets = read_stefan_file()
    elif args.center == "uncentered":
        offsets = np.zeros(40, dtype=np.complex128)
    elif args.center == "empirical":     # offsets = true: compute_offsets, :105-125
        offsets = True
    elif args.center == "fit":
        offsets = None
    elif args.center == "ellipse":       # offset + ellipse (Heydemann) correction per channel
        offsets = "ellipse"
    else:
        raise SystemExit(f"unknown --center {args.center}")
    mine = partition_files(files, args.rank, args.world)   # no communication between ranks
    handle = _lib.Handle(args.device)
    sched = NightScheduler(handle, offsets, args.onlyhigh)

    def jobs():
        # read and gate a few files ahead of the GPU (file reads release the interpreter lock)
        from collections import deque
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=2) as readers:
            ahead = deque()
            it = iter(mine)
            for f in it:
                ahead.append(readers.submit(_plan_file, f, args, folder))
                if len(ahead) < 4:
                    continue
                j = ahead.popleft().result()
                if j is not None:
                    yield j
            while ahead:
                j = ahead.popleft().result()
                if j is not None:
                    yield j

    t0 = time.time()
    names = sched.run(jobs())
    if os.environ.get("GPPD_CLI_TIMING"):     # tools/night_cli.py: the night without interpreter start-up
        import json
        print(json.dumps({"files_written": len(names), "run_seconds": time.time() - t0,
                          "main_thread_seconds": {"waiting_for_planned_files": sched.t_plan,
                                                  "wait_results_and_request_write": sched.t_finish,
                                                  "submit": sched.t_submit}}), file=sys.stderr)
    return 0


if __name__ == "__main__":
    sys.exit(main())
