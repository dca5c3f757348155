"""The table entry points of include/gppd.h held against each other, output for output, and
the status each entry point returns for the option combinations no path runs.

One seeded table, bright and FAINT, runs through gppd_process_table_f32, gppd_submit_table_f32
(slot 3), gppd_submit_fits_rows (big-endian 332-byte records), gppd_file_submit / _wait / _write
(a FITS file), gppd_process_table_f32_dev and gppd_process_tables_f32_dev (next to a table of
the other kind, so that the FAINT and bright chains run side by side).  They share one staging
and launch sequence, so every output must be the same bytes: demodulated VOLT, params, chi2,
info, states and the fitted centres or ellipses."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import make_case

N = 3000
REC = 332                   # TIME (1J) + VOLT (80E) + POWER_LASER (1E) + LAMBDA_LASER (1E)
OK, ERR_ARG, ERR_UNSUPPORTED = 0, 1, 5


@pytest.fixture(scope="module")
def tables(gp, ora):
    return {"bright": make_case(gp.synthetic, N, k=81), "faint": make_case(gp.synthetic, N, k=82, faint=True, ora=ora)}


@pytest.fixture(scope="module")
def fits_files(gp, tables, tmp_path_factory):
    d = tmp_path_factory.mktemp("entry_points")
    return {kind: gp.synthetic.make_fits(str(d / (kind + ".fits")), tab, tab["header"]) for kind, tab in tables.items()}


class Case:
    """One table and one mode, with the host arguments every entry point shares."""

    def __init__(self, gp, tab, offsets, window, keepraw, flags=0, mask=0, n=None):
        self.gp, self.L, self.h = gp, gp._lib.lib(), gp.default_handle()
        self.tab, self.n = tab, N if n is None else n
        self.tu, self.volt, self.mjd = tab["time_us"], tab["volt"], tab["mjd"]
        self.window = window
        self.empirical = offsets is True
        self.ellipse = isinstance(offsets, str) and offsets == "ellipse"
        self.stefan = None if offsets is None or self.empirical or self.ellipse else \
            np.ascontiguousarray(offsets, dtype=np.complex128).view(np.float64)
        self.o = gp.api._options(keepraw=keepraw, empirical=self.empirical, ellipse=self.ellipse)
        self.o.flags |= flags
        self.o.group_mask = mask
        fs = tab["faintstates"]
        self.t1 = None if fs is None else np.ascontiguousarray(fs.timer1, dtype=np.float64)
        self.t2 = None if fs is None else np.ascontiguousarray(fs.timer2, dtype=np.float64)
        self.wrows, self.nwin = gp.table_windows(self.tu, self.mjd, window)
        self.nf = 144 if keepraw else 80

    def timers(self):
        p = self.gp._lib.ptr
        return (p(self.t1), 0 if self.t1 is None else self.t1.size, p(self.t2), 0 if self.t2 is None else self.t2.size)

    def results(self):
        nfits = self.nwin * 32
        return dict(params=np.zeros((nfits, 6)), chi2=np.zeros(nfits),
                    info=np.zeros((nfits, 4), dtype=np.int32),
                    state=np.zeros(self.n, dtype=np.int8) if self.t1 is not None else None)

    def extra(self, slot, ntables=1, index=0):
        """the centres / ellipses the last call on `slot` fitted, as bytes"""
        _lib = self.gp._lib
        if self.empirical:
            c = np.empty((ntables, 40), dtype=np.complex128)
            _lib.check(self.L.gppd_centres(self.h.raw, slot, ntables, _lib.ptr(c.view(np.float64))))
            return c[index].tobytes()
        if self.ellipse:
            e, st = self.gp.ellipses(self.h, slot, ntables)
            return e[index].tobytes() + st[index].tobytes()
        return b""


def _host_table(c, slot=None):
    """gppd_process_table_f32 (slot None) or gppd_submit_table_f32 on `slot` + gppd_wait"""
    _lib = c.gp._lib
    r = c.results()
    vout = np.zeros((c.n, c.nf), dtype=np.float32)
    args = (c.n, _lib.ptr(c.tu, _lib._i32p), c.mjd, _lib.ptr(c.volt, _lib._fp), _lib.ptr(c.stefan)) + c.timers() + (
        float(c.window or 0.0), C.byref(c.o), _lib.ptr(vout, _lib._fp), _lib.ptr(r["params"]), _lib.ptr(r["chi2"]),
        _lib.ptr(r["info"], _lib._i32p), _lib.ptr(r["state"], _lib._i8p))
    if slot is None:
        rc = c.L.gppd_process_table_f32(c.h.raw, *args)
        slot = 0
    else:
        rc = c.L.gppd_submit_table_f32(c.h.raw, slot, *args)
        if rc == OK:
            rc = c.L.gppd_wait(c.h.raw, slot)
    return rc, dict(r, volt=vout, extra=c.extra(slot) if rc == OK else None)


def _records(c):
    rng = np.random.default_rng(5)
    rec = rng.integers(0, 256, size=(c.n, REC), dtype=np.uint8)
    rec[:, 0:4] = c.tu[:c.n].astype(">i4").view(np.uint8).reshape(c.n, 4)
    rec[:, 4:324] = c.volt[:c.n].astype(">f4").view(np.uint8).reshape(c.n, 320)
    return rec


def _volt_of_records(c, out, rec):
    """VOLT (native float32) of the output records; the other fields must pass through"""
    rb = REC + 4 * (c.nf - 80)
    out = np.asarray(out).reshape(c.n, rb)
    assert np.array_equal(out[:, :4], rec[:, :4]) and np.array_equal(out[:, 4 + 4 * c.nf:], rec[:, 324:])
    return out[:, 4:4 + 4 * c.nf].copy().view(">f4").astype(np.float32)


def _fits_rows(c, slot=5):
    _lib = c.gp._lib
    rec = _records(c)
    r = c.results()
    out = np.zeros(c.n * (REC + 4 * (c.nf - 80)), dtype=np.uint8)
    rc = c.L.gppd_submit_fits_rows(
        c.h.raw, slot, c.n, rec.ctypes.data_as(C.c_void_p), REC, 0, 4, c.mjd, _lib.ptr(c.stefan), *c.timers(),
        float(c.window or 0.0), C.byref(c.o), out.ctypes.data_as(C.c_void_p), _lib.ptr(r["params"]),
        _lib.ptr(r["chi2"]), _lib.ptr(r["info"], _lib._i32p), _lib.ptr(r["state"], _lib._i8p))
    if rc == OK:
        rc = c.L.gppd_wait(c.h.raw, slot)
    if rc != OK:
        return rc, None
    return rc, dict(r, volt=_volt_of_records(c, out, rec), extra=c.extra(slot))


def _file(c, path, tmp_path, slot=6):
    """gppd_file_submit / gppd_file_wait / gppd_file_write; the status is the first that is not OK"""
    from gppd_b200 import fits
    _lib = c.gp._lib
    met = fits.scan_fits(path)[3]
    rc = c.L.gppd_file_submit(c.h.raw, slot, os.fsencode(path), met.data_offset, c.n, REC, 0, 4, c.mjd,
                              _lib.ptr(c.stefan), *c.timers(), float(c.window or 0.0), C.byref(c.o))
    if rc != OK:
        return rc, None
    r = c.results()
    rc = c.L.gppd_file_wait(c.h.raw, slot, _lib.ptr(r["params"]), _lib.ptr(r["chi2"]),
                            _lib.ptr(r["info"], _lib._i32p), _lib.ptr(r["state"], _lib._i8p))
    if rc != OK:
        assert c.L.gppd_file_drain(c.h.raw) == rc and c.L.gppd_file_drain(c.h.raw) == OK
        return rc, None
    extra = c.extra(slot)
    seg = (_lib.FileSegment * 1)()
    seg[0].kind = _lib.SEG_RECORDS
    out_path = str(tmp_path / "out.fits")
    _lib.check(c.L.gppd_file_write(c.h.raw, slot, os.fsencode(out_path), seg, 1, None, 0))
    _lib.check(c.L.gppd_file_drain(c.h.raw))
    rb = REC + 4 * (c.nf - 80)
    out = np.frombuffer(open(out_path, "rb").read(), dtype=np.uint8)
    assert out.size == (c.n * rb + 2879) // 2880 * 2880
    src = np.frombuffer(open(path, "rb").read(), dtype=np.uint8)[met.data_offset:met.data_offset + c.n * REC]
    return rc, dict(r, volt=_volt_of_records(c, out[:c.n * rb], src.reshape(c.n, REC)), extra=extra)


def _dev(c, other=None, slot=2):
    """gppd_process_table_f32_dev (other None) or gppd_process_tables_f32_dev on [table, other]"""
    import torch
    _lib = c.gp._lib
    dev = torch.device("cuda", c.h.device)
    cases = [c] if other is None else [c, other]
    T = len(cases)
    d = [dict(time=torch.from_numpy(x.tu[:x.n].copy()).to(dev), volt=torch.from_numpy(x.volt[:x.n].copy()).to(dev),
              out=torch.zeros((x.n, x.nf), dtype=torch.float32, device=dev),
              params=torch.zeros((x.nwin * 32, 6), dtype=torch.float64, device=dev),
              chi2=torch.zeros(x.nwin * 32, dtype=torch.float64, device=dev),
              info=torch.zeros((x.nwin * 32, 4), dtype=torch.int32, device=dev),
              state=torch.zeros(x.n, dtype=torch.int8, device=dev)) for x in cases]
    d_off = None if c.stefan is None else torch.from_numpy(c.stefan.copy()).to(dev)
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())
    torch.cuda.synchronize(dev)
    if other is None:
        rc = c.L.gppd_process_table_f32_dev(
            c.h.raw, slot, None, c.n, c.wrows, p(d[0]["time"]), c.mjd, p(d[0]["volt"]), p(d_off), *c.timers(),
            C.byref(c.o), p(d[0]["out"]), p(d[0]["params"]), p(d[0]["chi2"]), p(d[0]["info"]), p(d[0]["state"]))
    else:
        vp = lambda k: (C.c_void_p * T)(*[x[k].data_ptr() for x in d])
        i64 = lambda v: (C.c_int64 * T)(*v)
        dpp = lambda arrs: (_lib._dp * T)(*[C.cast(None, _lib._dp) if a is None else _lib.ptr(a) for a in arrs])
        rc = c.L.gppd_process_tables_f32_dev(
            c.h.raw, slot, None, T, i64([x.n for x in cases]), i64([x.wrows for x in cases]), vp("time"),
            (C.c_double * T)(*[x.mjd for x in cases]), vp("volt"), p(d_off), dpp([x.t1 for x in cases]),
            i64([0 if x.t1 is None else x.t1.size for x in cases]), dpp([x.t2 for x in cases]),
            i64([0 if x.t2 is None else x.t2.size for x in cases]), C.byref(c.o), vp("out"), vp("params"),
            vp("chi2"), vp("info"), vp("state"))
    if rc == OK:
        rc = c.L.gppd_wait(c.h.raw, slot)
    if rc != OK:
        return rc, None
    r = {k: v.cpu().numpy() for k, v in d[0].items() if k in ("params", "chi2", "info", "state")}
    if c.t1 is None:
        r["state"] = None
    return rc, dict(r, volt=d[0]["out"].cpu().numpy(), extra=c.extra(slot, T, 0))


def _entry_points(c, path, tmp_path, other):
    yield "gppd_submit_table_f32", _host_table(c, slot=3)
    yield "gppd_submit_fits_rows", _fits_rows(c)
    yield "gppd_file_*", _file(c, path, tmp_path)
    yield "gppd_process_table_f32_dev", _dev(c)
    yield "gppd_process_tables_f32_dev", _dev(c, other=other, slot=4)


def _offsets(gp, name):
    return {"stefan": gp.synthetic.stefan_centres(), "fit": None, "empirical": True, "ellipse": "ellipse"}[name]


@pytest.mark.gpu
@pytest.mark.parametrize("keepraw", [False, True])
@pytest.mark.parametrize("window", [None, 1.0])
@pytest.mark.parametrize("offsets", ["stefan", "fit", "empirical", "ellipse"])
@pytest.mark.parametrize("kind", ["bright", "faint"])
def test_table_entry_points_agree(gp, tables, fits_files, tmp_path, kind, offsets, window, keepraw):
    c = Case(gp, tables[kind], _offsets(gp, offsets), window, keepraw)
    other = Case(gp, tables["faint" if kind == "bright" else "bright"], _offsets(gp, offsets), window, keepraw)
    rc, ref = _host_table(c)
    assert rc == OK
    assert (ref["state"] is not None) == (kind == "faint") and (ref["extra"] != b"") == (offsets in ("empirical", "ellipse"))
    assert np.isfinite(ref["params"]).all() and ref["volt"].shape == (N, 144 if keepraw else 80)
    for name, (rc, got) in _entry_points(c, fits_files[kind], tmp_path, other):
        assert rc == OK, name
        for k in ("volt", "params", "chi2", "info"):
            assert got[k].tobytes() == ref[k].tobytes(), (name, k)
        assert (got["state"] is None) == (ref["state"] is None), name
        if ref["state"] is not None:
            assert got["state"].tobytes() == ref["state"].tobytes(), name
        assert got["extra"] == ref["extra"], name


@pytest.mark.gpu
@pytest.mark.parametrize("nwindow", [0, 700])
@pytest.mark.parametrize("fitoffsets", [False, True])
@pytest.mark.parametrize("kind", ["bright", "faint"])
def test_array_entry_points_agree(gp, tables, kind, fitoffsets, nwindow):
    import torch
    tab = tables[kind]
    t, z = gp.synthetic.to_complex(tab, None if fitoffsets else gp.synthetic.stefan_centres())
    state = tab["state"]
    out, params, chi2, info = gp.demodulateall(t, z, faintparam=state, fitoffsets=fitoffsets, raw=True,
                                               nwindow=nwindow, return_info=True)
    L, h = gp._lib.lib(), gp.default_handle()
    dev = torch.device("cuda", h.device)
    nfits = params.shape[0]
    d_t, d_z = torch.from_numpy(t).to(dev), torch.from_numpy(np.ascontiguousarray(z.T)).to(dev)
    d_s = None if state is None else torch.from_numpy(state).to(dev)
    d_o = torch.zeros_like(d_z)
    d_p = torch.zeros((nfits, 6), dtype=torch.float64, device=dev)
    d_c = torch.zeros(nfits, dtype=torch.float64, device=dev)
    d_i = torch.zeros((nfits, 4), dtype=torch.int32, device=dev)
    o = gp.api._options(fitoffsets=fitoffsets)
    p = lambda x: None if x is None else C.c_void_p(x.data_ptr())
    torch.cuda.synchronize(dev)
    gp._lib.check(L.gppd_demodulate_f64_dev(h.raw, 1, None, N, nwindow, p(d_t), p(d_z), p(d_s), C.byref(o),
                                            p(d_o), p(d_p), p(d_c), p(d_i)))
    gp._lib.check(L.gppd_wait(h.raw, 1))
    assert d_o.cpu().numpy().T.tobytes() == np.ascontiguousarray(out).tobytes()
    assert d_p.cpu().numpy().tobytes() == params.tobytes() and d_c.cpu().numpy().tobytes() == chi2.tobytes()
    assert d_i.cpu().numpy().tobytes() == info.tobytes()


def _array_status(gp, tab, flags, mask, n, dev):
    """(gppd_demodulate_f64, gppd_demodulate_f64_dev) status"""
    import torch
    L, h, _lib = gp._lib.lib(), gp.default_handle(), gp._lib
    t, z = gp.synthetic.to_complex(tab)
    zt = np.ascontiguousarray(z.T)
    o = _lib.Options()
    o.flags, o.group_mask = flags, mask
    out = np.empty_like(zt)
    par, chi2 = np.empty((32, 6)), np.empty(32)
    rc_host = L.gppd_demodulate_f64(h.raw, n, 0, _lib.ptr(t), _lib.ptr(zt.view(np.float64)), None, C.byref(o),
                                    _lib.ptr(out.view(np.float64)), _lib.ptr(par), _lib.ptr(chi2), None, None)
    d_t, d_z = torch.from_numpy(t).to(dev), torch.from_numpy(zt).to(dev)
    d_o, d_p, d_c = torch.empty_like(d_z), torch.empty((32, 6), dtype=torch.float64, device=dev), \
        torch.empty(32, dtype=torch.float64, device=dev)
    p = lambda x: C.c_void_p(x.data_ptr())
    torch.cuda.synchronize(dev)
    rc_dev = L.gppd_demodulate_f64_dev(h.raw, 1, None, n, 0, p(d_t), p(d_z), None, C.byref(o), p(d_o), p(d_p),
                                       p(d_c), None)
    L.gppd_wait(h.raw, 1)
    return rc_host, rc_dev


# name: (flags, group_mask, n, status of every table entry point, of both array entry points)
ERRORS = {
    "ellipse_fitoffsets": (128 | 2, 0, N, ERR_ARG, ERR_UNSUPPORTED),
    "ellipse_empirical": (128 | 32, 0, N, ERR_ARG, ERR_UNSUPPORTED),
    "ellipse_empirical_partial_mask": (128 | 32, 0x0f, N, ERR_ARG, ERR_UNSUPPORTED),
    "ellipse_partial_mask": (128, 0x0f, N, ERR_UNSUPPORTED, ERR_UNSUPPORTED),
    "partial_mask": (0, 0x0f, N, ERR_UNSUPPORTED, OK),
    "ellipse": (128, 0, N, OK, ERR_UNSUPPORTED),
    "empirical_fitoffsets": (32 | 2, 0, N, OK, ERR_ARG),
    "empirical": (32, 0, N, OK, ERR_ARG),
    "one_row": (0, 0, 1, ERR_ARG, ERR_ARG),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(ERRORS))
def test_entry_point_status(gp, tables, fits_files, tmp_path, case):
    import torch
    flags, mask, n, want_table, want_arrays = ERRORS[case]
    tab, other = tables["faint"], tables["bright"]
    c = Case(gp, tab, None, None, False, flags=flags, mask=mask, n=n)
    o = Case(gp, other, None, None, False, flags=flags, mask=mask)
    got = {"gppd_process_table_f32": _host_table(c)[0]}
    got.update((name, res[0]) for name, res in _entry_points(c, fits_files["faint"], tmp_path, o))
    assert got == {k: want_table for k in got}, case
    assert _array_status(gp, tab, flags, mask, n, torch.device("cuda", c.h.device)) == (want_arrays, want_arrays), case
