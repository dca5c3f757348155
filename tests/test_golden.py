"""Committed golden vectors (tests/golden/golden_small.npz, written by
tests/golden/make_golden.py from the CPU oracle -- the reference itself cannot run
here, see the script's header): the oracle must keep reproducing them bit for bit, and
the CUDA path is compared with them without any oracle call at run time.  The input
tables come from the seeded generator and are checked against the SHA-256 stored with
the vectors."""
import os
import sys

import numpy as np
import pytest

import fitref
from conftest import make_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_golden  # noqa: E402


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "golden_small.npz"))


def _inputs(gp, golden, name):
    st = golden["faint_state"] if name == "faint" else None
    tab = make_golden.small_inputs(gp, name, st)
    assert np.array_equal(make_golden.input_digest(tab), golden[f"{name}_sha256"]), "generator drifted"
    t, z = gp.synthetic.to_complex(tab, gp.synthetic.stefan_centres())
    return tab, t, z, st


@pytest.mark.parametrize("name", ["bright", "faint"])
def test_oracle_reproduces_golden(gp, ora, golden, name):
    tab, t, z, st = _inputs(gp, golden, name)
    if st is not None:      # segmentation is integer work: bit-exact
        fs = ora.FaintStates(golden["faint_timer1"], golden["faint_timer2"], 1.0, 2.0)
        assert np.array_equal(ora.buildstates(fs, t), st)
    o, p, l = ora.demodulateall(t, z, faintparam=st, nthreads=8)
    assert p.tobytes() == golden[f"{name}_params"].tobytes()
    assert l.tobytes() == golden[f"{name}_chi2"].tobytes()
    assert np.array_equal(o[:, :32].astype(np.complex64), golden[f"{name}_output"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bright", "faint"])
def test_gpu_against_golden(gp, golden, name):
    tab, t, z, st = _inputs(gp, golden, name)
    if st is not None:
        fs = gp.FaintStates(golden["faint_timer1"], golden["faint_timer2"], 1.0, 2.0)
        assert np.array_equal(gp.buildstates(fs, t), st)                 # bit-exact
    # objective parity on the fixed grid: one objective call at the start vector
    # (maxfun = 1 stops NEWUOA after its first evaluation); b = 5.5 is outside the harmonic
    # evaluator's range and goes through the fallback queue
    for g, (b, phi) in enumerate(golden[f"{name}_grid"]):
        _, _, _, info, trace = gp.demodulateall(t, z, faintparam=st, init=[b, phi], maxfun=1, raw=True,
                                                return_info=True, return_trace=True)
        f = trace[:, 0, 2]
        ref = golden[f"{name}_grid_chi2"][:, g]
        assert np.all(trace[:, 0, 0] == b) and np.all(trace[:, 0, 1] == phi)
        assert np.abs(f - ref).max() <= 1e-10 * np.abs(ref).max(), (b, phi)
        assert np.all(info[:, 2] == (1 if abs(b) > 5 else 2))
    # end to end: fits on the oracle's trajectory agree to 1e-9, the others within the
    # solver's stopping tolerance (DESIGN.md section 2)
    out, par, like = gp.demodulateall(t, z, faintparam=st, raw=True)
    gpar = golden[f"{name}_params"]
    same, stats = fitref.compare_fits(par, like, gpar, golden[f"{name}_chi2"])
    assert same.sum() >= fitref.MIN_COINCIDE
    assert np.abs(par[same][:, 2:6] - gpar[same][:, 2:6]).max() <= 1e-9 * np.abs(gpar[:, 2:6]).max()
    assert np.abs(like[same] - golden[f"{name}_chi2"][same]).max() <= 1e-9 * golden[f"{name}_chi2"].max()
    gout = golden[f"{name}_output"]
    err = np.abs(out[:, :32].astype(np.complex64) - gout).max(axis=0) / np.abs(gout).max(axis=0)
    assert err[same].max() <= 2.0 ** -22
    assert err.max() <= 4 * fitref.FORK_HARD


# ---- BASELINE-size vectors (1e5 rows): tests/golden/golden_1e5.npz ---------------------
@pytest.fixture(scope="module")
def golden_full():
    return np.load(os.path.join(ROOT, "tests", "golden", "golden_1e5.npz"))


def _full_inputs(gp, ora, name):
    return make_golden, make_golden.full_size_inputs(gp, ora, make_case, name)


@pytest.mark.parametrize("name", ["bright", "faint"])
def test_oracle_reproduces_golden_full_size(gp, ora, golden_full, name):
    mg, (tab, t, z) = _full_inputs(gp, ora, name)
    assert np.array_equal(mg.input_digest(tab), golden_full[f"{name}_sha256"]), "generator drifted"
    if name == "faint":
        st = tab["state"]
        starts = golden_full["faint_state_starts"]
        assert np.array_equal(np.concatenate([[0], np.flatnonzero(np.diff(st)) + 1]), starts)
        assert np.array_equal(st[starts], golden_full["faint_state_values"])
    o, p, l, nf = ora.demodulateall(t, z, faintparam=tab["state"], nthreads=8, return_nfev=True)
    assert p.tobytes() == golden_full[f"{name}_params"].tobytes()
    assert l.tobytes() == golden_full[f"{name}_chi2"].tobytes()
    assert np.array_equal(nf, golden_full[f"{name}_nfev"])
    assert np.array_equal(o[::mg.FULL_STRIDE, :32].astype(np.complex64), golden_full[f"{name}_output"])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["bright", "faint"])
def test_gpu_against_golden_full_size(gp, ora, golden_full, name):
    """The METROLOGY-table path (the one bench.py times) on a 1e5-row table against the
    committed vectors; no oracle fit at run time (the oracle only rebuilds the FAINT
    states the generator needs)."""
    mg, (tab, t, z) = _full_inputs(gp, ora, name)
    assert np.array_equal(mg.input_digest(tab), golden_full[f"{name}_sha256"]), "generator drifted"
    fs = tab["faintstates"]
    fs_g = gp.FaintStates(fs.timer1, fs.timer2, 1.0, 2.0) if name == "faint" else None
    vout, par, chi2, info, st = gp.process_table(tab["time_us"], tab["volt"], tab["mjd"],
                                                 offsets=gp.synthetic.stefan_centres(), faintparam=fs_g)
    if name == "faint":
        assert np.array_equal(st, tab["state"])
    gpar, gchi = golden_full[f"{name}_params"], golden_full[f"{name}_chi2"]
    same, stats = fitref.compare_fits(par, chi2, gpar, gchi, info[:, 0], golden_full[f"{name}_nfev"])
    print("golden 1e5 %s: forks %d / 32" % (name, stats["forks"]))
    assert same.sum() >= fitref.MIN_COINCIDE
    assert np.abs(par[same][:, 2:6] - gpar[same][:, 2:6]).max() <= 1e-9 * np.abs(gpar[:, 2:6]).max()
    assert (np.abs(chi2 - gchi)[same] <= 1e-9 * gchi[same]).all()
    gout = golden_full[f"{name}_output"]
    got = vout[::mg.FULL_STRIDE, 0:64:2] + 1j * vout[::mg.FULL_STRIDE, 1:64:2]
    err = np.abs(got - gout).max(axis=0) / np.abs(gout).max(axis=0)
    assert err[same].max() <= 2.0 ** -22 and err.max() <= 4 * fitref.FORK_HARD
