#!/usr/bin/env python
"""Regenerates tests/golden/golden_small.npz.

PROVENANCE: the reference (Julia + OptimPackNextGen) cannot run in this image and ships
no test vectors, so these are outputs of the in-repo CPU oracle (oracle/, a restatement
of the reference's algorithm), frozen so that later edits of the oracle or of the
synthetic generator cannot drift unnoticed, and so that the GPU path has fixed vectors
to be compared with.  They pin the oracle to itself, not to the reference ("parity
unpinned", DESIGN.md section 2).

    python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import gppd_b200 as gp
    import oracle
    from conftest import make_case
    oracle.build()
    out = {}
    off = gp.synthetic.stefan_centres()
    for name, faint in (("bright", False), ("faint", True)):
        tab = make_case(gp.synthetic, SMALL_ROWS, k=SMALL_SEEDS[name], faint=faint, ora=oracle)
        t, z = gp.synthetic.to_complex(tab, off)
        st = tab["state"]
        assert np.array_equal(input_digest(small_inputs(gp, name, st)), input_digest(tab))
        o, p, l = oracle.demodulateall(t, z, faintparam=st, nthreads=8)
        out[f"{name}_sha256"] = input_digest(tab)
        if faint:
            out["faint_state"] = st.astype(np.int8)
            out["faint_timer1"] = tab["faintstates"].timer1
            out["faint_timer2"] = tab["faintstates"].timer2
        out[f"{name}_params"] = p            # (32, 6): c.re, c.im, a.re, a.im, b, phi (b >= 0)
        out[f"{name}_chi2"] = l
        out[f"{name}_output"] = o[:, :32].astype(np.complex64)   # float32 like the VOLT column
        # objective values on a fixed grid (independent of any solver trajectory)
        grid = [(0.1, -1.0), (0.7, 0.3), (1.9, 2.5), (-2.4, -0.2), (4.9, 3.0), (5.5, 1.0)]
        vals = np.empty((32, len(grid)))
        for ch in range(32):
            fc = np.exp(1j * np.angle(z[:, 32 + ch // 4]))
            w = pw = None
            if faint:
                pw, w = oracle.compute_mean_var_power(st, z[:, ch])
            for g, (b, phi) in enumerate(grid):
                vals[ch, g] = oracle.chi2(t, z[:, ch], fc, b, phi, weight=w, power=pw)[0]
        out[f"{name}_grid"] = np.array(grid)
        out[f"{name}_grid_chi2"] = vals
    path = os.path.join(ROOT, "tests", "golden", "golden_small.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")
    full = full_size_vectors(gp, oracle, make_case)
    path = os.path.join(ROOT, "tests", "golden", "golden_1e5.npz")
    np.savez_compressed(path, **full)
    print(path, os.path.getsize(path), "bytes")


SMALL_ROWS = 1000
SMALL_SEEDS = {"bright": 76, "faint": 77}
FULL_ROWS = 100_000
FULL_STRIDE = 1009          # rows of the output kept in the file


def small_inputs(gp, name, state=None):
    """The 1000-row bright / FAINT tables of golden_small.npz, rebuilt from the seeded
    generator (the file keeps their SHA-256 and the FAINT states, not the tables)."""
    return gp.synthetic.make_table(SMALL_ROWS, k=SMALL_SEEDS[name], faint=state is not None, state=state)


def full_size_inputs(gp, oracle, make_case, name):
    """BASELINE.json configs 1 / 2: one bright and one FAINT table of 1e5 rows (seeded
    generator: the inputs are not stored, only their SHA-256)."""
    faint = name == "faint"
    tab = make_case(gp.synthetic, FULL_ROWS, k=43 if faint else 41, faint=faint, jitter=True, ora=oracle)
    t, z = gp.synthetic.to_complex(tab, gp.synthetic.stefan_centres())
    return tab, t, z


def input_digest(tab):
    import hashlib
    h = hashlib.sha256()
    h.update(np.ascontiguousarray(tab["time_us"]).tobytes())
    h.update(np.ascontiguousarray(tab["volt"]).tobytes())
    return np.frombuffer(h.digest(), dtype=np.uint8)


def full_size_vectors(gp, oracle, make_case):
    out = {}
    for name in ("bright", "faint"):
        tab, t, z = full_size_inputs(gp, oracle, make_case, name)
        o, p, l, nf = oracle.demodulateall(t, z, faintparam=tab["state"], nthreads=8, return_nfev=True)
        out[f"{name}_sha256"] = input_digest(tab)
        out[f"{name}_params"] = p
        out[f"{name}_chi2"] = l
        out[f"{name}_nfev"] = nf
        out[f"{name}_output"] = o[::FULL_STRIDE, :32].astype(np.complex64)
        if name == "faint":     # run-length form of the segmentation
            st = tab["state"]
            chg = np.flatnonzero(np.diff(st)) + 1
            out["faint_state_starts"] = np.concatenate([[0], chg]).astype(np.int32)
            out["faint_state_values"] = st[out["faint_state_starts"]].astype(np.int8)
    return out


if __name__ == "__main__":
    main()
