"""BASELINE.json configs[2] through the command line: a synthetic night directory of FITS
files (70 % bright / 30 % FAINT, 1e5 rows each) demodulated recursively by
bin/GPPupilDemodulation (-r), timed end to end (file read, H2D, kernels, D2H, file write).

    python tools/night_cli.py [files] [rows] [base directory]

The base directory defaults to /dev/shm (tmpfs: the code without the box's disk); pass a
directory on a real file system to include it.  Ten distinct tables are generated and copied
under different names (generating 100 takes a minute of NumPy time and changes nothing for
the I/O path)."""
import json, os, sys, time, shutil, subprocess
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import gppd_b200 as gp
import oracle
from conftest import make_case

nfiles = int(sys.argv[1]) if len(sys.argv) > 1 else 100
rows = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000
base = sys.argv[3] if len(sys.argv) > 3 else ("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp")
d = os.path.join(base, "gppd_night"); out = os.path.join(base, "gppd_night_out")
shutil.rmtree(d, ignore_errors=True); shutil.rmtree(out, ignore_errors=True)
t0 = time.time()
made = {}
for k in range(nfiles):
    sub = os.path.join(d, "sub%d" % (k % 4))
    os.makedirs(sub, exist_ok=True)
    path = os.path.join(sub, "GRAVI_%03d.fits" % k)
    if k % 10 in made:
        shutil.copyfile(made[k % 10], path)
        continue
    faint = (k % 10) in (3, 6, 9)
    tab = make_case(gp.synthetic, rows, k=k, faint=faint, ora=oracle)
    gp.synthetic.make_fits(path, tab, tab["header"])
    made[k % 10] = path
tgen = time.time() - t0
res = {"workload": "night directory of %d FITS files x %d rows (30 %% FAINT), bin/GPPupilDemodulation -r" % (nfiles, rows),
       "base_directory": base, "input_gb": nfiles * rows * 332 / 1e9, "generation_seconds": tgen}
env = dict(os.environ, GPPD_CLI_TIMING="1")
for label, extra in (("native", []), ("python_records", ["--no-native"]), ("ellipse", ["-c", "ellipse"])):
    runs, inner, detail = [], [], None
    for _ in range(3):                      # page cache / first-touch effects make single runs noisy
        shutil.rmtree(out, ignore_errors=True)
        t0 = time.time()
        r = subprocess.run([os.path.join(ROOT, "bin", "GPPupilDemodulation"), "-r", "-d", out] + extra + [d],
                           capture_output=True, text=True, env=env)
        runs.append(time.time() - t0)
        for line in r.stderr.splitlines():
            if line.startswith("{") and "run_seconds" in line:
                inner.append(json.loads(line)["run_seconds"])
                detail = json.loads(line).get("main_thread_seconds")
        if r.returncode:
            print(r.stderr[-2000:], file=sys.stderr)
    nout = len(os.listdir(out)) if os.path.isdir(out) else 0
    dt, di = min(runs), (min(inner) if inner else None)
    res[label] = {"files_written": nout, "returncode": r.returncode, "command_seconds": dt,
                  "command_seconds_of_each_run": runs, "night_seconds_inside_the_process": di,
                  "main_thread_seconds_last_run": detail, "files_per_s": nout / dt, "diode_samples_per_s_command": nout * rows * 32 / dt,
                  "diode_samples_per_s_night": (nout * rows * 32 / di) if di else None}
res["note"] = ("command = wall clock of the whole command including interpreter start-up, library load and "
               "CUDA context creation; night = first file submitted to last file written, inside the process. "
               "native: records read / written by the library's I/O threads (gppd_file_*); python_records: "
               "the same files through gppd_submit_fits_rows with Python reading and writing the records; "
               "ellipse: the native path with --center ellipse (offset + ellipse correction per channel)")
print(json.dumps(res))
shutil.rmtree(d, ignore_errors=True); shutil.rmtree(out, ignore_errors=True)
