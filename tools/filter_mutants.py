"""Mutation check of the sphere filters' error bounds: does the suite notice when a bound is weakened?

For each mutant: copy the tree to a temporary directory, apply one textual change to a bound of the FP32 or the tensor
filter, build there (rtiow_b200/build.py), run tests/test_filter_bypass_gpu.py (and, with --existing, pytest on the given
arguments without that file: the existing suite) and report which tests failed and the differing ray / path / pixel counts
their messages give.  The copy is removed afterwards; every test run is a child process that ends before the next starts.
Needs a B200.

    python tools/filter_mutants.py [--only fp32-slack-0,...] [--existing "tests -m gpu"] [--json out.json]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import shlex
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent

# name -> (file, text, replacement): each text must occur exactly once
MUTANTS = {
    "fp32-slack-0": ("rtiow_b200/csrc/rt_scene.cuh", "#define RT_FILTER_SLACK 5.7220458984375e-06f", "#define RT_FILTER_SLACK 0.0f"),
    "tensor-slack-0": ("rtiow_b200/csrc/capi.cu", "const double slack = 1.5625e-5 * R * R;", "const double slack = 0.0 * R * R;"),
    "sigma-0": ("rtiow_b200/csrc/capi.cu", "sc.filter_sigma = (float)(16.0 * ", "sc.filter_sigma = (float)(0.0 * "),
    "r2-margin-0": ("rtiow_b200/csrc/capi.cu", "(float)(R * R * (1.0 + 1e-6))", "(float)(R * R)"),
    "tensor-slack/16": ("rtiow_b200/csrc/capi.cu", "const double slack = 1.5625e-5 * R * R;", "const double slack = 1.5625e-5 / 16 * R * R;"),
}
NEW_TESTS = "tests/test_filter_bypass_gpu.py"
COUNT = re.compile(r"(\d+) of (\d+) (rays|paths|pixels) differ")


def _copy(dst: Path):
    skip = {".git", "__pycache__", ".pytest_cache"}
    shutil.copytree(ROOT, dst, symlinks=True,
                    ignore=lambda d, names: [n for n in names if n in skip or (Path(d).name == "rtiow_b200" and n == "lib")])


def _pytest(tree: Path, files, timeout):
    env = dict(os.environ, COLUMNS="1000", PYTHONDONTWRITEBYTECODE="1")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", "-rf", *files], cwd=tree, env=env,
                       capture_output=True, text=True, timeout=timeout)
    failed = [ln[len("FAILED "):] for ln in r.stdout.splitlines() if ln.startswith("FAILED ")]
    tail = r.stdout.strip().splitlines()[-1:] or [r.stderr.strip()[-300:]]
    return failed, tail[0]


def _summary(failed):
    """per failed test: its id and the differing count its message reports"""
    out = []
    for f in failed:
        test, _, msg = f.partition(" - ")
        m = COUNT.search(msg)
        out.append({"test": test, "differ": f"{m.group(1)} of {m.group(2)} {m.group(3)}" if m else msg[:160]})
    return out


def run(name, existing, timeout):
    path, old, new = MUTANTS[name]
    with tempfile.TemporaryDirectory(prefix="filter_mutant_") as tmp:
        tree = Path(tmp) / "repo"
        _copy(tree)
        src = tree / path
        text = src.read_text()
        assert text.count(old) == 1, f"{name}: the text to mutate occurs {text.count(old)} times in {path}"
        src.write_text(text.replace(old, new))
        t0 = time.time()
        b = subprocess.run([sys.executable, "-m", "rtiow_b200.build", "--force"], cwd=tree, capture_output=True, text=True, timeout=timeout)
        if b.returncode != 0:
            return {"mutant": name, "error": "build failed: " + (b.stdout + b.stderr)[-2000:]}
        rep = {"mutant": name, "change": f"{path}: {old!r} -> {new!r}"}
        failed, tail = _pytest(tree, [NEW_TESTS], timeout)
        rep["new"] = _summary(failed); rep["new_tail"] = tail
        if existing:
            failed, tail = _pytest(tree, shlex.split(existing) + [f"--ignore={NEW_TESTS}"], timeout)
            rep["existing"] = _summary(failed); rep["existing_tail"] = tail
        rep["seconds"] = round(time.time() - t0, 1)
        return rep


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--only", default=",".join(MUTANTS), help="comma-separated mutant names (default: all)")
    ap.add_argument("--existing", default="", help='pytest arguments of the existing suite to run against each mutant too, e.g. "tests -m gpu"')
    ap.add_argument("--json", help="write the report here as well")
    ap.add_argument("--timeout", type=float, default=1800.0, help="seconds per build / test run")
    a = ap.parse_args()
    reports = []
    for name in a.only.split(","):
        rep = run(name, a.existing, a.timeout)
        reports.append(rep)
        print(f"== {name}  ({rep.get('seconds', '-')} s)  {rep.get('change', '')}")
        if "error" in rep:
            print("   " + rep["error"])
            continue
        for key in ("new", "existing"):
            if key not in rep:
                continue
            print(f"   {key}: {len(rep[key])} failed   [{rep[key + '_tail']}]")
            for f in rep[key]:
                print(f"      {f['test']}: {f['differ']}")
        sys.stdout.flush()
    if a.json:
        Path(a.json).parent.mkdir(parents=True, exist_ok=True)
        Path(a.json).write_text(json.dumps(reports, indent=1))
    missed = [r["mutant"] for r in reports if "new" in r and not r["new"]]
    print("not caught by " + NEW_TESTS + ": " + (", ".join(missed) or "none"))


if __name__ == "__main__":
    main()
