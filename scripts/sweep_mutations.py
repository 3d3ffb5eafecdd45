"""Mutation check of the per-env tester parameter tests: build the library with one deliberate defect in the parameter kernels
(kernels_params.cuh) and show that tests/test_gpu_agent_params.py fails on it.

    python scripts/sweep_mutations.py [--out FILE]

Mutants (each built in a temporary directory from a copy of cavgym_b200/csrc: params_m2.cu recompiled, linked with the other
objects of the in-tree build, loaded through CAVGYM_LIB; the tests run on the two-body pedestrians scenarios):
  row_of_previous_body   body b reads row b - 1 of both arrays (body 0 reads row 0);
  next_env               slot e reads slot e + 1's parameters (the last slot its own);
  threshold_from_epsilon the threshold is read from the epsilon array (the scenario's value where that is unset);
  step_ignores           the step kernel takes the scenario's values;
  record_ignores         the recording kernel takes the scenario's values.
A sixth defect the issue lists, ghost lanes reading slot hi, is not built: a ghost lane steps a copy of env hi - 1 with every
side effect switched off (no store, no counter, no episode row, no record row), so which parameters it reads cannot change
anything a caller or a test can observe.  A mutant is caught when pytest fails; the first failing test is reported.  Needs the
in-tree build (build() first) and a GPU.
"""
import argparse
import concurrent.futures
import os
import re
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cavgym_b200.csrc import build  # noqa: E402

STEP = ("advance<R, M, true, GENERIC, NoPhase, EnvTester<R>>(sc, buf, io, e, t_global, env, ext, NoPhase(), false, nullptr, "
        "EnvTester<R>{params});")
RECORD = "advance<R, M, true, GENERIC, Phase, EnvTester<R>>(sc, buf, at, e, t_global + t, env, ext, phase, ghost, nullptr, tester);"
MUTANTS = {
    "row_of_previous_body": [("p.epsilon[(int64_t)b * n + e]", "p.epsilon[(int64_t)(b > 0 ? b - 1 : 0) * n + e]"),
                             ("p.threshold[(int64_t)b * n + e]", "p.threshold[(int64_t)(b > 0 ? b - 1 : 0) * n + e]")],
    "next_env": [("p.epsilon[(int64_t)b * n + e]", "p.epsilon[(int64_t)b * n + (e + 1 < n ? e + 1 : e)]"),
                 ("p.threshold[(int64_t)b * n + e]", "p.threshold[(int64_t)b * n + (e + 1 < n ? e + 1 : e)]")],
    "threshold_from_epsilon": [("return p.threshold ? p.threshold[(int64_t)b * n + e] : body.threshold;",
                                "return p.epsilon ? R(p.epsilon[(int64_t)b * n + e]) : body.threshold;")],
    "step_ignores": [(STEP, "advance<R, M, true, GENERIC>(sc, buf, io, e, t_global, env, ext);")],
    "record_ignores": [(RECORD, "advance<R, M, true, GENERIC, Phase>(sc, buf, at, e, t_global + t, env, ext, phase, ghost);")],
}
UNITS = ("params_m2",)
TESTS = "pedestrians_rc_seed0 or pedestrians_proximity_seed3 or rc_pedestrians or proximity"


def build_mutant(name, work):
    tree = os.path.join(work, name)
    shutil.copytree(os.path.join(ROOT, "cavgym_b200", "csrc"), os.path.join(tree, "cavgym_b200", "csrc"),
                    ignore=shutil.ignore_patterns("build", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    csrc = os.path.join(tree, "cavgym_b200", "csrc")
    path = os.path.join(csrc, "kernels_params.cuh")
    text = open(path).read()
    for old, new in MUTANTS[name]:
        if text.count(old) != 1:
            raise RuntimeError(f"{name}: the code to mutate is not there exactly once: {old}")
        text = text.replace(old, new)
    open(path, "w").write(text)
    objs = [os.path.join(tree, unit + ".o") for unit in UNITS]
    for unit, obj in zip(UNITS, objs):
        proc = subprocess.run([build.NVCC] + build.FLAGS + ["-c", os.path.join(csrc, unit + ".cu"), "-o", obj], capture_output=True, text=True)
        if proc.returncode:
            raise RuntimeError(f"{name}: {proc.stderr[-2000:]}")
    others = sorted(os.path.join(build.OBJ_DIR, f) for f in os.listdir(build.OBJ_DIR)
                    if f.endswith(".o") and f[:-2] not in UNITS and not f.endswith(".stub.o"))
    lib = os.path.join(tree, "libcavgym_sm100.so")
    proc = subprocess.run([build.NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs + others
                          + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"], capture_output=True, text=True)
    if proc.returncode:
        raise RuntimeError(f"{name}: {proc.stderr[-2000:]}")
    return lib


def run_tests(lib):
    env = dict(os.environ, CAVGYM_LIB=lib)
    proc = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider", "tests/test_gpu_agent_params.py",
                           "-k", TESTS], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    failed = re.findall(r"^FAILED (\S+)", proc.stdout, flags=re.M)
    where = re.findall(r"^E\s+(.*)$", proc.stdout, flags=re.M)
    return proc.returncode, (failed[0] if failed else ""), (where[0].strip()[:160] if where else "")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report here")
    args = ap.parse_args()
    names = list(MUTANTS)
    lines = []
    with tempfile.TemporaryDirectory() as work:
        with concurrent.futures.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as pool:
            libs = dict(zip(names, pool.map(lambda n: build_mutant(n, work), names)))
        for name in names:
            rc, failed, where = run_tests(libs[name])
            line = f"{name:26s} {'caught' if rc == 1 else 'NOT CAUGHT' if rc == 0 else f'pytest exit {rc}'}  {failed}  | {where}"
            print(line, flush=True)
            lines.append(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    return 0 if all(" caught " in line for line in lines) else 1


if __name__ == "__main__":
    sys.exit(main())
