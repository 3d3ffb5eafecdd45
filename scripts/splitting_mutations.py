"""Mutation check of the parking-rollout tests: build the library with one deliberate defect in rollout_until_kernel and show
that tests/test_gpu_splitting.py fails on it.

    python scripts/splitting_mutations.py [--out FILE]

Mutants (each built in a temporary directory from a copy of cavgym_b200/csrc: until_m2.cu recompiled, linked with the other
objects of the in-tree build, loaded through CAVGYM_LIB; the tests run on the two-body pedestrians):
  score_not_read          the score starts at -inf instead of the caller's value;
  parked_steps_once_more  an env that reaches the level takes one more step before it parks;
  salt_ignored            a non-zero salt draws on the engine's own streams;
  final_danger_counted    the danger of a step that ends the episode without a tester win enters the score.
All four are logic defects: no index or trap changes.  A mutant is caught when pytest fails; the first failing test is
reported.  Needs the in-tree build (build() first) and a GPU.
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

MUTANTS = {
    "score_not_read": ("R s = score[e];", "R s = R(-INFINITY);"),
    "parked_steps_once_more": ("      if ((double)s >= level) { st = UNTIL_PARKED; break; }\n",
                               "      if (st == UNTIL_PARKED) break;\n      if ((double)s >= level) st = UNTIL_PARKED;\n"),
    "salt_ignored": ("  if (salt != 0) buf.seed ^= splitmix64(salt);\n", ""),
    "final_danger_counted": ("        else st = UNTIL_FINISHED;\n",
                             "        else { s = rmax(s, danger<R, M, GENERIC>(sc, env)); st = UNTIL_FINISHED; }\n"),
}
UNITS = ("until_m2",)


def build_mutant(name, work):
    tree = os.path.join(work, name)
    shutil.copytree(os.path.join(ROOT, "cavgym_b200", "csrc"), os.path.join(tree, "cavgym_b200", "csrc"),
                    ignore=shutil.ignore_patterns("build", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    csrc = os.path.join(tree, "cavgym_b200", "csrc")
    path = os.path.join(csrc, "kernels_until.cuh")
    old, new = MUTANTS[name]
    text = open(path).read()
    if text.count(old) != 1:
        raise RuntimeError(f"{name}: the code to mutate is not there exactly once: {old}")
    open(path, "w").write(text.replace(old, new))
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
    proc = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider", "tests/test_gpu_splitting.py",
                           "-k", "homogeneous_2_bodies or salt"],
                          cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
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
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    return 0 if all(" caught " in line for line in lines) else 1


if __name__ == "__main__":
    sys.exit(main())
