"""Mutation check of the recorded-rollout tests: build the library with one deliberate defect in rollout_record_kernel and
show that tests/test_gpu_rollout_record.py fails on it.

    python scripts/rollout_record_mutations.py [--out FILE]

Mutants (each built in a temporary directory from a copy of cavgym_b200/csrc: record_m2.cu and record_m5.cu recompiled,
linked with the other objects of the in-tree build, loaded through CAVGYM_LIB; the tests run on the two-body pedestrians
and the five-body bus stop):
  observation_before_reset  the observation row is stored before the auto-reset at the top of the step;
  frozen_rows_skipped       a finished env leaves the loop without auto-reset, as rollout_kernel does, writing no more rows;
  timestep_latched          a frozen row's timestep is the latched t_ep instead of 0;
  action_not_zeroed         a frozen row's action is the env's held action instead of 0.
Ghost lanes are not mutated: a ghost steps a copy of the batch's last env on that env's own random stream, so what it could
write is what the env itself writes.  A mutant is caught when pytest fails; the first failing test is reported.  Needs the
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

OBSERVATION = """    if (!ghost && rec.observation) {
#pragma unroll
      for (int b = 0; b < M; ++b)
#pragma unroll
        for (int c = 0; c < 4; ++c) rec.observation[row * (M * 4) + ((int64_t)b * 4 + c) * n + e] = env.s[b][c];
    }
"""
RESET = """    if (CAV_UNLIKELY(env.done != 0) && auto_reset) {
      reset_env<R, M>(sc, buf, nullptr, e, env);
      was_reset = true;
    }
"""
ROW = """    const int64_t row = (int64_t)t * n;
    const bool stepped = env.done == 0;
"""
MUTANTS = {
    "observation_before_reset": (RESET + ROW + OBSERVATION,
                                 "    const int64_t row = (int64_t)t * n;\n" + OBSERVATION + RESET + "    const bool stepped = env.done == 0;\n"),
    "frozen_rows_skipped": (RESET, "    if (CAV_UNLIKELY(env.done != 0) && !auto_reset) break;\n" + RESET),
    "timestep_latched": ("rec.timestep[row + e] = stepped ? env.t_ep : 0;", "rec.timestep[row + e] = env.t_ep;"),
    "action_not_zeroed": ("= stepped ? env.held[b][0] : R(0);", "= env.held[b][0];"),
}
UNITS = ("record_m2", "record_m5")


def build_mutant(name, work):
    tree = os.path.join(work, name)
    shutil.copytree(os.path.join(ROOT, "cavgym_b200", "csrc"), os.path.join(tree, "cavgym_b200", "csrc"),
                    ignore=shutil.ignore_patterns("build", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    csrc = os.path.join(tree, "cavgym_b200", "csrc")
    path = os.path.join(csrc, "kernels_small.cuh")
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
    proc = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider", "tests/test_gpu_rollout_record.py",
                           "-k", "(homogeneous_2_bodies or synced_bus_stop) and not against_the_oracle"],
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
