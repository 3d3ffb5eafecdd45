"""Mutation check of the episode regeneration tests: build the library with one deliberate defect in the regeneration kernel
(kernels_regen.cuh) or in what it shares with the transition, and show that tests/test_gpu_regenerate.py fails on it.

    python scripts/regenerate_mutations.py [--out FILE]

Mutants (each built in a temporary directory from a copy of cavgym_b200/csrc: regen_m2.cu recompiled, linked with the other
objects of the in-tree build, loaded through CAVGYM_LIB, so only the regeneration kernels carry the defect; the tests run on
the two-body pedestrians scenarios):
  agent_draws_by_slot    the agents' Philox draws are keyed by the slot's own global id instead of env_id[e];
  spawn_draws_by_slot    the spawn draws of the reset are keyed by the slot's own global id;
  episode_off_by_one     the reset draws episode episodes[e] + 1;
  scene_tester           the kernel takes the scenario's tester parameters (SceneTester's values) instead of the slot's;
  log_row_slot_id        the episode row carries the slot's own global id.
A mutant is caught when pytest fails; the first failing test is reported.  Needs the in-tree build (build() first) and a GPU.
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

# (file, code, mutated code): only regen_m2.cu is recompiled, so a change to a shared header reaches the regeneration kernels only
MUTANTS = {
    "agent_draws_by_slot": [("transition_body.inc", "(uint64_t)key(buf, e)", "(uint64_t)(buf.shard + e)", 2)],
    "spawn_draws_by_slot": [("transition.cuh", "const uint64_t g = (uint64_t)key(buf, e);", "const uint64_t g = (uint64_t)(buf.shard + e);", 1)],
    "episode_off_by_one": [("kernels_regen.cuh", "env.episode = episodes[e] - 1;", "env.episode = episodes[e];", 1)],
    "scene_tester": [("kernels_regen.cuh", "const EnvTester<R> tester{params};", "const EnvTester<R> tester{AgentParams<R>{nullptr, nullptr}};", 1)],
    "log_row_slot_id": [("transition.cuh", "buf.ep_log_capacity, key(buf, e), episode};", "buf.ep_log_capacity, buf.shard + e, episode};", 1)],
}
UNITS = ("regen_m2",)
TESTS = "pedestrians_rc_seed0 or epsilon or threshold"


def build_mutant(name, work):
    tree = os.path.join(work, name)
    shutil.copytree(os.path.join(ROOT, "cavgym_b200", "csrc"), os.path.join(tree, "cavgym_b200", "csrc"),
                    ignore=shutil.ignore_patterns("build", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    csrc = os.path.join(tree, "cavgym_b200", "csrc")
    for file, old, new, count in MUTANTS[name]:
        path = os.path.join(csrc, file)
        text = open(path).read()
        if text.count(old) != count:
            raise RuntimeError(f"{name}: the code to mutate is not there {count} time(s): {old}")
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
    proc = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider", "tests/test_gpu_regenerate.py",
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
