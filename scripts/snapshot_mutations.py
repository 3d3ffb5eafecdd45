"""Mutation check of the snapshot tests: build the library with one deliberate defect in the snapshot code and show that
tests/test_gpu_snapshot.py fails on it.

    python scripts/snapshot_mutations.py [--out FILE]

Mutants (each built in a temporary directory from a copy of cavgym_b200/csrc, linked with the other objects of the in-tree
build, loaded through CAVGYM_LIB):
  drop_<section>  move_envs gives one of the eleven row sections (state, action, agent, cs, liveness, t_ep, episode,
                  winner, active, done, err) zero rows: it is neither saved nor loaded nor forked;
  pdl             the snapshot kernels are launched with the programmatic-stream-serialisation attribute, so a save, load
                  or fork may start while a replay_tma_kernel (which releases its dependents at entry) still runs.
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

DROPS = {
    "state": ("add_rows(reals, buf.state, p, m * 4)", "add_rows(reals, buf.state, p, 0)"),
    "action": ("add_rows(reals, buf.action, p, m * 2)", "add_rows(reals, buf.action, p, 0)"),
    "agent": ("add_rows(reals, buf.agent, p, m * CAV_AGENT_WORDS)", "add_rows(reals, buf.agent, p, 0)"),
    "cs": ("add_rows(reals, buf.cs, p, m * 2)", "add_rows(reals, buf.cs, p, 0)"),
    "liveness": ("add_rows(ints, buf.liveness, q, m)", "add_rows(ints, buf.liveness, q, 0)"),
    "t_ep": ("add_rows(ints, buf.t_ep, q, 1)", "add_rows(ints, buf.t_ep, q, 0)"),
    "episode": ("add_rows(ints, buf.episode, q, 1)", "add_rows(ints, buf.episode, q, 0)"),
    "winner": ("add_rows(ints, buf.winner, q, 1)", "add_rows(ints, buf.winner, q, 0)"),
    "active": ("add_rows(ints, buf.active, q, 1)", "add_rows(ints, buf.active, q, 0)"),
    "done": ("add_rows(bytes, buf.done, snap + L.u8_offset, 1)", "add_rows(bytes, buf.done, snap + L.u8_offset, 0)"),
    "err": ("add_rows(bytes, buf.err, snap + L.u8_offset + k, 1)", "add_rows(bytes, buf.err, snap + L.u8_offset + k, 0)"),
}
PDL_LAUNCH = """{
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = dim3(kSnapThreads); cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, snapshot_kernel<T>, t);
}"""


def mutate(name, csrc):
    if name == "pdl":
        path, old, new = os.path.join(csrc, "kernels_snapshot.cuh"), "snapshot_kernel<T><<<grid, kSnapThreads, 0, stream>>>(t);", PDL_LAUNCH
    else:
        (old, new), path = DROPS[name[len("drop_"):]], os.path.join(csrc, "engine.cu")
    text = open(path).read()
    if text.count(old) != 1:
        raise RuntimeError(f"{name}: the code to mutate is not there exactly once: {old}")
    open(path, "w").write(text.replace(old, new))


def build_mutant(name, work):
    tree = os.path.join(work, name)
    shutil.copytree(os.path.join(ROOT, "cavgym_b200", "csrc"), os.path.join(tree, "cavgym_b200", "csrc"),
                    ignore=shutil.ignore_patterns("build", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    csrc = os.path.join(tree, "cavgym_b200", "csrc")
    mutate(name, csrc)
    obj, lib = os.path.join(tree, "engine.o"), os.path.join(tree, "libcavgym_sm100.so")
    others = sorted(os.path.join(build.OBJ_DIR, f) for f in os.listdir(build.OBJ_DIR)
                    if f.endswith(".o") and f != "engine.o" and not f.endswith(".stub.o"))
    for cmd in ([build.NVCC] + build.FLAGS + ["-c", os.path.join(csrc, "engine.cu"), "-o", obj],
                [build.NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib, obj] + others
                + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"]):
        proc = subprocess.run(cmd, capture_output=True, text=True)
        if proc.returncode:
            raise RuntimeError(f"{name}: {proc.stderr[-2000:]}")
    return lib


def run_tests(name, lib):
    selection = "chained_replay_train" if name == "pdl" else "not chained_replay_train"
    env = dict(os.environ, CAVGYM_LIB=lib)
    proc = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider", "tests/test_gpu_snapshot.py",
                           "-k", selection], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    failed = re.findall(r"^FAILED (\S+)", proc.stdout, flags=re.M)
    where = re.findall(r"^>\s+(.*)$", proc.stdout, flags=re.M)
    return proc.returncode, (failed[0] if failed else ""), (where[0].strip() if where else "")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the report here")
    args = ap.parse_args()
    names = ["drop_" + s for s in DROPS] + ["pdl"]
    lines = []
    with tempfile.TemporaryDirectory() as work:
        with concurrent.futures.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as pool:
            libs = dict(zip(names, pool.map(lambda n: build_mutant(n, work), names)))
        for name in names:
            rc, failed, where = run_tests(name, libs[name])
            line = f"{name:16s} {'caught' if rc == 1 else 'NOT CAUGHT' if rc == 0 else f'pytest exit {rc}'}  {failed}  | {where}"
            print(line, flush=True)
            lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    return 0 if all(" caught " in line for line in lines) else 1


if __name__ == "__main__":
    sys.exit(main())
