"""Mutation check of the per-instantiation and pair-sweep tests: build the library with one deliberate defect confined to one
(body count, scenario family) instantiation of the thread-per-env kernels, or to one case of the warp-per-env pair sweep, and
show that the tests of that cell fail on it.

    python scripts/instantiation_mutations.py build DIR          # compile every mutant into DIR (no GPU needed)
    python scripts/instantiation_mutations.py run DIR [--out F]  # run each mutant's tests against DIR/<mutant>.so (GPU)

Mutants (each built from a copy of cavgym_b200/csrc: the named translation units recompiled, linked with the other objects of
the in-tree build; the tests load it through CAVGYM_LIB).  The first four are confined to one instantiation of the
thread-per-env kernels, the last two to the warp-per-env pair sweep:
  rolled_zone_loop_skips_last_m6_generic  transition_rolled, generic M = 6 only: the ego-zone loop stops before the last body;
  record_launcher_m7_generic_runs_homogeneous
                                          the recording rollout's launcher at M = 7 runs the GENERIC = false kernel for a
                                          generic scenario;
  until_launcher_m8_generic_runs_homogeneous
                                          the same in the parking rollout's launcher at M = 8;
  tma_step_m1_drops_reward_rows           the TMA step kernel at M = 1 stages no reward row out;
  dense_within_round_16_dropped           the warp-per-env sweep inside a tile skips rotation round 16 (lanes 0..15 against
                                          lanes 16..31 at offset 16);
  dense_lower_tiles_skipped_in_a_one_tile_pass
                                          a final pass with only tile A does not sweep the tiles below it (65..96, 129..160 bodies).
Each is a logic defect that only drops work or picks another compiled kernel over the same buffers: no index grows, so a
mutant can give wrong answers but never touches memory the correct build does not.  A mutant is caught when pytest fails;
the first failing test is reported.  Needs the in-tree build (build() first).
"""
import argparse
import concurrent.futures
import os
import re
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cavgym_b200.csrc import build  # noqa: E402

ROLLED = ('#define CAV_BODY_LOOP _Pragma("unroll 1")\n',
          '#undef CAV_MUT_SKIP_LAST\n#define CAV_MUT_SKIP_LAST(M, G) ((M) == 6 && (G))\n#define CAV_BODY_LOOP _Pragma("unroll 1")\n')
UNROLLED = ('#define CAV_BODY_LOOP _Pragma("unroll")\n', '#define CAV_MUT_SKIP_LAST(M, G) false\n#define CAV_BODY_LOOP _Pragma("unroll")\n')
ZONE_LOOP = ("    for (int b = 1; b < M; ++b) {\n      if (!is_pedestrian(b)) continue;   // environment.py:192,199\n",
             "    for (int b = 1; b < M - (CAV_MUT_SKIP_LAST(M, GENERIC) ? 1 : 0); ++b) {\n      if (!is_pedestrian(b)) continue;\n")

# name -> ([(file, old, new)], translation units to recompile, pytest arguments)
MUTANTS = {
    "rolled_zone_loop_skips_last_m6_generic": (
        [("transition.cuh",) + UNROLLED, ("transition.cuh",) + ROLLED, ("transition_body.inc",) + ZONE_LOOP],
        ("small_m6", "record_m6", "until_m6"),
        ["tests/test_gpu_instantiations.py", "-k", "generic_m6 and replayed"]),
    "record_launcher_m7_generic_runs_homogeneous": (
        [("kernels_small.cuh",
          "  else rollout_record_kernel<R, M, true><<<grid_for(buf, synced), synced, 0, stream>>>(sc, buf, rec, t_global, n_steps, auto_reset);\n",
          "  else if constexpr (M == 7) rollout_record_kernel<R, M, false><<<grid_for(buf, plain), plain, 0, stream>>>(sc, buf, rec, t_global, n_steps, auto_reset);\n"
          "  else rollout_record_kernel<R, M, true><<<grid_for(buf, synced), synced, 0, stream>>>(sc, buf, rec, t_global, n_steps, auto_reset);\n")],
        ("record_m7",),
        ["tests/test_gpu_rollout_record.py", "-k", "matrix_generic_7_bodies and changes_nothing"]),
    "until_launcher_m8_generic_runs_homogeneous": (
        [("kernels_until.cuh",
          "  else\n    rollout_until_kernel<R, M, true>",
          "  else if constexpr (M == 8)\n    rollout_until_kernel<R, M, false><<<grid_for(buf, plain), plain, 0, stream>>>(sc, buf, score, status, level, t_global, n_steps);\n"
          "  else\n    rollout_until_kernel<R, M, true>")],
        ("until_m8",),
        ["tests/test_gpu_splitting.py", "-k", "matrix_generic_8_bodies and (level_inf or running_max)"]),
    "tma_step_m1_drops_reward_rows": (
        [("kernels_tma.cuh",
          "      for (int b = 0; b < M; ++b) out(io.reward_out, b, sizeof(R), L::oReward + b * L::kRow);\n",
          "      for (int b = 0; b < (M == 1 ? 0 : M); ++b) out(io.reward_out, b, sizeof(R), L::oReward + b * L::kRow);\n")],
        ("small_m1",),
        ["tests/test_gpu_instantiations.py", "-k", "m1 and replayed"]),
    "dense_within_round_16_dropped": (
        [("kernels_dense.cuh", "any |= broad_overlap(pi, pj) && (r < 16 || lane < 16);", "any |= broad_overlap(pi, pj) && (r < 16);"),
         ("kernels_dense.cuh", "if ((r < 16 || lane < 16) && broad_overlap(sm.bp[i], pj))", "if ((r < 16) && broad_overlap(sm.bp[i], pj))")],
        ("dense",),
        ["tests/test_gpu_dense.py", "-k", "pair_sweep"]),
    "dense_lower_tiles_skipped_in_a_one_tile_pass": (
        [("kernels_dense.cuh", "        if (__any_sync(kFull, broad_overlap(ui, pA) || broad_overlap(ui, pB))) sweep(it, it + 32, true);",
          "        if (haveB && __any_sync(kFull, broad_overlap(ui, pA) || broad_overlap(ui, pB))) sweep(it, it + 32, true);")],
        ("dense",),
        ["tests/test_gpu_dense.py", "-k", "pair_sweep"]),
}


def build_mutant(name, out_dir):
    tree = os.path.join(out_dir, "src", name)
    shutil.rmtree(tree, ignore_errors=True)
    shutil.copytree(os.path.join(ROOT, "cavgym_b200", "csrc"), os.path.join(tree, "cavgym_b200", "csrc"),
                    ignore=shutil.ignore_patterns("build", "__pycache__"))
    shutil.copytree(os.path.join(ROOT, "include"), os.path.join(tree, "include"))
    csrc = os.path.join(tree, "cavgym_b200", "csrc")
    edits, units, _ = MUTANTS[name]
    for file, old, new in edits:
        path = os.path.join(csrc, file)
        text = open(path).read()
        if text.count(old) != 1:
            raise RuntimeError(f"{name}: the code to mutate is not in {file} exactly once: {old!r}")
        open(path, "w").write(text.replace(old, new))
    objs = [os.path.join(tree, unit + ".o") for unit in units]
    for unit, obj in zip(units, objs):
        proc = subprocess.run([build.NVCC] + build.FLAGS + ["-c", os.path.join(csrc, unit + ".cu"), "-o", obj], capture_output=True, text=True)
        if proc.returncode:
            raise RuntimeError(f"{name}: {proc.stderr[-2000:]}")
    others = sorted(os.path.join(build.OBJ_DIR, f) for f in os.listdir(build.OBJ_DIR)
                    if f.endswith(".o") and f[:-2] not in units and not f.endswith(".stub.o"))
    lib = os.path.join(out_dir, name + ".so")
    proc = subprocess.run([build.NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", lib] + objs + others
                          + ["-lcudart_static", "-lpthread", "-ldl", "-lrt"], capture_output=True, text=True)
    if proc.returncode:
        raise RuntimeError(f"{name}: {proc.stderr[-2000:]}")
    shutil.rmtree(tree)
    return lib


def run_tests(name, lib):
    env = dict(os.environ, CAVGYM_LIB=lib)
    proc = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider"] + MUTANTS[name][2],
                          cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    failed = re.findall(r"^FAILED (\S+)", proc.stdout, flags=re.M)
    where = re.findall(r"^E\s+(.*)$", proc.stdout, flags=re.M)
    return proc.returncode, (failed[0] if failed else ""), (where[0].strip()[:160] if where else "")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("what", choices=("build", "run"))
    ap.add_argument("dir")
    ap.add_argument("--out", default=None, help="also write the report here")
    args = ap.parse_args()
    names = list(MUTANTS)
    os.makedirs(args.dir, exist_ok=True)
    if args.what == "build":
        with concurrent.futures.ThreadPoolExecutor(max_workers=len(names)) as pool:
            for lib in pool.map(lambda n: build_mutant(n, args.dir), names):
                print("built", lib, flush=True)
        return 0
    lines = []
    for name in names:
        rc, failed, where = run_tests(name, os.path.join(args.dir, name + ".so"))
        line = f"{name:44s} {'caught' if rc == 1 else 'NOT CAUGHT' if rc == 0 else f'pytest exit {rc}'}  {failed}  | {where}"
        print(line, flush=True)
        lines.append(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")
    return 0 if all(" caught " in line for line in lines) else 1


if __name__ == "__main__":
    sys.exit(main())
