"""Mutation run of the candidate certificate: does tests/test_gpu_certificate.py fail when the threshold is weakened?

    python tools/certificate_mutations.py OUT_DIR [--build-only | --run-only] [--mutants eta0,kth,...] [--timeout S]

For the baseline and each mutant the tree is copied to OUT_DIR/<id> (sources, tests, oracle; object files too, so that
only the edited translation unit recompiles), ONE exact string replacement is applied to the copy's
lidar_global_registration_b200/csrc/candidates_tc.cu -- the target text must occur exactly once, so the script fails
loudly when the source drifts -- and the library is rebuilt.  Then tests/test_gpu_certificate.py runs once under a
timeout and the failing tests are logged to OUT_DIR/mutations.log.  Mutants are never written into the repository.

Every mutation changes threshold arithmetic or which already-loaded value is chosen, never an index, a loop bound over
memory, a barrier or a launch shape: a mutant can give wrong answers but cannot fault.  --build-only (no GPU needed)
and --run-only split the two halves, e.g. to compile the mutants in parallel before the GPU run.
"""
import argparse
import os
import re
import shutil
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TU = os.path.join("lidar_global_registration_b200", "csrc", "candidates_tc.cu")

# id -> (what it weakens, exact target text, replacement)
MUTATIONS = {
    "eta0": ("the FP16 rounding term eta = 0",
             "sts_f32(st.s_const + 4u, ab * 4.8828125e-4f * 1.001953125f + 2.384185791015625e-7f * sqrtf((float) p.dim));",
             "sts_f32(st.s_const + 4u, 0.f);"),
    "gfac1": ("the reference's FP32 rounding factor gfac = 1",
              "sts_f32(st.s_const + 12u, 1.f + 2.2f * (float) (p.dim + 4) * 5.9604644775390625e-8f);",
              "sts_f32(st.s_const + 12u, 1.f);"),
    "slop": ("A-resident accumulation slop cut to its bare 1e-6",
             ": ab * ab * 1.52587890625e-5f + 1e-6f);",
             ": 1e-6f);"),
    "ks_slop": ("K-streamed slop cut to the A-resident 2^-16 constant",
                "KS ? ab * ab * ((float) p.ksteps * 4.76837158203125e-7f) + 1e-6f",
                "KS ? ab * ab * 1.52587890625e-5f + 1e-6f"),
    "eta_nobmax": ("eta and slop without the train-side bound bmax (ab = |a16|)",
                   "const float ab = sqrtf(na) + (DP ? p.prep->bmax[p.train_side] : p.bmax);",
                   "const float ab = sqrtf(na);"),
    "kth": ("kth_smallest picks the (k-1)-th smallest value",
            "if (s == k - 1) T = st.tk[s];",
            "if (s == k - 2) T = st.tk[s];"),
    "merge_self": ("EH = 2 merge counts the thread's own published values (j = 0..2 instead of 1..3)",
                   "for (uint32_t j = 1; j < 4; ++j) {",
                   "for (uint32_t j = 0; j < 3; ++j) {"),
}

SKIP_DIRS = {".git", "profiles", "build", "__pycache__", ".pytest_cache"}


def copy_tree(dst):
    def ignore(d, names):
        return [n for n in names if n in SKIP_DIRS or (os.path.abspath(os.path.join(d, n)) == os.path.abspath(dst))]
    if os.path.exists(dst):
        shutil.rmtree(dst)
    shutil.copytree(ROOT, dst, ignore=ignore, symlinks=True)   # copy2: mtimes kept, untouched objects stay current


def mutate(tree, mid):
    if mid == "baseline":
        return
    _, old, new = MUTATIONS[mid]
    path = os.path.join(tree, TU)
    text = open(path).read()
    n = text.count(old)
    if n != 1:
        raise SystemExit("mutation %s: target text occurs %d times in %s (expected exactly once)" % (mid, n, TU))
    open(path, "w").write(text.replace(old, new))


def build(tree):
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from lidar_global_registration_b200 import build as b; b.build()\n"
            "from oracle import oracle as orc; orc.build()\n") % tree
    r = subprocess.run([sys.executable, "-c", code], cwd=tree, capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit("build of %s failed:\n%s%s" % (tree, r.stdout, r.stderr))


def run_tests(tree, timeout):
    t0 = time.time()
    cmd = [sys.executable, "-m", "pytest", "-q", "-rf", "-p", "no:cacheprovider", "tests/test_gpu_certificate.py"]
    try:
        r = subprocess.run(cmd, cwd=tree, capture_output=True, text=True, timeout=timeout)
        out, rc = r.stdout + r.stderr, r.returncode
    except subprocess.TimeoutExpired as e:
        out, rc = (e.stdout or b"").decode(errors="replace") if isinstance(e.stdout, bytes) else (e.stdout or ""), "timeout"
    failed = sorted(set(re.findall(r"^FAILED (\S+)", out, re.M)))
    summary = [l for l in out.splitlines() if re.search(r"\d+ (passed|failed)", l)]
    return rc, failed, (summary[-1] if summary else out.strip().splitlines()[-1:] or ["(no output)"]), time.time() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--build-only", action="store_true")
    ap.add_argument("--run-only", action="store_true")
    ap.add_argument("--mutants", default=",".join(["baseline"] + list(MUTATIONS)))
    ap.add_argument("--timeout", type=float, default=900)
    a = ap.parse_args()
    ids = a.mutants.split(",")
    for mid in ids:
        if mid != "baseline" and mid not in MUTATIONS:
            raise SystemExit("unknown mutation " + mid)
    os.makedirs(a.out_dir, exist_ok=True)
    trees = {mid: os.path.join(os.path.abspath(a.out_dir), mid) for mid in ids}
    if not a.run_only:
        for mid in ids:
            copy_tree(trees[mid])
            mutate(trees[mid], mid)
        with ThreadPoolExecutor(max_workers=len(ids)) as ex:   # one nvcc per tree: only candidates_tc.cu recompiles
            list(ex.map(build, [trees[m] for m in ids]))
        print("built: " + ", ".join(ids))
    if a.build_only:
        return
    log = open(os.path.join(a.out_dir, "mutations.log"), "w")
    for mid in ids:
        # the test file is not part of the build: run the repository's current one
        shutil.copy2(os.path.join(ROOT, "tests", "test_gpu_certificate.py"), os.path.join(trees[mid], "tests"))
        rc, failed, summary, secs, out = run_tests(trees[mid], a.timeout)
        what = "unmodified tree" if mid == "baseline" else MUTATIONS[mid][0]
        line = "%-11s %-78s rc=%s %5.0f s  %s" % (mid, what, rc, secs, summary)
        print(line, flush=True)
        log.write(line + "\n")
        for f in failed:
            log.write("    FAILED " + f + "\n")
        log.flush()
        open(os.path.join(a.out_dir, mid + ".pytest.log"), "w").write(out)
    log.close()


if __name__ == "__main__":
    main()
