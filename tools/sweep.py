"""Build variants of libdsac_b200.so here (CPU box), measure each on the GPU box.

    python tools/sweep.py build          # here: writes variants/*.so (shipped to the GPU box by gpurun, git-ignored)
    python tools/sweep.py run            # on the GPU box: one tools/sweep_one.py process per variant -> gpurun_out/sweep.jsonl

Variants: the kernels of the last commit ("old": kernels.cuh / refine.cuh from git HEAD with the current host code),
and the working tree's kernels with experiment macros.  Development aid only."""
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
VAR = os.path.join(ROOT, "variants")
# (name, extra nvcc flags)
VARIANTS = [("cur", "")]


def build():
    os.makedirs(VAR, exist_ok=True)
    code = "import sys; sys.path.insert(0, %r); from dsac_b200 import build as b; b.build(out=sys.argv[1], csrc=(sys.argv[2] or None))" % ROOT
    old = os.path.join(VAR, "src_old")
    if os.environ.get("SWEEP_OLD_REF"):
        shutil.rmtree(old, ignore_errors=True)
        shutil.copytree(os.path.join(ROOT, "dsac_b200", "csrc"), old)
        for f in ("kernels.cuh", "refine.cuh"):
            with open(os.path.join(old, f), "wb") as fh:
                fh.write(subprocess.check_output(["git", "-C", ROOT, "show", os.environ["SWEEP_OLD_REF"] + ":dsac_b200/csrc/" + f]))
        subprocess.check_call([sys.executable, "-c", code, os.path.join(VAR, "old.so"), old])
        print("built old.so")
    for name, flags in VARIANTS:
        env = dict(os.environ, DSAC_EXTRA_NVCC_FLAGS=flags)
        subprocess.check_call([sys.executable, "-c", code, os.path.join(VAR, name + ".so"), ""], env=env)
        print("built", name)


def run():
    out = os.path.join(ROOT, "gpurun_out", "sweep.jsonl")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    libs = sorted(f for f in os.listdir(VAR) if f.endswith(".so"))
    only = os.environ.get("SWEEP_ONLY")
    if only:
        libs = [l for l in libs if l[:-3] in only.split(",")]
    with open(out, "a") as fh:
        for l in libs:
            env = dict(os.environ, DSAC_B200_LIB=os.path.join(VAR, l))
            try:
                r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sweep_one.py")], env=env, capture_output=True, text=True, timeout=300)
                lines = [x for x in r.stdout.splitlines() if x.startswith("SWEEP ")]
                msg = lines[-1][6:] if lines else '{"lib": "%s", "error": %r}' % (l, (r.stderr or r.stdout)[-600:])
            except subprocess.TimeoutExpired:
                msg = '{"lib": "%s", "error": "timeout"}' % l
            fh.write(msg + "\n"); fh.flush()
            print(l, msg[:1500])


if __name__ == "__main__":
    {"build": build, "run": run}[sys.argv[1]]()
