"""Recipe for `oracle/_ref/`: a mirror of a checkout of the original project (fschmid56/EfficientAT), made by build()
wherever such a checkout exists.  It is git-ignored and travels with the working tree to machines that have no checkout.

    python oracle/make_ref.py [--src CHECKOUT]

The checkout is read from $EAT_REFERENCE_ROOT, else from its default location (SRC).  Without one, an existing mirror is
left as it is.  The mirror is used by measurement and test infrastructure only, never by efficientat_b200/:
  * `bench.py` `gpu_baseline` / `--impl reference-gpu` and `cpu_baseline` (baseline/ref_step.py): the UNMODIFIED
    reference modules timed on the same hardware, the bar BASELINE.md section 3 names;
  * `tests/test_gpu_refscripts.py`, `tests/test_gpu_zz_f4.py`: the reference's own `ex_audioset.py`, `inference.py` and
    `windowed_inference.py` run unchanged against this package (SURVEY.md section 8 rows f1, f4);
  * `tests/golden/make_golden.py`.
Large non-code assets (images/, the wandb/ run directory) are skipped.
"""
import argparse
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
DST = os.path.join(HERE, "_ref")
SKIP_DIRS = {".git", "images", "wandb", "__pycache__"}
SRC = os.environ.get("EAT_REFERENCE_ROOT", "/root/reference")


def make(src=SRC, dst=DST):
    if not os.path.isdir(src):
        return None
    n = 0
    for root, dirs, files in os.walk(src):
        dirs[:] = [d for d in dirs if d not in SKIP_DIRS]
        rel = os.path.relpath(root, src)
        out = os.path.join(dst, rel) if rel != "." else dst
        os.makedirs(out, exist_ok=True)
        for f in files:
            if f.endswith((".pyc", ".pt")):
                continue
            s, d = os.path.join(root, f), os.path.join(out, f)
            if not os.path.exists(d) or os.path.getmtime(d) < os.path.getmtime(s) or os.path.getsize(d) != os.path.getsize(s):
                shutil.copyfile(s, d)           # contents only: the checkout's read-only modes would block a refresh
                n += 1
    return dst, n


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default=SRC)
    a = ap.parse_args()
    r = make(a.src)
    print("reference checkout not found, nothing mirrored" if r is None else f"{r[0]}: {r[1]} files updated")
    sys.exit(0)
