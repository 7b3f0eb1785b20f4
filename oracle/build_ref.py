"""Snapshot the UNMODIFIED reference's hot-path Python packages into the git-ignored `oracle/_ref/` (test / baseline
infrastructure).  The reference is pure Python — there is nothing to compile — so "building" the real reference is a
verbatim file copy made by this committed recipe; the copy is never committed (`oracle/_ref/` is in .gitignore) but it
travels to the GPU box with the gpurun snapshot, where `/root/reference` does not exist.

    python oracle/build_ref.py            # copies lvdm/ scheduler/ pipeline/ utils/ ode_solver/ model_scope/ (*.py only)

Consumers: `bench.py --impl reference` (the CPU arm: reference `UNetModel` + `Decoder`, unmodified, on the full
BASELINE config), `scripts/ref_gpu_bench.py` (the same modules in bf16 on the B200: the north star's GPU denominator)
and `oracle/make_goldens.py`.  The import shims for `diffusers` / `pytorch_lightning` base classes live in `oracle/shim/`.
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = "/root/reference"
DST = os.path.join(HERE, "_ref")
PACKAGES = ("lvdm", "scheduler", "pipeline", "utils", "ode_solver", "model_scope")


def build_ref(src: str = SRC, dst: str = DST) -> str | None:
    if not os.path.isdir(src):
        return None
    n = 0
    for pkg in PACKAGES:
        for root, _, files in os.walk(os.path.join(src, pkg)):
            rel = os.path.relpath(root, src)
            for f in files:
                if not f.endswith(".py"):
                    continue
                os.makedirs(os.path.join(dst, rel), exist_ok=True)
                shutil.copyfile(os.path.join(root, f), os.path.join(dst, rel, f))
                n += 1
    if n == 0:          # present but empty or unreadable: no snapshot
        return None
    with open(os.path.join(dst, "SNAPSHOT.txt"), "w") as fh:
        fh.write(f"verbatim copy of {n} .py files of {src} ({', '.join(PACKAGES)}) made by oracle/build_ref.py; not committed\n")
    return dst


if __name__ == "__main__":
    out = build_ref()
    print(f"reference snapshot: {out}" if out else f"{SRC} not present: nothing copied")
    sys.exit(0)
