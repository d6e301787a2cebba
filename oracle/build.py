"""TEST INFRASTRUCTURE.  Builds the C oracle (gcc) and, when NVSF_REFERENCE names a checkout of
the reference project, the reference extensions via build_ref.sh / build_ref_chamfer.sh."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "raymarching_oracle.c")
OUT_DIR = os.path.join(HERE, "_build")
OUT = os.path.join(OUT_DIR, "libnvsf_oracle.so")

# -ffp-contract=off: the oracle spells out every fused multiply-add with fmaf().
CFLAGS = ["-O2", "-march=x86-64-v3", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
          "-shared", "-fvisibility=hidden", "-Wall", "-Wextra"]


def build_oracle(force=False):
    os.makedirs(OUT_DIR, exist_ok=True)
    if not force and os.path.exists(OUT) and os.path.getmtime(OUT) >= os.path.getmtime(SRC):
        return OUT
    # the system gcc (not $CC, which may point at a toolchain without libgomp); OpenMP is
    # only used to time the oracle as a multi-core CPU baseline, so fall back without it.
    for flags in (CFLAGS, [f for f in CFLAGS if f != "-fopenmp"]):
        cmd = ["gcc"] + flags + ["-o", OUT, SRC, "-lm"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode == 0:
            return OUT
    sys.stderr.write(r.stdout + r.stderr)
    raise RuntimeError("gcc failed building the oracle")


def build_ref():
    """Compile the unmodified reference extensions for sm_100a (no-op without NVSF_REFERENCE)."""
    out = []
    for script in ("build_ref.sh", "build_ref_chamfer.sh"):
        r = subprocess.run(["bash", os.path.join(HERE, script)], capture_output=True, text=True)
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError(f"oracle/{script} failed")
        out.append(r.stdout.strip())
    return "\n".join(out)


if __name__ == "__main__":
    print(build_oracle(force="--force" in sys.argv))
    print(build_ref())
