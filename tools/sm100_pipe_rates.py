"""Measure the per-SM issue rates of FFMA, FFMA2, FADD2 and the MUFU ex2 / rcp ops (alone and mixed with FFMA2) on the
local GPU, with the card's name, power limit and clocks.  The .cu next to this script is compiled into a temporary
directory, so the tree stays untouched.
    python tools/sm100_pipe_rates.py"""
import subprocess
import sys
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent


def main() -> int:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True)
    print(q.stdout.strip() if q.returncode == 0 else "nvidia-smi: " + q.stderr.strip())
    with tempfile.TemporaryDirectory() as tmp:
        exe = Path(tmp) / "sm100_pipe_rates"
        subprocess.run(["/usr/local/cuda/bin/nvcc", "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
                        str(HERE / "sm100_pipe_rates.cu"), "-o", str(exe)], check=True)
        return subprocess.run([str(exe)]).returncode


if __name__ == "__main__":
    sys.exit(main())
