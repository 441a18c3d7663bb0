"""Build the C++ host side (libllama.so, kuiper_decode, and the reference's demo programs when a
reference checkout is present) with CMake + Ninja, in-tree under kuiper/_build/<variant>/.

variants: "llama2" (default arithmetic), "qwen2" (-DQWEN2_SUPPORT=ON), "llama3" (-DLLAMA3_SUPPORT=ON)
-- the same compile-time switches the reference uses (CMakeLists.txt:16-26 there).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
VARIANTS = {"llama2": [], "qwen2": ["-DQWEN2_SUPPORT=ON"], "llama3": ["-DLLAMA3_SUPPORT=ON"]}


def reference_checkout() -> Path | None:
    """The reference checkout named by KUIPER_REFERENCE_DIR whose demo programs are built unchanged,
    or None when the variable is unset or the demo sources cannot be read."""
    d = os.environ.get("KUIPER_REFERENCE_DIR")
    if not d:
        return None
    try:
        return Path(d) if (Path(d) / "demo" / "main.cpp").is_file() else None
    except OSError:
        return None


def build_dir(variant: str) -> Path:
    return HERE / "_build" / variant


def binary(variant: str, name: str) -> Path:
    return build_dir(variant) / name


def build(variant: str = "llama2", verbose: bool = False) -> Path:
    if variant not in VARIANTS:
        raise ValueError(f"unknown variant {variant!r}")
    cmake = shutil.which("cmake")
    if cmake is None:
        raise RuntimeError("cmake not found on PATH")
    out = build_dir(variant)
    out.mkdir(parents=True, exist_ok=True)
    cfg = [cmake, "-S", str(HERE), "-B", str(out), "-DCMAKE_BUILD_TYPE=Release",
           "-DCMAKE_CXX_COMPILER=/usr/bin/g++", *VARIANTS[variant]]
    if shutil.which("ninja"):
        cfg += ["-G", "Ninja"]
    reference = reference_checkout()
    if reference is not None:
        cfg.append(f"-DKUIPER_REFERENCE_DIR={reference}")
    quiet = {} if verbose else {"stdout": subprocess.PIPE, "stderr": subprocess.STDOUT}
    for cmd in (cfg, [cmake, "--build", str(out), "-j", str(min(32, os.cpu_count() or 4))]):
        r = subprocess.run(cmd, text=True, **quiet)
        if r.returncode != 0:
            raise RuntimeError(f"{' '.join(cmd)} failed:\n{r.stdout or ''}")
    return out


if __name__ == "__main__":
    for v in (sys.argv[1:] or ["llama2", "qwen2"]):
        print(build(v, verbose=True))
