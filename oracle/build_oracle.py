"""oracle/ (test infrastructure): compiles the CPU restatement.

  oracle/_build/oracle_cli        single-threaded CPU mapper (SAM out)
  oracle/_build/liboracle.so      C entry points for tests (ctypes)
and, when /root/reference is present, the real reference through build_ref.sh -> oracle/_ref/.
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
OUT = HERE / "_build"


def _newer(target: Path, sources) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(s).stat().st_mtime > t for s in sources if Path(s).exists())


def build(force=False):
    OUT.mkdir(exist_ok=True)
    deps = sorted(HERE.glob("*.hpp")) + sorted((HERE.parent / "bitmapperbs_b200/csrc/host").glob("*.hpp")) + [HERE.parent / "bitmapperbs_b200/csrc/bmbs_refine_ends.h"]
    cli = OUT / "oracle_cli"
    if force or _newer(cli, [HERE / "oracle_cli.cpp", *deps]):
        subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-Wno-sign-compare", str(HERE / "oracle_cli.cpp"), "-o", str(cli), "-lz"], check=True)
    lib = OUT / "liboracle.so"
    if (HERE / "oracle_capi.cpp").exists() and (force or _newer(lib, [HERE / "oracle_capi.cpp", *deps])):
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-Wno-sign-compare", str(HERE / "oracle_capi.cpp"), "-o", str(lib), "-lz"], check=True)
    subprocess.run(["bash", str(HERE / "build_ref.sh")], check=True)
    return cli, lib


if __name__ == "__main__":
    build("--force" in sys.argv)
