"""Build liblora_b200.so (the CUDA library + C ABI) in-tree with nvcc for sm_100a.

The built .so sits next to this file so that it travels with the repository snapshot to the
GPU box (the JIT cache under ~/.cache would not)."""
from __future__ import annotations

import os
import shutil
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
CSRC = PKG / "csrc"
LIB = PKG / "liblora_b200.so"
HOST_EMUL = ROOT / "build" / "host_emul.so"

NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "-shared", "--use_fast_math=false"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and Path(cand).exists():
            return cand
    raise RuntimeError("nvcc not found: cannot build liblora_b200.so")


def _stale(target: Path, sources) -> bool:
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any(Path(s).stat().st_mtime > t for s in sources)


def _sources():
    return sorted(CSRC.glob("*.cu")) + sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.h")) + [ROOT / "include" / "lora_b200.h"]


TRANSLATION_UNITS = ("lora_b200.cu", "k1_rows.cu", "k1_packed.cu", "channelizer.cu", "gateway.cu")


def build(force: bool = False, verbose: bool = False) -> Path:
    """Every translation unit is compiled to build/obj/*.o (in parallel, only when stale) and linked into the .so."""
    srcs = _sources()
    if not (force or _stale(LIB, srcs)):
        return LIB
    from concurrent.futures import ThreadPoolExecutor
    obj_dir = ROOT / "build" / "obj"
    obj_dir.mkdir(parents=True, exist_ok=True)
    cflags = [f for f in NVCC_FLAGS if f not in ("-shared",) and not f.startswith("--use_fast_math")]
    headers = [p for p in srcs if p.suffix != ".cu"]

    def compile_one(name):
        obj = obj_dir / (name + ".o")
        if force or _stale(obj, [CSRC / name, *headers]):
            cmd = [_nvcc(), *cflags, "-c", "-o", str(obj), str(CSRC / name)]
            if verbose:
                print(" ".join(cmd))
            subprocess.run(cmd, check=True)
        return obj

    with ThreadPoolExecutor(len(TRANSLATION_UNITS)) as ex:
        objs = list(ex.map(compile_one, TRANSLATION_UNITS))
    cmd = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(LIB), *map(str, objs)]
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB


def build_host_emul(force: bool = False) -> Path:
    """CPU build of the kernels' __host__ __device__ phase functions (non-GPU tests only)."""
    if force or _stale(HOST_EMUL, _sources()):
        HOST_EMUL.parent.mkdir(exist_ok=True)
        cmd = [_nvcc(), "-O2", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
               "-shared", "-o", str(HOST_EMUL), str(CSRC / "host_emul.cu")]
        subprocess.run(cmd, check=True)
    return HOST_EMUL


SHIM = ROOT / "build" / "lora_shim_demo"


def build_shim(force: bool = False) -> Path:
    """The C++ drop-in body of gr::lora::decoder_impl (host/decoder_impl.cc) + a file-replay main,
    compiled against host/gr_stub (GNU Radio is not installed here) and linked to liblora_b200.so."""
    host = PKG / "host"
    srcs = [host / "decoder_impl.cc", host / "shim_main.cc", host / "decoder_impl.h", host / "lora" / "decoder.h",
            host / "gr_stub" / "gnuradio" / "sync_block.h", ROOT / "include" / "lora_b200.h"]
    build()
    if force or _stale(SHIM, srcs) or SHIM.stat().st_mtime < LIB.stat().st_mtime:
        SHIM.parent.mkdir(exist_ok=True)
        cmd = [os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-I", str(host / "gr_stub"), "-I", str(host), "-I",
               str(ROOT / "include"), "-o", str(SHIM), str(host / "decoder_impl.cc"), str(host / "shim_main.cc"),
               "-L", str(PKG), "-llora_b200", f"-Wl,-rpath,{PKG}"]
        subprocess.run(cmd, check=True)
    return SHIM


CHAN_SHIM = ROOT / "build" / "chan_shim_demo"


def build_chan_shim(force: bool = False) -> Path:
    """The C++ drop-in body of gr::lora::channelizer_impl (host/channelizer_impl.cc) + a file-in / file-out main."""
    host = PKG / "host"
    srcs = [host / "channelizer_impl.cc", host / "chan_shim_main.cc", host / "channelizer_impl.h", host / "lora" / "channelizer.h",
            host / "gr_stub" / "gnuradio" / "hier_block2.h", host / "gr_stub" / "gnuradio" / "sync_block.h", ROOT / "include" / "lora_b200.h"]
    build()
    if force or _stale(CHAN_SHIM, srcs) or CHAN_SHIM.stat().st_mtime < LIB.stat().st_mtime:
        CHAN_SHIM.parent.mkdir(exist_ok=True)
        cmd = ["g++", "-O2", "-std=c++17", "-I", str(host / "gr_stub"), "-I", str(host), "-I", str(ROOT / "include"), "-o", str(CHAN_SHIM),
               str(host / "channelizer_impl.cc"), str(host / "chan_shim_main.cc"), "-L", str(PKG), "-llora_b200", f"-Wl,-rpath,{PKG}"]
        subprocess.run(cmd, check=True)
    return CHAN_SHIM


if __name__ == "__main__":
    print(build(verbose=True))
