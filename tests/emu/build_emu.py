"""TEST INFRASTRUCTURE ONLY: compile the product's .cu files with g++ against tests/emu/cuda_runtime.h (a functional CPU
emulation of the CUDA constructs they use) into tests/emu/_build/libd3h_tets_emu.so.  See tests/emu/cuda_runtime.h."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "d3human-code_b200", "csrc")
OUT = os.path.join(HERE, "_build", "libd3h_tets_emu.so")
OUT_SAN = os.path.join(HERE, "_build", "libd3h_tets_emu_san.so")
OUT_TSAN = os.path.join(HERE, "_build", "libd3h_tets_emu_tsan.so")
SOURCES = ["d3h_api.cu", "d3h_classify.cu", "d3h_sort.cu", "d3h_scan.cu", "d3h_surface.cu", "d3h_backward.cu", "d3h_mesh.cu", "d3h_lbs.cu", "d3h_mlp.cu"]


def build(force=False, sanitize=False, tsan=False):
    """sanitize=True: the same sources with -fsanitize=address,alignment,bounds (a second library, loaded by
    tests/test_emu_sanitize.py in a child process that preloads libasan): out-of-bounds accesses to any torch buffer,
    misaligned vector loads / stores and out-of-range local array indices abort the run."""
    out = OUT_TSAN if tsan else (OUT_SAN if sanitize else OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, f) for f in ("cuda_runtime.h", "emu_core.cpp")]
    deps += [os.path.join(ROOT, "include", h) for h in ("d3h_tets.h", "d3h_mesh.h", "d3h_lbs.h", "d3h_mlp.h")]
    if not force and os.path.isfile(out) and all(os.path.getmtime(d) <= os.path.getmtime(out) for d in deps):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    # -ffp-contract=off: the float pipeline must round like the GPU build (-fmad=false); -x c++ for the .cu files
    cmd = ["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-ffp-contract=off", "-fno-strict-aliasing", "-w",
           "-DD3H_CPU_EMU=1", "-I", HERE]
    if tsan:   # every emulated CUDA thread is a ThreadSanitizer fibre (tests/emu/emu_core.cpp, EMU_TSAN)
        cmd += ["-fsanitize=thread", "-DEMU_TSAN=1", "-fno-omit-frame-pointer"]
    elif sanitize:
        cmd += ["-fsanitize=address,alignment,bounds", "-fno-sanitize-recover=all", "-fno-omit-frame-pointer"]
    for s in SOURCES:
        cmd += ["-x", "c++", os.path.join(CSRC, s)]
    if tsan:
        # the scheduler's own bookkeeping is shared by all fibres on purpose: it is compiled WITHOUT instrumentation, so
        # that ThreadSanitizer only watches the kernels (it still calls the fibre / annotation API)
        core_obj = os.path.join(os.path.dirname(out), "emu_core_tsan.o")
        core = ["g++", "-O1", "-g", "-std=c++17", "-fPIC", "-c", "-w", "-DD3H_CPU_EMU=1", "-DEMU_TSAN=1", "-I", HERE,
                os.path.join(HERE, "emu_core.cpp"), "-o", core_obj]
        res = subprocess.run(core, capture_output=True, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stderr[-6000:])
            raise RuntimeError("g++ failed building the emulator core")
        cmd += ["-x", "none", core_obj, "-o", out]
    else:
        cmd += ["-x", "c++", os.path.join(HERE, "emu_core.cpp"), "-o", out]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stderr[-6000:])
        raise RuntimeError("g++ failed building the emulated library")
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, sanitize="--sanitize" in sys.argv, tsan="--tsan" in sys.argv))
