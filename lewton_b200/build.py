"""Build lewton_b200/liblewton_b200.so for sm_100a with nvcc (in-tree, so it travels to the GPU box).

Also enforces the parity-critical property of the fused kernel at build time: its SASS must not
contain a fused multiply-add (ptxas 12.9 contracts packed f32x2 mul+add even with explicit .rn;
kernel_long.cuh is written so that no such pair exists -- this check keeps it that way).
"""
import os
import re
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "liblewton_b200.so")
SOURCES = ["lwb_api.cu", "host_objects.cuh", "path_generic.cuh", "path_long.cuh", "path_chain.cuh", "path_mixed.cuh", "path_mid.cuh",
           "tables_host.cpp", "frontend.cpp", "lwb_common.h", "kernels_generic.cuh", "kernel_long.cuh", "kernel_short.cuh", "kernel_mid.cuh", "kernel_chain.cuh", "kernel_prologue.cuh", "floor1_eval.cuh",
           "floor1_inverse_db.inc", "Makefile"]


def _stale():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + [os.path.join(HERE, "..", "include", h)
                                                       for h in ("lewton_b200.h", "lewton_frontend.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def check_no_fma(so=SO):
    """No FFMA/FFMA2/DFMA in any of our kernels: every rounding of the reference is kept."""
    if shutil.which("cuobjdump") is None:
        return None
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    bad = re.findall(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P[0-9T]\s+)?(FFMA2?|DFMA)\b.*$", sass, re.M)
    return len(bad)


def hot_kernel_registers(log):
    """Registers per thread of every k_long<OutT, CS> instantiation (CS = 1 planar, 2..8 interleaved) from ptxas -v
    output.  The headline kernel is bound by per-warp latency and touchy about its allocation: at 254-255 registers
    (two more live values, or a changed helper template that only its sibling k_long_s uses) it lost 3-4 % (A/B on one
    box, DESIGN.md 4.4); 250 / 252 is the allocation the measured planar numbers belong to, 253-254 the one of the
    interleaved instantiations (DESIGN.md 4.7)."""
    regs = {}
    for m in re.finditer(r"Compiling entry function '(_ZN3lwb6k_longI([fs])Li(\d+)EE[^']*)'.*?Used (\d+) registers", log, re.S):
        regs[f"k_long<{'float' if m.group(2) == 'f' else 'int16_t'}, {m.group(3)}>"] = int(m.group(4))
    return regs


def build(force=False, verbose=False):
    if force or _stale():
        if shutil.which("nvcc") is None:
            raise RuntimeError("nvcc not found: lewton_b200 has no CPU fallback and cannot be built without CUDA")
        r = subprocess.run(["make", "-C", CSRC, "-B"], capture_output=True, text=True)
        if verbose or r.returncode:
            print(r.stdout)
            print(r.stderr)
        if r.returncode:
            raise RuntimeError("nvcc build of liblewton_b200.so failed")
        regs = hot_kernel_registers(r.stdout + r.stderr)
        if len(regs) != 16:
            print(f"lewton_b200 build: WARNING: found {len(regs)} of the 16 k_long instantiations in the ptxas log")
        if any(v > (252 if k.endswith(", 1>") else 254) for k, v in regs.items()):
            print(f"lewton_b200 build: WARNING: {regs} -- k_long above 252 registers (planar) / 254 (interleaved) has "
                  "measured 3-4 % slower; look at what changed in kernel_long.cuh's shared helpers")
        n = check_no_fma()
        if n:
            os.remove(SO)
            raise RuntimeError(f"{n} fused multiply-add instructions in the kernels' SASS: bit parity with "
                               "the reference would be lost (see kernel_long.cuh vadd_p/vsub_p)")
    return SO


if __name__ == "__main__":
    print(build(force=True, verbose=True))
