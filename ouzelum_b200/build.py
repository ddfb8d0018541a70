"""Build libouzelum_b200.so in-tree with nvcc for sm_100a (B200).  `python ouzelum_b200/build.py [--force] [-v]`
(run it as a script: importing the package first would try to load the library being built).

Flags that matter:
  -gencode arch=compute_100a,code=sm_100a   Blackwell-only SASS (no PTX fallback for other archs)
  -fmad=false                                no implicit contraction: every float op is individually rounded and fused
                                             multiply-adds are explicit (fmaf) => bit-exact against the op-ordered CPU oracles
  -lineinfo                                  ncu source-page attribution
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libouzelum_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# Floating-point contract: EVERY translation unit is compiled without FMA contraction (-fmad=false); fused multiply-adds are
# written explicitly (fmaf / fma) where they pay.  The env-step arithmetic is therefore bit-exact against the op-ordered CPU
# oracles wherever it is instantiated (quad_step.cu, quadcopter.cu AND the one-launch EKFLeeLanded step), and the estimator /
# controller device functions give identical bits in the fused kernel and in the stand-alone companion kernels.
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "-Xcompiler", "-fPIC", "-fmad=false"]


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "ouzelum_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs, procs = [], []
    for src in sources():
        name = os.path.basename(src)
        obj = os.path.join(objdir, name[:-3] + ".o")
        cmd = [NVCC] + FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
        objs.append(obj)
    for cmd, pr in procs:
        out, err = pr.communicate()
        if verbose or pr.returncode != 0:
            sys.stderr.write(out + err)
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed:\n" + " ".join(cmd))
    cmd = [NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", OUT] + objs
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed:\n" + " ".join(cmd))
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
