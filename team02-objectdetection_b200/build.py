"""Build libb200seg.so in-tree with nvcc for sm_100a (no torch headers, plain C ABI).

    python team02-objectdetection_b200/build.py [--force] [--verbose]

The .so lands next to the Python package (b200seg/libb200seg.so) so that it travels with the repo
snapshot to the GPU box.  cudart is linked statically; the driver API (cuTensorMapEncodeTiled) is
resolved at run time through cudaGetDriverEntryPoint, so the library loads on a GPU-less host.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "b200seg", "libb200seg.so")
SOURCES = ["runtime.cu", "hbm_ops.cu", "conv_simt.cu", "conv_tc.cu", "conv_rs.cu", "softmax_ce.cu", "train_ops.cu", "conv_wgrad_tc.cu", "mbconv.cu", "adam.cu", "preprocess.cu", "generic_ops.cu", "tail_fused.cu", "stem_mb1.cu", "bn_cluster.cu", "seg_metrics.cu", "postprocess.cu", "softmax_ce_ex.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
         "-Xcompiler", "-fPIC"]


def _newest(paths):
    return max(os.path.getmtime(p) for p in paths)


def build(force=False, verbose=False):
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps = srcs + [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "seg_metrics.cuh"), os.path.join(HERE, "..", "include", "b200seg.h"), __file__]
    if not force and os.path.exists(OUT) and os.path.getmtime(OUT) >= _newest(deps):
        return OUT
    objs = []
    procs = []
    for s in srcs:
        o = s[:-3] + ".o"
        cmd = [NVCC, *FLAGS, "-c", s, "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            print(" ".join(cmd)); print(out)
        if p.returncode:
            raise RuntimeError("nvcc failed: " + " ".join(cmd))
    link = [NVCC, "-shared", "-o", OUT, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        print(r.stdout)
        raise RuntimeError("link failed")
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
