"""Resident blocks per SM of the lane-per-env step kernels (graphenvs_b200/csrc/ge_lane.cu) at the dynamic shared memory their
launches ask for (lane_smem), from cudaOccupancyMaxActiveBlocksPerMultiprocessor on the device, with their registers and local
memory (cudaFuncGetAttributes).  The staged kernels' residency is set by the adjacency tile each one-tile block stages, so this is
the number to check whenever that tile changes.

Compiles a small probe that includes ge_lane.cu (nvcc, sm_100a) in a temporary directory and prints one JSON line per kernel and N:

    python profiles/lane_occupancy.py [--N 10 33 50 64] [--out FILE]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PROBE = r"""
#include <cstdio>
#include <cstdlib>
#include "ge_lane.cu"
extern "C" int ge_set_error(int code, const char *, ...) { return code; }
int ge_grant_smem(const void *, size_t) { return GE_OK; }

template <class K> static void probe(const char *name, K kernel, int N, size_t smem) {
    if (smem > 48 * 1024) cudaFuncSetAttribute((const void *)kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int blocks = -1;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks, kernel, LANE_T, smem);
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, (const void *)kernel);
    printf("{\"kernel\": \"%s\", \"N\": %d, \"dyn_smem\": %zu, \"static_smem\": %zu, \"blocks_per_sm\": %d, \"regs\": %d, "
           "\"local_bytes\": %zu, \"status\": \"%s\"}\n", name, N, smem, a.sharedSizeBytes, blocks, a.numRegs, a.localSizeBytes,
           cudaGetErrorString(e));
}

int main(int argc, char **argv) {
    cudaDeviceProp p;
    cudaGetDeviceProperties(&p, 0);
    printf("{\"device\": \"%s\", \"sms\": %d, \"smem_per_sm\": %zu, \"reserved_smem_per_block\": %zu}\n", p.name,
           p.multiProcessorCount, p.sharedMemPerMultiprocessor, p.reservedSharedMemPerBlock);
    for (int i = 1; i < argc; ++i) {
        ge_batch d = {};
        d.kind = GE_LONGEST_PATH; d.parenting = 2; d.N = atoi(argv[i]); d.NW = (d.N + 31) / 32;
        const size_t smem = lane_smem(&d);
        probe("lane_step_kernel<1, 1>", lane_step_kernel<true, true>, d.N, smem);
        probe("lane_step_kernel<1, 0>", lane_step_kernel<true, false>, d.N, smem);
    }
    probe("lane_step_kernel<0, 1>", lane_step_kernel<false, true>, 0, 0);
    return 0;
}
"""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--N", type=int, nargs="+", default=[10, 33, 50, 64])
    ap.add_argument("--out", default=None, help="also append the lines to this file")
    args = ap.parse_args()
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    csrc = os.path.join(ROOT, "graphenvs_b200", "csrc")
    with tempfile.TemporaryDirectory() as td:
        src, exe = os.path.join(td, "probe.cu"), os.path.join(td, "probe")
        open(src, "w").write(PROBE)
        subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-I", os.path.join(ROOT, "include"),
                               "-I", csrc, src, "-o", exe])
        out = subprocess.check_output([exe] + [str(n) for n in args.N]).decode()
    lines = [json.loads(s) for s in out.splitlines() if s.strip()]
    for rec in lines:
        print(json.dumps(rec))
    if args.out:
        with open(args.out, "a") as f:
            for rec in lines:
                f.write(json.dumps(rec) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
