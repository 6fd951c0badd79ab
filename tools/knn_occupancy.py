"""Resident CTAs per SM of the histogram-select kNN kernels at the dynamic shared memory their launches request.

The kernels are internal to the library, so their cubin is extracted from it (cuobjdump) and loaded through the
driver API; cuOccupancyMaxActiveBlocksPerMultiprocessor then answers for the registers the compiler gave each
kernel and the per-thread buffer of `cap` candidate entries plus 16-bit bins (kp_grid.cu, hq_smem).

    python tools/knn_occupancy.py [--lib kinectpy_b200/libkinectpy_b200.so] [--entry-bytes 4]

--entry-bytes 8 sizes the buffer as builds before the 4-byte entry did, so that their libraries can be compared.
Prints one JSON line.  Needs a CUDA device."""
import argparse
import ctypes as C
import glob
import json
import os
import re
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (label, mangled-name suffix, threads per CTA, bins, slack: capacity = k + slack) of the launches in kp_knn_batch_level0 / _mid
KERNELS = [
    ("k_knn_hist_b<64,1,64>", "k_knn_hist_bILi64ELi1ELi64EEEvNS_12KnnBatchArgsE", 64, 64, 8),      # k > 32, level 0
    ("k_knn_mid_b", "k_knn_mid_bENS_12KnnBatchArgsE", 64, 64, 24),                                 # k > 32, mid level
    ("k_knn_hist_b<32,1,128>", "k_knn_hist_bILi32ELi1ELi128EEEvNS_12KnnBatchArgsE", 128, 32, 8),   # k <= 32, level 0
]
CU_FUNC_ATTRIBUTE_NUM_REGS = 4
CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES = 8
CU_DEVICE_ATTRIBUTE_MAX_SHARED_MEMORY_PER_MULTIPROCESSOR = 81


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed: CUresult %d" % (what, rc))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=os.path.join(ROOT, "kinectpy_b200", "libkinectpy_b200.so"))
    ap.add_argument("--entry-bytes", type=int, default=4, choices=[4, 8])
    ap.add_argument("--ks", default="50,20", help="neighbour counts to size the buffers for")
    args = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(args.lib)], cwd=tmp, check=True, capture_output=True)
        cubin, names = None, {}
        for f in sorted(glob.glob(os.path.join(tmp, "*.cubin"))):
            data = open(f, "rb").read()
            for _, kname, *_ in KERNELS:
                m = re.search(rb"_Z\w*?kp_grid_cu_\w*?" + re.escape(kname.encode()) + rb"(?!\w)", data)
                if m:
                    cubin, names[kname] = f, m.group(0)
        if cubin is None or len(names) != len(KERNELS):
            raise RuntimeError("kNN kernels not found in %s" % args.lib)
        cu = C.CDLL("libcuda.so.1")
        check(cu.cuInit(0), "cuInit")
        dev, ctx, mod = C.c_int(), C.c_void_p(), C.c_void_p()
        check(cu.cuDeviceGet(C.byref(dev), 0), "cuDeviceGet")
        check(cu.cuDevicePrimaryCtxRetain(C.byref(ctx), dev), "cuDevicePrimaryCtxRetain")
        check(cu.cuCtxSetCurrent(ctx), "cuCtxSetCurrent")
        check(cu.cuModuleLoad(C.byref(mod), cubin.encode()), "cuModuleLoad")
        smem_sm = C.c_int()
        check(cu.cuDeviceGetAttribute(C.byref(smem_sm), CU_DEVICE_ATTRIBUTE_MAX_SHARED_MEMORY_PER_MULTIPROCESSOR, dev), "cuDeviceGetAttribute")
        rows = []
        for k in [int(x) for x in args.ks.split(",")]:
            for label, kname, T, nb, slack in KERNELS:
                if (nb == 32) != (k <= 32):
                    continue
                fn = C.c_void_p()
                check(cu.cuModuleGetFunction(C.byref(fn), mod, names[kname]), "cuModuleGetFunction")
                regs = C.c_int()
                check(cu.cuFuncGetAttribute(C.byref(regs), CU_FUNC_ATTRIBUTE_NUM_REGS, fn), "cuFuncGetAttribute")
                cap = k + slack
                smem = T * (cap * args.entry_bytes + nb * 2)
                check(cu.cuFuncSetAttribute(fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, smem), "cuFuncSetAttribute")
                n = C.c_int()
                check(cu.cuOccupancyMaxActiveBlocksPerMultiprocessor(C.byref(n), fn, T, C.c_size_t(smem)), "cuOccupancyMaxActiveBlocksPerMultiprocessor")
                rows.append({"kernel": label, "k": k, "cap": cap, "entry_bytes": args.entry_bytes, "threads": T, "regs": regs.value,
                             "dyn_smem_bytes": smem, "ctas_per_sm": n.value, "warps_per_sm": n.value * T // 32})
        cu.cuModuleUnload(mod)
        cu.cuDevicePrimaryCtxRelease(dev)
    print(json.dumps({"lib": os.path.relpath(os.path.abspath(args.lib), ROOT), "smem_per_sm": smem_sm.value, "kernels": rows}))


if __name__ == "__main__":
    main()
