#!/usr/bin/env python
"""Cost of the per-sample log-weights and posterior-predictive draws (gwi_sample_log_weights / gwi_draw_samples) on the
BASELINE workloads: gwi_model_create time and device memory with and without keep_sample_index, the time of one
log-weight pass and of one draw call (E draws from the events, one each, and E draws from the injections), and the
host likelihood call for scale.  Times are host wall clock around the call and a device synchronise, after warm-up,
median of --repeat calls.  Prints one JSON line per workload, preceded by one with the GPU name and power limit.

    python tools/draw_probe.py --workloads cfg1 cfg2 cfg3 cfg5
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from gwinferno_b200 import capi, workloads  # noqa: E402


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")[:2]]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # no nvidia-smi: the name from the runtime, no power limit
        return {"gpu": "unknown", "power_limit": "unknown", "error": str(e)}


def mem_used():
    free, total = C.c_size_t(), C.c_size_t()
    rt = capi.cudart()
    rt.cudaMemGetInfo.argtypes = [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    capi._cuda_check(rt.cudaMemGetInfo(C.byref(free), C.byref(total)), "cudaMemGetInfo")
    return total.value - free.value


def timed(fn, repeat):
    fn()
    capi.synchronize()
    ts = []
    for _ in range(repeat):
        t0 = time.perf_counter()
        fn()
        capi.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def probe(name, repeat):
    pe, inj, const, z_range = workloads.shard_catalog(name, 0, 1, scale=1.0, all_reduce_minmax=lambda lo, hi: (lo, hi))
    weights, params_fn = workloads.build_model(const["family"], pe, inj, z_range=z_range)
    low, lam, _ = workloads.lower_workload(weights, params_fn, pe, inj)
    cat = capi.Catalog(low.pe_cols, low.inj_cols, const["total_inj"])
    E, P = cat.n_events, low.spec.n_params
    n_cat = int(cat.offsets[-1]) + cat.n_inj
    row = {"workload": name, "events": E, "pe_samples": int(cat.offsets[-1]), "injections": cat.n_inj}
    lib = capi.load_library()
    for keep in (False, True):
        capi.synchronize()
        m0 = mem_used()
        t0 = time.perf_counter()
        mdl = capi.Model(cat, low.spec, keep_sample_index=keep)
        t_create = time.perf_counter() - t0
        tag = "with_index" if keep else "without_index"
        row[f"model_create_s_{tag}"] = t_create
        row[f"model_device_bytes_{tag}"] = mem_used() - m0
        row[f"n_padded_{tag}"] = mdl.info()["n_padded"]
        row[f"loglike_host_s_{tag}"] = timed(lambda: mdl.loglike_host(lam, E), repeat)
        if keep:
            lam_d, out_d, idx_d = capi.DeviceBuffer(P), capi.DeviceBuffer(n_cat), capi.DeviceBuffer(2 * E)
            lam_d.upload(lam)
            row["sample_log_weights_s"] = timed(lambda: capi._check(lib.gwi_sample_log_weights(mdl.handle, C.c_void_p(lam_d.ptr), C.c_void_p(out_d.ptr), None)), repeat)
            m0 = mem_used()
            row["draw_samples_s"] = timed(lambda: capi._check(lib.gwi_draw_samples(mdl.handle, C.c_void_p(lam_d.ptr), 7, 1, E, C.c_void_p(idx_d.ptr), None)), repeat)
            row["draw_scratch_device_bytes"] = mem_used() - m0  # allocated by the first (warm-up) draw call
            for b in (lam_d, out_d, idx_d):
                b.free()
        mdl.close()
    cat.close()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", nargs="+", default=["cfg1", "cfg2", "cfg3", "cfg5"], choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--repeat", type=int, default=10)
    args = ap.parse_args()
    print(json.dumps(gpu_identity()), flush=True)
    for name in args.workloads:
        print(json.dumps(probe(name, args.repeat)), flush=True)


if __name__ == "__main__":
    main()
