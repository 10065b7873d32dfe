"""FastGlobalRegistration timings on seeded scenes (bench.py is not involved).

    python tools/bench_fgr.py [--sizes 20000,100000,200000] [--runs 5] [--out FILE]

Per size: random 33-dim features and clouds of n points per fragment (the two feature sets, 2 x n x 132 B, fit in
the B200's 126 MB L2 up to n of about 400 k, so the matcher reads them from L2 after the first pass).  CUDA-event
times, median of --runs after one warm-up, of each stage:
  matcher   one-way cphb_feature_nn with preallocated outputs (launch + decode, no allocation or copy in the window)
  matching  cphb_fgr_advanced_matching: normalisation, two-way matcher, cross check, tuple test, truncation
  gnc       the pose loop kernel alone (cphb_icp_result.loop_ms of cphb_fast_global_registration)
  evaluate  cphb_evaluate_registration on the original clouds with the final pose
  fgr       the whole cphb_fast_global_registration call
The matcher's rate is pairs/s and two shares of peak: instruction issue (one FSUB + one FFMA per feature per pair
against SM count x 128 FP32 lanes x the card's max SM clock) and FLOP (FSUB 1 + FFMA 2 against SM x 128 x 2 x clock).
Comparison points, labelled: a chunked torch.cdist + argmin (speed reference only, not bit-exact) and the CPU
oracle (warmed, on a 200-row sample, extrapolated)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().split("\n")[0]
    name, pl, clk = [x.strip() for x in q.split(",")]
    return {"name": name, "power_limit_w": float(pl), "max_sm_clock_mhz": float(clk)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="20000,100000,200000")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import cupoch_b200 as cph
    import fgr_oracle as F
    R = cph.registration
    _ = cph._lib.lib()
    info = card()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    peak = sms * 128 * 2 * info["max_sm_clock_mhz"] * 1e6  # FP32 FLOP/s (an FMA counted as 2)
    out = {"card": info, "sm_count": sms, "fp32_peak_flops": peak, "runs": a.runs, "sizes": []}

    def timed(fn):
        fn()
        ts = []
        for _ in range(a.runs):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    import ctypes as C
    L = cph._lib.lib()
    F.feature_nn(np.zeros((1, 33), np.float32), np.zeros((1, 33), np.float32))  # builds the oracle library
    for n in [int(s) for s in a.sizes.split(",")]:
        rng = np.random.default_rng(n)
        fs = torch.from_numpy(rng.uniform(0, 100, (n, 33)).astype(np.float32)).cuda()
        ft = torch.from_numpy(rng.uniform(0, 100, (n, 33)).astype(np.float32)).cuda()
        ps = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
        pt = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
        Fs, Ft = R.Feature(fs), R.Feature(ft)
        S, T = cph.geometry.PointCloud(ps), cph.geometry.PointCloud(pt)
        opt = R.FastGlobalRegistrationOption()
        copt = opt._c()
        idx = cph.utility.DeviceArray((n,), np.int32)
        d2 = cph.utility.DeviceArray((n,), np.float32)
        pairs = cph.utility.DeviceArray((opt.maximum_tuple_count, 2), np.int32)
        corr = cph.utility.DeviceArray((n, 2), np.int32)
        counts = (C.c_int64 * 4)()
        sc, tc = S._cloud(False), T._cloud(False)
        res = cph._lib.IcpResult()
        row = {"n": n}
        row["matcher_one_way_ms"] = timed(lambda: L.cphb_feature_nn(Fs.data.ptr, n, Ft.data.ptr, n, 33, idx.ptr, d2.ptr,
                                                                     None, None, None))
        row["matching_ms"] = timed(lambda: L.cphb_fgr_advanced_matching(S._points.ptr, n, T._points.ptr, n, Fs.data.ptr, n,
                                                                        Ft.data.ptr, n, 33, C.byref(copt), pairs.ptr, counts,
                                                                        None))
        gnc = []

        def fgr():
            L.cphb_fast_global_registration(C.byref(sc), C.byref(tc), Fs.data.ptr, n, Ft.data.ptr, n, 33, C.byref(copt),
                                            C.byref(res), corr.ptr, None, None)
            gnc.append(res.loop_ms)
        row["fgr_end_to_end_ms"] = timed(fgr)
        row["gnc_ms"] = float(np.median(gnc[1:]))
        row["pairs"], row["mutual"] = int(counts[0]), int(counts[1])
        Tf = (C.c_float * 16)(*res.transformation)
        row["evaluate_ms"] = timed(lambda: L.cphb_evaluate_registration(C.byref(sc), C.byref(tc),
                                                                        opt.maximum_correspondence_distance, Tf,
                                                                        C.byref(res), corr.ptr, None))
        pairs_n = float(n) * n
        sec = row["matcher_one_way_ms"] * 1e-3
        row["matcher_pairs_per_s"] = pairs_n / sec
        row["matcher_share_of_fp32_issue_peak"] = pairs_n * 33 * 2 / sec / (sms * 128 * info["max_sm_clock_mhz"] * 1e6)
        row["matcher_share_of_fp32_flop_peak"] = pairs_n * 33 * 3 / sec / peak

        def cdist():
            for c in range(0, n, 16384):
                torch.cdist(ft[c:c + 16384], fs).argmin(1)
        row["torch_cdist_argmin_ms_speed_reference_not_bit_exact"] = timed(cdist)
        m = 200
        fs_h, ft_h = fs.cpu().numpy(), ft[:m].cpu().numpy()
        t0 = time.perf_counter()
        F.feature_nn(fs_h, ft_h)
        row["cpu_oracle_ms_for_%d_rows" % m] = (time.perf_counter() - t0) * 1e3
        row["cpu_oracle_ms_extrapolated_all_rows"] = row["cpu_oracle_ms_for_%d_rows" % m] * n / m
        out["sizes"].append(row)
        print(json.dumps(row), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    print(json.dumps({"card": info, "sm_count": sms}))


if __name__ == "__main__":
    main()
