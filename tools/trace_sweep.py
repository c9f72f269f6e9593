"""Per-CTA timeline of the NN-1 sweep (development tool): builds a -DPCD_SWEEP_TRACE variant of the
library, runs BASELINE config 2 and prints when CTAs start, reach their first tile, leave the loop
and finish, relative to the earliest CTA start.  It passes the tiling the library would choose, which
keeps the full sweep on shapes the pruned chain serves (whose bucketing pass writes other stamps).

    python tools/trace_sweep.py [B N M]
"""
import importlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
VARIANT = os.path.join(ROOT, "tools", "libpcdist_trace.so")


def main():
    spec = importlib.util.spec_from_file_location("_b", os.path.join(ROOT, "3dpointcloudattack_b200", "build.py"))
    b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)
    b.build(extra_flags=["-DPCD_SWEEP_TRACE"], out=VARIANT)
    if "--build-only" in sys.argv:
        return
    os.environ["PCDIST_LIBRARY"] = VARIANT
    import ctypes
    import numpy as np
    import torch
    pcd = importlib.import_module("3dpointcloudattack_b200")
    synth = importlib.import_module("3dpointcloudattack_b200.synth")
    F = pcd.functional
    lib = pcd._lib.load()
    args = [int(a) for a in sys.argv[1:] if a.isdigit()]
    B, N, M = (args + [32, 4096, 4096])[:3] if len(args) < 3 else args[:3]
    ori = synth.face_clouds(min(B, 4), N, seed=1).cuda().repeat((B + 3) // 4, 1, 1)[:B].contiguous()
    adv = (ori + 0.01 * torch.randn_like(ori))[:, :M].contiguous()
    trace = torch.zeros(4096 * 8, dtype=torch.int64, device="cuda")
    R, mt = ctypes.c_int(), ctypes.c_int()
    assert lib.pcd_nn1_query_tiling(B, N, M, ctypes.byref(R), ctypes.byref(mt)) == 0
    F.force_tiling(R.value, mt.value)
    for _ in range(3):
        F.nn1(ori, adv, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    torch.cuda.synchronize()
    fn = lib.pcd_debug_set_sweep_trace
    fn.restype = ctypes.c_int; fn.argtypes = [ctypes.c_void_p]
    assert fn(trace.data_ptr()) == 0
    F.nn1(ori, adv, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    torch.cuda.synchronize()
    fn(None)
    F.force_tiling(0, 0)
    t = trace.cpu().numpy().reshape(-1, 8)
    t = t[t[:, 0] > 0]
    t0 = t[:, 0].min()
    start, loop_end, end, smid, first = (t[:, 0] - t0) / 1e3, (t[:, 1] - t0) / 1e3, (t[:, 2] - t0) / 1e3, t[:, 3], (t[:, 4] - t0) / 1e3
    def q(x):
        return "min %.1f  p10 %.1f  med %.1f  p90 %.1f  max %.1f" % (x.min(), np.percentile(x, 10), np.median(x), np.percentile(x, 90), x.max())
    print(f"B={B} N={N} M={M}: {len(t)} CTAs on {len(set(smid.tolist()))} SMs  (times in us after the first CTA start)")
    print("  CTA start        ", q(start))
    print("  first tile ready ", q(first))
    print("  loop end         ", q(loop_end))
    print("  CTA end          ", q(end))
    print("  CTA busy (end-start)", q(end - start))
    # per SM: when the first / the last of its co-resident CTAs finished
    sm_first, sm_last = {}, {}
    for i in range(len(t)):
        k = int(smid[i])
        sm_first[k] = min(sm_first.get(k, 1e9), float(end[i])); sm_last[k] = max(sm_last.get(k, 0.0), float(end[i]))
    print("  per SM: first CTA done", q(np.array(list(sm_first.values()))))
    print("  per SM: last CTA done ", q(np.array(list(sm_last.values()))))
    # per-SM: co-resident CTAs
    order = np.argsort(end)
    print("  earliest-finishing CTAs:", [(int(i), round(float(end[i]), 1)) for i in order[:5]])
    print("  latest-finishing CTAs:  ", [(int(i), round(float(end[i]), 1)) for i in order[-5:]])
    # phase cycles of warp 0 of every CTA (clock64): row switch | compute | convert + barrier wait | flush
    row_c, comp_c = t[:, 5].astype(np.float64), t[:, 6].astype(np.float64)
    bar_c, flush_c = (t[:, 7] >> 32).astype(np.float64), (t[:, 7] & 0xffffffff).astype(np.float64)
    tot = row_c + comp_c + bar_c + flush_c
    early = end < np.median(end)                      # the CTA of each SM that finishes first / last
    for name, sel in (("first-finishing CTAs", early), ("last-finishing CTAs", ~early)):
        print(f"  {name}: cycles/1000  row switch {row_c[sel].mean()/1e3:.1f}  compute {comp_c[sel].mean()/1e3:.1f}  "
              f"convert+barrier {bar_c[sel].mean()/1e3:.1f}  flush {flush_c[sel].mean()/1e3:.1f}  (sum {tot[sel].mean()/1e3:.1f} = "
              f"{tot[sel].mean()/1.965e3:.1f} us at 1.965 GHz)")
    ts = np.unique(t[:, :3])
    print("  globaltimer granularity (ns):", int(np.diff(ts).min()) if len(ts) > 1 else -1)


if __name__ == "__main__":
    main()
