"""The pruned NN-1 chain against the full sweep, per kernel, on the shapes it serves.

    python tools/nn1_prune_bench.py [--reps 20] [--model-only]

For face clouds (sigma 0.01) from configs[1] (B=32, N=M=4096) to configs[4] (B=512, N=M=16384) and for unrelated uniform clouds (B=32,
N=M=4096, the worst case) it prints one JSON line each with
  k1_us / k2_us / k3_us   nn1_bucket, nn1_pruned_sweep and the fix-up (torch.profiler kernel times, median over reps,
                          L2 overwritten before every rep)
  old_us                  the full chain (arm + sweep + fix-up) at the same inputs, selected by passing the tiling that the
                          library would choose for it (an explicit tiling keeps the full sweep)
  kept_pairs_frac         evaluated pairs / B*N*M, both directions, from a numpy model of the bucketing, the seeds and the two
                          filter stages (box against U, then point against the lane's running minimum, candidates in index
                          order); float64 minima, so it is a model, not a count
  k2_gpairs_per_s         evaluated pairs per second of the pruned sweep, from the model's pair count

    python tools/nn1_prune_bench.py --count

runs the same workloads on a -DPCD_SWEEP_TRACE build of the library (tools/libpcdist_trace.so, built if missing) and prints
what the pruned sweep counted instead of times: counted_pairs_frac (evaluated chunks * 32 * 32 / B*N*M, exact for whole
chunks), and per item the evaluated chunks, arg-min re-scans and tie passes.  It also reads the bucketing pass's phase stamps
(%globaltimer, thread 0 of every CTA) and prints k1_phases_us: the median over CTAs of each phase (start -> loads and joint
box -> codes -> sort pass 1 -> sort pass 2 -> gather and stores), and k1_span_us, first CTA start to last CTA end.  The
stamps of the trace build add barriers of their own, so the phases are a breakdown, not the release kernel's time.
"""
import argparse
import ctypes
import importlib
import importlib.util
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
TRACE_LIB = os.path.join(ROOT, "tools", "libpcdist_trace.so")
if "--count" in sys.argv:          # before the package import: the library path is read once, at import
    os.environ["PCDIST_LIBRARY"] = TRACE_LIB
synth = importlib.import_module("3dpointcloudattack_b200.synth")

BITS = 5
MARGIN_REL, MARGIN_ABS, LB_SCALE = 40.0 * 2.0 ** -24, 2.0 ** -100, 1.0 - 2.0 ** -20


def _spread(v):
    out = np.zeros_like(v)
    for k in range(BITS):
        out |= ((v >> k) & 1) << (3 * k)
    return out


def model_sample(rows, cols):
    """Evaluated (row chunk, column chunk) pairs of one sample, both directions, mirroring nn1_bucket / nn1_pruned_sweep."""
    both = np.concatenate([rows, cols]).astype(np.float64)
    lo, hi = both.min(0), both.max(0)
    cell = np.where(hi > lo, 2.0 ** BITS / np.where(hi > lo, hi - lo, 1), 0)
    sides = []
    for p in (rows, cols):
        q = np.clip((p - lo) * cell, 0, 2 ** BITS - 1).astype(np.int64)
        code = _spread(q[:, 0]) | (_spread(q[:, 1]) << 1) | (_spread(q[:, 2]) << 2)
        s = p[np.argsort(code, kind="stable")].astype(np.float64)
        nc = (len(s) + 31) // 32
        ch = [s[k * 32:(k + 1) * 32] for k in range(nc)]
        sides.append((ch, np.array([c.min(0) for c in ch]), np.array([c.max(0) for c in ch]),
                      np.array([(c ** 2).sum(1).max() for c in ch])))
    kept = 0
    for own, opp in ((sides[0], sides[1]), (sides[1], sides[0])):
        ch_o, lo_o, hi_o, n_o = own
        ch_c, lo_c, hi_c, n_c = opp
        for c, pts in enumerate(ch_o):
            cs = c * len(ch_c) // len(ch_o)
            seeds = [k for k in (cs - 1, cs, cs + 1) if 0 <= k < len(ch_c)]
            cand = np.concatenate([ch_c[k] for k in seeds])
            best = ((pts[:, None, :] - cand[None]) ** 2).sum(-1).min(1)
            kept += len(pts) * len(cand)
            # box stage against U = the largest seed minimum
            gap = np.maximum(np.maximum(lo_c - hi_o[c], lo_o[c] - hi_c), 0)
            lb = (gap ** 2).sum(1) * LB_SCALE
            keep = ~(lb - (MARGIN_REL * (n_o[c] + n_c) + MARGIN_ABS) > best.max())
            keep[seeds] = False
            # point stage, in index order, against each point's running minimum
            pn = (pts ** 2).sum(1)
            for k in np.flatnonzero(keep):
                g = np.maximum(np.maximum(lo_c[k] - pts, pts - hi_c[k]), 0)
                lbp = (g ** 2).sum(1) * LB_SCALE
                if (~(lbp - (MARGIN_REL * (pn + n_c[k]) + MARGIN_ABS) > best)).any():
                    best = np.minimum(best, ((pts[:, None, :] - ch_c[k][None]) ** 2).sum(-1).min(1))
                    kept += len(pts) * len(ch_c[k])
    return kept


K1_PHASES = ("loads_box", "codes", "sort1", "sort2", "gather_store")     # the ends of nn1_bucket's phases: stamps 1 .. 5


def counts(adv, ori):
    """The pruned sweep's own counters over one call (trace build): items, evaluated chunks, arg-min re-scans, tie passes,
    and the bucketing pass's phase stamps (8 words per CTA: its start, then the end of each phase of K1_PHASES)."""
    import torch
    pcd = importlib.import_module("3dpointcloudattack_b200")
    F, lib = pcd.functional, pcd._lib.load()
    a, o = torch.from_numpy(adv).cuda(), torch.from_numpy(ori).cuda()
    F.nn1(a, o, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    buf = torch.zeros(4, dtype=torch.int64, device="cuda")
    fn = lib.pcd_debug_set_prune_counters
    fn.restype, fn.argtypes = ctypes.c_int, [ctypes.c_void_p]
    torch.cuda.synchronize()
    assert fn(buf.data_ptr()) == 0
    F.nn1(a, o, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    torch.cuda.synchronize()
    assert fn(None) == 0
    items, chunks, scans, ties = buf.tolist()
    B, N, M = a.shape[0], a.shape[1], o.shape[1]
    stamps = torch.zeros(2 * B * 8, dtype=torch.int64, device="cuda")
    st = lib.pcd_debug_set_sweep_trace
    st.restype, st.argtypes = ctypes.c_int, [ctypes.c_void_p]
    assert st(stamps.data_ptr()) == 0
    F.nn1(a, o, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
    torch.cuda.synchronize()
    assert st(None) == 0
    t = stamps.cpu().numpy().reshape(-1, 8).astype(np.float64)
    end = len(K1_PHASES)
    phases = {name: round(float(np.median(t[:, k + 1] - t[:, k])) / 1e3, 2) for k, name in enumerate(K1_PHASES)}
    return {"counted_pairs_frac": chunks * 32 * 32 / (B * N * M), "chunks_per_item": chunks / items,
            "rescans_per_item": scans / items, "tie_passes_per_item": ties / items,
            "k1_phases_us": phases, "k1_span_us": round(float(t[:, end].max() - t[:, 0].min()) / 1e3, 2)}


def inputs(kind, B, n):
    if kind == "uniform":
        rs = np.random.RandomState(5)
        return rs.rand(B, n, 3).astype(np.float32), rs.rand(B, n, 3).astype(np.float32)
    ori = synth.face_clouds(min(B, 8), n, seed=1234)
    adv = synth.perturb(ori, 0.01, seed=99)
    rep = (B + ori.shape[0] - 1) // ori.shape[0]
    return (adv.numpy().repeat(rep, 0)[:B].copy(), ori.numpy().repeat(rep, 0)[:B].copy())


def gpu_times(adv, ori, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    pcd = importlib.import_module("3dpointcloudattack_b200")
    F, lib = pcd.functional, pcd._lib.load()
    a, o = torch.from_numpy(adv).cuda(), torch.from_numpy(ori).cuda()
    B, N, M = a.shape[0], a.shape[1], o.shape[1]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    R, mt = ctypes.c_int(), ctypes.c_int()
    assert lib.pcd_nn1_query_tiling(B, N, M, ctypes.byref(R), ctypes.byref(mt)) == 0
    groups = {"k1": ("nn1_bucket_kernel",), "k2": ("nn1_pruned_sweep_kernel",), "k3": ("nn1_fixup",),
              "old": ("nn1_arm_kernel", "nn1_sweep_kernel", "nn1_fixup")}
    out = {}
    for chain, tiling in (("new", (0, 0)), ("old", (R.value, mt.value))):
        F.force_tiling(*tiling)
        try:
            for _ in range(3):
                F.nn1(a, o, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
            torch.cuda.synchronize()
            per = {k: [] for k in groups}
            for _ in range(reps):
                flush.fill_(1)
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    F.nn1(a, o, F.FORM_SUM_FIRST, F.NORM_FMA, cache=False)
                    torch.cuda.synchronize()
                ev = [(e.name, e.device_time) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
                for k, names in groups.items():
                    per[k].append(sum(t for n_, t in ev if any(s in n_ for s in names)))
        finally:
            F.force_tiling(0, 0)
        keys = ("old",) if chain == "old" else ("k1", "k2", "k3")
        for k in keys:
            out[k + "_us"] = float(np.median(per[k]))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--model-only", action="store_true")
    ap.add_argument("--model-samples", type=int, default=2)
    ap.add_argument("--count", action="store_true")
    args = ap.parse_args()
    if args.count and not os.path.exists(TRACE_LIB):
        spec = importlib.util.spec_from_file_location("_b", os.path.join(ROOT, "3dpointcloudattack_b200", "build.py"))
        b = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(b)
        b.build(extra_flags=["-DPCD_SWEEP_TRACE"], out=TRACE_LIB)
    for name, kind, B, n in (("configs1", "face", 32, 4096), ("face_b32_n8192", "face", 32, 8192), ("face_b16_n16384", "face", 16, 16384),
                             ("face_b64_n16384", "face", 64, 16384), ("configs4", "face", 512, 16384), ("uniform", "uniform", 32, 4096)):
        adv, ori = inputs(kind, B, n)
        S = min(args.model_samples, B)
        frac = sum(model_sample(adv[b], ori[b]) for b in range(S)) / (S * n * n)
        res = {"workload": name, "B": B, "N": n, "kept_pairs_frac": frac}
        if args.count:
            res.update(counts(adv, ori))
        elif not args.model_only:
            import torch
            res["gpu"] = torch.cuda.get_device_name(0)
            res.update(gpu_times(adv, ori, args.reps))
            res["k2_gpairs_per_s"] = frac * B * n * n / (res["k2_us"] * 1e-6) / 1e9
            res["new_over_old"] = (res["k1_us"] + res["k2_us"] + res["k3_us"]) / res["old_us"]
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
