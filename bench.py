#!/usr/bin/env python
"""bench.py -- Chamfer+Hausdorff fwd+bwd throughput of the B200 point-set distance path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

One "step" = one fused bidirectional Chamfer + Hausdorff forward AND backward over the batch
(BASELINE.json configs[1]: B=32, N=M=4096, fp32, synthetic face clouds, adv = ori + N(0, 0.01^2)),
through the reference-shaped Python surface (distance.chamfer / distance.hausdorff on the same
tensors -> one sweep) and loss.backward().  Unit of work = ALGORITHMIC pairs B*N*M per step (the
reference evaluates the matrix twice; we count it once), 8 FLOP per pair.

value      device-timed (CUDA events per step, L2 flushed between steps outside the event pairs),
           inputs resident in HBM, max over ranks.
e2e        same step from pinned HOST buffers: H2D of adv and ori, fwd+bwd, D2H of the four
           loss vectors and the gradient w.r.t. adv; host<->device copies inside the timed region.
roofline   the sweep kernel alone, timed live with CUDA events recorded inside the C ABI around
           its launch (event arguments of pcd_nn1_forward); peak = fp32 FMA rate measured in the same
           run by an FFMA micro-kernel (MEASURED_PEAKS.json has no CUDA-core fp32 figure).
cpu_baseline  the reference's torch CPU path (oracle/ref_torch_port.py: op-for-op restatement)
           on the host cores, on a bounded sample (B_chunk samples of the same workload).

Multi-GPU: one process per GPU, the batch is sharded (weak scaling: 32 samples per GPU); no
collective inside the loop, one NCCL all-gather of losses and perturbed clouds at the end.
"""
import argparse
import importlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "Chamfer+Hausdorff fwd+bwd Gpair-dist/s"
UNIT = "Gpair/s"
B_PER_GPU, NPTS, SIGMA = 32, 4096, 0.01
FLOP_PER_PAIR = 8.0
BWD_BYTES_PER_POINT_DIR = 68.0          # SURVEY.md section 8d
NCU_COUNTERS = os.path.join(ROOT, "profiles", "r2_ncu_counters.json")   # written by tools/ncu_counters.py from an ncu --set full capture


def sweep_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one nn1_sweep_kernel launch at the headline workload, read from the
    committed counter file by kernel name (None if the file or the kernel is missing)."""
    try:
        with open(NCU_COUNTERS) as f:
            d = json.load(f)
        for name, c in d["kernels"].items():
            if "nn1_sweep_kernel" in name:
                return int(c["dram__bytes_read.sum"] + c["dram__bytes_write.sum"]), name, d.get("source", "")
    except Exception:
        pass
    return None, None, None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons with NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.stop_flag = threading.Event()
        self.sm, self.reasons, self.max_mhz = [], set(), None
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._nvml_index(pynvml, index))
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as e:                       # NVML missing: report, never fail the bench
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    @staticmethod
    def _nvml_index(pynvml, local_index):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if local_index < len(ids) and ids[local_index].isdigit():
                return int(ids[local_index])
        return local_index

    def run(self):
        if self.h is None:
            return
        try:
            import pynvml
            h = self.h
            names = {
                pynvml.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                pynvml.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                pynvml.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            }
            while not self.stop_flag.is_set():
                self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.005)
        except Exception as e:                       # NVML missing: report, never fail the bench
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def summary(self):
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(sm)}


def dump_outputs(out_dir, rank, world, **arrays):
    """Write what the timed step returns to its caller (the loss, the four per-sample loss vectors of
    distance.chamfer / distance.hausdorff and the gradient w.r.t. adv, 1.6 MB per rank) as float32
    <name>.npy, so that two builds can be compared output for output on the same seeded inputs."""
    import numpy as np
    suffix = "" if world == 1 else f"_rank{rank}"
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), t.detach().float().cpu().numpy())


def make_inputs(B, first_sample):
    synth = importlib.import_module("3dpointcloudattack_b200.synth")
    ori = synth.face_clouds(B, NPTS, seed=1234, first_sample=first_sample)
    adv = synth.perturb(ori, SIGMA, seed=99, first_sample=first_sample)
    return adv, ori


# ----------------------------------------------------------------------------- reference arm
def cpu_reference_run(steps, warmup, b_chunk=2):
    """The reference's torch CPU path on the host cores: `steps` timed steps, each a bounded
    sample (b_chunk samples of the B=32 workload). Returns (Gpair/s, ms_per_step, cores)."""
    import torch
    from oracle import ref_torch_port as RP
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    adv, ori = make_inputs(b_chunk, 0)
    for _ in range(warmup):
        RP.chamfer_hausdorff_fwd_bwd(adv, ori)
    t0 = time.perf_counter()
    for _ in range(steps):
        RP.chamfer_hausdorff_fwd_bwd(adv, ori)
    dt = time.perf_counter() - t0
    pairs = float(b_chunk) * NPTS * NPTS * steps
    return pairs / dt / 1e9, dt / steps * 1e3, torch.get_num_threads(), b_chunk


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    gps, ms, cores, b_chunk = cpu_reference_run(args.steps, args.warmup)
    sample = f"{b_chunk} of {B_PER_GPU} samples per step (N=M={NPTS}), reference builds the pair matrix twice"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": gps, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"chamfer+hausdorff fwd+bwd B={B_PER_GPU} N=M={NPTS} fp32 (configs[1]), CPU sample B={b_chunk}"},
        "cpu_baseline": {"value": gps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": gps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------------- CW attack loop
CW_ITERS = 100


def _cw_dist_func(pcd):
    cd, hd = pcd.dist_utils.ChamferDist(method="avg"), pcd.dist_utils.HausdorffDist(method="avg")

    def dist(adv, ori, weights, batch_avg=False):
        return cd(adv, ori, weights=weights, batch_avg=batch_avg) + hd(adv, ori, weights=weights, batch_avg=batch_avg)
    return dist


def run_cw(pcd, dev, rank, world, B):
    """CW-style attack (attack/CW/CW_attack.py loop shape) against a random-init PointNet(106),
    B samples per GPU, N=4096, dist = w*(Chamfer(avg)+Hausdorff(avg)), kappa=30, Adam 1e-2,
    ClipPointsLinf(0.18).  Returns local iterations/s (eager and CUDA-graph)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import victims
    torch.manual_seed(0)
    model = victims.PointNetVictim(106).to(dev).eval()
    ori_h, _ = make_inputs(B, rank * B)[1], None
    data = ori_h.to(dev)
    target = torch.arange(B, device=dev) % 106
    out = {}
    for mode in ("eager", "graph"):
        atk = pcd.cw_loop.CWAttack(model, pcd.cw_loop.UntargetedLogitsAdvLoss(kappa=30.), _cw_dist_func(pcd),
                                   attack_lr=1e-2, init_weight=10., max_weight=80., binary_step=1, num_iter=CW_ITERS,
                                   clip_func=pcd.cw_loop.ClipPointsLinf(0.18), global_batch=B * world,
                                   use_graph=(mode == "graph"))
        atk.attack(data, target, seed=1, first_sample=rank * B)         # warm-up (and graph capture check)
        torch.cuda.synchronize()
        atk.attack(data, target, seed=2, first_sample=rank * B)
        out[mode] = CW_ITERS / (atk.loop_ms * 1e-3)        # CUDA events around the iteration loop
    return out


def cw_cpu_baseline(iters=4):
    """The reference-shaped CW iteration on the host cores at B=1 (BASELINE configs[0])."""
    import torch
    from oracle import ref_torch_port as RP
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import victims
    torch.manual_seed(0)
    model = victims.PointNetVictim(106).eval()
    for p in model.parameters():
        p.requires_grad_(False)
    data = make_inputs(1, 0)[1]
    target = torch.zeros(1, dtype=torch.long)
    RP.cw_iterations_cpu(model, data, target, 1)
    t0 = time.perf_counter()
    RP.cw_iterations_cpu(model, data, target, iters)
    return iters / (time.perf_counter() - t0)


# ---------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    pcd = importlib.import_module("3dpointcloudattack_b200")
    F = pcd.functional
    lib = pcd._lib.load()                      # raises if libpcdist.so is missing: no fallback

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    B = B_PER_GPU
    adv_h, ori_h = make_inputs(B, rank * B)
    adv_h, ori_h = adv_h.pin_memory(), ori_h.pin_memory()
    adv = adv_h.to(dev).requires_grad_(True)
    ori = ori_h.to(dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    gw = torch.tensor([1.0, 1.0, 1.0, 1.0], device=dev)     # loss = CD1 + CD2 + HD1 + HD2

    def loss_fn(a, o):
        c1, c2 = pcd.distance.chamfer(a, o)
        h1, h2 = pcd.distance.hausdorff(a, o)                 # same tensors -> served by the same sweep
        losses = torch.stack([c1, c2, h1, h2])
        return losses.sum(), (losses,)

    def step(a, o):
        loss, (losses,) = loss_fn(a, o)
        loss.backward()
        return losses

    ev = lambda: torch.cuda.Event(enable_timing=True)
    sweep_ev = [(ev(), ev()) for _ in range(args.steps)]
    for a, b in sweep_ev:                                     # materialise the cudaEvent handles
        a.record(); b.record()
    torch.cuda.synchronize()

    for _ in range(args.warmup):
        adv.grad = None
        step(adv, ori)
    torch.cuda.synchronize()

    # clocks are sampled across every timed loop below (eager, graph replay, e2e)
    # (rank 0 only: eight processes polling NVML every few ms contend on driver locks and delay launches)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    # ---------------- eager loop: kernel-level timing (sweep events live inside the C ABI) -------
    launches0 = F.launches()
    eager_ev, bwd_ev = [], []
    for k in range(args.steps):
        flush.zero_()
        adv.grad = None
        e0, e1, e2 = ev(), ev(), ev()
        F.time_next_sweep(sweep_ev[k][0], sweep_ev[k][1])     # events passed per call through the C ABI
        e0.record()
        loss, _ = loss_fn(adv, ori)
        e1.record()
        loss.backward()
        e2.record()
        eager_ev.append((e0, e2)); bwd_ev.append((e1, e2))
    torch.cuda.synchronize()
    launches_per_step = (F.launches() - launches0) // args.steps
    eager_ms = [a.elapsed_time(b) for a, b in eager_ev]
    sweep_ms = [a.elapsed_time(b) for a, b in sweep_ev]
    bwd_ms = [a.elapsed_time(b) for a, b in bwd_ev]

    # the backward kernel alone: one pcd_nn1_backward launch (pre-zeroed gradient buffer) between two events
    def time_backward_kernel(a_t, o_t, reps):
        import ctypes
        Bq, Nq = a_t.shape[0], a_t.shape[1]
        r = F.nn1(o_t, a_t.detach(), F.FORM_SUM_FIRST, F.NORM_FMA, row_sum_scale=1.0 / Nq, col_sum_scale=1.0 / Nq, cache=False)
        g = torch.zeros_like(a_t)
        wv = torch.ones(Bq, device=dev)
        ws_ = (ctypes.c_int64 * 4)(1, 1, 1, 1)
        out = []
        for _ in range(reps + 2):
            g.zero_()
            flush.zero_()
            b0, b1 = ev(), ev()
            b0.record()
            st_ = lib.pcd_nn1_backward(o_t.data_ptr(), *o_t.stride(), a_t.data_ptr(), *a_t.stride(), Bq, Nq, Nq, 0, 0,
                                       r.row_arg.data_ptr(), r.col_arg.data_ptr(), r.row_min.data_ptr(), r.col_min.data_ptr(),
                                       None, None, wv.data_ptr(), wv.data_ptr(), r.row_argmax.data_ptr(),
                                       wv.data_ptr(), wv.data_ptr(), r.col_argmax.data_ptr(), ws_, 1.0 / Nq, 1.0 / Nq,
                                       None, 0, 0, 0, g.data_ptr(), *g.stride(), 1, torch.cuda.current_stream().cuda_stream)
            pcd._lib.check(st_, "pcd_nn1_backward")
            b1.record()
            out.append((b0, b1))
        torch.cuda.synchronize()
        ms = sorted(x.elapsed_time(y) for x, y in out[2:])
        return ms[len(ms) // 2]

    bwdk_med_ms = time_backward_kernel(adv.detach(), ori, args.steps)

    # ---------------- timed region: the same step captured once as a CUDA graph and replayed -----
    graphed = pcd.graph.GraphedLoss(loss_fn, adv, ori, warmup=3)
    for _ in range(args.warmup):
        graphed.replay()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    step_ev = []
    for k in range(args.steps):
        flush.zero_()
        torch.cuda._sleep(400000)          # ~200 us of device-side spin BEFORE the first event: the host enqueues the
        e0, e1 = ev(), ev()                # events and the graph launch meanwhile, so no host launch latency is timed
        e0.record()
        graphed.replay()
        e1.record()
        step_ev.append((e0, e1))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    step_ms = [a.elapsed_time(b) for a, b in step_ev]
    total_ms = sum(step_ms)
    launches = launches_per_step * args.steps
    losses = graphed.aux[0]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank, world, loss=graphed.loss, chamfer_1=losses[0], chamfer_2=losses[1],
                     hausdorff_1=losses[2], hausdorff_2=losses[3], grad_adv=graphed.grad)
    # the replayed graph must reproduce the eager result bit for bit
    ref_losses = step(adv.detach().clone().requires_grad_(True), ori)
    if not torch.equal(ref_losses, losses):
        raise RuntimeError("graph replay and eager step disagree")

    # ---------------- e2e: pinned host buffers, copies inside the timed region -------------------
    loss_h = torch.empty((4, B), dtype=torch.float32).pin_memory()
    grad_h = torch.empty_like(adv_h).pin_memory()
    # public API: PipelinedLoss(host adv, host ori).replay() -- ONE graph whose three branches (8 + 12 + 12 samples)
    # upload, compute and download independently, so the copies overlap the kernels
    piped = pcd.graph.PipelinedLoss(loss_fn, adv_h, ori_h, chunks=3)
    e2e_pipe_ms = []
    for k in range(args.warmup + args.steps):
        flush.zero_()
        torch.cuda._sleep(400000)
        e0, e1 = ev(), ev()
        e0.record()
        piped.replay()
        e1.record()
        torch.cuda.synchronize()
        if k >= args.warmup:
            e2e_pipe_ms.append(e0.elapsed_time(e1))
    pipe_losses = torch.cat([a[0] for a in piped.aux_host], 1).clone()
    pipe_grad = piped.grad_host.clone()
    e2e_ms, e2e_eager_ms = [], []
    for k in range(args.warmup + args.steps):                  # monolithic: GraphedLoss.replay(host adv, host ori) + two copies back
        flush.zero_()
        e0, e1 = ev(), ev()
        e0.record()
        _, (l_d,), g_d = graphed.replay(adv_h, ori_h)
        loss_h.copy_(l_d, non_blocking=True)
        grad_h.copy_(g_d, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        if k >= args.warmup:
            e2e_ms.append(e0.elapsed_time(e1))
    adv_d = torch.empty_like(adv_h, device=dev).requires_grad_(True)
    ori_d = torch.empty_like(ori_h, device=dev)
    for k in range(args.warmup + args.steps):                  # eager drop-in surface, same copies
        flush.zero_()
        adv_d.grad = None
        e0, e1 = ev(), ev()
        e0.record()
        with torch.no_grad():
            adv_d.copy_(adv_h, non_blocking=True)
            ori_d.copy_(ori_h, non_blocking=True)
        l_d = step(adv_d, ori_d)
        loss_h.copy_(l_d.detach(), non_blocking=True)
        grad_h.copy_(adv_d.grad, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        if k >= args.warmup:
            e2e_eager_ms.append(e0.elapsed_time(e1))
    if not torch.equal(pipe_losses, loss_h) or float((pipe_grad - grad_h).abs().max()) > 1e-5 * float(grad_h.abs().max()):
        raise RuntimeError("pipelined and monolithic host-to-host steps disagree")
    e2e_single_ms = sum(e2e_ms) / len(e2e_ms)
    e2e_total_ms = sum(e2e_pipe_ms)
    sampler.stop_flag.set()
    if rank == 0:
        sampler.join(timeout=2)
    h2d = adv_h.numel() * 4 + ori_h.numel() * 4
    d2h = loss_h.numel() * 4 + grad_h.numel() * 4

    # ---------------- secondary metric: CW attack iterations/s (device-resident loop, section 8f-1) ----
    cw = run_cw(pcd, dev, rank, world, B)

    # ---------------- the other BASELINE configs (tools/bench_configs.py) ---------------------------
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import bench_configs as BC
    fp32_peak = F.fp32_peak_flops(2048)
    gpu_ref = BC.gpu_reference(pcd, adv, ori, flush) if rank == 0 else None
    c2 = BC.config2(pcd, dev, rank, with_reference=(rank == 0 and world == 1))
    c3 = BC.config3(pcd, dev, rank, world, with_reference=(rank == 0 and world == 1))
    c4 = BC.config4(pcd, dev, rank, world, flush, fp32_peak, load_peaks()[0])
    # the backward kernel where it is large enough for the HBM roofline: the 8-GPU shard of configs[4] (B=64, N=16384, 143 MB)
    synth = importlib.import_module("3dpointcloudattack_b200.synth")
    o_l = synth.face_clouds(4, 16384, seed=4321).to(dev).repeat(16, 1, 1).contiguous()
    a_l = o_l + SIGMA * torch.randn(o_l.shape, device=dev, generator=torch.Generator(device=dev).manual_seed(7))
    bwl_ms = time_backward_kernel(a_l, o_l, 7)
    bwl_gbs = 2.0 * 64 * 16384 * BWD_BYTES_PER_POINT_DIR / (bwl_ms * 1e-3) / 1e9
    backward_large = {"workload": "nn1_bwd_kernel<2> at B=64 N=M=16384 (143 MB algorithmic)", "ms": bwl_ms, "achieved": bwl_gbs,
                      "unit": "GB/s", "peak": load_peaks()[0], "frac": bwl_gbs / load_peaks()[0]}
    del o_l, a_l

    # ---------------- max over ranks, final all-gather (the only collective of the path) ---------
    cw_t = torch.tensor([cw["eager"], cw["graph"], c2["iters_per_s_eager"]], device=dev, dtype=torch.float64)
    t = torch.tensor([total_ms, e2e_total_ms, c3["ms_per_iteration"], c4["ms_per_step"], c4["sweep_ms"]], device=dev, dtype=torch.float64)
    gather_ms = None
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(cw_t, op=dist.ReduceOp.MIN)
        all_loss = torch.empty((world, 4, B), device=dev)
        all_adv = torch.empty((world,) + tuple(adv.shape), device=dev)
        g0, g1 = ev(), ev()
        g0.record()
        dist.all_gather_into_tensor(all_loss, losses.detach().contiguous())
        dist.all_gather_into_tensor(all_adv, adv.detach().contiguous())
        g1.record(); torch.cuda.synchronize()
        gather_ms = g0.elapsed_time(g1)
    total_ms, e2e_total_ms = float(t[0]), float(t[1])
    # strong-scaling configs: the slowest rank decides (MAX over ranks), throughput is the GLOBAL batch over that time
    c3["ms_per_iteration"] = float(t[2]); c3["iters_per_s"] = 1e3 / float(t[2])
    c3["sample_iters_per_s"] = c3["global_batch"] * 1e3 / float(t[2])
    c4["ms_per_step"] = float(t[3]); c4["sweep_ms_slowest_rank"] = float(t[4])
    c4["value"] = c4["pairs_per_step_global"] / (float(t[3]) * 1e-3) / 1e9; c4["unit"] = UNIT
    c2["iters_per_s_eager"] = float(cw_t[2])
    c2["sample_iters_per_s"] = float(cw_t[2]) * 64 * world

    pairs_step_rank = float(B) * NPTS * NPTS
    value = pairs_step_rank * world * args.steps / (total_ms * 1e-3) / 1e9
    e2e_value = pairs_step_rank * world * args.steps / (e2e_total_ms * 1e-3) / 1e9

    if rank == 0:
        hbm_gbs, hbm_src = load_peaks()
        sweep_avg_ms = sum(sweep_ms) / len(sweep_ms)
        achieved = FLOP_PER_PAIR * pairs_step_rank / (sweep_avg_ms * 1e-3) / 1e12
        bwd_avg_ms = bwdk_med_ms                              # nn1_bwd_kernel<2> alone (gradient buffer pre-zeroed by the forward)
        bwd_autograd_ms = sum(bwd_ms) / len(bwd_ms)
        bwd_bytes = 2.0 * B * NPTS * BWD_BYTES_PER_POINT_DIR
        cpu = None
        if world == 1:                                        # reported baseline: rank 0 at N=1 only
            gps, ms, cores, b_chunk = cpu_reference_run(steps=3, warmup=1)
            cpu = {"value": gps, "unit": UNIT, "cores": cores, "kind": "port",
                   "sample": f"{b_chunk} of {B} samples x 3 steps (N=M={NPTS}); torch CPU op-for-op port of "
                             f"attack/CW/CW_utils/distance.py (pair matrix built twice), {ms:.0f} ms/step"}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"chamfer+hausdorff fwd+bwd B={B}/GPU N=M={NPTS} fp32 sigma={SIGMA} (BASELINE configs[1])",
                       "global_batch": B * world, "pairs_per_step": pairs_step_rank * world,
                       "parallelism": f"batch-sharded x{world}, no collective in the loop",
                       "l2": "256 MiB memset (+ 200 us device spin so the launch is queued) between timed steps, outside the per-step event pairs",
                       "timed_step": "CUDA graph replay of forward+backward (captured once, bit-identical to the eager step)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_total_ms / args.steps,
                    "api": "pcdist.graph.PipelinedLoss(loss_fn, pinned adv, pinned ori, chunks=3).replay(): one CUDA graph, per "
                           "slice (8 + 12 + 12 samples) H2D -> forward+backward -> D2H of the 4 loss vectors and the gradient; "
                           "slices overlap, earlier slices on higher-priority streams",
                    "monolithic_ms_per_step": e2e_single_ms,
                    "monolithic_value": pairs_step_rank * world / (e2e_single_ms * 1e-3) / 1e9,
                    "eager_api_ms_per_step": sum(e2e_eager_ms) / len(e2e_eager_ms),
                    "eager_api_value": pairs_step_rank * world / (sum(e2e_eager_ms) / len(e2e_eager_ms) * 1e-3) / 1e9},
            "eager": {"ms_per_step": sum(eager_ms) / len(eager_ms),
                      "value": pairs_step_rank * world / (sum(eager_ms) / len(eager_ms) * 1e-3) / 1e9,
                      "note": "same step without CUDA-graph capture (python/autograd launch overhead included)"},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
            "roofline": {"bound": "fp32", "kernel": "nn1_sweep_kernel", "achieved": achieved, "peak": fp32_peak / 1e12,
                         "unit": "TFLOP/s", "frac": achieved / (fp32_peak / 1e12), "traffic": sweep_traffic()[0],
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of %s in profiles/r2_ncu_counters.json "
                                           "(%s); algorithmic input bytes = 3.15 MB (both clouds, streamed raw)" % sweep_traffic()[1:],
                         "peak_source": "FFMA/FFMA2 micro-kernel measured in this run (pcd_fp32_probe_launch between CUDA events)",
                         "ms_per_launch": sweep_avg_ms, "flop_per_pair": FLOP_PER_PAIR},
            "roofline_backward": {"bound": "hbm", "kernel": "nn1_bwd_kernel<2>", "achieved": bwd_bytes / (bwd_avg_ms * 1e-3) / 1e9,
                                  "peak": hbm_gbs, "unit": "GB/s", "frac": bwd_bytes / (bwd_avg_ms * 1e-3) / 1e9 / hbm_gbs,
                                  "peak_source": hbm_src, "ms": bwd_avg_ms,
                                  "loss_backward_ms_with_autograd": bwd_autograd_ms,
                                  "note": "algorithmic 68 B per (point, direction) = 17.8 MB: too small for the HBM roofline (launch "
                                          "latency); one pcd_nn1_backward launch between two events, L2 flushed, median; "
                                          "backward_large is the same kernel at 143 MB"},
            "backward_large": backward_large,
            "cpu_baseline": cpu,
            "gpu_reference": gpu_ref,
            "configs2": c2,
            "configs3": c3,
            "configs4": c4,
            "cw_attack": {"metric": "CW attack iters/s", "iters_per_s_graph": float(cw_t[1]), "iters_per_s_eager": float(cw_t[0]),
                          "sample_iters_per_s_graph": float(cw_t[1]) * B * world,
                          "config": f"PointNet(106) random init, B={B}/GPU N={NPTS}, w*(Chamfer+Hausdorff avg) + logits loss kappa=30, "
                                    f"Adam 1e-2, ClipPointsLinf 0.18, {CW_ITERS} iters; slowest rank; every rank attacks its own {B} samples",
                          "cpu_reference_iters_per_s_B1": cw_cpu_baseline() if world == 1 else None,
                          "note": "iters_per_s = loop iterations per second with B samples per GPU advancing together; "
                                  "sample_iters_per_s = iterations x samples over all GPUs; CPU figure is the reference-shaped "
                                  "loop at B=1 (its only supported batch size) on the host cores"},
            "step_ms_min_med_max": [min(step_ms), sorted(step_ms)[len(step_ms) // 2], max(step_ms)],
            "final_allgather_ms": gather_ms,
        }
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's outputs (loss, per-sample Chamfer/Hausdorff, gradient) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl != "ours":
            ap.error("--dump-outputs needs --impl ours")
        os.makedirs(args.dump_outputs, exist_ok=True)
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
