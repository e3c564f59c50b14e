#!/usr/bin/env python
"""Benchmark of the cascade-MVS depth hot path on B200 (contract: task prompt §④).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned (depth_l, confidence_l; at N > 1 also
depth_0_all_ranks, the gathered depth maps of that step) as DIR/<name>.npy, float32.  Inputs and
weights are seeded, so two builds run with the same arguments can be compared output for output.

A *step* is one `CascadeMVSNet.forward` (FeatureNet + three cascade stages) over
one batch of synthetic DTU-shaped views per GPU: BASELINE.json configs[1] —
640x512, V=3, D=48/32/8, variance cost, B=1 per GPU.  Metric: depth-maps/sec.

  value        whole-job depth-maps/s, inputs resident in HBM when timing starts: K CUDA-graph
               replays through the streaming engine (PipelinedCascade: 3 slots, one compute stream
               each, so 3 independent reference views are in flight); at N > 1 every rank keeps its
               K depth maps and the ranks all-gather them inside the timed region, in chunks of 5
               steps on a side stream while the next forwards run
  one_view_at_a_time  the same K replays strictly one after the other on one stream (the latency
               of a single depth map; rounds 1 and 2 reported this as `value` until the slots got
               their own streams)
  e2e          the same through the public API with HOST (pinned) inputs: H2D copy of imgs+proj and
               D2H read of depth_0 + confidence_2 every step, inside the timed region (3-slot
               pipeline on every rank)
  roofline     the fused warp+variance kernel (K1): algorithmic bytes of its three launches /
               their CUDA-event time (L2 flushed), vs MEASURED_PEAKS.json hbm_gbs
  roofline_k2  the three CostRegNet stacks: ms, GB/s, TFLOP/s, tensor-pipe % (from profiles/)
  parity       this run's GPU output vs the oracle on the same inputs and weights (N = 1)
  sustained    >= 2 s of back-to-back replays with clocks / power sampled
  fallbacks    tf32 layers that ran on the CUDA-core fallback kernel (must be 0)
  other_configs    single-view graph-replay timings of cfg3 / cfg4 / cfg5 (N = 1)
  throughput_modes cfg2 depth maps/s when the caller gives the GPU more than one reference view at
                   a time: a batch of 4 per forward, or 3 single-view graphs in flight on 3 streams
                   (`value` stays one view at a time, the reference eval loop's batch size)
  sharded_configs  cfg4 (batch of N views) and cfg5 (batch of 4N) sharded over the N ranks with one
                   all_gather at the end: ms per batch, bit-equality with one GPU (N > 1)
  cpu_baseline the CPU oracle port of the reference path on this box's host cores (N = 1)
  --impl reference : the reference arm = the same CPU port, fastest thread count
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W_IMG, H_IMG, VIEWS = 640, 512, 3
N_DEPTHS = (8, 32, 48)          # level 0..2  (BASELINE writes coarse->fine 48/32/8)
RATIOS = (1, 2, 4)
METRIC = "depth-maps/sec at 640x512 V=3 D=48/32/8"
FALLBACK_HBM_GBS = 6650.0       # /opt/skills/guides/B200_PROFILING.md fallback
# identical in both arms (the driver compares the two lines' config.workload)
WORKLOAD = ("cfg2: 640x512, V=3, D=48/32/8, variance cost, B=1 per GPU "
            "(BASELINE.json configs[1])")
K2_ALGO_BYTES = 1846.8e6        # SURVEY.md 8(d): layer-by-layer fp32 activation traffic, cfg2
K2_ALGO_FLOP = 81.1e9           # 2*27*N*(8*Cin3d+120) summed over the three stages


def k1_algorithmic_bytes(V, G=1, W=W_IMG, H=H_IMG, n_depths=N_DEPTHS):
    """SURVEY.md §8(d): 4*[V*C*h*w + Cin3d*D*h*w + D*h*w] + 48*(V-1) per stage."""
    per = []
    for l in (2, 1, 0):
        C, D, h, w = 8 * 2 ** l, n_depths[l], H >> l, W >> l
        cin3d = C if G == 1 else G
        per.append(4 * (V * C * h * w + cin3d * D * h * w + D * h * w) + 48 * (V - 1))
    return per


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(",") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                pw.append(float(r[3]))
                for n, v in zip(names, r[4:8]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "power_w_max": max(pw) if pw else None,
                "reasons": sorted(reasons)}


def cpu_port_forward_factory(threads):
    """The CPU reference arm / cpu_baseline: oracle port of the reference path."""
    import torch
    from casmvsnet_pl_b200 import ABN, synth
    from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet
    from oracle import casmvs_oracle as O
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    m = CascadeMVSNet(n_depths=list(N_DEPTHS), interval_ratios=list(RATIOS), norm_act=ABN)
    synth.randomize_model_(m, 0)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    imgs, pm, dmin, dint = synth.make_inputs(B=1, V=VIEWS, W=W_IMG, H=H_IMG, seed=0)

    def fwd():
        return O.cascade_forward(sd, imgs, pm, dmin, dint, N_DEPTHS, RATIOS, 1)
    return fwd


def best_cpu_threads(cores):
    """torch/oneDNN over-subscribe badly on many-core hosts (128 threads measured 7x
    slower than 8 on the GPU box), so the CPU arm uses the thread count that is
    FASTEST for it: probed on the coarsest stage (128x160, D=48) of the workload."""
    import torch
    from casmvsnet_pl_b200 import ABN, synth
    from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet
    from oracle import casmvs_oracle as O
    torch.manual_seed(0)
    m = CascadeMVSNet(n_depths=list(N_DEPTHS), interval_ratios=list(RATIOS), norm_act=ABN)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    feats = synth.make_level_feats(1, VIEWS, 2, W_IMG, H_IMG)
    pm = synth.projection_matrices(VIEWS, W_IMG, H_IMG)[:, 2].unsqueeze(0)
    dv = O.initial_hypotheses(425.0, 2.65 * 4, 48, 1, H_IMG // 4, W_IMG // 4).contiguous()
    cands = sorted({t for t in (4, 8, 16, 32, 64, cores) if t <= cores})
    best, best_t = None, None
    for t in cands:
        torch.set_num_threads(t)
        with torch.no_grad():
            O.predict_depth(feats, pm, dv, sd, "cost_reg_2.", 1)
            t0 = time.perf_counter()
            O.predict_depth(feats, pm, dv, sd, "cost_reg_2.", 1)
            dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, best_t = dt, t
    return best_t


def dump_outputs(out_dir, arrays):
    """arrays: name -> tensor; written as out_dir/<name>.npy in float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy().astype(np.float32))


def time_cpu_port(steps, warmup, threads, want_result=False):
    fwd = cpu_port_forward_factory(threads)
    for _ in range(warmup):
        fwd()
    ts = []
    res = None
    for _ in range(steps):
        t0 = time.perf_counter()
        res = fwd()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    if want_result:
        return ts[len(ts) // 2], sum(ts), res
    return ts[len(ts) // 2], sum(ts)


def run_reference_arm(args, rank):
    if rank != 0:
        return
    import torch
    avail = len(os.sched_getaffinity(0))
    cores = best_cpu_threads(avail)
    steps = max(1, args.steps)
    med, total, res = time_cpu_port(steps, max(1, min(args.warmup, 2)), cores, want_result=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    value = steps / total
    sample = (f"{steps} full forwards of the cfg2 workload (640x512, V=3, D=48/32/8, B=1) on "
              f"{cores} torch threads (fastest of 4..{avail} available; more threads are slower); "
              f"oracle port of the reference PyTorch-CPU path "
              f"(/root/reference does not travel to the GPU box)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "depth-maps/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "device": "cpu",
                   "torch_threads": torch.get_num_threads()},
        "cpu_baseline": {"value": value, "unit": "depth-maps/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "depth-maps/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def pin_to_gpu_numa(local_rank):
    """Bind this rank (and the pinned buffers it allocates afterwards) to the CPUs that
    `nvidia-smi topo -m` lists as local to its GPU.  Best effort; returns a description."""
    import re
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True,
                             timeout=30).stdout
        for line in out.splitlines():
            toks = line.replace("\x1b[4m", "").replace("\x1b[0m", "").split()
            if not toks or toks[0] != f"GPU{local_rank}":
                continue
            for t in toks[1:]:
                if re.fullmatch(r"\d+(-\d+)?(,\d+(-\d+)?)*", t) and ("-" in t or "," in t):
                    cpus = set()
                    for part in t.split(","):
                        lo, _, hi = part.partition("-")
                        cpus.update(range(int(lo), int(hi or lo) + 1))
                    cpus &= os.sched_getaffinity(0)
                    if cpus:
                        os.sched_setaffinity(0, cpus)
                        return f"rank bound to GPU{local_rank}-local CPUs {t}"
    except Exception as e:                                   # noqa: BLE001
        return f"not bound ({type(e).__name__})"
    return "not bound (no CPU affinity column)"


SHARDED_CONFIGS = {
    # BASELINE.json configs[3], configs[4]: a batch of reference views sharded over the ranks,
    # ONE all_gather of the per-view depth maps at the end (SURVEY.md 8e; replaces the loop at
    # reference eval.py:213-229)
    "cfg4": dict(W=1152, H=864, V=5, n_depths=(8, 32, 48), views_per_gpu=1),
    "cfg5": dict(W=1920, H=1056, V=7, n_depths=(8, 32, 64), views_per_gpu=4),
}


def run_sharded_config(name, rank, world, dev, precision, reps=3):
    """cfg4 / cfg5 through dist.sharded_depth_inference on `world` GPUs: ms per batch (CUDA
    events, max over ranks, barrier on both sides, inputs resident on each rank's GPU) and
    bit-equality of the gathered result with a single-GPU evaluation of the same views."""
    import torch
    import torch.distributed as dist
    from casmvsnet_pl_b200 import ABN, synth
    from casmvsnet_pl_b200.dist import shard_bounds, sharded_depth_inference
    from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet
    c = SHARDED_CONFIGS[name]
    B = c["views_per_gpu"] * world
    torch.manual_seed(0)
    model = CascadeMVSNet(n_depths=list(c["n_depths"]), norm_act=ABN, precision=precision)
    synth.randomize_model_(model, 0)
    model = model.eval().to(dev).requires_grad_(False)
    lo, hi = shard_bounds(B, rank, world)
    # every rank materialises only its own shard (view i is seeded with i, so any rank can
    # regenerate any view); the (B, ...) tensors are views of untouched virtual memory
    shard = [synth.make_inputs(B=1, V=c["V"], W=c["W"], H=c["H"], seed=i) for i in range(lo, hi)]
    dmin, dint = shard[0][2], shard[0][3]
    imgs_l = torch.cat([s[0] for s in shard]).to(dev)
    pm_l = torch.cat([s[1] for s in shard]).to(dev)

    class ShardView:
        """Stands for the (B, ...) batch: only this rank's rows exist."""
        def __init__(self, t):
            self.t, self.shape, self.device = t, (B,) + tuple(t.shape[1:]), t.device

        def __getitem__(self, sl):
            assert sl.start == lo and sl.stop == hi
            return self.t

    def engine(i, p, a, b):
        with torch.no_grad():
            return model(i, p, a, b)

    def once():
        return sharded_depth_inference(engine, ShardView(imgs_l), ShardView(pm_l), dmin, dint)

    out = once()                                          # warm-up (weight packing, smem opt-in)
    ts = []
    for _ in range(reps):
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = once()
        e1.record()
        dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ts.append(ms.item())
    # bit-equality with one GPU: rank 0 evaluates a view of ANOTHER rank's shard on its own GPU
    probe = min(B - 1, hi)                                # first view of rank 1 (or last view)
    ok = None
    if rank == 0:
        pi, pp, _, _ = synth.make_inputs(B=1, V=c["V"], W=c["W"], H=c["H"], seed=probe)
        r1 = engine(pi.to(dev), pp.to(dev), dmin, dint)
        ok = bool(torch.equal(r1["depth_0"][0], out["depth_0"][probe]) and
                  torch.equal(r1["confidence_2"][0], out["confidence_2"][probe]) and
                  torch.equal(out["depth_0"][lo:hi], engine(imgs_l, pm_l, dmin, dint)["depth_0"]))
    del model
    torch.cuda.empty_cache()
    ts.sort()
    return {"config": f"{name}: {c['W']}x{c['H']}, V={c['V']}, D={'/'.join(map(str, c['n_depths'][::-1]))}, "
                      f"batch of {B} ref views over {world} GPUs ({c['views_per_gpu']}/GPU)",
            "ms_per_batch": ts[len(ts) // 2], "views_per_s": B / (ts[len(ts) // 2] * 1e-3),
            "gathered_shape": list(out["depth_0"].shape),
            "bit_equal_to_single_gpu": ok,
            "collective": "one all_gather_into_tensor per output key at the end (depth_0, confidence_2)"}


OTHER_CONFIGS = {
    # single-GPU timings of the remaining BASELINE.json configs (one reference view each); their
    # parity against the oracle is in tests/test_gpu_cascade.py::test_full_size_parity_vs_oracle
    "cfg3": dict(W=640, H=512, V=3, G=8, n_depths=(8, 32, 48)),
    "cfg4_view": dict(W=1152, H=864, V=5, G=1, n_depths=(8, 32, 48)),
    "cfg5_view": dict(W=1920, H=1056, V=7, G=1, n_depths=(8, 32, 64)),
}


def run_other_configs(dev, precision, reps=20):
    import torch
    from casmvsnet_pl_b200 import ABN, synth
    from casmvsnet_pl_b200.graph import GraphedCascade
    from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet
    out = {}
    for name, c in OTHER_CONFIGS.items():
        torch.manual_seed(0)
        model = CascadeMVSNet(n_depths=list(c["n_depths"]), num_groups=c["G"], norm_act=ABN,
                              precision=precision)
        synth.randomize_model_(model, 0)
        model = model.eval().to(dev).requires_grad_(False)
        imgs, pm, dmin, dint = synth.make_inputs(B=1, V=c["V"], W=c["W"], H=c["H"], seed=0)
        g = GraphedCascade(model, imgs.to(dev), pm.to(dev), dmin, dint, warmup=2)
        for _ in range(3):
            g()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            g()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out[name] = {"config": f"{c['W']}x{c['H']}, V={c['V']}, G={c['G']}, "
                               f"D={'/'.join(map(str, c['n_depths'][::-1]))}, one reference view",
                     "ms_per_view": ms, "views_per_s": 1e3 / ms, "how": "CUDA-graph replay, inputs resident"}
        del g, model
        torch.cuda.empty_cache()
    return out


def run_throughput_modes(model, dev, reps=30):
    """cfg2 with more than one independent reference view on the GPU at once (inputs resident)."""
    import torch
    from casmvsnet_pl_b200 import synth
    from casmvsnet_pl_b200.graph import GraphedCascade
    out = {}
    imgs, pm, dmin, dint = synth.make_inputs(B=1, V=VIEWS, W=W_IMG, H=H_IMG, seed=0)

    def clock(fn, n_maps):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n_maps
        return {"ms_per_depth_map": ms, "depth_maps_per_s": 1e3 / ms}

    BATCH = 4
    g = GraphedCascade(model, imgs.expand(BATCH, -1, -1, -1, -1).contiguous().to(dev),
                       pm.expand(BATCH, *pm.shape[1:]).contiguous().to(dev), dmin, dint, warmup=2)
    out["batch_of_4_per_forward"] = clock(lambda: [g() for _ in range(reps)], reps * BATCH)
    del g
    torch.cuda.empty_cache()
    K = 3
    gs = [GraphedCascade(model, imgs.to(dev), pm.to(dev), dmin, dint, warmup=1) for _ in range(K)]
    streams = [torch.cuda.Stream() for _ in range(K)]

    def in_flight():
        main_s = torch.cuda.current_stream()
        for s_ in streams:
            s_.wait_stream(main_s)
        for i in range(reps * K):
            with torch.cuda.stream(streams[i % K]):
                gs[i % K].graph.replay()
        for s_ in streams:
            main_s.wait_stream(s_)
    out["3_single_view_graphs_in_flight"] = clock(in_flight, reps * K)
    del gs
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("CASMVS_PRECISION", "tf32"),
                    choices=["fp32", "tf32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-sharded-configs", action="store_true",
                    help="skip the cfg4 / cfg5 sharded-batch runs at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch
    import torch.distributed as dist
    from casmvsnet_pl_b200 import ABN, _lib, ops, synth
    from casmvsnet_pl_b200.models.mvsnet import CascadeMVSNet

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a B200; no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    numa = pin_to_gpu_numa(local_rank) if world > 1 else None

    torch.manual_seed(0)
    model = CascadeMVSNet(n_depths=list(N_DEPTHS), interval_ratios=list(RATIOS), norm_act=ABN,
                          precision=args.precision)
    synth.randomize_model_(model, 0)
    model = model.eval().to(dev).requires_grad_(False)
    B = 1
    K = args.steps
    imgs_h, pm_h, dmin, dint = synth.make_inputs(B=B, V=VIEWS, W=W_IMG, H=H_IMG, seed=rank)
    imgs_h, pm_h = imgs_h.pin_memory(), pm_h.pin_memory()
    imgs_d, pm_d = imgs_h.to(dev), pm_h.to(dev)
    # multi-GPU: every rank keeps the depth maps of its own views on the device and the path's
    # single collective type (SURVEY.md 8e: all-gather of per-view depth maps) collects them
    # inside the timed region, chunk by chunk (gather_chunk below)
    nkeep = max(K, args.warmup, 3)
    store = torch.empty(nkeep * B, H_IMG, W_IMG, device=dev) if world > 1 else None
    gathered = torch.empty(world * nkeep * B, H_IMG, W_IMG, device=dev) if world > 1 else None

    graphed = None
    pipe = None
    if not args.no_graph:
        from casmvsnet_pl_b200.graph import GraphedCascade, PipelinedCascade
        graphed = GraphedCascade(model, imgs_d, pm_d, dmin, dint)
        # the streaming engine: three slots (static inputs + captured graph + result buffers
        # each), one compute stream per slot -> consecutive views overlap each other on the GPU
        pipe = PipelinedCascade(model, imgs_d, pm_d, dmin, dint)

    # multi-GPU: the depth maps are gathered in chunks of GATHER_EVERY steps on a side stream while
    # the next forwards run (the same single collective type, all_gather_into_tensor, issued as
    # the results appear: at N = 8 a gather of 8 x 1.3 MB per step left to the end of the timed
    # region costs ~0.1 ms per step, 10 % of the step)
    GATHER_EVERY = 5
    comm = torch.cuda.Stream() if world > 1 else None
    works = []

    def gather_chunk(k0, k1, events):
        for ev in events:
            comm.wait_event(ev)
        with torch.cuda.stream(comm):
            works.append(dist.all_gather_into_tensor(gathered[world * k0 * B: world * k1 * B],
                                                     store[k0 * B: k1 * B], async_op=True))

    def gather_finish():
        while works:
            works.pop(0).wait()                      # the current stream waits for the collective
        torch.cuda.current_stream().wait_stream(comm)

    def run_resident(steps):
        """K forwards, inputs resident: through the streaming engine (3 views in flight)."""
        if pipe is not None:
            res = pipe.run_resident(steps, keep=(lambda k: store[k * B:(k + 1) * B]) if world > 1 else None,
                                    every=GATHER_EVERY if world > 1 else 0,
                                    on_chunk=gather_chunk if world > 1 else None)
        else:
            res = None
            with torch.no_grad():
                for k in range(steps):
                    res = model(imgs_d, pm_d, dmin, dint)
                    if world > 1:
                        store[k * B:(k + 1) * B].copy_(res["depth_0"])
                        if (k + 1) % GATHER_EVERY == 0 or k + 1 == steps:
                            ev = torch.cuda.Event()
                            ev.record()
                            gather_chunk(k + 1 - ((k % GATHER_EVERY) + 1), k + 1, [ev])
        if world > 1:
            gather_finish()
        return res

    def run_one_at_a_time(steps):
        """K forwards, inputs resident, one view at a time on one stream (the latency form)."""
        with torch.no_grad():
            for _ in range(steps):
                graphed() if graphed is not None else model(imgs_d, pm_d, dmin, dint)

    out_depth_h = torch.empty(B, H_IMG, W_IMG).pin_memory()
    out_conf_h = torch.empty(B, H_IMG // 4, W_IMG // 4).pin_memory()

    def run_e2e(steps):
        # every step: H2D of that step's inputs from pinned memory, forward, D2H of its results
        if pipe is not None:
            # copies of neighbouring steps overlap the compute, and the (three) slots replay on
            # their own streams so that consecutive views overlap each other, on every rank
            k0 = 0
            for k in range(steps):
                pipe.submit(imgs_h, pm_h, keep=store[k * B:(k + 1) * B] if world > 1 else None)
                if world > 1 and ((k + 1) % GATHER_EVERY == 0 or k + 1 == steps):
                    gather_chunk(k0, k + 1, list(pipe.compute_done))
                    k0 = k + 1
            pipe.drain()
        else:
            with torch.no_grad():
                k0 = 0
                for k in range(steps):
                    res = model(imgs_h.to(dev, non_blocking=True), pm_h.to(dev, non_blocking=True),
                                dmin, dint)
                    if world > 1:
                        store[k * B:(k + 1) * B].copy_(res["depth_0"])
                    out_depth_h.copy_(res["depth_0"], non_blocking=True)   # eval.py:224-226
                    out_conf_h.copy_(res["confidence_2"], non_blocking=True)
                    torch.cuda.current_stream().synchronize()
                    if world > 1 and ((k + 1) % GATHER_EVERY == 0 or k + 1 == steps):
                        ev = torch.cuda.Event()
                        ev.record()
                        gather_chunk(k0, k + 1, [ev])
                        k0 = k + 1
        if world > 1:
            gather_finish()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """barrier + sync | CUDA events around fn(steps) | barrier + sync; max over ranks."""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(steps)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    run_resident(args.warmup)
    run_e2e(3)
    torch.cuda.synchronize()

    fb0 = _lib.fallback_count()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    n0 = _lib.launch_count()
    last = []
    ms_total = timed(lambda steps: last.append(run_resident(steps)), K)
    launches = _lib.launch_count() - n0
    if args.dump_outputs:
        # copied now: the e2e and latency runs below replay into the same result buffers
        dumped = {k: v.cpu() for k, v in last[0].items()}
        if world > 1:
            # gathered[] holds each chunk of steps k0..K-1 rank by rank
            k0 = (K - 1) // GATHER_EVERY * GATHER_EVERY
            rows = [(world * k0 + r * (K - k0) + K - 1 - k0) * B for r in range(world)]
            dumped["depth_0_all_ranks"] = torch.stack([gathered[i:i + B] for i in rows]).cpu()
        if rank == 0:
            dump_outputs(args.dump_outputs, dumped)
    if graphed is not None:      # graph replays launch the captured libcasmvs kernels
        launches += graphed.kernels_per_replay * K
    run_e2e(max(3, args.warmup))     # copy engines / PCIe links idled during the resident timing
    ms_e2e = timed(run_e2e, K)
    run_one_at_a_time(3)
    ms_single = timed(run_one_at_a_time, K)
    clocks = sampler.stop() if sampler else None

    # ---- sustained: the same resident step back to back for >= 2 s (clocks settle below boost)
    sus_sampler = ClockSampler(local_rank) if rank == 0 else None
    if sus_sampler:
        sus_sampler.start()
    chunk = max(50, int(0.25 / max(ms_total / K * 1e-3, 1e-6)))
    sus_steps, sus_ms = 0, 0.0
    while sus_ms < 2000.0:
        sus_ms += timed((lambda n: pipe.run_resident(n)) if pipe is not None
                        else (lambda n: [model(imgs_d, pm_d, dmin, dint) for _ in range(n)]), chunk)
        sus_steps += chunk
    sus_clocks = sus_sampler.stop() if sus_sampler else None
    sustained = None
    if rank == 0:
        sustained = {"seconds": sus_ms * 1e-3, "steps": sus_steps,
                     "depth_maps_per_s": world * B * sus_steps / (sus_ms * 1e-3),
                     "sm_mhz_median": sus_clocks["sm_mhz"], "power_w_max": sus_clocks["power_w_max"],
                     "reasons": sus_clocks["reasons"],
                     "what": "CUDA-graph replays of the resident step back to back (3 views in flight), "
                             "no collective"}
    fallbacks = _lib.fallback_count() - fb0

    extras_failed = {}
    # ---- K1 roofline: the three launches of one depth map, CUDA events, L2 flushed ----
    roofline = None
    hot = None
    if rank == 0:
        try:
            peak, peak_src = measured_peak_hbm()
            flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2
            per_stage_bytes = k1_algorithmic_bytes(VIEWS)
            stage_ms, stage_ms_mat = [], []
            with torch.no_grad():
                feats = model.feature(imgs_d.reshape(B * VIEWS, 3, H_IMG, W_IMG))
                for i, l in enumerate((2, 1, 0)):
                    f = feats[f"level_{l}"]
                    f = f.view(B, VIEWS, *f.shape[1:])
                    D = N_DEPTHS[l]
                    h, w = f.shape[-2:]
                    pml = pm_d[:, :, l].contiguous()
                    # the shipped cascade hands K1 the hypothesis LADDER (first + step*d, generated
                    # in the kernel); the materialised (B,D,h,w) form of the public API is timed too
                    lad = ops.Ladder(dmin + 3.0 * l, dint * RATIOS[l], D, B, h, w, dev)
                    dv = lad.materialize()
                    use_ladder = model.fuse_hypotheses and ops.ladder_supported(VIEWS, f.shape[2], 1)
                    forms = [("ladder", lambda: ops.warp_cost_ladder(f, pml, lad, 1))] if use_ladder else []
                    forms.append(("tensor", lambda: ops.warp_cost(f, pml, dv, 1, ops.NHWC)))
                    res_ms = {}
                    for name, fn in forms:
                        ts = []
                        for it in range(3 + 10):
                            flush.zero_()
                            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                            e0.record()
                            fn()
                            e1.record()
                            torch.cuda.synchronize()
                            if it >= 3:
                                ts.append(e0.elapsed_time(e1))
                        res_ms[name] = sum(ts) / len(ts)
                    stage_ms.append(res_ms.get("ladder", res_ms["tensor"]))
                    stage_ms_mat.append(res_ms["tensor"])
            tot_bytes = sum(per_stage_bytes)
            tot_ms = sum(stage_ms)
            achieved = tot_bytes / (tot_ms * 1e-3) / 1e9
            roofline = {"kernel": "warp_var_smem kernel (K1, TMA-staged fused warp+variance), 3 launches / depth map",
                        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                        "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                        "per_stage": [{"level": l, "algorithmic_bytes": b, "ms": m,
                                       "GBps": b / (m * 1e-3) / 1e9}
                                      for l, b, m in zip((2, 1, 0), per_stage_bytes, stage_ms)],
                        "l2": "flushed (256 MiB memset) before every timed launch",
                        "hypotheses": ("ladder first + step*d generated in the kernel (what "
                                       "CascadeMVSNet.forward runs); algorithmic bytes keep the API-level "
                                       "D*h*w hypothesis term (SURVEY.md 8d)") if stage_ms != stage_ms_mat
                                      else "materialised (B,D,h,w) tensor",
                        "materialised_hypotheses": {"ms": stage_ms_mat,
                                                    "frac": tot_bytes / (sum(stage_ms_mat) * 1e-3) / 1e9 / peak}}
            prof = os.path.join(ROOT, "profiles", "k1_traffic.json")
            if os.path.isfile(prof):
                try:
                    roofline["traffic"] = json.load(open(prof)).get("dram_bytes_per_depth_map")
                except Exception:
                    pass
            # hot path only (features resident): K4+K1+K2+K3 x 3 stages
            def hot_only():
                depth_l = None
                for l in (2, 1, 0):
                    f = feats[f"level_{l}"]
                    f = f.view(B, VIEWS, *f.shape[1:])
                    depth_l, _ = model.run_stage(l, f, pm_d[:, :, l].contiguous(), depth_l, dmin, dint)
            with torch.no_grad():
                for _ in range(3):
                    hot_only()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    hot_only()
                e1.record()
                torch.cuda.synchronize()
                hot_ms = e0.elapsed_time(e1) / args.steps
            hot = {"ms_per_depth_map": hot_ms, "depth_maps_per_s": 1e3 / hot_ms,
                   "what": "features resident -> depth/confidence (K4,K1,K2,K3 x 3 stages), no FeatureNet"}
        except Exception as e:                                       # noqa: BLE001
            extras_failed["roofline_k1"] = f"{type(e).__name__}: {e}"[:300]
            print(f"WARNING: bench extra 'roofline_k1' failed: {e}", file=sys.stderr)

    # ---- K2 roofline: the three CostRegNet stacks (11 layers each), CUDA events, L2 flushed
    roofline_k2 = None
    if rank == 0:
        try:
            stage_ms = []
            with torch.no_grad():
                for l in (2, 1, 0):
                    f = feats[f"level_{l}"]
                    f = f.view(B, VIEWS, *f.shape[1:])
                    D = N_DEPTHS[l]
                    h, w = f.shape[-2:]
                    dv = ops.uniform_hypotheses(dmin + 3.0 * l, dint * RATIOS[l], D, B, h, w, dev)
                    cost = ops.warp_cost(f, pm_d[:, :, l].contiguous(), dv, 1, ops.NHWC,
                                         round_tf32=(args.precision == "tf32"))
                    reg = getattr(model, f"cost_reg_{l}")
                    # the 11 launches of a stack as ONE captured graph: launched eagerly from
                    # Python the coarsest stack (0.19 ms of GPU work) is bound by the host
                    for _ in range(2):
                        reg(cost)
                    torch.cuda.synchronize()
                    _lib.check(_lib.load().casmvs_settle_weight_images(), "settle_weight_images")
                    stack = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(stack):
                        reg(cost)
                    ts = []
                    for it in range(3 + 10):
                        flush.zero_()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        stack.replay()
                        e1.record()
                        torch.cuda.synchronize()
                        if it >= 3:
                            ts.append(e0.elapsed_time(e1))
                    stage_ms.append(sum(ts) / len(ts))
                    del cost, stack
            k2_ms = sum(stage_ms)
            roofline_k2 = {"kernel": "CostRegNet x3 (33 tcgen05 conv launches / depth map)",
                           "algorithmic_bytes": K2_ALGO_BYTES, "flop": K2_ALGO_FLOP, "ms": k2_ms,
                           "per_stage_ms": dict(zip(("level_2", "level_1", "level_0"), stage_ms)),
                           "GBps": K2_ALGO_BYTES / (k2_ms * 1e-3) / 1e9,
                           "frac_hbm": K2_ALGO_BYTES / (k2_ms * 1e-3) / 1e9 / peak,
                           "TFLOPps": K2_ALGO_FLOP / (k2_ms * 1e-3) / 1e12,
                           "bound": "hbm (fp32 activations, Cout <= 64: 44 FLOP/B << ridge)",
                           "tensor_pipe_pct": None,
                           "l2": "flushed before every timed stack (each stack = one captured graph)"}
            prof = os.path.join(ROOT, "profiles", "k2_tensor_pipe.json")
            if os.path.isfile(prof):
                try:
                    roofline_k2["tensor_pipe_pct"] = json.load(open(prof))
                except Exception:
                    pass
        except Exception as e:                                       # noqa: BLE001
            extras_failed["roofline_k2"] = f"{type(e).__name__}: {e}"[:300]
            print(f"WARNING: bench extra 'roofline_k2' failed: {e}", file=sys.stderr)

    cpu_baseline = None
    parity = None
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        try:
            avail = len(os.sched_getaffinity(0))
            cores = best_cpu_threads(avail)
            med, total, ref_out = time_cpu_port(3, 1, cores, want_result=True)
            # parity of THIS run's GPU output against the oracle on the same seed-0 inputs/weights
            with torch.no_grad():
                got = graphed() if graphed is not None else model(imgs_d, pm_d, dmin, dint)
            torch.cuda.synchronize()
            parity = {}
            for l in (2, 1, 0):
                d, r = got[f"depth_{l}"].cpu(), ref_out[f"depth_{l}"]
                parity[f"rel_l1_depth_{l}"] = ((d - r).abs().mean() / r.abs().mean()).item()
            gen = torch.Generator().manual_seed(1)
            gt = ref_out["depth_0"] + 5.6 * torch.randn(ref_out["depth_0"].shape, generator=gen)
            a = (got["depth_0"].cpu() - gt).abs().mean().item()
            b = (ref_out["depth_0"] - gt).abs().mean().item()
            parity.update({"rel_l1": parity["rel_l1_depth_0"], "abs_err_ours_mm": a,
                           "abs_err_oracle_mm": b, "abs_err_delta": abs(a - b),
                           "confidence_2_max_delta": (got["confidence_2"].cpu() -
                                                      ref_out["confidence_2"]).abs().max().item(),
                           "against": "oracle.cascade_forward on the same seed-0 inputs and weights "
                                      "(the cpu_baseline run)", "tolerance": "rel_l1 < 1e-3 (north_star)"})
            parity["ok"] = bool(parity["rel_l1"] < 1e-3 and parity["abs_err_delta"] < 1e-3)
            if not parity["ok"]:
                print(f"WARNING: parity against the oracle FAILED: {parity}", file=sys.stderr)
            cpu_baseline = {"value": 1.0 / med, "unit": "depth-maps/s", "cores": cores, "kind": "port",
                            "sample": "1 warm-up + 3 timed full forwards of the same cfg2 workload "
                                      f"(median {med:.2f} s/depth-map), oracle port of the reference "
                                      f"PyTorch-CPU path on {cores} torch threads (fastest of "
                                      f"4..{avail} available)"}
        except Exception as e:                                       # noqa: BLE001
            extras_failed["cpu_baseline_parity"] = f"{type(e).__name__}: {e}"[:300]
            print(f"WARNING: bench extra 'cpu_baseline_parity' failed: {e}", file=sys.stderr)

    other = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            other = run_other_configs(dev, args.precision)
        except Exception as e:                                       # noqa: BLE001
            extras_failed["other_configs"] = f"{type(e).__name__}: {e}"[:300]

    modes = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            modes = run_throughput_modes(model, dev)
        except Exception as e:                                       # noqa: BLE001
            extras_failed["throughput_modes"] = f"{type(e).__name__}: {e}"[:300]

    pipelined = pipe is not None
    sharded = None
    if world > 1 and not args.no_sharded_configs:
        del graphed, pipe
        torch.cuda.empty_cache()
        sharded = {}
        for name in SHARDED_CONFIGS:
            try:
                sharded[name] = run_sharded_config(name, rank, world, dev, args.precision)
            except Exception as e:                                  # noqa: BLE001
                sharded[name] = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0:
        maps = world * B * args.steps
        value = maps / (ms_total * 1e-3)
        h2d = imgs_h.numel() * 4 + pm_h.numel() * 4
        d2h = out_depth_h.numel() * 4 + out_conf_h.numel() * 4
        line = {
            "metric": METRIC, "value": value, "unit": "depth-maps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else f"f32 (conv products {args.precision}, fp32 accumulate)",
            "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "step": ("CascadeMVSNet.forward = FeatureNet (cuDNN fp32 convs + fused FPN "
                                "kernel) + 3 cascade stages") if args.precision == "fp32" else
                               ("CascadeMVSNet.forward = FeatureNet (own kernels: planar tcgen05 "
                                "convs, RGB block, FPN merges) + 3 cascade stages (K4, K1, K2 x 11 "
                                "layers on tcgen05, K3)"),
                       "parallelism": f"dp{world} (independent reference views per rank; the {args.steps} "
                                      f"per-rank depth maps are gathered by all_gather_into_tensor in chunks of "
                                      f"{GATHER_EVERY} steps on a side stream while the next forwards run, all "
                                      "inside the timed region)" if world > 1 else "single GPU",
                       "numa": numa,
                       "precision": args.precision,
                       "cuda_graph": not args.no_graph,
                       "in_flight": ("3 independent reference views on 3 streams (PipelinedCascade slots), "
                                     "value and e2e alike; one_view_at_a_time = the serial latency")
                                    if not args.no_graph else "1",
                       "l2": "per-step working set (>1 GB of intermediates) exceeds the 126 MB L2; "
                             "K1 roofline launches are preceded by an explicit L2 flush"},
            "e2e": {"value": maps / (ms_e2e * 1e-3), "unit": "depth-maps/s",
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps,
                    "how": ("pinned host inputs -> H2D -> CUDA-graph forward -> D2H of depth_0 + "
                            "confidence_2, every step; copies of neighbouring steps overlap compute "
                            "(PipelinedCascade: 3 slots, one compute stream per slot, so consecutive views "
                            "also overlap each other on the GPU)") if pipelined else
                           "pinned host inputs -> H2D -> forward -> D2H, serial"},
            "one_view_at_a_time": {"ms_per_step": ms_single / args.steps,
                                   "value": world * B * args.steps / (ms_single * 1e-3),
                                   "what": "the same K forwards replayed one after the other on one "
                                           "stream (latency of a single depth map); `value` keeps "
                                           "3 independent views in flight on 3 streams"},
            "parity": parity,
            "extras_failed": extras_failed or None,
            "sharded_configs": sharded,
            "other_configs": other,
            "throughput_modes": modes,
            "fallbacks": fallbacks,
            "sustained": sustained,
            "roofline_k2": roofline_k2,
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline,
            "hot_path": hot,
            "cpu_baseline": cpu_baseline,
        }
        print(json.dumps(line), flush=True)
    if fallbacks:           # the tests assert 0; here the line itself carries the evidence
        print(f"WARNING: {fallbacks} tf32 layers fell back to the CUDA-core kernel", file=sys.stderr)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
