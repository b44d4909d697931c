#!/usr/bin/env python
"""bench.py -- PointFlow iterations / second on synthetic DTU-shaped input.

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on host cores
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as .npy

A "step" is one pass of the hot path (the 3-iteration point_flow loop, reference
pointmvsnet/model.py:297-303) over one reference view per GPU; metric = PointFlow
iterations per second (one iteration = one point_flow call), whole job over all ranks.
Multi-GPU (torchrun, one rank per GPU): reference views are sharded over ranks, the only
collective is the NCCL all-gather of the final depth maps inside every step (weak scaling).

Prints ONE JSON line on rank 0.  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (no __pycache__)

CONFIGS = {
    # name: (H, W, V, D)   V counts the reference view (dataset.py:84): "3 src views" = V 4
    "C2": (512, 640, 4, 96),
    "C3": (512, 640, 6, 96),
    "C4": (960, 1280, 4, 96),
    "C5": (1184, 1600, 6, 96),
    "small": (64, 128, 3, 48),
}
IMG_SCALES = (0.125, 0.25, 0.5)      # config.py:70
INTER_SCALES = (1.0, 0.75, 0.15)     # config.py:71
METRIC = "PointFlow iters/sec"


def load_pretrained_hot_path_weights():
    """The reference's shipped hot-path weights (outputs/dtu_wde3/model_pretrained.pth, keys flow_edge_conv.* /
    flow_mlp.*), committed as the fixture tests/golden/flow_weights.npz (SURVEY.md a16)."""
    import numpy as np
    z = np.load(os.path.join(ROOT, "tests", "golden", "flow_weights.npz"))
    return {k: torch.from_numpy(z[k]) for k in z.files}


def survey_8d_bytes_per_pass(H, W, V, B=1):
    """SURVEY.md 8(d) algorithmic bytes of one 3-iteration pass, per stage (fp32, int64 indices as the public API
    mandates, single-pass BatchNorm ideal): the numerators of `roofline_stage`."""
    fetch = knn = chain = 0
    prev = (H // 8) * (W // 8)
    for s in IMG_SCALES:
        h, w = int(H * s), int(W * s)
        P = h * w * B
        fetch += 28 * V * H * W * B + 4 * prev * B + 2720 * P + 60 * P
        knn += 5 * P * 140
        chain += 5 * P * 3108
        prev = h * w
    return {"fetch": fetch, "knn": knn, "edgeconv_mlp": chain}


def workload_name(cfg, H, W, V, D):
    return "%s: DTU-shape %dx%d, %d src views (V=%d), %d depth hyp, %d flow iters, B=1 per pass" % (
        cfg, W, H, V - 1, V, D, len(IMG_SCALES))


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


DUMP_LIMIT_BYTES = 64 * 1000 * 1000


def pass_outputs(outs, prefix=""):
    """[(depth, prob)] per iteration of one pass -> {name: tensor} under the reference's prediction names
    (flow1, flow1_prob, ..., model.py:297-303)."""
    arrays = {}
    for i, (depth, prob) in enumerate(outs):
        arrays["%sflow%d" % (prefix, i + 1)] = depth
        arrays["%sflow%d_prob" % (prefix, i + 1)] = prob
    return arrays


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT_BYTES):
    """Writes {name: tensor} as <out_dir>/<name>.npy in float32.  When the arrays hold more than `limit` bytes in
    all, each one is cut to the same fraction of its elements: a sample drawn with a fixed seed, flattened, in
    ascending element order, so that two runs with the same arguments write the same positions."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.detach().float().cpu() for k, v in arrays.items()}
    total = sum(t.numel() * 4 for t in host.values())
    frac = min(1.0, (limit - 256 * len(host)) / max(total, 1))  # 256 B per file for the .npy header
    for name, t in host.items():
        if frac < 1.0:
            keep = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:int(t.numel() * frac)]
            t = t.reshape(-1)[keep.sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy())


# --------------------------------------------------------------------------------------
# algorithmic bytes per kernel launch class over ONE pass (DESIGN.md "Kernels")
# --------------------------------------------------------------------------------------
def algorithmic_bytes_per_pass(H, W, V, B=1):
    """dict kernel-name -> (bytes per pass, launches per pass).  fp32, int32 internal indices."""
    out = {}

    def add(name, nbytes):
        b, n = out.get(name, (0, 0))
        out[name] = (b + nbytes, n + 1)

    pyr_bytes = 28 * V * H * W * B  # V*(16*HW/4 + 32*HW/16 + 64*HW/64)*4
    for c, (hh, ww) in zip((16, 32, 64), ((H // 2, W // 2), (H // 4, W // 4), (H // 8, W // 8))):
        add("transpose", 2 * B * V * c * hh * ww * 4)
    prev = (H // 8) * (W // 8)
    for s in IMG_SCALES:
        h, w = int(H * s), int(W * s)
        P = h * w * B
        R = 5 * P
        # model.py:184 materialised once per iteration: read the pyramids, write [B,V,h,w,112] fp32
        add("warp_source", pyr_bytes + B * V * h * w * 448)
        add("fused_fetch", pyr_bytes + 4 * prev * B + 2720 * P + 60 * P)
        add("knn3d", R * (12 + 64))
        for (cin, cout2, c) in ((136, 64, 32), (32, 64, 32), (64, 128, 64)):
            add("gemm_%dx%d" % (cin, cout2), R * 4 * (cin + cout2))
            add("edge_stats_%d" % c, R * (8 * c + 64))
            add("edge_apply_%d" % c, R * (8 * c + 64 + 4 * (c if cin == 136 else 2 * c)))
        for (cin, cout) in ((224, 64), (64, 64), (64, 16)):
            add("gemm_%dx%d" % (cin, cout), R * 4 * (cin + cout))
        add("flow_head", R * 64 + P * 28)
        prev = h * w
    return out


def sample_clocks_start(local_gpu):
    try:
        f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        p = subprocess.Popen(
            ["nvidia-smi", "-i", str(local_gpu),
             "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
            stdout=f, stderr=subprocess.DEVNULL)
        return p, f
    except Exception:
        return None, None


def sample_clocks_stop(p, f):
    if p is None:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    time.sleep(0.15)
    p.terminate()
    try:
        p.wait(timeout=5)
    except Exception:
        p.kill()
    f.flush()
    f.seek(0)
    sm, mx, reasons = [], [], set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for line in f.read().strip().splitlines():
        parts = [x.strip() for x in line.split(",")]
        if len(parts) < 7:
            continue
        try:
            sm.append(float(parts[0]))
            mx.append(float(parts[1]))
        except ValueError:
            continue
        for nm, val in zip(names, parts[3:7]):
            if val.lower().startswith("active"):
                reasons.add(nm)
    f.close()
    try:
        os.unlink(f.name)
    except OSError:
        pass
    sm.sort()
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------
# CPU legs (the oracle is executed here ONLY as the reported baseline / reference arm)
# --------------------------------------------------------------------------------------
def cpu_reference_pass(cfg_name, steps, warmup, budget_s=200.0):
    """Times the reference algorithm (oracle/pointflow_oracle.py, a restatement of the
    reference's Python; /root/reference itself does not exist on the GPU box) on the host
    cores.  A step is ALWAYS one whole 3-iteration pass of the same workload (same inputs, same
    pretrained weights); when `steps + warmup` passes do not fit the time budget, FEWER passes are
    timed (never a part of a pass) and the count actually timed is returned.
    Returns (iters_per_s, ms_per_step, info)."""
    from oracle import pointflow_oracle as O
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    H, W, V, D = CONFIGS[cfg_name]
    cores = os.cpu_count() or 1
    inp = make_pointflow_inputs(H, W, V, 1, D, seed=0)
    params = O.params_from_state_dict(load_pretrained_hot_path_weights())
    scales, inters = IMG_SCALES, INTER_SCALES

    def one(sc, it):
        with torch.no_grad():
            O.point_flow_pass(inp["coarse_depth"], inp["depth_interval"], inp["pyramids"], inp["cam_params_list"],
                              inp["mean"], inp["std"], inp["img_hw"], params, img_scales=sc, inter_scales=it)

    # Give the reference its best thread count: PyTorch's CPU kernels on these per-call tensors
    # get slower with too many threads (all 128 host threads are ~10x slower than 16 on the B200 host), so
    # iteration 1 is timed at a few pool sizes and the fastest is kept; `cores` reports it.
    t_begin = time.time()
    best = None
    for nt in sorted({t for t in (8, 16, 32, 64, cores) if t <= cores}):
        torch.set_num_threads(nt)
        if best is None:
            one(scales[:1], inters[:1])  # allocator / thread-pool warm-up
        t0 = time.time()
        one(scales[:1], inters[:1])
        dt = time.time() - t0
        if best is None or dt < best[1]:
            best = (nt, dt)
        if dt > 4 * best[1]:
            break
    torch.set_num_threads(best[0])
    n_sub = sum(int(round(sc * 8)) ** 2 for sc in scales)  # 21 equal-sized sub-cloud calls per pass
    est_pass = best[1] * n_sub
    left = budget_s - (time.time() - t_begin)
    n_warm = warmup if est_pass * (warmup + 1) < left else (1 if est_pass * 2 < left else 0)
    n_timed = int(max(1, min(steps, (left - n_warm * est_pass) // max(est_pass, 1e-3))))
    for _ in range(n_warm):
        one(scales, inters)
    times = []
    for _ in range(n_timed):
        t0 = time.time()
        one(scales, inters)
        times.append(time.time() - t0)
    ms = 1e3 * sum(times) / len(times)
    value = len(scales) / (ms / 1e3)
    sample = "%d whole pass(es) of the same workload timed (%d requested), %d warm-up pass(es)" % (n_timed, steps, n_warm)
    return value, ms, {"cores": best[0], "host_cores": cores, "sample": sample, "kind": "port",
                       "steps_timed": n_timed, "warmup_done": n_warm}


def run_reference_arm(args):
    rank, world, local = dist_env()
    if rank != 0:
        return
    H, W, V, D = CONFIGS[args.config]
    value, ms, info = cpu_reference_pass(args.config, max(1, args.steps), args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "iters/s", "n_gpus": args.gpus,
        # steps / warmup are the counts actually RUN (whole passes; fewer than requested when they would not fit
        # the few-minute bound), so that steps * ms_per_step is the measured time
        "steps": info["steps_timed"], "warmup": info["warmup_done"], "steps_requested": args.steps,
        "warmup_requested": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.config, H, W, V, D), "step": "one whole 3-iteration pass",
                   "weights": "pretrained hot-path weights (tests/golden/flow_weights.npz)"},
        "cpu_baseline": {"value": value, "unit": "iters/s", "cores": info["cores"], "kind": info["kind"],
                         "host_cores": info["host_cores"], "sample": info["sample"]},
        "e2e": {"value": value, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def per_iteration_kernel_ms(recs, n_iter):
    """Profile records [(kernel name, ms)] in launch order -> mean kernel-time per iteration size.

    Every iteration of a pass starts with the `cam_setup` launch (csrc/api.cu, pmvs_point_flow_iter);
    launches before the first one of a pass (the pyramid transposes) are not part of an iteration.
    Returns a list of n_iter floats (ms, summed kernel time of that iteration averaged over the
    recorded passes) or None if the records do not have that structure."""
    sums = [0.0] * n_iter
    counts = [0] * n_iter
    it = -1
    seen = 0
    for name, ms in recs:
        if name == "cam_setup":
            it = seen % n_iter
            seen += 1
            counts[it] += 1
        elif name == "transpose":
            it = -1
        if it >= 0:
            sums[it] += ms
    if seen == 0 or seen % n_iter != 0 or len(set(counts)) != 1:
        return None
    return [s / counts[0] for s in sums]


# --------------------------------------------------------------------------------------
# this repo's arm
# --------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from pointmvsnet_b200 import _lib
    from pointmvsnet_b200.point_flow import PointFlow, PointFlowPass
    from pointmvsnet_b200.synthetic import make_pointflow_inputs, make_flow_params
    from pointmvsnet_b200.parallel import gather_depth_maps, state_dict_from_params

    rank, world, local = dist_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback in the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL_DEBUG=VERSION (this image's default) makes NCCL print a banner on stdout; stdout must
        # carry ONE JSON line, so the banner is switched off (any other explicit level is kept)
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=dev)
    H, W, V, D = CONFIGS[args.config]
    n_iter = len(IMG_SCALES)

    # Every rank owns G different reference views (different seeds): weak scaling.  The G views of a
    # rank are independent passes (own inputs, own workspace, own BatchNorm buffers) whose CUDA
    # graphs are replayed concurrently on G streams - small launches of one view fill the SMs the
    # other view leaves idle.  G = 1 is the plain "one pass per step".
    import copy
    G = max(1, args.views_in_flight)
    hosts = [make_pointflow_inputs(H, W, V, 1, D, seed=rank * G + g, pin_memory=True) for g in range(G)]
    to_dev = lambda h: {k: ([t.to(dev) for t in v] if isinstance(v, list) else (v.to(dev) if torch.is_tensor(v) else v))
                        for k, v in h.items()}
    gpu_ins = [to_dev(h) for h in hosts]
    gpu_in = gpu_ins[0]
    pf = PointFlow().to(dev)
    pf.load_reference_state_dict(load_pretrained_hot_path_weights())
    pf.train()  # BN batch statistics, test.py:58

    def capture_set():
        """G captured passes (one per view in flight); views > 0 get their own module copy so that
        the BatchNorm running-statistics side effect is neither shared nor skipped."""
        pipes = []
        with torch.no_grad():
            for g in range(G):
                m = PointFlow(flow_edge_conv=copy.deepcopy(pf.flow_edge_conv), flow_mlp=copy.deepcopy(pf.flow_mlp)).to(dev)
                m.train()
                pipes.append(PointFlowPass(m, IMG_SCALES, INTER_SCALES).capture(gpu_ins[g]))
        return pipes

    set_a = capture_set()
    launches_per_pass = set_a[0].launches_per_pass
    h_f, w_f = set_a[0].outs[-1][0].shape[-2:]
    final_depths = torch.empty(G, 1, h_f, w_f, device=dev)   # the step's result: G final depth maps
    gathered = [torch.empty_like(final_depths) for _ in range(world)] if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    stream = torch.cuda.current_stream(dev)
    side = [torch.cuda.Stream(device=dev) for _ in range(G)]

    def replay_set(pipes):
        if G == 1:
            pipes[0].replay()
            final_depths[0].copy_(pipes[0].outs[-1][0][0])
            return
        for g in range(G):
            side[g].wait_stream(stream)
            with torch.cuda.stream(side[g]):
                pipes[g].replay()
                final_depths[g].copy_(pipes[g].outs[-1][0][0])
        for g in range(G):
            stream.wait_stream(side[g])

    def step():
        replay_set(set_a)
        if world > 1:
            gather_depth_maps(final_depths, gathered)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(nsteps, body):
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(nsteps)]
        ends = [torch.cuda.Event(enable_timing=True) for _ in range(nsteps)]
        barrier()
        for i in range(nsteps):
            flush.zero_()  # evict L2 between steps (untimed)
            starts[i].record(stream)
            body()
            ends[i].record(stream)
        barrier()
        total_ms = sum(s.elapsed_time(e) for s, e in zip(starts, ends))
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    for _ in range(max(3, args.warmup)):
        step()
    clk_p, clk_f = sample_clocks_start(local) if rank == 0 else (None, None)
    total_ms = timed(args.steps, step)
    clocks = sample_clocks_stop(clk_p, clk_f) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the last timed step's results: every view's pass outputs, and with several ranks the gathered depth maps
        arrays = {}
        for g, pipe in enumerate(set_a):
            arrays.update(pass_outputs(pipe.outs, "view%d_" % g))
        for r, t in enumerate(gathered or []):
            arrays["rank%d_final_depth" % r] = t
        dump_outputs(args.dump_outputs, arrays)
    ms_per_step = total_ms / args.steps
    value = world * G * n_iter / (ms_per_step / 1e3)

    # ---- end-to-end: host buffers in, host result out, copies inside the timed region -----
    # Two sets of captured graphs with their own static input buffers alternate; the H2D copies of
    # step i+1 (pinned host memory, copy stream) overlap the compute of step i; the D2H read of the
    # step's final depth maps closes every step.  Every step's H2D and D2H are inside the timed region.
    host_out = torch.empty(final_depths.shape, dtype=torch.float32).pin_memory()
    h2d = G * (sum(p.numel() * 4 for p in hosts[0]["pyramids"]) + sum(
        hosts[0][k].numel() * 4 for k in ("coarse_depth", "cam_params_list", "depth_interval", "mean", "std")))
    d2h = host_out.numel() * 4
    sets = [set_a, capture_set()]
    copy_stream = torch.cuda.Stream(device=dev)
    copied = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def copy_set(pipes):
        for g in range(G):
            pipes[g].copy_inputs(hosts[g], non_blocking=True)

    def e2e_run(nsteps):
        """returns total device time (ms) from the first H2D to the last D2H"""
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        flush.zero_()
        torch.cuda.synchronize(dev)
        t0.record(stream)
        copy_stream.wait_stream(stream)
        with torch.cuda.stream(copy_stream):
            copy_set(sets[0])
            copied[0].record(copy_stream)
        for i in range(nsteps):
            cur, nxt = i % 2, (i + 1) % 2
            if i + 1 < nsteps:
                with torch.cuda.stream(copy_stream):
                    if i >= 1:
                        copy_stream.wait_event(consumed[nxt])  # step i-1 finished reading those buffers
                    copy_set(sets[nxt])
                    copied[nxt].record(copy_stream)
            stream.wait_event(copied[cur])
            flush.zero_()  # cold L2 for every step (timed: ~40 us of the step)
            replay_set(sets[cur])
            consumed[cur].record(stream)
            if world > 1:
                gather_depth_maps(final_depths, gathered)
            host_out.copy_(final_depths, non_blocking=True)
        t1.record(stream)
        barrier()
        t = torch.tensor([t0.elapsed_time(t1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()

    e2e_run(3)
    e2e_ms = e2e_run(args.steps) / args.steps
    e2e_value = world * G * n_iter / (e2e_ms / 1e3)

    # ---- per-kernel CUDA-event timing (eager, not captured) for the roofline ---------------
    roofline = None
    roofline_stage = None
    roofline_gemm = None
    kernel_table = None
    by_size = None
    if rank == 0:
        with torch.no_grad():
            eager = PointFlowPass(pf, IMG_SCALES, INTER_SCALES)
            run = lambda: eager.run(gpu_in["pyramids"], gpu_in["coarse_depth"], gpu_in["cam_params_list"],
                                    gpu_in["depth_interval"], gpu_in["mean"], gpu_in["std"], gpu_in["img_hw"])
            run()
            torch.cuda.synchronize(dev)
            _lib.profile_enable(True)
            reps = 5
            for _ in range(reps):
                flush.zero_()
                run()
            torch.cuda.synchronize(dev)
            _lib.profile_enable(False)
            recs = _lib.profile_collect()
        agg = {}
        for name, ms in recs:
            a = agg.setdefault(name, [0.0, 0])
            a[0] += ms
            a[1] += 1
        by_size = None
        try:  # SURVEY 8d: per-iteration-size rates next to the pass rate (kernel time, one view in flight)
            it_ms = per_iteration_kernel_ms(recs, n_iter)
            if it_ms is not None:
                by_size = [{"flow_hw": [int(H * sc), int(W * sc)], "points": 5 * int(H * sc) * int(W * sc),
                            "kernel_ms": round(m, 4), "iters_per_s": round(1e3 / m, 1)}
                           for sc, m in zip(IMG_SCALES, it_ms)]
        except Exception:
            by_size = None
        alg = algorithmic_bytes_per_pass(H, W, V)
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        traffic = {}
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json")))
        except Exception:
            pass
        kernel_table = {}
        tot = sum(a[0] for a in agg.values())
        for name, (ms, cnt) in sorted(agg.items(), key=lambda kv: -kv[1][0]):
            per_pass_ms = ms / reps
            ab = alg.get(name, (0, 0))[0]
            gbps = ab / (per_pass_ms * 1e-3) / 1e9 if per_pass_ms > 0 else None
            kernel_table[name] = {"ms_per_pass": round(per_pass_ms, 5), "share": round(ms / tot, 4),
                                  "launches_per_pass": cnt // reps,
                                  "alg_GBps": round(gbps, 1) if gbps is not None else None,
                                  "hbm_frac": round(gbps / hbm_peak, 4) if gbps is not None else None}
        # tensor-pipe view of the contraction kernels: executed TF32 FLOPs (3 products per element
        # for 3xTF32) over their summed time, against half the measured dense bf16 GEMM rate
        # (kind::tf32 runs at half the bf16 rate; MEASURED_PEAKS.json has no TF32 figure)
        gemm_ms = sum(ms for name, (ms, cnt) in agg.items() if name.startswith("gemm_")) / reps
        mac_per_pt = 136 * 64 + 32 * 64 + 64 * 128 + 224 * 64 + 64 * 64 + 64 * 16
        pts = sum(5 * int(H * sc) * int(W * sc) for sc in IMG_SCALES)
        mode = _lib.lib.pmvs_get_gemm_mode()
        flops = 2.0 * mac_per_pt * pts * (3 if mode == 3 else 1)
        tf32_peak = float(peaks.get("bf16_tflops", 1590.0)) / 2.0
        roofline_gemm = None
        if gemm_ms > 0 and mode != 0:
            ach = flops / (gemm_ms * 1e-3) / 1e12
            roofline_gemm = {"kernels": "gemm_* (tcgen05 kind::tf32, mode %d)" % mode, "bound": "tensor",
                             "achieved": round(ach, 1), "peak": round(tf32_peak, 1), "unit": "TFLOP/s",
                             "frac": round(ach / tf32_peak, 4), "ms_per_pass": round(gemm_ms, 4),
                             "peak_source": "MEASURED_PEAKS.json bf16_tflops / 2 (TF32 runs at half the bf16 rate)",
                             "note": "the contractions are memory bound (25 FLOP/B): see kernels[*].alg_GBps"}
        # SURVEY.md 8(d) stage rooflines: the stage's single-pass algorithmic bytes over the summed event time of
        # the kernels that implement it (the pyramid `transpose` launches and the BN running-statistics update are
        # layout / bookkeeping outside 8(d)'s three stages and only enter the whole-pass line)
        surv = survey_8d_bytes_per_pass(H, W, V)
        stage_of = lambda n: ("fetch" if n in ("warp_source", "fused_fetch", "cam_setup") else
                              "knn" if n == "knn3d" else
                              "edgeconv_mlp" if (n.startswith("gemm_") or n.startswith("edge_") or n == "flow_head") else None)
        st_ms = {}
        for name, (ms, cnt) in agg.items():
            k = stage_of(name)
            if k is not None:
                st_ms[k] = st_ms.get(k, 0.0) + ms / reps
        roofline_stage = []
        for k, nb in list(surv.items()) + [("whole_pass", sum(surv.values()))]:
            ms = st_ms.get(k, 0.0) if k != "whole_pass" else tot / reps
            if ms > 0:
                gb = nb / (ms * 1e-3) / 1e9
                roofline_stage.append({"stage": k, "bound": "hbm", "alg_bytes_per_pass": int(nb), "ms_per_pass": round(ms, 4),
                                       "achieved": round(gb, 1), "peak": hbm_peak, "unit": "GB/s",
                                       "frac": round(gb / hbm_peak, 4), "numerator": "SURVEY.md 8(d)"})
        dom = max(agg.items(), key=lambda kv: kv[1][0])[0]
        dom_ms_per_launch = agg[dom][0] / agg[dom][1]
        dom_bytes_per_launch = alg.get(dom, (0, 1))[0] / max(1, alg.get(dom, (0, 1))[1])
        achieved = dom_bytes_per_launch / (dom_ms_per_launch * 1e-3) / 1e9
        roofline = {"kernel": dom, "bound": "hbm", "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s",
                    "frac": round(achieved / hbm_peak, 4), "traffic": traffic.get(dom),
                    "traffic_source": ("static: ncu capture of one pass, profiles/dram_traffic.json (%s)" %
                                       traffic.get("_capture", "see its _comment")) if traffic.get(dom) else None,
                    "numerator": "bytes this kernel must read + write once given its boundaries (DESIGN.md 3); the "
                                 "SURVEY 8(d) stage figures are in roofline_stage",
                    "peak_source": peak_src,
                    "avg_launch_ms": round(dom_ms_per_launch, 5),
                    "alg_bytes_per_launch": int(dom_bytes_per_launch),
                    "kernel_sum_ms_per_pass": round(tot / reps, 4)}

    # ---- reported CPU baseline (rank 0, N=1 only) -------------------------------------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, ms, info = cpu_reference_pass(args.config, 1, 0, budget_s=60.0)
        cpu_baseline = {"value": round(v, 4), "unit": "iters/s", "cores": info["cores"], "kind": info["kind"],
                        "host_cores": info["host_cores"], "sample": info["sample"], "ms_per_pass": round(ms, 1)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": round(value, 2), "unit": "iters/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": round(ms_per_step, 5), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.config, H, W, V, D),
                       "step": "%d reference view(s) in flight per GPU: one 3-iteration point_flow pass each (B=1, own "
                               "BatchNorm statistics), CUDA-graph replays on %d stream(s) + NCCL all-gather of the "
                               "final depth maps" % (G, G),
                       "views_in_flight": G,
                       "l2": "flushed between steps (256 MiB memset, untimed); per-step CUDA events, max over ranks",
                       "parallelism": "dp%d over reference views" % world, "bn": "batch statistics (train mode)",
                       "weights": "pretrained hot-path weights of the reference (tests/golden/flow_weights.npz)",
                       "options": {k: _lib.get_option(k) for k in ("edge", "knn", "fetch", "gemm")}},
            "e2e": {"value": round(e2e_value, 2), "unit": "iters/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": round(e2e_ms, 5),
                    "how": "pinned host -> device copy of every step's inputs on a copy stream, double-buffered "
                           "against the previous step's compute; final depth map read back every step; "
                           "one CUDA-event pair around all steps; a 256 MiB L2 flush runs "
                           "inside every timed step"},
            "gpu_launches": int(launches_per_pass * G * args.steps),
            "launches_per_step": int(launches_per_pass * G),
            "clocks": clocks, "roofline": roofline, "roofline_stage": roofline_stage, "roofline_gemm": roofline_gemm,
            "cpu_baseline": cpu_baseline,
            "kernels": kernel_table,
            "per_iteration_size": by_size,
        }
        result_line = json.dumps(line)
    else:
        result_line = None
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return result_line


def run_subcloud(args):
    """BASELINE C5 style: ONE reference view refined by all ranks (parallel.SubCloudShardedPass): the view's
    pyramids are owned per source view and all-gathered every step, iteration 1 is replicated, iterations 2 / 3 are
    split by sub-cloud, the depth map is all-reduced after every split iteration.  A latency configuration (strong
    scaling): value = iterations / time, NOT multiplied by the number of GPUs; bound 21 / (1 + 1 + 2) = 5.25x at 8."""
    import torch.distributed as dist
    from pointmvsnet_b200 import _lib
    from pointmvsnet_b200.point_flow import PointFlow
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    from pointmvsnet_b200.parallel import SubCloudShardedPass, gather_view_pyramids, shard_views

    rank, world, local = dist_env()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            del os.environ["NCCL_DEBUG"]
        dist.init_process_group("nccl", device_id=dev)
    H, W, V, D = CONFIGS[args.config]
    n_iter = len(IMG_SCALES)
    host = make_pointflow_inputs(H, W, V, 1, D, seed=0, pin_memory=True)   # the same view on every rank
    own = shard_views(V, rank, world)
    host_own = [lv[:, own].contiguous().pin_memory() for lv in host["pyramids"]]
    dev_own = [torch.empty_like(t, device=dev) for t in host_own]
    small = {k: host[k].to(dev) for k in ("coarse_depth", "cam_params_list", "depth_interval", "mean", "std")}
    pf = PointFlow().to(dev)
    pf.load_reference_state_dict(load_pretrained_hot_path_weights())
    pf.train()
    sp = SubCloudShardedPass(pf, rank, world, IMG_SCALES, INTER_SCALES)
    outs = [(torch.empty(1, 1, int(H * s), int(W * s), device=dev), torch.empty(1, 5, int(H * s), int(W * s), device=dev))
            for s in IMG_SCALES]
    host_out = torch.empty(1, 1, int(H * IMG_SCALES[-1]), int(W * IMG_SCALES[-1])).pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream(dev)

    def step(copy_in):
        if copy_in:
            for d, h in zip(dev_own, host_own):
                d.copy_(h, non_blocking=True)
        with torch.no_grad():
            pyr = gather_view_pyramids(dev_own, V, rank, world)
            cl = PointFlow.pyramids_to_channels_last(pyr)
            depth = sp.run(cl, small["coarse_depth"], small["cam_params_list"], small["depth_interval"], small["mean"],
                           small["std"], host["img_hw"], outs=outs)
        if copy_in:
            host_out.copy_(depth, non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(nsteps, copy_in):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        total = 0.0
        for _ in range(nsteps):
            barrier()
            flush.zero_()
            t0.record(stream)
            step(copy_in)
            t1.record(stream)
            torch.cuda.synchronize(dev)
            total += t0.elapsed_time(t1)
        t = torch.tensor([total], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item() / nsteps

    for d, h in zip(dev_own, host_own):
        d.copy_(h)
    for _ in range(max(3, args.warmup)):
        step(False)
    n0 = _lib.launch_count()
    step(False)
    torch.cuda.synchronize(dev)
    launches = _lib.launch_count() - n0
    clk_p, clk_f = sample_clocks_start(local) if rank == 0 else (None, None)
    ms = timed(args.steps, False)
    clocks = sample_clocks_stop(clk_p, clk_f) if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the pass returns the final depth map (the probabilities of other ranks' sub-clouds are not gathered)
        dump_outputs(args.dump_outputs, {"flow%d" % n_iter: outs[-1][0]})
    e2e_ms = timed(args.steps, True)
    line = None
    if rank == 0:
        h2d = sum(t.numel() * 4 for t in host_own)
        line = json.dumps({
            "metric": METRIC, "value": round(n_iter / (ms / 1e3), 2), "unit": "iters/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms, 5), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_name(args.config, H, W, V, D),
                       "step": "ONE reference view per step refined by all %d GPU(s): pyramids owned per source view and "
                               "all-gathered, iteration 1 replicated, iterations 2/3 split by sub-cloud (4 / 16 units), "
                               "depth map all-reduced after each split iteration; eager launches (NCCL inside the step)" % world,
                       "parallelism": "sub-cloud sharding over %d ranks (latency configuration, bound 5.25x at 8)" % world,
                       "l2": "flushed before every step (256 MiB memset, untimed); per-step CUDA events, max over ranks",
                       "weights": "pretrained hot-path weights of the reference (tests/golden/flow_weights.npz)"},
            "e2e": {"value": round(n_iter / (e2e_ms / 1e3), 2), "unit": "iters/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": host_out.numel() * 4, "ms_per_step": round(e2e_ms, 5),
                    "how": "pinned host -> device copy of this rank's own views' pyramids, all-gather, pass, final "
                           "depth map read back, all inside the timed region"},
            "gpu_launches": int(launches * args.steps), "launches_per_step": int(launches), "clocks": clocks,
        })
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


def run_oplevel(args):
    """The operator-level drop-in (an UNCHANGED reference model.py over this package's stand-alone operators,
    pointmvsnet_b200/point_flow_oplevel.py): one reference view per step, eager launches, fp32 (TF32 off for the
    stock flow_mlp convolutions).  Reported next to the fused path so that mode has a number."""
    from pointmvsnet_b200 import _lib
    from pointmvsnet_b200.point_flow import PointFlow
    from pointmvsnet_b200.point_flow_oplevel import point_flow_pass_oplevel
    from pointmvsnet_b200.synthetic import make_pointflow_inputs
    rank, world, local = dist_env()
    if rank != 0:
        return None
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    H, W, V, D = CONFIGS[args.config]
    inp = make_pointflow_inputs(H, W, V, 1, D, seed=0, device=dev)
    pf = PointFlow().to(dev)
    pf.load_reference_state_dict(load_pretrained_hot_path_weights())
    pf.train()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        return point_flow_pass_oplevel(pf.flow_edge_conv, pf.flow_mlp, inp["coarse_depth"], inp["depth_interval"],
                                       inp["pyramids"], inp["cam_params_list"], inp["mean"], inp["std"], inp["img_hw"])

    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize(dev)
    n0 = _lib.launch_count()
    total = 0.0
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(args.steps):
        flush.zero_()
        t0.record()
        outs = step()
        t1.record()
        torch.cuda.synchronize(dev)
        total += t0.elapsed_time(t1)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, pass_outputs(outs))
    ms = total / args.steps
    return json.dumps({
        "metric": METRIC, "value": round(len(IMG_SCALES) / (ms / 1e3), 2), "unit": "iters/s", "n_gpus": 1,
        "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(args.config, H, W, V, D), "mode": "oplevel",
                   "step": "one reference view: the reference closure's control flow (21 cal_sub_flow calls) over the "
                           "stand-alone operators, eager launches, device-resident inputs"},
        "gpu_launches": int(_lib.launch_count() - n0),
    })


class _StdoutToStderr(object):
    """Route fd 1 to fd 2 while libraries (NCCL, CUDA, torchrun children) may chat; restore it
    for the single JSON line."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--views-in-flight", type=int, default=4,
                    help="independent reference views whose passes run concurrently on one GPU (default 4: measured "
                         "1 -> 2 -> 4 views = 1.00 / 1.11 / 1.17x the single-view rate at C2)")
    ap.add_argument("--mode", default="fused", choices=["fused", "oplevel"],
                    help="fused: the PointFlow module (default); oplevel: the reference closure over the stand-alone "
                         "operators (what an unchanged model.py runs)")
    ap.add_argument("--parallel", default="views", choices=["views", "subcloud"],
                    help="views: whole reference views per GPU (throughput, default); subcloud: all GPUs refine ONE "
                         "view, iterations 2/3 split by sub-cloud (BASELINE C5, latency)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32, at "
                         "most 64 MB in all; a fixed, seeded sample of each array beyond that); the inputs depend "
                         "only on the arguments, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        with _StdoutToStderr():
            if args.mode == "oplevel":
                line = run_oplevel(args)
            else:
                line = run_subcloud(args) if args.parallel == "subcloud" else run_ours(args)
        if line is not None:
            print(line, flush=True)


if __name__ == "__main__":
    main()
