#!/usr/bin/env python
"""bench.py -- point-clouds/sec of the SECOND LiDAR-inference hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b2second|reference] [--config car.fhd]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path (voxelize -> sparse middle -> BEV -> RPN -> decode/NMS) over one batch
of synthetic clouds per GPU.  Frames shard over GPUs (weak scaling: the per-GPU batch is fixed) and every
step ends with the single all-gather of detection records (N > 1).

Prints ONE JSON line (rank 0):
  value     whole-job clouds/s with the clouds already resident in HBM, CUDA-event timed per step, L2
            flushed between steps, max over ranks
  e2e       same metric through the reference-facing call -- net(example), the VoxelNet.forward contract, bound to
            the fused engine by b2second.fastpath.accelerate -- with HOST (pinned) clouds: H2D of the points and D2H of
            the detection records inside the timed region
  roofline  the dominant hand-written kernel, timed live with CUDA events (eager replay of the same pipeline):
            k_conv3x3_tc2 (tcgen05 3x3 RPN layers; bound "tensor": algorithmic fp32 flops per launch / average
            launch time against MEASURED_PEAKS.json bf16_tflops, with the 3xF16 ceiling spelled out; `traffic`
            from the committed ncu capture), and as `second_kernel` the sparse middle layers (bound "hbm":
            SURVEY.md §8d bytes / time against hbm_gbs)
  configs   short runs of the other BASELINE.json configurations (car.lite, pointpillars xyres_16, all.fhd at 32
            frames split over the ranks, NuScenes at ~300 k points per cloud) and the bs=1 latency of the headline
            config, each with its stage split and RPN tensor rate
  cpu_baseline  the same network through the CPU oracle (`port`: C voxelizer/NMS + torch-CPU sparse conv/RPN)
            on a bounded sample of the same workload, host cores of this box
--dump-outputs DIR: after the timed steps, the detections of the last timed step of each timed path (resident:
  engine.infer, e2e: net(example)) go to DIR as float32 .npy files, so that two builds can be compared output for
  output (same arguments -> same seeded clouds and weights).
--impl reference: the reference arm = the reference's CPU implementation of the path.  spconv 1.x is not
  in the reference tree and cannot be installed (no network), so this is the oracle port timed with all host
  threads (DESIGN.md "reference arm").
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(REPO, "second.pytorch_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "point-clouds/sec (KITTI car.fhd synthetic, ~17k voxels)"
UNIT = "clouds/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b2second", choices=["b2second", "reference"])
    ap.add_argument("--config", default="car.fhd")
    ap.add_argument("--batch", type=int, default=32,
                    help="frames per GPU per step (serving batch; measured clouds/s at 8/16/32/64: 1950/2320/2460/2516)")
    ap.add_argument("--points", type=int, default=29000, help="points per synthetic cloud (29k -> ~17k voxels)")
    ap.add_argument("--cpu-frames", type=int, default=24,
                    help="frames in the bounded CPU-baseline sample (~0.4 s each on 16 host threads -> ~10 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--sparse", default="tc", choices=["tc", "fma"],
                    help="sparse-conv inner product: tc = tcgen05 3xF16 split, fma = fp32 FMA tiles")
    ap.add_argument("--rpn", default="auto", choices=["auto", "tc", "cudnn"],
                    help="RPN implementation: tc = hand-written tcgen05 3xF16 implicit GEMM, cudnn = torch fp32")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the detections of the last timed step of each timed path to DIR/<path>_<field>.npy")
    return ap.parse_args()


def make_clouds(name, count, points, seed0=0):
    from b2second import config, synth
    cfg = config.get_config(name)
    out = []
    for s in range(count):
        if "nuscenes" in name:
            out.append(synth.nuscenes_cloud(seed0 + s, points))
        else:
            out.append(synth.kitti_cloud(seed0 + s, points, cfg.point_cloud_range))
    return out


def pinned_slab(clouds):
    """the clouds of one batch in ONE pinned host buffer (what a serving loop's ring buffer looks like); returns the
    per-frame views.  The engine recognises frames that lie back to back and moves the batch with one copy."""
    total = sum(c.shape[0] for c in clouds)
    slab = torch.empty(total, clouds[0].shape[1], dtype=torch.float32).pin_memory()
    views, off = [], 0
    for c in clouds:
        n = c.shape[0]
        slab[off:off + n].copy_(torch.from_numpy(c))
        views.append(slab[off:off + n])
        off += n
    return views


def device_slab(host_views, dev):
    """the same batch resident in HBM, again as views of one buffer"""
    rows = [int(h.shape[0]) for h in host_views]
    slab = torch.cat(list(host_views), 0).to(dev)
    out, off = [], 0
    for n in rows:
        out.append(slab[off:off + n])
        off += n
    return out


def workload_desc(args, n_voxels=None):
    d = {"workload": "%s.config inference, synthetic KITTI-range clouds" % args.config,
         "points_per_cloud": args.points, "frames_per_gpu_per_step": args.batch,
         "parallelism": "frames sharded dp%d, one all-gather of detections" % args.gpus,
         "l2": "flushed between steps (512 MiB write), per-step CUDA events",
         "rpn": args.rpn, "sparse_conv": args.sparse,
         "precision": "fp32-grade (tcgen05 kind::f16 on a 3-term fp16 hi/lo split, fp32 accumulation)"}
    if n_voxels is not None:
        d["active_voxels_per_cloud"] = n_voxels
    return d


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_path_clouds_per_s(name, clouds, threads):
    """the oracle port end to end on `clouds` (list of numpy clouds); returns (clouds/s, stage seconds)."""
    from b2second import config, loader, models
    oracle = loader.oracle_spconv()
    cfg = config.get_config(name)
    torch.set_num_threads(threads)
    net = models.build_network(cfg, oracle).eval()
    models.synthetic_weights_(net, name, seed=0)
    anchors = torch.from_numpy(net.anchors()[None])
    # warm (allocations, MKL thread pools, oracle scratch grid)
    res = net.voxel_generator.generate(clouds[0], cfg.max_voxels)
    t0 = time.perf_counter()
    for pts in clouds:
        res = net.voxel_generator.generate(pts, cfg.max_voxels)
        coords = np.pad(res["coordinates"], ((0, 0), (1, 0)))
        ex = {"anchors": anchors, "voxels": torch.from_numpy(res["voxels"]),
              "num_points": torch.from_numpy(res["num_points_per_voxel"]), "coordinates": torch.from_numpy(coords)}
        with torch.no_grad():
            net(ex)
    dt = time.perf_counter() - t0
    return len(clouds) / dt, dt


CPU_KIND = ("port: mirror model (b2second.models, reference state-dict keys) on the oracle spconv package -- C voxelizer "
            "and NMS (single thread, as upstream) + torch-CPU sparse conv / RPN; the unmodified reference cannot run "
            "here (spconv 1.x absent, /root/reference not on the GPU box)")


def cpu_threads():
    """torch-CPU intra-op threads for the CPU arm.  The sparse middle is thousands of tiny gather/mm/index_add
    calls; on the 128-core GPU host, 128 intra-op threads made the same path ~200x SLOWER than 8-16 threads
    (measured round 1), so the arm uses the thread count that the path can actually exploit."""
    env = os.environ.get("B2S_CPU_THREADS")
    if env:
        return int(env)
    return min(os.cpu_count() or 1, 16)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = cpu_threads()
    clouds = make_clouds(args.config, max(1, args.cpu_frames), args.points)
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_path_clouds_per_s(args.config, clouds[:1], threads)
    vals = []
    t_all = time.perf_counter()
    for _ in range(args.steps):
        v, _ = cpu_path_clouds_per_s(args.config, clouds, threads)
        vals.append(v)
        if time.perf_counter() - t_all > 150:   # keep the whole run within a few minutes
            break
    value = float(np.mean(vals))
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
            "warmup": args.warmup, "ms_per_step": 1e3 * len(clouds) / value, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": workload_desc(args),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                             "kind_detail": CPU_KIND,
                             "sample": "%d clouds per step, %d steps, whole hot path on host cores"
                                       % (len(clouds), len(vals))},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_detections(out_dir, path, dets):
    """one step's per-frame detection dicts (the reference's list of dicts) as float32 arrays: the rows of all frames
    concatenated in frame order, <path>_frame.npy holding each row's frame index."""
    arrays = {f: np.concatenate([np.asarray(d[f], dtype=np.float32) for d in dets])
              for f in ("box3d_lidar", "scores", "label_preds")}
    arrays["frame"] = np.repeat(np.arange(len(dets)), [len(d["scores"]) for d in dets]).astype(np.float32)
    if sum(a.nbytes for a in arrays.values()) > DUMP_LIMIT_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write more than %d bytes" % DUMP_LIMIT_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for f, a in arrays.items():
        np.save(os.path.join(out_dir, "%s_%s.npy" % (path, f)), a)


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active")
                                                         for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ GPU arm
def _peaks():
    try:
        return json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def _timed(fn, steps, warmup, flush, world, dev):
    """W untimed steps, then K steps each bracketed by CUDA events (L2 flushed between steps, outside the pair);
    barrier + synchronize on both sides; max over ranks.  Returns total ms."""
    import torch.distributed as dist
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    evs = []
    for i in range(steps):
        flush.fill_(float(i))          # evict L2 between steps (outside the event pair)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn(warmup + i)
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def _rpn_tensor_rate(eng, stages, peaks):
    """algorithmic fp32 TFLOP/s of the k_conv3x3_tc2 launches of one step (stage "rpn") against the measured bf16 peak."""
    rstats = [s for s in eng.rpn_layer_stats() if s["v2"]]
    rpn_ms = stages.get("rpn", 0.0)
    if not rstats or rpn_ms <= 0:
        return None
    bf16 = float(peaks.get("bf16_tflops", 1687.0))
    n_l = len(rstats)
    flops = sum(s["flops"] for s in rstats) / n_l
    launch_ms = rpn_ms / n_l
    ach = flops / (launch_ms * 1e-3) / 1e12
    executed = sum(s["flops"] * s["tiles_computed_frac"] for s in rstats) / n_l
    return {"launches": n_l, "ms_per_launch": launch_ms, "achieved": ach, "peak": bf16, "frac": ach / bf16,
            "algorithmic_flops_per_launch": flops, "executed_flops_per_launch": executed,
            "executed_tflops": executed / (launch_ms * 1e-3) / 1e12,
            "tiles_computed_frac": [round(s["tiles_computed_frac"], 3) for s in rstats],
            "bytes_moved_per_launch": sum(s["bytes"] for s in rstats) / n_l,
            "algorithmic_bytes_per_launch_fp32": sum(s["bytes_fp32_algorithmic"] for s in rstats) / n_l}


def _group_stages(stages):
    grouped = {}
    for k, v in stages.items():
        g = "sparse_conv" if k.startswith("sparse_conv") else ("rulebook" if k.startswith("rulebook") else k)
        grouped[g] = grouped.get(g, 0.0) + v
    return grouped


def measure_config(name, B, points, steps, warm, dev, world, rank, flush, peaks):
    """short run of one BASELINE configuration through net(example): resident clouds/s, e2e clouds/s, stage split."""
    from b2second import config, fastpath, loader, models
    sp = loader.product_spconv()
    cfg = config.get_config(name)
    net = models.build_network(cfg, sp).eval()
    models.synthetic_weights_(net, name, seed=0)
    net = fastpath.accelerate(net.to(dev), max_points=points + 1000, output="host")
    eng = net.b2s_fastpath.engine(B)
    uniq = make_clouds(name, min(2 * B, 4), points, seed0=1000 * rank + 7)   # a few distinct clouds, tiled over the slots
    clouds = [uniq[i % len(uniq)] for i in range(2 * B)]
    host = [pinned_slab(clouds[s * B:(s + 1) * B]) for s in range(2)]
    devc = [device_slab(hs, dev) for hs in host]
    anchors = torch.from_numpy(net.anchors()[None]).to(dev)
    ms_res = _timed(lambda i: eng.infer(devc[i % 2]), steps, warm, flush, world, dev)
    ms_e2e = _timed(lambda i: net({"points": host[i % 2], "anchors": anchors}), steps, warm, flush, world, dev)
    eng.check_status()
    out = {"config": name, "frames_per_gpu_per_step": B, "points_per_cloud": int(np.mean([c.shape[0] for c in clouds])),
           "steps": steps, "ms_per_step": ms_res / steps, "clouds_per_s": world * B * steps / (ms_res / 1e3),
           "e2e_ms_per_step": ms_e2e / steps, "e2e_clouds_per_s": world * B * steps / (ms_e2e / 1e3)}
    if rank == 0:
        eng.load_points(devc[0])
        stages = eng.run_timed(iters=3)
        out["active_voxels_per_cloud"] = int(eng.num_voxels[0].item()) // B
        out["stage_ms_eager"] = _group_stages(stages)
        out["rpn_3x3_tensor"] = _rpn_tensor_rate(eng, stages, peaks)
        out["gpu_launches_per_step"] = eng.kernel_launches_per_step()
    del eng, net
    torch.cuda.empty_cache()
    return out


def run_gpu_arm(args):
    import torch.distributed as dist
    from b2second import config, dist as b2dist, fastpath, loader, models

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    sp = loader.product_spconv()
    cfg = config.get_config(args.config)
    net = models.build_network(cfg, sp).eval()
    models.synthetic_weights_(net, args.config, seed=0)
    B = args.batch
    # the public call: net(example) (VoxelNet.forward contract), bound to the fused engine
    net = fastpath.accelerate(net.to(dev), max_points=args.points + 1000, output="host", rpn_impl=args.rpn,
                              sparse_impl=args.sparse)
    fast = net.b2s_fastpath
    eng = fast.engine(B)
    args.rpn = eng.rpn_impl
    gather = b2dist.DetectionGatherer(B, eng.post_max, eng.code + 2, dev) if world > 1 else None
    if gather is not None:
        fast.post_run = lambda e: gather.gather_records(e.det_record)     # the one collective of a step
    # distinct clouds per rank and per slot; two alternating batches so consecutive steps differ
    n_sets = 2
    clouds = make_clouds(args.config, n_sets * B, args.points, seed0=1000 * rank)
    host = [pinned_slab(clouds[s * B:(s + 1) * B]) for s in range(n_sets)]
    devc = [device_slab(hs, dev) for hs in host]
    anchors = torch.from_numpy(net.anchors()[None]).to(dev)
    flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    h2d_bytes = sum(int(h.numel()) * 4 for h in host[0])
    d2h_bytes = eng.det_record.numel() * 4 + 4

    def step_resident(i):
        eng.infer(devc[i % n_sets])        # device->device staging of the batch + one graph replay
        if gather is not None:
            gather.gather_records(eng.det_record)

    last = {}

    def step_e2e(i):
        # pinned host clouds in, host tensors out: H2D of the points, the graph, the all-gather (N > 1) and ONE D2H
        # of the detection records all happen inside this call
        last["e2e"] = net({"points": host[i % n_sets], "anchors": anchors})

    warm = max(args.warmup, 3)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if os.environ.get("B2S_PROFILE"):      # `ncu --profile-from-start off`: capture steady-state steps only
        for i in range(warm):
            step_resident(i)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for i in range(int(os.environ["B2S_PROFILE"])):
            step_resident(i)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    ms_res = _timed(step_resident, args.steps, warm, flush, world, dev)
    if args.dump_outputs:      # the detection records the last resident step left on the device, before e2e reuses them
        last["resident"] = eng.detections()
    ms_e2e = _timed(step_e2e, args.steps, warm, flush, world, dev)
    if args.dump_outputs and rank == 0:
        for path in ("resident", "e2e"):
            dump_detections(args.dump_outputs, path, last[path])
    clocks = sampler.stop() if rank == 0 else None
    eng.check_status()
    frames = world * B * args.steps
    value = frames / (ms_res / 1e3)
    e2e = frames / (ms_e2e / 1e3)
    peaks = _peaks()
    # ---- short runs of the other BASELINE configs (every rank takes part: all.fhd is split over the ranks)
    extra = []
    if not args.no_configs and args.config == "car.fhd":
        k = max(3, min(5, args.steps))
        plan = [("car.fhd", 1, args.points),                                  # bs=1 latency of the headline config
                ("car.lite", B, args.points),
                ("pointpillars.car.xyres_16", B, args.points),
                ("all.fhd", max(1, 32 // world), args.points),               # BASELINE config 4: bs=32 over the ranks
                ("nuscenes.all.pp.largea", 4, 300000)]                       # BASELINE config 5: ~300 k points / cloud
        del devc
        for name, b, pts in plan:
            try:
                extra.append(measure_config(name, b, pts, k, 3, dev, world, rank, flush, peaks))
            except Exception as e:      # a side measurement must not take the headline line down
                extra.append({"config": name, "error": "%s: %s" % (type(e).__name__, e)})
        devc = [device_slab(hs, dev) for hs in host]
    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant hand-written kernel, measured live (eager replay, CUDA events per stage)
    eng.load_points(devc[0])
    stages = eng.run_timed(iters=5)
    stats = eng.sparse_layer_stats()
    n_vox = int(eng.num_voxels[0].item()) // B
    conv_ms = sum(v for k, v in stages.items() if k.startswith("sparse_conv"))
    conv_bytes = sum(s["bytes"] for s in stats)
    conv_flops = sum(s["flops"] for s in stats)
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    sparse_roof = {"kernel": "k_sparse_conv%s (all %d sparse layers of one step, %d frames)"
                             % ("_tc" if args.sparse == "tc" else "", len(stats), B),
                   "bound": "hbm", "achieved": conv_bytes / (conv_ms * 1e-3) / 1e9 if conv_ms > 0 else 0.0,
                   "peak": hbm_peak, "unit": "GB/s", "algorithmic_bytes_per_step": conv_bytes,
                   "algorithmic_flops_per_step": conv_flops, "ms_per_step": conv_ms,
                   "achieved_tflops": conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0,
                   "useful_mma_frac_per_layer": [round(s["useful_mma_frac"], 3) for s in stats]}
    sparse_roof["frac"] = sparse_roof["achieved"] / hbm_peak
    rt = _rpn_tensor_rate(eng, stages, peaks)
    if rt is not None and stages.get("rpn", 0.0) >= 0.5 * conv_ms:
        # dominant kernel = k_conv3x3_tc2 (dense RPN 3x3 layers, implicit GEMM on tcgen05, 3xF16 split for fp32-grade
        # results).  `achieved` counts ALGORITHMIC fp32 flops per launch (2*px*9*cin*cout) over the average launch
        # duration; the tensor pipe executes 3 fp16 MMAs per algorithmic MAC, so bf16_peak/3 is this arithmetic's
        # ceiling -- reported alongside.
        traffic = None
        try:   # dram read+write bytes per launch from the committed ncu --set full capture of this kernel
            tj = json.load(open(os.path.join(REPO, "profiles", "r2_traffic.json")))
            traffic = tj["k_conv3x3_tc2"]["dram_bytes_per_launch"] * B / tj["frames_in_capture"]
        except Exception:
            pass
        roofline = {"kernel": "k_conv3x3_tc2 (per launch; %d launches per step, %d frames)" % (rt["launches"], B),
                    "bound": "tensor", "achieved": rt["achieved"], "peak": rt["peak"], "unit": "TFLOP/s",
                    "frac": rt["frac"], "traffic": traffic,
                    "traffic_source": "profiles/r2_traffic.json (ncu --set full)" if traffic else None,
                    "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst)" if peaks else "fallback",
                    "algorithmic_flops_per_launch": rt["algorithmic_flops_per_launch"],
                    "algorithmic_bytes_per_launch": rt["algorithmic_bytes_per_launch_fp32"],
                    "bytes_moved_per_launch": rt["bytes_moved_per_launch"],
                    "ms_per_launch": rt["ms_per_launch"],
                    "executed_flops_per_launch": rt["executed_flops_per_launch"],
                    "tiles_computed_frac_per_layer": rt["tiles_computed_frac"],
                    "issued_f16_tflops": 3 * rt["executed_tflops"],
                    "frac_of_pipe_issued": 3 * rt["executed_tflops"] / rt["peak"],
                    "note": "`achieved` = the layer's full algorithmic fp32 flops (2*B*H*W*9*Cin*Cout) / launch time.  "
                            "fp32-parity arithmetic: each executed MAC = 3 fp16 MMAs (hi*hi, hi*lo, lo*hi) with fp32 "
                            "accumulation, so 1/3 of the bf16/fp16 peak is the ceiling for EXECUTED flops "
                            "(frac_of_pipe_issued); output tiles whose whole receptive field is empty BEV are not "
                            "computed but filled with the layer's data-independent constant (csrc/rpn_bg.cu), which "
                            "is why `frac` can exceed 1/3 -- tiles_computed_frac_per_layer says by how much",
                    "second_kernel": sparse_roof}
    else:
        roofline = dict(sparse_roof, traffic=None, peak_source="measured" if peaks else "fallback")
    cpu_baseline = None
    if not args.no_cpu_baseline:
        threads = cpu_threads()
        sample = clouds[:max(1, args.cpu_frames)]
        v, dt = cpu_path_clouds_per_s(args.config, sample, threads)
        n1 = max(1, min(4, args.cpu_frames // 6))
        v1, dt1 = cpu_path_clouds_per_s(args.config, clouds[:n1], 1)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "kind_detail": CPU_KIND,
                        "sample": "%d clouds of the same workload (%.1f s), whole hot path: C voxelizer + torch-CPU "
                                  "sparse conv/RPN + C NMS" % (len(sample), dt),
                        "one_thread": {"value": v1, "unit": UNIT, "cores": 1,
                                       "sample": "%d clouds (%.1f s)" % (n1, dt1)}}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warm, "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "b2second",
            "config": workload_desc(args, n_vox),
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "ms_per_step": ms_e2e / args.steps,
                    "api": "net(example) = VoxelNet.forward(example) bound by b2second.fastpath.accelerate; example = "
                           "{'points': pinned host clouds, 'anchors'}; returns the reference's list of dicts (host)"},
            "gpu_launches": eng.kernel_launches_per_step() * args.steps,
            "gpu_launches_per_step": eng.kernel_launches_per_step(),
            "clocks": clocks, "roofline": roofline, "stage_ms_eager": _group_stages(stages),
            "cpu_baseline": cpu_baseline, "configs": extra}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the b2second arm has no CPU fallback "
                         "(use --impl reference for the CPU baseline)")
    run_gpu_arm(args)


if __name__ == "__main__":
    main()
