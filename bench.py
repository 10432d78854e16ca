#!/usr/bin/env python3
"""Benchmark of the B200-native PIN-SLAM hot path (contract: see the task statement / DESIGN.md §4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload at N=1: BASELINE.json configs[1] -- the fused kNN + SDF-MLP query (K1) over a batch of
200 000 query points, K=8 neighbours, 32-d features, 2x64 decoder, C=33 probe cells, with the
analytic d sdf / d x.  One *step* is one pass of the hot path over that batch.

  value     whole-job throughput, inputs resident in HBM, in ALGORITHMIC GB/s
            (bytes per query from SURVEY.md §8d: 12 + 4C + 16 N_occ + K_v (4F+4) + 28; N_occ and K_v
            are measured on the workload) -- per-step CUDA-event time on the launching stream, L2
            flushed between steps; max over ranks
  e2e       the same metric through the reference-facing call (NeuralPoints.query_sdf on HOST,
            pinned, query points; results copied back to the host) with the copies inside the timed
            region
  roofline  achieved algorithmic GB/s of the K1 kernel / measured HBM copy peak (MEASURED_PEAKS.json)
  cpu_baseline / --impl reference
            the UNMODIFIED reference classes (oracle/_ref, vendored by oracle/make_ref.py) on the host
            cores, in a process that never loads this repo's CUDA library
  roofline_variants / mapper_dp / per_frame
            K1 on maps >> L2 and in decode-every-neighbour mode; BASELINE configs[4] data-parallel
            training (NCCL all-reduce inside the timed region, every N); configs[2] per-frame loop
            next to the reference's own Tracker/Mapper in PyTorch-CUDA mode
N>1: the query path has no exchange step -- every rank runs the same per-GPU batch on its own map
replica (weak scaling); no collective on the data path.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_QUERY = 200_000
FALLBACK_HBM_GBS = 6650.0


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
    p = os.path.join(ROOT, "profiles", "k1_traffic.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["dram_bytes_per_launch"])
        except Exception:
            return None
    return None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


MAP_SCALE = 1.0  # --map-scale: the synthetic map grows by scale^2 at constant point density (SURVEY.md 8d: M = 250 k / 1 M runs)


def build_workload(device):
    import torch

    from pin_slam_b200.config import HotPathConfig
    from pin_slam_b200.model import Decoder
    from pin_slam_b200.synthetic import build_map, surface_queries

    cfg = HotPathConfig.cfg2(device=str(device), feature_std=0.1, local_map_radius=1e4)
    npm = build_map(cfg, n_surface=int(3_000_000 * MAP_SCALE**2), seed=0, extent=80.0 * MAP_SCALE)
    torch.manual_seed(42)
    dec = Decoder(cfg, cfg.geo_mlp_hidden_dim, cfg.geo_mlp_level, 1)
    q = surface_queries(npm, N_QUERY, seed=1, sigma=0.1)
    return cfg, npm, dec, q


def workload_stats(npm, q, k):
    """Measured N_occ (occupied probes / query) and K_v (selected valid neighbours / query)."""
    import torch

    from pin_slam_b200 import ops

    _, idx = ops.radius_search(npm.map_handle(False), q[:50000].contiguous())
    n_occ = float((idx >= 0).sum(1).float().mean())
    _, _, _, cnt = ops.knn_search(npm.map_handle(True), q, k)
    k_v = float(torch.clamp(cnt, max=k).float().mean())
    return n_occ, k_v, float((cnt >= k).float().mean())


def bytes_per_query(c, n_occ, k_v, f):
    return 12 + 4 * c + 16 * n_occ + k_v * (4 * f + 4) + 28


def _ref_subprocess(mode, device, extra, timeout=900):
    """Run oracle/ref_arm.py (the unmodified reference classes from oracle/_ref) in a clean process: it never imports
    pin_slam_b200 and never maps libpinb200.so.  Returns the parsed JSON line or {"error": ...}."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_arm.py"), mode, "--device", device] + [str(x) for x in extra]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)
        return {"error": (r.stderr or r.stdout)[-300:]}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)[:300]}


def run_reference(args):
    """--impl reference: the reference's own implementation of the path -- the unmodified `NeuralPoints` / `Decoder` /
    `Tracker.query_source_points` classes vendored into oracle/_ref by oracle/make_ref.py -- on the host CPU, all
    200 000 queries of BASELINE configs[1] per step.  This process imports neither pin_slam_b200 nor libpinb200.so:
    the workload (map, decoder, queries) is built with the reference's classes from the same seeded generators."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import ref_arm

    if not ref_arm.available():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref is missing (oracle/make_ref.py needs the "
                                                              "reference checkout; run build() in the build container)"}))
        return
    a = argparse.Namespace(device="cpu", steps=args.steps, warmup=args.warmup, sample=0, frames=12)
    r = ref_arm.run_query(a)
    bq = bytes_per_query(r["n_probe"], r["occupied_probes_mean"], r["valid_knn_mean"], r["feature_dim"])
    dt = r["s_per_step"]
    val = bq * r["n_query"] / dt / 1e9
    line = {
        "impl": "reference", "metric": "kNN+MLP fused query throughput (algorithmic bytes)", "value": val, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {
            "workload": "BASELINE configs[1]: fused kNN+SDF-MLP query, 200k query pts, K=8, F=32, 2x64 decoder, "
                        "C=33 probes, with d sdf/dx",
            "n_query": r["n_query"], "nn_k": r["nn_k"], "feature_dim": r["feature_dim"], "decoder": r["decoder"],
            "weighted_first": r["weighted_first"], "n_probe": r["n_probe"], "map_points": r["map_points"],
            "local_points": r["local_points"], "buffer_size": r["buffer_size"],
            "occupied_probes_mean": round(r["occupied_probes_mean"], 3), "valid_knn_mean": round(r["valid_knn_mean"], 3),
            "bytes_per_query": round(bq, 1), "l2": "n/a (host CPU)",
            "parallelism": "replicas (no collective on the query path)"},
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": r["threads"], "host_cores": r["host_cores"],
                         "kind": "reference",
                         "threads_tried_s_per_20000_queries": r["threads_tried_s_per_20000_queries"],
                         "sample": f"all {r['n_query']} queries per step through the unmodified reference "
                                   "Tracker.query_source_points (oracle/_ref), torch CPU ops at the fastest thread count "
                                   "of the ones tried"},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "queries_per_s": r["queries_per_s"],
    }
    print(json.dumps(line))


def workload_config(cfg, npm, n_occ, k_v, bq, sample=None):
    return {
        "workload": "BASELINE configs[1]: fused kNN+SDF-MLP query, 200k query pts, K=8, F=32, 2x64 decoder, "
                    "C=33 probes, with d sdf/dx",
        "n_query": N_QUERY if sample is None else sample, "nn_k": cfg.query_nn_k, "feature_dim": cfg.feature_dim,
        "decoder": f"{cfg.geo_mlp_level}x{cfg.geo_mlp_hidden_dim}", "weighted_first": cfg.weighted_first,
        "n_probe": int(npm.neighbor_K), "map_points": int(npm.count()), "local_points": int(npm.local_count()),
        "buffer_size": int(npm.buffer_size), "occupied_probes_mean": round(n_occ, 3), "valid_knn_mean": round(k_v, 3),
        "bytes_per_query": round(bq, 1), "l2": "flushed between timed steps (512 MiB memset)",
        "parallelism": "replicas (no collective on the query path)",
    }


def frame_benchmark(dev, n_frames=12, warm_iters=100):
    """BASELINE configs[2]: per-frame tracker (3 GN iterations) + mapper (5 training iterations) on synthetic
    64x1024 KITTI-shaped scans; frames/s over tracker+mapper only.  Also times the reference's op sequence
    (oracle port, PyTorch eager) on the same GPU and map state for the same two stages."""
    import torch

    from pin_slam_b200 import ops
    from pin_slam_b200.frame_loop import FrameLoop

    loop = FrameLoop(device=dev)
    loop.step(0, timed=False, map_iters=warm_iters)   # frame 0 bootstraps the map (untimed, like the reference's init)
    loop.step(1, timed=False)
    l0 = ops.launch_count()
    info = [loop.step(f) for f in range(2, 2 + n_frames)]
    launches = (ops.launch_count() - l0) / n_frames
    trk = sorted(t for t, _ in loop.times)[len(loop.times) // 2]
    mp = sorted(m for _, m in loop.times)[len(loop.times) // 2]
    prep = sorted(loop.prep_times)[len(loop.prep_times) // 2]
    out = {"workload": "BASELINE configs[2]: tracker GN x3 + mapper x5 per frame, 64x1024 synthetic KITTI scan, "
                       "run_kitti.yaml parameters (F=8, K=6, 1x64, weighted_first=False, bs 16384)",
           "frames": n_frames, "tracker_ms_median": trk, "mapping_ms_median": mp,
           "frames_per_s": 1000.0 / (trk + mp), "prep_ms_median": prep,
           "frames_per_s_with_prep": 1000.0 / (trk + mp + prep), "kernel_launches_per_frame": launches,
           "source_points": info[-1]["n_source"], "scan_points": info[-1]["n_scan"],
           "local_map_points": info[-1]["local_points"], "pool_samples": info[-1]["pool"],
           "final_translation_error_m": info[-1]["trans_err_m"],
           "translation_error_m_per_frame": [round(i["trans_err_m"], 4) for i in info]}
    # the >= 10x denominator of north_star: the reference's OWN Tracker / Mapper in PyTorch-CUDA mode on this GPU, same
    # scans, same preprocessing, 3 registration + 5 training iterations per frame (clean subprocess, oracle/_ref)
    del loop
    torch.cuda.empty_cache()
    ref = _ref_subprocess("frames", "cuda", ["--frames", n_frames])
    out["reference_cuda_baseline"] = ref
    if "frames_per_s" in ref:
        out["speedup_vs_reference_cuda"] = out["frames_per_s"] / ref["frames_per_s"]
        out["speedup_vs_reference_cuda_with_prep"] = out["frames_per_s_with_prep"] / ref["frames_per_s_with_prep"]
    return out


def replica_benchmark(dev, n_frames=8, n_track_iter=10, n_map_iter=20):
    """BASELINE configs[3]: Replica-shaped RGB-D frames (640 x 480 pinhole depth + colour of an analytic room),
    run_replica.yaml parameters: colour decoder head on, K = 6, F = 8, photometric point-to-implicit registration
    (fixed `n_track_iter` GN iterations, no host sync) + `n_map_iter` map-training iterations (SDF + colour branches)
    per frame; and the dense per-pixel query (SDF + colour + both gradients) of a whole frame as a K1 roofline."""
    import torch

    from pin_slam_b200 import ops
    from pin_slam_b200.frame_loop import FrameLoop

    loop = FrameLoop(device=dev, rgbd=True, n_track_iter=n_track_iter, n_map_iter=n_map_iter)
    loop.step(0, timed=False, map_iters=100)
    loop.step(1, timed=False)
    l0 = ops.launch_count()
    info = [loop.step(f) for f in range(2, 2 + n_frames)]
    launches = (ops.launch_count() - l0) / n_frames
    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    trk, mp, prep = med([t for t, _ in loop.times]), med([m for _, m in loop.times]), med(loop.prep_times)
    out = {"workload": "BASELINE configs[3]: Replica-shaped RGB-D, 640x480 depth + colour, run_replica.yaml (voxel 0.05 m, "
                       "K=6, F=8, 1x64 SDF + colour decoders, weighted_first, photometric GN x%d + mapper x%d per frame)"
                       % (n_track_iter, n_map_iter),
           "frames": n_frames, "frame_pixels": int(loop.last_frame_points), "tracker_ms_median": trk,
           "mapping_ms_median": mp, "prep_ms_median": prep, "frames_per_s": 1000.0 / (trk + mp),
           "frames_per_s_with_prep": 1000.0 / (trk + mp + prep), "kernel_launches_per_frame": launches,
           "source_points": info[-1]["n_source"], "scan_points": info[-1]["n_scan"],
           "local_map_points": info[-1]["local_points"], "pool_samples": info[-1]["pool"],
           "translation_error_m_per_frame": [round(i["trans_err_m"], 4) for i in info]}
    # dense per-pixel query of one frame: SDF + colour heads with both gradients
    from pin_slam_b200.synthetic import rgbd_frame, rgbd_pose

    npm, cfg = loop.neural_points, loop.cfg
    gt = rgbd_pose(2 + n_frames)
    pts, _ = rgbd_frame(gt, seed=99, device=dev)
    world = (pts @ gt[:3, :3].float().to(dev).T + gt[:3, 3].float().to(dev)).contiguous()
    n = world.shape[0]
    flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    o = {}
    fn = lambda: npm.query_sdf(world, loop.sdf_mlp, need_grad=True, color_decoder=loop.color_mlp, color_grad=True, out=o)  # noqa: E731
    for _ in range(3):
        fn()
    ms = []
    for _ in range(8):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    t = sorted(ms)[4]
    _, idx = ops.radius_search(npm.map_handle(False), world[:50000].contiguous())
    n_occ = float((idx >= 0).sum(1).float().mean())
    k_v = float(torch.clamp(o["nn_count"], max=cfg.query_nn_k).float().mean())
    # SURVEY 8(d) with the colour head on: two feature rows per neighbour, colour (3) + colour gradient (9) outputs
    bq = 12 + 4 * npm.neighbor_K + 16 * n_occ + k_v * (2 * 4 * cfg.feature_dim + 4) + 28 + 4 * (3 + 9)
    peak, _ = hbm_peak()
    ach = bq * n / (t * 1e-3) / 1e9
    out["dense_query"] = {"pixels": n, "ms": t, "bytes_per_query": round(bq, 1), "occupied_probes_mean": round(n_occ, 2),
                          "valid_knn_mean": round(k_v, 2),
                          "kernels": "pinb::search_kernel + pinb::wsq_decode_kernel<8,true,false> (SDF + d/dq) + "
                                     "pinb::wsq_decode_kernel<8,true,false> (colour head + its Jacobian, all 3 channels in one pass)",
                          "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak}}
    return out


def mapper_benchmark(args, standalone=True):
    """BASELINE configs[4]: mapper-only data-parallel training.  A 2M-sample replay pool sharded over the ranks,
    per-GPU batch 16384 (weak scaling), K1 forward + loss heads + K2 backward + ONE NCCL all-reduce of
    [feature grads | decoder grads | certainty increments] + K3 Adam per iteration.  value = samples/s (all ranks)."""
    import types

    import torch
    import torch.distributed as dist

    from pin_slam_b200 import ops
    from pin_slam_b200.config import HotPathConfig
    from pin_slam_b200.model import Decoder
    from pin_slam_b200.synthetic import build_map, surface_queries
    from pin_slam_b200.utils.mapper import Mapper

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and standalone:
        dist.init_process_group("nccl", device_id=dev)
    cfg = HotPathConfig.kitti(device=str(dev), feature_std=0.05, bs_new_sample=0, local_map_radius=1e4)
    npm = build_map(cfg, n_surface=2_000_000, seed=0, extent=80.0)   # identical replica on every rank (same seed)
    torch.manual_seed(42)
    dec = Decoder(cfg, cfg.geo_mlp_hidden_dim, cfg.geo_mlp_level, 1)
    ds = types.SimpleNamespace(processed_frame=0, lose_track=False, stop_status=False, gt_pose_provided=False,
                               odom_poses=None, pgo_poses=None, gt_poses=None)
    mapper = Mapper(cfg, ds, npm, {"sdf": dec, "semantic": None, "color": None})
    pool_total = 2_000_000
    n = pool_total // world                                        # this rank's shard of the replay pool
    g = torch.Generator().manual_seed(100 + rank)
    coord = surface_queries(npm, n, seed=200 + rank, sigma=0.15)
    mapper.global_coord_pool = coord
    mapper.coord_pool = coord
    mapper.sdf_label_pool = (0.15 * torch.randn(n, generator=g)).to(dev)
    mapper.weight_pool = (torch.rand(n, generator=g) * 0.8 + 0.6).to(dev)
    mapper.time_pool = torch.zeros(n, dtype=torch.int32, device=dev)
    mapper.pool_sample_count = n
    torch.manual_seed(1000 + rank)                                  # per-rank batch draws

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    mapper.mapping(max(args.warmup, 3))
    barrier()
    l0 = ops.launch_count()
    reps = []
    for _ in range(3):  # median of three timed regions (each: args.steps iterations, max over ranks)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        mapper.mapping(args.steps)
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        reps.append(float(t[0]))
    t = torch.tensor([sorted(reps)[1]], dtype=torch.float64)
    ms = float(t[0]) / args.steps
    res = {
        "metric": "mapper training throughput (samples/s, all GPUs)", "value": cfg.bs * world / (ms * 1e-3),
        "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "BASELINE configs[4]: mapper-only, 2M-sample pool sharded over ranks, bs/GPU 16384, "
                               "run_kitti.yaml parameters, NCCL all-reduce of feature+decoder grads per iteration",
                   "local_points": int(npm.local_count()), "pool_per_rank": n,
                   "allreduce_floats": int(mapper.allreduce_floats()) if hasattr(mapper, "allreduce_floats") else
                   int(npm.local_geo_features.numel() + dec.flat_parameters().numel() + npm.local_count()),
                   "parallelism": f"dp{world}"},
        "gpu_launches": (ops.launch_count() - l0) // 3, "ms_per_step_of_3_regions": [round(r / args.steps, 4) for r in reps],
        "collective": "ncclAllReduce enqueued by pinb200_map_iterations on the kernel stream (one host call per "
                      "mapping())" if world > 1 else "none (single GPU)"}
    if standalone:
        if rank == 0:
            print(json.dumps(res))
        if world > 1:
            dist.destroy_process_group()
    return res


def dump_outputs(path, out):
    """The K1 output tensors as <path>/<name>.npy: floating outputs in float32, integer ones (nn_count) in float64
    (exact); scratch buffers (names starting with "_") are not outputs."""
    import numpy as np

    os.makedirs(path, exist_ok=True)
    for name, t in sorted(out.items()):
        if name.startswith("_"):
            continue
        a = t.detach().cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float32 if a.dtype.kind == "f" else np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-frame", action="store_true", help="skip the per-frame tracker+mapper measurement")
    ap.add_argument("--no-variants", action="store_true", help="skip the map >> L2 / decode-every-neighbour K1 variants")
    ap.add_argument("--no-mapper", action="store_true", help="skip the data-parallel map-training measurement")
    ap.add_argument("--map-scale", type=float, default=1.0,
                    help="query workload only: scale the synthetic map (points ~ scale^2, same density); "
                         "1.55 ~ 250 k points, 3.1 ~ 1 M points (map >> L2).  The default (1.0, 106 k points) is the "
                         "configuration every committed number refers to")
    ap.add_argument("--workload", default="query", choices=["query", "mapper"],
                    help="query = BASELINE configs[1] (default, the headline); mapper = configs[4] data-parallel training")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="query workload: write what the last timed step returned (sdf, grad, sdf_std, certainty, "
                         "nn_count of all 200 000 queries, ~6 MB) as DIR/<name>.npy; the inputs are seeded, so runs "
                         "with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "query"):
        ap.error("--dump-outputs writes the outputs of the query workload of --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    global MAP_SCALE
    MAP_SCALE = float(args.map_scale)
    if args.impl == "reference":
        run_reference(args)
        return
    if args.workload == "mapper":
        mapper_benchmark(args)
        return

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback for the hot path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from pin_slam_b200 import ops

    cfg, npm, dec, q = build_workload(dev)
    k = cfg.query_nn_k
    n_occ, k_v, full_k = workload_stats(npm, q, k)
    bq = bytes_per_query(npm.neighbor_K, n_occ, k_v, cfg.feature_dim)
    flush = torch.empty(512 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    out = {}

    def step():
        return npm.query_sdf(q, dec, need_grad=True, out=out)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def time_k1(fn, steps):
        """Per-step CUDA-event times (ms) of `fn` on the launching stream, L2 flushed before every step."""
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in evs:
            flush.zero_()
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for a, b in evs]

    for _ in range(args.warmup):
        step()
    barrier()

    # ---- device-resident throughput: per-step CUDA events on the launching stream, L2 flushed in between
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ops.launch_count()
    barrier()
    step_ms = time_k1(step, args.steps)
    barrier()
    launches = ops.launch_count() - launches0
    total_ms = sum(step_ms)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)

    # ---- end to end through the public call with host buffers
    q_host = q.cpu().pin_memory()
    res_host = {n: torch.empty(s, dtype=d).pin_memory() for n, s, d in
                [("sdf", (N_QUERY,), torch.float32), ("grad", (N_QUERY, 3), torch.float32),
                 ("sdf_std", (N_QUERY,), torch.float32), ("nn_count", (N_QUERY,), torch.int32),
                 ("certainty", (N_QUERY,), torch.float32)]}
    E2E_CHUNKS = 2

    def e2e_step():
        # the public host-facing call: pinned host queries in, pinned host results out; the batch is cut into pieces on
        # two streams so that the PCIe copies overlap the kernels (pin_slam_b200/model/neural_points.py)
        npm.query_sdf_host(q_host, dec, res_host, chunks=E2E_CHUNKS, need_grad=True)

    for _ in range(3):
        e2e_step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)

    t = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = float(t[0]), float(t[1])
    ms_per_step = total_ms / args.steps
    value = bq * N_QUERY * world / (ms_per_step * 1e-3) / 1e9
    e2e_val = bq * N_QUERY * world / (e2e_ms / args.steps * 1e-3) / 1e9
    peak, peak_src = hbm_peak()
    kernel_ms = sorted(step_ms)[len(step_ms) // 2]
    achieved = bq * N_QUERY / (ms_per_step * 1e-3) / 1e9
    split = ops.uses_split(N_QUERY, cfg.weighted_first)
    k1_kernels = ("pinb::search_kernel + pinb::wsq_decode_kernel<%d,true,false>" % cfg.feature_dim) if split else \
        "pinb::query_kernel<%d,%s,false>" % (cfg.feature_dim, "true" if cfg.weighted_first else "false")

    line = None
    if rank == 0:
        line = {
            "metric": "kNN+MLP fused query throughput (algorithmic bytes)", "value": value, "unit": "GB/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(cfg, npm, n_occ, k_v, bq),
            "queries_per_s": N_QUERY * world / (ms_per_step * 1e-3),
            "e2e": {"value": e2e_val, "unit": "GB/s", "h2d_bytes_per_step": 12 * N_QUERY,
                    "d2h_bytes_per_step": 28 * N_QUERY, "ms_per_step": e2e_ms / args.steps,
                    "call": "NeuralPoints.query_sdf_host(pinned host queries) -> pinned host sdf/grad/std/nn_count/certainty, "
                            "%d pieces pipelined over 2 streams" % E2E_CHUNKS},
            "gpu_launches": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(), "peak_source": peak_src, "kernel": k1_kernels,
                         "kernel_ms_median": kernel_ms,
                         "note": "K1 = the two launches of the query pipeline (neighbour search, then the warp-specialised "
                                 "gather + tcgen05 decoder with forward-mode d/dq); achieved = algorithmic bytes/query x "
                                 "queries / mean CUDA-event time of the "
                                 "pipeline; traffic = dram bytes of both launches (ncu, profiles/k1_traffic.json)"},
            "clocks": clocks,
        }
    # ---- the other regimes of SURVEY.md 8(d): maps >> L2, and decode-every-neighbour against the compute roof
    if world == 1 and not args.no_variants:
        variants = []
        from pin_slam_b200.config import HotPathConfig
        from pin_slam_b200.model import Decoder
        from pin_slam_b200.synthetic import build_map, surface_queries

        for scale, wf in ((1.55, True), (3.1, True), (1.0, False)):
            try:
                vcfg = HotPathConfig.cfg2(device=str(dev), feature_std=0.1, local_map_radius=1e4)
                vcfg.weighted_first = wf
                vnpm = npm if scale == 1.0 else build_map(vcfg, n_surface=int(3_000_000 * scale * scale), seed=0,
                                                          extent=80.0 * scale)
                if scale == 1.0:
                    vnpm.config = vcfg
                torch.manual_seed(42)
                vdec = Decoder(vcfg, vcfg.geo_mlp_hidden_dim, vcfg.geo_mlp_level, 1)
                vq = q if scale == 1.0 else surface_queries(vnpm, N_QUERY, seed=1, sigma=0.1)
                vo = {}
                fn = lambda: vnpm.query_sdf(vq, vdec, need_grad=True, out=vo)  # noqa: E731
                for _ in range(3):
                    fn()
                ms = sorted(time_k1(fn, 8))[4]
                vn_occ, vk_v, _ = workload_stats(vnpm, vq, k)
                vbq = bytes_per_query(vnpm.neighbor_K, vn_occ, vk_v, vcfg.feature_dim)
                ach = vbq * N_QUERY / (ms * 1e-3) / 1e9
                v = {"workload": "cfg2 %s, map x%.2f" % ("weighted_first" if wf else "decode-every-neighbour", scale),
                     "map_points": int(vnpm.count()), "weighted_first": wf, "ms_per_step": ms,
                     "bytes_per_query": round(vbq, 1),
                     "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak}}
                if not wf:
                    # dense [N*K, D] x [D, 64] x [64, 64] chain, forward + backward to the input: 2 flops per MAC
                    D, H = vcfg.feature_dim + 3, 64
                    flops = 2.0 * (D * H + H * H + H) * k * 2 * N_QUERY
                    sm_peak = 148 * 128 * 2 * 1.965e9 / 1e12  # fp32 SIMT FMA peak of this part (TFLOP/s)
                    v["compute_roofline"] = {"bound": "fp32 (3xTF32 on tensor cores counts as fp32 work)",
                                             "achieved": flops / (ms * 1e-3) / 1e12, "peak": sm_peak, "unit": "TFLOP/s",
                                             "frac": flops / (ms * 1e-3) / 1e12 / sm_peak}
                variants.append(v)
                if scale != 1.0:
                    del vnpm
                    torch.cuda.empty_cache()
            except Exception as e:  # noqa: BLE001
                variants.append({"workload": "map x%.2f wf=%s" % (scale, wf), "error": repr(e)[:200]})
        npm.config = cfg
        if line is not None:
            line["roofline_variants"] = variants
    # ---- BASELINE configs[4]: data-parallel map training, every N (the collective is inside the timed region)
    if not args.no_mapper:
        del flush
        torch.cuda.empty_cache()
        try:
            md = mapper_benchmark(argparse.Namespace(steps=args.steps, warmup=args.warmup), standalone=False)
            if line is not None:
                line["mapper_dp"] = {"ms_per_iter": md["ms_per_step"], "samples_per_s": md["value"],
                                     "allreduce_bytes": 4 * md["config"]["allreduce_floats"],
                                     "bs_per_gpu": 16384, "n_gpus": world, "gpu_launches": md["gpu_launches"],
                                     "workload": md["config"]["workload"]}
        except Exception as e:  # noqa: BLE001
            if line is not None:
                line["mapper_dp"] = {"error": repr(e)[:300]}
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            # the reference itself (unmodified classes, oracle/_ref), clean subprocesses: CPU on the host cores over a
            # bounded sample, and its own PyTorch-CUDA mode on this GPU over the full batch
            r = _ref_subprocess("query", "cpu", ["--steps", 2, "--warmup", 1, "--sample", 50000])
            if "queries_per_s" in r:
                line["cpu_baseline"] = {"value": bq * r["queries_per_s"] / 1e9, "unit": "GB/s", "cores": r["threads"],
                                        "host_cores": r["host_cores"], "kind": "reference",
                                        "queries_per_s": r["queries_per_s"],
                                        "threads_tried_s_per_20000_queries": r["threads_tried_s_per_20000_queries"],
                                        "sample": "50000 of the 200000 queries per step, 2 steps, unmodified reference "
                                                  "Tracker.query_source_points (oracle/_ref) on CPU tensors at the "
                                                  "fastest thread count tried"}
            else:
                line["cpu_baseline"] = r
            g = _ref_subprocess("query", "cuda", ["--steps", 3, "--warmup", 2])
            if "queries_per_s" in g:
                line["reference_cuda_baseline"] = {
                    "value": bq * g["queries_per_s"] / 1e9, "unit": "GB/s", "ms_per_step": g["s_per_step"] * 1e3,
                    "what": "unmodified reference Tracker.query_source_points (oracle/_ref) in PyTorch-CUDA mode on this "
                            "B200, all 200k queries per step"}
                line["speedup_vs_reference_cuda"] = g["s_per_step"] * 1e3 / ms_per_step
            else:
                line["reference_cuda_baseline"] = g
        if world == 1 and not args.no_frame:
            try:
                line["per_frame"] = frame_benchmark(dev)
            except Exception as e:  # noqa: BLE001
                line["per_frame"] = {"error": repr(e)[:300]}
            try:
                line["per_frame_replica"] = replica_benchmark(dev)
            except Exception as e:  # noqa: BLE001
                import traceback

                line["per_frame_replica"] = {"error": repr(e)[:300], "trace": traceback.format_exc()[-600:]}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
