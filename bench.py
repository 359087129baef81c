#!/usr/bin/env python
"""bench.py -- predict_instances throughput of the B200 path (and of the reference CPU path).

  python bench.py --gpus N --steps K --warmup W            # our arm (one rank per GPU under torchrun)
  python bench.py --impl reference --steps K --warmup W     # the reference's CPU path (oracle)

One JSON line.  What it holds (BASELINE.json: "instances/sec (predict_instances end-to-end) 2D 1024^2 r=32 & 3D 128x512^2 r=96"):

  value / e2e / roofline        configs[1]: StarDist2D.predict_instances on one synthetic 1024x1024 image (default Config2D,
                                n_rays 32, grid (1,1)), K timed steps.  `value` = instances/s with the padded input resident
                                in HBM; `e2e` = host image in -> host labels + polygons out through the public API.
                                N > 1: every rank processes its own copy of the image (weak scaling, no data-path collective).
  value_3d / e2e_3d / roofline_3d   configs[2]: StarDist3D.predict_instances on a 128x512x512 volume, Rays_GoldenSpiral(96),
                                default Config3D; same two timings over the same number of steps.
  big_2d / big_3d               configs[3] / [4]: predict_instances_big on a tiled 8192x8192 image / a 512^3 anisotropic volume,
                                blocks sharded over the N ranks (strong scaling: the image is fixed, value = instances of the
                                whole image / max-over-ranks wall time incl. the device-to-device tile gather and the D2H of
                                the assembled label map on rank 0).
  cpu_baseline                  the reference's CPU path timed on this box's host cores (see --impl reference).

--steps K sets the timed steps of configs[1] and configs[2]; the predict_instances_big runs of configs[3] / [4] are timed
over fixed passes (2 for the image, 1 for the volume, each after one warm-up pass).  --dump-outputs DIR writes what the
last timed step of configs[1] / [2] returned, as float32 / float64 .npy files; of the 3-D label volume only the voxels at
dump_voxels_3d() are written.
"""
import argparse, json, os, sys, time, threading, subprocess
import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPE = (1024, 1024)
N_RAYS = 32
PROB_THRESH = 0.5          # the reference's default thresholds (base.py:241)
NMS_THRESH = 0.4
SHAPE_3D = (128, 512, 512)
N_RAYS_3D = 96
PROB_THRESH_3D = 0.7       # SURVEY 8d (R2): 0.7 / 0.3 for the 3-D workload
NMS_THRESH_3D = 0.3
BIG_2D = dict(shape=(8192, 8192), block_size=2304, min_overlap=128, context=96)
BIG_3D = dict(shape=(512, 512, 512), block_size=304, min_overlap=32, context=32, anisotropy=(2, 1, 1))
REF_SAMPLE_3D = (64, 256, 256)     # CPU arms time one eighth of the 3-D volume per step (bounded sample; instances/s is intensive)
METRIC = "instances/sec (predict_instances end-to-end)"
DUMP_LIMIT = 64 << 20          # bytes written by --dump-outputs at most


def dump_voxels_3d(n):
    """flat indices of the voxels of the 3-D label volume that --dump-outputs writes (labels_3d_sample.npy): a fixed sample"""
    return np.sort(np.random.default_rng(0).choice(n, 1 << 21, replace=False))


W2D = "StarDist2D predict_instances, 1024x1024, n_rays=32, seeded synthetic U-Net weights (configs[1])"
W3D = "StarDist3D predict_instances, 128x512x512, Rays_GoldenSpiral n_rays=96, seeded synthetic U-Net weights (configs[2])"


class ClockSampler(threading.Thread):
    """samples nvidia-smi SM clocks / throttle reasons while the timed region runs"""
    def __init__(self, gpu_index=0, period=0.2):
        super().__init__(daemon=True)
        self.gpu, self.period, self.samples, self._halt = gpu_index, period, [], threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                self.samples.append([v.strip() for v in out.split(",")])
            except Exception:
                pass
            self._halt.wait(self.period)

    def stop(self):
        self._halt.set(); self.join(timeout=5)
        sm = [int(s[0]) for s in self.samples if s and s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples if len(s) >= 6 for i in range(4) if s[2 + i].lower().startswith("active")})
        return {"sm_mhz": int(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def conv_flops(config, shape):
    """algorithmic FLOPs of one forward pass (2*pixels*Cin*Cout*k^d per conv layer, SURVEY 8d)"""
    from stardist_b200.models.weights import unet_layers
    sp = np.array(shape, dtype=np.float64)
    fl = 0.0
    for l in unet_layers(config):
        if l['kind'] in ('conv', 'head'):
            fl += 2.0 * np.prod(sp) * l['cin'] * l['cout'] * np.prod(l['k'])
        elif l['kind'] == 'pool':
            sp = sp / np.array(l['pool'])
        elif l['kind'] == 'up':
            sp = sp * np.array(l['pool'])
    return fl


def nms_algorithmic_bytes(n_px, n_cand, n_kept, n_pairs, n_rays, nd):
    """SURVEY 8d: threshold scan 4 B/px + candidate rows (4R + 4 + 4 nd B) read and written sorted + 1 B keep flag,
    two rows per evaluated pair, label paint 4 B/px written + one row per survivor read"""
    row = 4 * n_rays + 4 + 4 * nd
    return 4.0 * n_px + 2.0 * n_cand * row + n_cand + 2.0 * n_pairs * row + 4.0 * n_px + n_kept * row


# ====================================================================================== reference (CPU) arm
def _ref_worker(args):
    """one process, fixed thread count: times `steps` passes of the reference CPU path on the 2-D image or the 3-D sample"""
    import torch
    t = int(args.threads)
    torch.set_num_threads(t)
    import bench_data
    from oracle import pipeline2d, pipeline3d
    st = {}
    def tic(k, t0): st[k] = st.get(k, 0.0) + time.perf_counter() - t0
    if args.dim == 2:
        from stardist_b200.models.config import Config2D
        cfg = Config2D(n_rays=N_RAYS)
        w = bench_data.bench_weights_2d(cfg)
        img, _ = bench_data.synthetic_image(SHAPE, seed=0)
        def step():
            t0 = time.perf_counter(); prob, dist, pads = pipeline2d.predict(cfg, w, img); tic("unet", t0)
            t0 = time.perf_counter(); pa, da, pts = pipeline2d.candidates(cfg, prob, dist, pads, img.shape, PROB_THRESH); tic("threshold_gather", t0)
            t0 = time.perf_counter(); labels, res = pipeline2d.instances(cfg, img.shape, pa, da, pts, NMS_THRESH); tic("nms_labels", t0)
            return len(res['prob'])
    else:
        from stardist_b200.rays3d import rays_from_json
        cfg = bench_data.bench_config_3d(N_RAYS_3D)
        w = bench_data.bench_weights_3d(cfg)
        rays = rays_from_json(cfg.rays_json)
        img, _ = bench_data.synthetic_volume(REF_SAMPLE_3D, seed=0)
        def step():
            t0 = time.perf_counter(); prob, dist = pipeline3d.predict(cfg, w, img); tic("unet", t0)
            t0 = time.perf_counter(); pa, da, pts = pipeline3d.candidates(cfg, prob, dist, img.shape, PROB_THRESH_3D); tic("threshold_gather", t0)
            t0 = time.perf_counter(); labels, res = pipeline3d.instances(cfg, rays, img.shape, pa, da, pts, NMS_THRESH_3D); tic("nms_labels", t0)
            return len(res['prob'])
    for _ in range(args.warmup): step()
    st.clear()
    t0 = time.perf_counter(); n = 0
    for _ in range(args.steps): n += step()
    dt = time.perf_counter() - t0
    print(json.dumps({"threads": t, "dim": args.dim, "instances": n, "seconds": dt, "steps": args.steps,
                      "stages_ms": {k: 1000 * v / args.steps for k, v in st.items()}}))


def _run_worker(dim, threads, steps, warmup, timeout=900):
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"): env.pop(k, None)
    env["OMP_NUM_THREADS"] = str(threads); env["MKL_NUM_THREADS"] = str(threads)
    env.setdefault("OMP_WAIT_POLICY", "PASSIVE")     # torch and the reference extension bring two OpenMP runtimes into one process
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference-worker", "--dim", str(dim), "--threads", str(threads),
                        "--steps", str(steps), "--warmup", str(warmup)], capture_output=True, text=True, timeout=timeout, env=env)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if not lines:
        raise RuntimeError("reference worker failed: " + r.stderr[-400:])
    return json.loads(lines[-1])


def reference_numbers(steps, warmup, budget_s=240.0):
    """the reference's CPU implementation of the path on this box's host cores: reference C++/OpenMP NMS + polyhedron_to_label
    (oracle/_ref, compiled unmodified from the reference's sources), numpy glue restated from nms.py / base.py, torch-CPU fp32
    U-Net standing in for TF-CPU (not installable here).  Thread sweep on the full 1024^2 image, best thread count reported
    (the stack does not scale monotonically with cores: two OpenMP runtimes, per-survivor fork/join in the C++ NMS)."""
    cores = os.cpu_count() or 1
    sweep = sorted({t for t in (8, 16, 32, 64, 128, cores) if t <= cores} | {min(cores, 8)})
    t_start = time.perf_counter()
    tried = {}
    for t in sweep:
        if tried and time.perf_counter() - t_start > 0.35 * budget_s:
            break
        try:
            r = _run_worker(2, t, 1, 1)
            tried[t] = r["instances"] / r["seconds"]
        except Exception as e:
            tried[t] = 0.0
    best_t = max(tried, key=tried.get)
    r2 = _run_worker(2, best_t, max(1, min(steps, 5)), min(1, warmup))
    out = {"threads_sweep_2d_instances_per_s": {str(k): v for k, v in tried.items()}, "best_threads": best_t, "cores": cores,
           "value_2d": r2["instances"] / r2["seconds"], "ms_per_step_2d": 1000 * r2["seconds"] / r2["steps"], "steps_2d": r2["steps"],
           "stages_ms_2d": r2["stages_ms"]}
    try:
        t3 = best_t
        r3 = _run_worker(3, t3, max(1, min(steps, 2)), 0 if time.perf_counter() - t_start > 0.5 * budget_s else 1)
        out.update({"value_3d": r3["instances"] / r3["seconds"], "ms_per_step_3d": 1000 * r3["seconds"] / r3["steps"], "steps_3d": r3["steps"],
                    "stages_ms_3d": r3["stages_ms"], "threads_3d": t3})
    except Exception as e:
        out["error_3d"] = repr(e)[:300]
    return out


def cpu_baseline_record(ref):
    return {"value": ref["value_2d"], "unit": "instances/s", "cores": ref["best_threads"], "host_cores": ref["cores"], "kind": "reference",
            "sample": "full 1024x1024 image, %d steps at the best of the thread sweep %s; NMS = reference C++/OpenMP (oracle/_ref), U-Net = torch-CPU fp32 "
                      "stand-in for TF-CPU (not installable here), labels = numpy restatement" % (ref["steps_2d"], sorted(int(k) for k in ref["threads_sweep_2d_instances_per_s"])),
            "threads_sweep_instances_per_s": ref["threads_sweep_2d_instances_per_s"], "stages_ms": ref["stages_ms_2d"], "ms_per_step": ref["ms_per_step_2d"],
            "value_3d": ref.get("value_3d"), "stages_ms_3d": ref.get("stages_ms_3d"), "ms_per_step_3d": ref.get("ms_per_step_3d"),
            "sample_3d": "one %dx%dx%d sub-volume (1/8 of 128x512x512; instances/s is intensive in the volume) per step, %s steps, %s threads; "
                         "NMS + polyhedron_to_label = reference C++/OpenMP" % (REF_SAMPLE_3D + (ref.get("steps_3d"), ref.get("threads_3d")))}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    ref = reference_numbers(args.steps, args.warmup)
    v = ref["value_2d"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "instances/s",
        "n_gpus": 0, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ref["ms_per_step_2d"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": W2D, "workload_3d": W3D, "prob_thresh": PROB_THRESH, "weights": "seeded Glorot body + fitted heads (bench_data.py)",
                   "nms_thresh": NMS_THRESH, "prob_thresh_3d": PROB_THRESH_3D, "nms_thresh_3d": NMS_THRESH_3D,
                   "timed_steps": "2-D: %d steps of the full image at the best thread count; 3-D: %s steps of a 1/8 sub-volume" % (ref["steps_2d"], ref.get("steps_3d"))},
        "value_3d": ref.get("value_3d"),
        "cpu_baseline": cpu_baseline_record(ref),
        "e2e": {"value": v, "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "e2e_3d": {"value": ref.get("value_3d"), "unit": "instances/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ====================================================================================== B200 arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps of the 2-D and the 3-D workload (device and e2e timing each); the big-image runs use fixed passes")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-3d", action="store_true")
    ap.add_argument("--skip-big", action="store_true")
    ap.add_argument("--dim", type=int, default=2)          # reference-worker only
    ap.add_argument("--threads", type=int, default=8)      # reference-worker only
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of the 2-D and the 3-D workload returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "reference-worker":
        return _ref_worker(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from stardist_b200 import Config2D, StarDist2D, StarDist3D, _lib
    import bench_data
    warm = max(3, args.warmup)
    if os.environ.get("STARDIST_B200_NMS3D_VARIANT"):
        _lib.load().sdb_nms3d_set_variant(int(os.environ["STARDIST_B200_NMS3D_VARIANT"]))
    if os.environ.get("STARDIST_B200_NMS2D_TAIL"):
        _lib.load().sdb_nms2d_set_tail(int(os.environ["STARDIST_B200_NMS2D_TAIL"]))
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        if world > 1: dist.barrier()
        torch.cuda.synchronize()

    def reduce_max_sum(vals):
        t = torch.tensor(vals, dtype=torch.float64, device="cuda")
        if world == 1: return list(vals), list(vals)
        a = t.clone(); dist.all_reduce(a, op=dist.ReduceOp.MAX); b = t.clone(); dist.all_reduce(b, op=dist.ReduceOp.SUM)
        return a.tolist(), b.tolist()

    STAGES = (("net_begin", "net_end", "unet"), ("net_end", "cand_end", "threshold_sort_gather"),
              ("cand_end", "nms_end", "nms"), ("nms_end", "label_end", "coord_label"))

    def time_device(model, x_dev, shape, pthr, nthr, steps):
        """device-resident timing: CUDA events around predict_instances_device, L2 flushed between steps;
        also returns what the last step computed"""
        n_inst = 0; dev_ms = 0.0; stage = {}; n_cand = 0; last = None
        for _ in range(steps):
            flush.zero_()
            model._events = []
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            labels, res = model.predict_instances_device(x_dev, shape, prob_thresh=pthr, nms_thresh=nthr)
            e1.record(); torch.cuda.synchronize()
            dev_ms += e0.elapsed_time(e1); n_inst += len(res['prob']); n_cand += getattr(model, '_last_n_cand', 0)
            ev = dict(model._events); model._events = None
            for a, b, k in STAGES:
                if a in ev and b in ev: stage[k] = stage.get(k, 0.0) + ev[a].elapsed_time(ev[b])
            last = (labels, res)
        return dev_ms, n_inst, n_cand, stage, last

    def dump(arrays):
        """--dump-outputs: one float32 / float64 .npy per array (integers up to 2^24 are exact in float32)"""
        if not args.dump_outputs or rank != 0:
            return
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in arrays.items():
            a = np.asarray(a)
            a = a.astype(np.float64 if a.dtype in (np.float64, np.int64) else np.float32)
            dumped[0] += a.nbytes
            assert dumped[0] <= DUMP_LIMIT, "--dump-outputs would exceed %d bytes" % DUMP_LIMIT
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    dumped = [0]

    def time_e2e(model, img, pthr, nthr, steps, warmup=2):
        model._stats = {}
        for _ in range(warmup): model.predict_instances(img, prob_thresh=pthr, nms_thresh=nthr)
        model._stats = {}
        barrier(); t0 = time.perf_counter(); n = 0
        for _ in range(steps):
            flush.zero_()
            labels, res = model.predict_instances(img, prob_thresh=pthr, nms_thresh=nthr)
            n += len(res['prob'])
        torch.cuda.synchronize(); s = time.perf_counter() - t0
        (s_max, _), (_, n_sum) = reduce_max_sum([s, float(n)])
        return {"value": n_sum / s_max, "unit": "instances/s", "h2d_bytes_per_step": int(model._stats.get('h2d_bytes', 0) // max(1, steps)),
                "d2h_bytes_per_step": int(model._stats.get('d2h_bytes', 0) // max(1, steps)), "ms_per_step": 1000 * s_max / steps}

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf_burst = peaks.get("bf16_tflops", 1700.0)
    peak_tf_sust = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_bw = peaks.get("hbm_gbs", 6650.0)
    src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        traffic = {}

    # ------------------------------------------------------------------ configs[1]: 2-D 1024^2
    cfg = Config2D(n_rays=N_RAYS)
    model = StarDist2D(cfg, name=None, basedir=None, weights=bench_data.bench_weights_2d(cfg))
    img, _ = bench_data.synthetic_image(SHAPE, seed=0)        # every rank works on an identical copy (weak scaling: fixed work per GPU)
    x_dev = torch.from_numpy(img[None, ..., None]).cuda()
    for _ in range(warm):
        model.predict_instances_device(x_dev, SHAPE, prob_thresh=PROB_THRESH, nms_thresh=NMS_THRESH)
    sampler = ClockSampler(local); sampler.start()
    _lib.launch_count(reset=True)
    _lib.profile_enable(True)
    barrier()
    dev_ms, n_inst, n_cand, stage, (labels, res) = time_device(model, x_dev, SHAPE, PROB_THRESH, NMS_THRESH, args.steps)
    launches = _lib.launch_count()
    prof_conv = _lib.profile_get("conv_tc")
    prof_nms = {k: _lib.profile_get("nms2d_" + k) for k in ("frontier", "pairs", "fast", "clip", "tail")}
    _lib.profile_enable(False)
    barrier()
    dump({"labels_2d": labels, "points_2d": res['points'], "prob_2d": res['prob'], "coord_2d": res['coord']})
    del labels, res
    (dev_ms_max, _, _), (_, n_total, _) = reduce_max_sum([dev_ms, float(n_inst), 0.0])
    value = n_total / (dev_ms_max / 1000.0)
    e2e = time_e2e(model, img, PROB_THRESH, NMS_THRESH, args.steps)
    clocks = None if not args.skip_3d else sampler.stop()      # otherwise sampled through the 3-D timed regions as well (the 2-D ones last ~0.1 s)

    out = None
    if rank == 0:
        fl = conv_flops(cfg, SHAPE)
        unet_ms = stage.get("unet", 0.0) / args.steps
        pairs_per_step = prof_nms["fast"]["units"] / args.steps if prof_nms["fast"]["units"] else 0.0
        conv_ms = prof_conv["ms"]
        ach = prof_conv["units"] / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
        roof = {"name": "conv_tc", "bound": "tensor", "kernel": "k_conv_tc* (tcgen05 3x3 convolutions + fused 1x1 heads, all launches of the forward pass)",
                "achieved": ach, "peak": peak_tf_burst, "unit": "TFLOP/s", "frac": ach / peak_tf_burst, "frac_of_sustained_peak": ach / peak_tf_sust,
                "traffic": None, "ms_per_step": conv_ms / args.steps, "launches_per_step": prof_conv["launches"] / args.steps,
                "algorithmic_flop_per_step": prof_conv["units"] / args.steps, "issued_flop_factor": 3, "unet_forward_ms": unet_ms,
                "unet_algorithmic_tflops": fl / (unet_ms / 1e3) / 1e12 if unet_ms > 0 else None,
                "peak_source": src + " bf16_tflops (burst: a ~1 ms kernel group timed alone)"}
        if "conv_tc" in traffic and roof["launches_per_step"]:
            roof["traffic"] = traffic["conv_tc"]["dram_bytes_per_step"] / roof["launches_per_step"]; roof["traffic_source"] = traffic["conv_tc"]["source"]
        post_ms = sum(stage.get(k, 0.0) for k in ("threshold_sort_gather", "nms", "coord_label")) / args.steps
        nms_bytes = nms_algorithmic_bytes(SHAPE[0] * SHAPE[1], n_cand / args.steps, n_inst / args.steps, pairs_per_step, N_RAYS, 2)
        roof_nms = {"name": "nms_labels_2d", "bound": "hbm", "kernel": "threshold/sort/gather + NMS (k_frontier2, k_pairs, k_fast, k_clip) + coord/label painting",
                    "achieved": nms_bytes / (post_ms / 1e3) / 1e9 if post_ms > 0 else 0.0, "peak": peak_bw, "unit": "GB/s",
                    "algorithmic_bytes_per_step": nms_bytes, "ms_per_step": post_ms, "candidates_per_step": n_cand / args.steps,
                    "pairs_per_step": pairs_per_step, "definition": "SURVEY 8d: 4 B/px scan + 2 x 140 B/candidate + 1 B keep + 2 rows per evaluated pair + 4 B/px paint + 1 row per survivor",
                    "traffic": traffic.get("nms_labels_2d", {}).get("dram_bytes_per_step"), "traffic_source": traffic.get("nms_labels_2d", {}).get("source"),
                    "peak_source": src + " hbm_gbs"}
        roof_nms["frac"] = roof_nms["achieved"] / peak_bw
        out = {
            "metric": METRIC, "value": value, "unit": "instances/s",
            "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": dev_ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": W2D, "prob_thresh": PROB_THRESH, "weights": "seeded Glorot body + fitted heads (bench_data.py)", "nms_thresh": NMS_THRESH,
                       "l2": "flushed (256 MiB write) between steps", "instances_per_image": n_total / (args.steps * world),
                       "candidates_per_image": n_cand / args.steps,
                       "stages_ms": {k: v / args.steps for k, v in stage.items()},
                       "nms_kernels_ms": {k: v["ms"] / args.steps for k, v in prof_nms.items()}},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
            "roofline": roof, "roofline_other": {"nms_labels_2d": roof_nms},
        }
    del x_dev

    # ------------------------------------------------------------------ configs[2]: 3-D 128x512x512
    if not args.skip_3d:
        dump3 = None
        try:
            steps3 = args.steps; warm3 = 2
            cfg3 = bench_data.bench_config_3d(N_RAYS_3D)
            model3 = StarDist3D(cfg3, name=None, basedir=None, weights=bench_data.bench_weights_3d(cfg3))
            vol, _ = bench_data.synthetic_volume(SHAPE_3D, seed=0)
            x3 = torch.from_numpy(vol[None, ..., None]).cuda()
            for _ in range(warm3):
                model3.predict_instances_device(x3, SHAPE_3D, prob_thresh=PROB_THRESH_3D, nms_thresh=NMS_THRESH_3D)
            torch.cuda.reset_peak_memory_stats()
            _lib.profile_enable(True)
            l0 = _lib.launch_count()
            barrier()
            dev_ms3, n_inst3, n_cand3, stage3, (labels3, res3) = time_device(model3, x3, SHAPE_3D, PROB_THRESH_3D, NMS_THRESH_3D, steps3)
            launches3 = _lib.launch_count() - l0
            prof_conv3 = _lib.profile_get("conv_tc")
            prof_n3 = {k: _lib.profile_get("nms3d_" + k) for k in ("pretest", "heavy", "heavy_bound", "hulls", "heavy_s4s3s5", "frontier", "paint")}
            _lib.profile_enable(False)
            if args.dump_outputs:
                dump3 = {"labels_3d_sample": labels3.reshape(-1)[dump_voxels_3d(labels3.size)],
                         "points_3d": res3['points'], "prob_3d": res3['prob'], "dist_3d": res3['dist']}
            del labels3, res3
            barrier()
            (dev3_max, _, _), (_, n3_total, _) = reduce_max_sum([dev_ms3, float(n_inst3), 0.0])
            peak_mem = torch.cuda.max_memory_allocated() / 2 ** 30
            del x3
            e2e3 = time_e2e(model3, vol, PROB_THRESH_3D, NMS_THRESH_3D, steps3, warmup=1)
            if clocks is None:
                clocks = sampler.stop()
                if rank == 0: out["clocks"] = clocks
            if rank == 0:
                fl3 = conv_flops(cfg3, SHAPE_3D)
                unet3 = stage3.get("unet", 0.0) / steps3
                c3ms = prof_conv3["ms"]
                ach3 = prof_conv3["units"] / (c3ms / 1e3) / 1e12 if c3ms > 0 else 0.0
                post3 = sum(stage3.get(k, 0.0) for k in ("threshold_sort_gather", "nms", "coord_label")) / steps3
                b3 = nms_algorithmic_bytes(int(np.prod(SHAPE_3D)), n_cand3 / steps3, n_inst3 / steps3, 0.0, N_RAYS_3D, 3)
                out["value_3d"] = n3_total / (dev3_max / 1000.0)
                out["ms_per_step_3d"] = dev3_max / steps3
                out["e2e_3d"] = e2e3
                out["gpu_launches_3d"] = int(launches3)
                out["config"].update({"workload_3d": W3D, "prob_thresh_3d": PROB_THRESH_3D, "nms_thresh_3d": NMS_THRESH_3D, "steps_3d": steps3, "warmup_3d": warm3,
                                      "instances_per_volume": n3_total / (steps3 * world), "candidates_per_volume": n_cand3 / steps3,
                                      "stages_ms_3d": {k: v / steps3 for k, v in stage3.items()},
                                      "nms3d_kernels_ms": {k: v["ms"] / steps3 for k, v in prof_n3.items() if v["launches"]},
                                      "peak_device_memory_gb_3d": peak_mem})
                out["roofline_3d"] = {"name": "conv_tc", "bound": "tensor", "kernel": "k_conv_tc4 as the 3x3x3 convolution (tcgen05) + 1x1x1 heads",
                                      "achieved": ach3, "peak": peak_tf_sust, "unit": "TFLOP/s", "frac": ach3 / peak_tf_sust, "traffic": None,
                                      "ms_per_step": c3ms / steps3, "launches_per_step": prof_conv3["launches"] / steps3,
                                      "algorithmic_flop_per_step": prof_conv3["units"] / steps3, "issued_flop_factor": 3, "unet_forward_ms": unet3,
                                      "unet_algorithmic_tflops": fl3 / (unet3 / 1e3) / 1e12 if unet3 > 0 else None,
                                      "peak_source": src + " bf16_tflops_sustained (kernels inside a ~0.1 s step)"}
                out["roofline_other"]["nms_labels_3d"] = {
                    "bound": "hbm", "kernel": "threshold/sort/gather + 3-D NMS (k_pretest, k_heavy, k_frontier) + k_paint3d + relabel",
                    "achieved": b3 / (post3 / 1e3) / 1e9 if post3 > 0 else 0.0, "peak": peak_bw, "unit": "GB/s", "frac": (b3 / (post3 / 1e3) / 1e9 / peak_bw) if post3 > 0 else 0.0,
                    "algorithmic_bytes_per_step": b3, "ms_per_step": post3, "traffic": traffic.get("nms_labels_3d", {}).get("dram_bytes_per_step"),
                    "definition": "SURVEY 8d: 4 B/voxel scan + 2 x 400 B/candidate + 1 B keep + 4 B/voxel paint + 1 row per survivor (pair rows not counted: no pair counter in 3-D)"}
            del model3, vol
            torch.cuda.empty_cache()
        except Exception as e:
            if rank == 0: out["error_3d"] = repr(e)[:400]
        if dump3 is not None:
            dump(dump3)
        if clocks is None:
            clocks = sampler.stop()
            if rank == 0: out["clocks"] = clocks

    # ------------------------------------------------------------------ configs[3] / [4]: predict_instances_big sharded over the ranks
    if not args.skip_big:
        def run_big(model_b, img_b, axes, spec, reps):
            kw = dict(axes=axes, block_size=spec["block_size"], min_overlap=spec["min_overlap"], context=spec["context"], show_progress=False)
            res = None
            times = []
            for it in range(reps + 1):                       # first pass = warm-up
                barrier(); t0 = time.perf_counter()
                labels, polys = model_b.predict_instances_big(img_b, **kw)
                torch.cuda.synchronize(); dt = time.perf_counter() - t0
                (dt_max,), _ = reduce_max_sum([dt])
                if it > 0: times.append(dt_max)
                if rank == 0: res = (int(len(polys['prob'])), int(labels.max()), tuple(labels.shape))
                del labels, polys
            return times, res
        try:
            tile, _ = bench_data.synthetic_image(SHAPE, seed=0)
            big_img = bench_data.TiledImage(tile, tuple(s // t for s, t in zip(BIG_2D["shape"], SHAPE)))
            times, res = run_big(model, big_img, 'YX', BIG_2D, 2)
            if rank == 0:
                t = float(np.median(times))
                from stardist_b200.big import BlockND
                nblk = len(BlockND.cover(BIG_2D["shape"], 'YX', BIG_2D["block_size"], BIG_2D["min_overlap"], BIG_2D["context"], (8, 8)))
                out["big_2d"] = {"workload": "StarDist2D predict_instances_big, tiled 8192x8192 (configs[3]), block %d / min_overlap %d / context %d -> %d blocks round-robin over %d rank(s)"
                                 % (BIG_2D["block_size"], BIG_2D["min_overlap"], BIG_2D["context"], nblk, world),
                                 "value": res[0] / t, "unit": "instances/s", "seconds": t, "instances": res[0], "scaling": "strong", "n_gpus": world, "blocks": nblk,
                                 "timed": "wall clock, host tiled image in -> assembled int32 label map + polygons on rank 0's host (max over ranks, median of 2 after 1 warm-up)"}
        except Exception as e:
            if rank == 0: out["big_2d"] = {"error": repr(e)[:400]}
        del model
        torch.cuda.empty_cache()
        if not args.skip_3d:
            try:
                cfg5 = bench_data.bench_config_3d(N_RAYS_3D, anisotropy=BIG_3D["anisotropy"])
                model5 = StarDist3D(cfg5, name=None, basedir=None, weights=bench_data.bench_weights_3d(cfg5))
                cell, _ = bench_data.synthetic_volume(bench_data.CELL_3D, seed=0)
                big_vol = bench_data.TiledImage(cell, tuple(s // t for s, t in zip(BIG_3D["shape"], cell.shape)))
                times, res = run_big(model5, big_vol, 'ZYX', BIG_3D, 1)
                if rank == 0:
                    t = float(np.median(times))
                    from stardist_b200.big import BlockND
                    nblk = len(BlockND.cover(BIG_3D["shape"], 'ZYX', BIG_3D["block_size"], BIG_3D["min_overlap"], BIG_3D["context"], (4, 4, 4)))
                    out["big_3d"] = {"workload": "StarDist3D predict_instances_big, tiled 512x512x512, rays anisotropy (2,1,1) (configs[4]), block %d / min_overlap %d / context %d -> %d blocks round-robin over %d rank(s)"
                                     % (BIG_3D["block_size"], BIG_3D["min_overlap"], BIG_3D["context"], nblk, world),
                                     "value": res[0] / t, "unit": "instances/s", "seconds": t, "instances": res[0], "scaling": "strong", "n_gpus": world, "blocks": nblk,
                                     "timed": "wall clock, host tiled volume in -> assembled label volume + polyhedra on rank 0's host (max over ranks, 1 pass after 1 warm-up)"}
                del model5
            except Exception as e:
                if rank == 0: out["big_3d"] = {"error": repr(e)[:400]}

    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            try:
                out["cpu_baseline"] = cpu_baseline_record(reference_numbers(2, 1, budget_s=150.0))
            except Exception as e:      # the baseline is a report, never a reason to lose the measurement
                out["cpu_baseline"] = {"error": repr(e)[:300]}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
