#!/usr/bin/env python
"""bench.py -- 480x640 4-iteration pose refinements/sec (BASELINE.json metric) on N B200s.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
           --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 5 --warmup 1      # restated reference CPU path (oracle)
    python bench.py --steps 20 --warmup 3 --dump-outputs DIR   # also write the last timed step's results as DIR/*.npy

One "step" = STEP_BATCHES (32) passes of the fused hot path (dim_refine: 4 x render -> bbox+zoom -> FlowNetS ->
se3 compose), each over one batch of 16 synthetic instances = 512 refinements; workload = BASELINE.json configs[1]
(C2: ~5k-vert mesh, 4 iters, batch 16 per GPU, random-init FlowNetS).  32 batches per step make the default
20-step timed region ~1.5-2 s long, so the clocks settle under the power cap, the clock sampler sees >= 15 samples and
the SUSTAINED tensor peak of MEASURED_PEAKS.json is the right roofline denominator.  Instances are independent:
N GPUs = N replicas of the per-GPU work, no data-path collective ("scaling": "weak").
The headline precision is DIM_PREC_FP16 (one fp16 tcgen05 pass; the mode whose -m gpu tests assert the north-star
1e-4 rot / 1e-3 trans tolerance at batch 16); the bf16 fast mode is reported as the labelled secondary `fast_mode`.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "mx-deepim_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "480x640 4-iter pose refinements/sec"
UNIT = "refinements/s"
N_ITER = 4
STEP_BATCHES = 32  # device batches per bench step
WORKLOAD = "C2: synthetic 5k-vert mesh (5151 verts / 10000 tris), 4 iters, batch=16 per GPU, FlowNetS random-init"


def conv_flops_per_instance_iter():
    from deepim_b200 import synth
    h, w, tot = 480, 640, 0
    for _, co, ci, k, s, p in synth.CONV_SPECS:
        ho, wo = synth.conv_out_hw(h, w, k, s, p)
        tot += 2 * ho * wo * co * ci * k * k
        h, w = ho, wo
    return tot  # 38.79 GFLOP (SURVEY 8(d): 38.876 incl. fc)


def measured_peaks():
    """MEASURED_PEAKS.json (driver-written): fp16 and bf16 share the tcgen05 kind::f16 rate, so the cuBLAS bf16 figures are the
    denominators.  `burst` for a region shorter than ~1 s (boost clocks), `sustained` for a long one (power-capped clocks)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        burst = d.get("bf16_tflops")
        return {"burst": burst, "sustained": d.get("bf16_tflops_sustained", burst), "hbm": d.get("hbm_gbs"), "src": "measured"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1])); smax = max(smax, float(f[2]))
                for n, v in zip(names, f[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def make_inputs(ctx, synth, mesh, B, n_sets, seed, dev, torch, z_mean=0.8, n_classes=1):
    """n_sets rotating input sets so consecutive steps never reuse L2-resident inputs."""
    K, means = synth.K_LINEMOD, synth.PIXEL_MEANS_RGB
    sets = []
    for s in range(n_sets):
        obs, ini = synth.sample_pose_pairs(B, seed * 100 + s, z_mean=z_mean)
        cls = (torch.arange(B, dtype=torch.int32, device=dev) % n_classes).contiguous()  # round-robin over the classes
        r = ctx.render(cls, torch.from_numpy(obs.astype(np.float32)).to(dev), K, want=("bgr", "mask"))
        g = torch.Generator(device=dev); g.manual_seed(seed * 100 + s)
        bg = torch.randint(0, 256, r["bgr"].shape, generator=g, device=dev, dtype=torch.int32).to(torch.uint8)
        m = r["mask"].permute(0, 2, 3, 1) > 0
        u8 = torch.where(m, r["bgr"].to(torch.uint8), bg).contiguous()     # [B,H,W,3] BGR uint8 (cv2.imread layout)
        sets.append({
            "img_dev": ctx.transform_image_u8(u8, means),                     # resident f32 blob for `value`
            "cls_dev": cls, "pose_dev": torch.from_numpy(ini).to(dev),
            "u8_host": u8.cpu().pin_memory(), "cls_host": cls.cpu().pin_memory(),
            "pose_host": torch.from_numpy(ini).pin_memory(), "obs": obs, "ini": ini,
        })
    torch.cuda.synchronize()
    return sets


def run_b200(args):
    import torch
    from deepim_b200 import _capi as capi
    from deepim_b200 import synth
    from deepim_b200.context import Context, launch_count

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    B, K_steps, W_steps, SB = args.batch, args.steps, max(args.warmup, 3), args.step_batches
    prec = capi.precision_id(args.precision)
    K = synth.K_LINEMOD
    means = synth.PIXEL_MEANS_RGB

    from deepim_b200.refiner import PoseRefiner
    workload = WORKLOAD
    if args.config == "c5":  # BASELINE.json configs[4]: rasteriser stress (secondary line; the headline stays C2)
        mesh = synth.make_blob(158, 316, diameter=0.25, tex_size=512, seed=4, name="stress")
        workload = ("C5: synthetic %d-vert / %d-tri mesh, diameter 0.25 m at 0.6 m (large on-screen footprint), 4 iters, batch=%d "
                    "per GPU, FlowNetS random-init" % (len(mesh.verts), len(mesh.faces), B))
    elif args.config == "c3":  # BASELINE.json configs[2]: 13 LINEMOD-scale meshes, instances round-robin over the classes
        meshes = synth.make_linemod_like_set(13)
        mesh = meshes[0]
        workload = ("C3: 13 synthetic LINEMOD-scale meshes (%d-%d verts), instances round-robin over classes, 4 iters, batch=%d per "
                    "GPU, FlowNetS random-init" % (min(len(m.verts) for m in meshes), max(len(m.verts) for m in meshes), B))
    else:
        mesh = synth.make_blob()  # C2
    if args.config != "c3":
        meshes = [mesh]
    workload += "; one bench step = %d device batches of %d = %d refinements" % (SB, B, SB * B)
    weights = synth.make_weights(0)
    refiner = PoseRefiner(meshes, weights, K, device=local_rank, max_batch=B, n_iter=N_ITER, pixel_means_rgb=means,
                          precision=args.precision, n_slots=args.slots)
    ctx = refiner.ctx
    sets = make_inputs(ctx, synth, mesh, B, 3, 1000 + rank, dev, torch, z_mean=0.6 if args.config == "c5" else 0.8,
                       n_classes=len(meshes))
    train_info = None
    if args.train_steps > 0:
        # The timed work does not depend on the weight VALUES; the ADD sanity of the line does.  Random-init weights make the
        # refinement drift, so the network is first trained with this repo's own training step (dim_train_forward_backward +
        # SGD, the reference's hyper-parameters) on the bench's own input pairs -- a recipe, not a checkpoint: seed 0,
        # `--train-steps` batches x 4 inner updates -- and the refiner then runs those weights (UNTIMED set-up).
        t_tr = time.time()
        weights, train_info = train_on_sets(meshes, sets, B, K, means, local_rank, args.train_steps, torch)
        for s_ in refiner.slots:
            s_["ctx"].load_weights(weights)
        train_info["wall_s"] = round(time.time() - t_tr, 1)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    outs = {}  # persistent result tensors per context: same device addresses every call -> the library replays its CUDA graph

    def batch_single(k, p):
        s = sets[k % len(sets)]
        outs[0] = ctx.refine(s["img_dev"], s["cls_dev"], s["pose_dev"], K, N_ITER, pixel_means_rgb=means, precision=p,
                             out=outs.get(0))
        return outs[0]

    def run_host(n_batches):
        """public host API, `slots` batches in flight: the H2D of batch k+1 overlaps the kernels of batch k"""
        pending, last = [], None
        for k in range(n_batches):
            s = sets[k % len(sets)]
            if len(pending) == len(refiner.slots):
                last = refiner.result(pending.pop(0))
            pending.append(refiner.submit(s["u8_host"], s["cls_host"], s["pose_host"]))
        for t in pending:
            last = refiner.result(t)
        return last

    # ---------------- device-resident arm (`value`): inputs already in HBM, `--slots` independent batches in
    # flight on as many streams / contexts (instances are independent, so consecutive batches overlap their tails)
    streams = [s_["stream"] for s_ in refiner.slots]
    ctxs = [s_["ctx"] for s_ in refiner.slots]

    def batch_multi(k, p):
        i = k % len(streams)
        with torch.cuda.stream(streams[i]):
            s = sets[k % len(sets)]
            outs[i] = ctxs[i].refine(s["img_dev"], s["cls_dev"], s["pose_dev"], K, N_ITER, pixel_means_rgb=means, precision=p,
                                     out=outs.get(i))
            return outs[i]

    def device_pass(p, n_steps, with_clocks):
        """n_steps x SB batches round-robin over the streams; CUDA events on torch's current stream bracket the region,
        every slot stream waits for the start event and is joined before the stop event."""
        sampler = None
        if with_clocks:
            sampler = ClockSampler(local_rank)
            sampler.start()
            time.sleep(0.3)
        barrier()
        launch_count(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for st_ in streams:
            st_.wait_event(e0)
        out = None
        for k in range(n_steps * SB):
            out = batch_multi(k, p)
        for st_ in streams:
            torch.cuda.current_stream().wait_stream(st_)
        e1.record()
        barrier()
        t1 = time.time()
        n_launch = launch_count()
        clocks = sampler.stop(t0, t1) if sampler else None
        return e0.elapsed_time(e1), n_launch, clocks, out

    for k in range(3):
        batch_single(k, prec)
    torch.cuda.synchronize()  # a context must only ever be driven from one stream at a time
    device_pass(prec, W_steps, False)                               # W warm-up steps of the timed configuration
    ms_total, launches, clocks, out = device_pass(prec, K_steps, True)
    dumped = None
    if args.dump_outputs:
        # each stream's persistent result tensors hold its latest batch until the next pass reuses them: the last
        # len(streams) batches of the last timed step, in batch order (a fixed sample of the step's SB batches)
        ks = range(max(0, K_steps * SB - len(streams)), K_steps * SB)
        dumped = {name: np.stack([outs[k % len(streams)][name].cpu().numpy() for k in ks]) for name in out}
    poses_last = out["poses"][-1].cpu().numpy()
    idx_last = (K_steps * SB - 1) % len(sets)

    # ---------------- secondary: the bf16 fast mode (fails the 1e-4 rot tolerance -- NOT the headline), same pass shape
    fast = None
    if prec != capi.PREC_BF16 and not args.no_fast_mode:
        kf = max(3, K_steps // 4)
        device_pass(capi.PREC_BF16, 1, False)
        ms_f, _, _, _ = device_pass(capi.PREC_BF16, kf, False)
        fast = (ms_f, kf)

    # ---------------- stage pass: a few steps on ONE stream with CUDA events between the stages (stage times are only
    # meaningful without a second batch interleaved on the SMs); explains the headline, does not produce it
    barrier()
    k_single = max(1, min(K_steps, 2))
    ctx.profile_enable(True)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    for k in range(k_single * SB):
        batch_single(k, prec)
    p1.record()
    barrier()
    ms_single = p0.elapsed_time(p1)
    stages, n_rec = ctx.profile_read()
    ctx.profile_enable(False)

    # ---------------- end-to-end arm (host buffers, H2D + D2H inside the timed region)
    run_host(2 * len(refiner.slots))
    barrier()
    tw0 = time.perf_counter()
    poses_host_last = run_host(K_steps * SB)   # every batch: pinned H2D of its inputs + D2H of its poses, results consumed
    barrier()
    ms_e2e = (time.perf_counter() - tw0) * 1e3
    assert np.isfinite(poses_host_last).all()

    t = torch.tensor([ms_total, ms_e2e, fast[0] if fast else 0.0], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e, ms_fast = float(t[0]), float(t[1]), float(t[2])
    n_ref = world * B * SB * K_steps                                      # refinements in the timed region, all ranks
    value = n_ref / (ms_total / 1e3)
    e2e_value = n_ref / (ms_e2e / 1e3)

    result = None
    if rank == 0:
        peaks = measured_peaks()
        flops_ii = conv_flops_per_instance_iter()
        # roofline of the conv tower IN THE SAME multi-stream pass that produced `value`: every tcgen05 FLOP of the timed
        # region over the whole region (the other kernels of the step run inside it: this is a lower bound of the conv
        # kernels' own rate).  Denominator: sustained bf16/fp16 peak when the region is >= 1 s, else the burst peak.
        long_run = ms_total >= 1000.0
        peak = peaks["sustained"] if long_run else peaks["burst"]
        step_tflops = flops_ii * N_ITER * B * SB * K_steps / (ms_total / 1e3) / 1e12
        conv_single = flops_ii * B * n_rec / (stages["conv"] / 1e3) / 1e12 if stages["conv"] > 0 else 0.0
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            traffic = json.load(open(tpath)).get("conv_igemm_bytes_per_launch")
        # ADD(-S) sanity of the last batch against the observed pose (blob is asymmetric -> ADD)
        s_last = sets[idx_last]
        def add(p, q, b):
            pts = meshes[b % len(meshes)].verts.astype(np.float64)
            return float(np.linalg.norm((pts @ p[:, :3].T + p[:, 3]) - (pts @ q[:, :3].T + q[:, 3]), axis=1).mean())
        add_init = float(np.mean([add(s_last["ini"][b], s_last["obs"][b], b) for b in range(B)]))
        add_final = float(np.mean([add(poses_last[b], s_last["obs"][b], b) for b in range(B)]))
        n_launch_kernels = 10  # conv1 + 9 implicit-GEMM launches per instance-batch iteration
        result = {
            "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": K_steps,
            "warmup": W_steps, "ms_per_step": round(ms_total / K_steps, 4), "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": args.precision,
            "data": "synthetic",
            "config": {"workload": workload, "batch_per_gpu": B, "batches_per_step": SB, "n_iter": N_ITER,
                       "precision": args.precision, "batches_in_flight": args.slots,
                       "parity": "DIM_PREC_FP16: tests/test_gpu_headline_b16.py asserts 1e-4 rot / 1e-3 trans per iteration at batch 16"
                                 if args.precision == "fp16" else "see tests/test_gpu_parity.py for this mode's bounds",
                       "l2": "per-batch working set (~1.6 GB of activations + 90 MB weights + 59 MB inputs) exceeds the "
                             "126 MB L2; 3 rotating input sets"},
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 2), "unit": UNIT,
                    "h2d_bytes_per_step": int(SB * (B * 480 * 640 * 3 + B * 4 + B * 96)),
                    "d2h_bytes_per_step": int(SB * N_ITER * B * (96 + 28)), "ms_per_step": round(ms_e2e / K_steps, 4),
                    "api": "PoseRefiner.submit/result -> dim_refine_host_async (uint8 BGR HWC pinned host images in, float64 poses out; %d batches in flight)" % args.slots, "timer": "host wall clock around K steps, bracketed by barrier + cuda synchronize"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "tensor", "kernel": "conv1_stack_kernel + conv_igemm_pair_kernel (conv2) + conv_igemm_persistent_kernel x8 (10 launches per batch-iteration)",
                         "achieved": round(step_tflops, 2), "peak": peak, "unit": "TFLOP/s",
                         "frac": round(step_tflops / peak, 4), "traffic": traffic,
                         "how": "algorithmic conv FLOPs of the timed region (38.79 GFLOP x %d instances x %d iterations x %d batches x %d steps) / "
                                "the CUDA-event duration of the same multi-stream region that produced `value`" % (B, N_ITER, SB, K_steps),
                         "peak_source": "%s bf16 %s (MEASURED_PEAKS.json; timed region %.2f s)" % (peaks["src"], "sustained" if long_run else "burst", ms_total / 1e3),
                         "frac_of_burst": round(step_tflops / peaks["burst"], 4), "frac_of_sustained": round(step_tflops / peaks["sustained"], 4),
                         "conv_tower_single_stream_tflops": round(conv_single, 2),
                         "launches_per_batch_iteration": n_launch_kernels},
            "stages_ms_per_batch_single_stream": {k: round(v / (k_single * SB), 4) for k, v in stages.items()},
            "single_stream": {"ms_per_batch": round(ms_single / (k_single * SB), 4),
                              "value": round(B * k_single * SB / (ms_single / 1e3), 2),
                              "note": "stage times come from this pass (one batch at a time, CUDA events between stages); "
                                      "`value` and `roofline` come from the pass with %d independent batches on %d streams" % (args.slots, args.slots)},
            "add_m": {"init": round(add_init, 5), "final": round(add_final, 5),
                      "acc_pct_at_0.1d": {"init": round(100.0 * float(np.mean([add(s_last["ini"][b], s_last["obs"][b], b) < 0.1 * meshes[b % len(meshes)].diameter for b in range(B)])), 2),
                                          "final": round(100.0 * float(np.mean([add(poses_last[b], s_last["obs"][b], b) < 0.1 * meshes[b % len(meshes)].diameter for b in range(B)])), 2)},
                      "weights": ("trained in this run by the repo's own training step on the bench's input pairs (untimed set-up): %s" % json.dumps(train_info))
                                 if train_info else "random-init weights: not expected to improve"},
        }
        if fast:
            result["fast_mode"] = {"dtype": "bf16", "value": round(world * B * SB * fast[1] / (ms_fast / 1e3), 2), "unit": UNIT,
                                   "steps": fast[1], "ms_per_step": round(ms_fast / fast[1], 4),
                                   "note": "secondary: single bf16 pass, bounded at 2e-3 rot by its tests (fails the north-star 1e-4); not the headline"}
        if world == 1 and not args.no_cpu_baseline:
            result["cpu_baseline"] = cpu_baseline_leg(sample=2, weights=weights, mesh=mesh)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    refiner.close()
    if result is not None:
        if dumped is not None:
            dump_outputs(args.dump_outputs, dumped)
        print(json.dumps(result), flush=True)


def dump_outputs(d, arrays):
    """DIR/<name>.npy, one leading axis over the dumped batches; the int32 bbox indices are widened (exactly) to float64."""
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def train_on_sets(meshes, sets, B, K, means, device, steps, torch):
    """`steps` data batches (4 inner updates each, deepim/core/module.py:1131-1137) of the training step on the bench's input
    pairs, cycling over the input sets; returns (inference weights, info)."""
    from deepim_b200 import synth, trainer
    from deepim_b200.context import Context
    tctx = Context(device, max_batch=B, max_classes=len(meshes), max_verts=max(len(m.verts) for m in meshes),
                   max_faces=max(len(m.faces) for m in meshes))
    for i, m in enumerate(meshes):
        tctx.upload_mesh(i, m)
    tr = trainer.Trainer(tctx, synth.make_train_weights(0))
    batches = []
    for s in sets:
        batches.append(trainer.make_device_batch(tctx, meshes, B, 0, K, means, poses=(s["obs"], s["ini"]), image_observed=s["img_dev"],
                                                 cls_np=s["cls_host"].numpy()))
    first = last = None
    for step in range(steps):
        batch, cls, tgt, depth_gt = batches[step % len(batches)]
        objs = trainer.fit_batch(tr, batch, cls, tgt, depth_gt, K, n_inner=4)
        if step == 0:
            first = [round(float(v), 4) for v in objs.cpu().numpy()]
    last = [round(float(v), 4) for v in objs.cpu().numpy()]
    w = tr.get_params()
    torch.cuda.synchronize()
    tctx.close()
    return w, {"steps": steps, "inner_updates_per_step": 4, "pairs": len(sets) * B, "lr": tr.lr, "momentum": tr.momentum, "wd": tr.wd,
               "objective_first_batch": first, "objective_last_batch": last,
               "recipe": "synth.make_train_weights(0), trainer.fit_batch on the bench's own input sets (reference hyper-parameters)"}


def cpu_baseline_leg(sample, weights=None, mesh=None, warm=True):
    """Restated reference CPU path (oracle port) on a bounded sample of the same workload."""
    import torch
    from deepim_b200 import synth
    from oracle import oracle as O

    mesh = mesh or synth.make_blob()
    weights = weights or synth.make_weights(0)
    cores = pick_cpu_threads(O, weights)
    K, means = synth.K_LINEMOD, synth.PIXEL_MEANS_RGB
    obs, ini = synth.sample_pose_pairs(sample, 4242)
    imgs = []
    for b in range(sample):
        r = O.render(mesh, obs[b], K)
        imgs.append(synth.transform_image(synth.composite_observed(r["bgr"], r["mask"], b)))
    imgs = np.stack(imgs)
    cls = np.zeros(sample, np.int32)
    if warm:
        O.refine(weights, [mesh], cls[:1], imgs[:1], ini[:1], K, 1, means.astype(np.float32))
    t = time.time()
    for b in range(sample):  # the reference runs one instance at a time (deepim/core/tester.py:83)
        O.refine(weights, [mesh], cls[b:b + 1], imgs[b:b + 1], ini[b:b + 1], K, N_ITER, means.astype(np.float32))
    dt = time.time() - t
    return {"value": round(sample / dt, 4), "unit": UNIT, "cores": cores, "kind": "port", "cpu_model": cpu_model(), "host_cores": os.cpu_count(),
            "stages_ms_per_iteration": cpu_stage_split(O, synth, mesh, weights, imgs[:1], ini[:1], K, means),
            "sample": "%d instances x %d iters of the C2 workload, batch 1 (restated reference CPU path: C rasteriser "
                      "+ C zoom + torch-CPU fp32 FlowNetS + float64 se3)" % (sample, N_ITER)}


def pick_cpu_threads(O, weights):
    """The restated CPU path is timed with the thread count that serves it best: at batch 1 torch's oneDNN convolutions get
    SLOWER beyond a few dozen threads on many-core hosts (measured 3.4 s / forward with 128 threads on the GPU box), and the
    reference arm must not be handicapped.  Best of 3 forwards per candidate (a single shot swung the pick 1.7x run to run)."""
    import torch
    cores = os.cpu_count() or 1
    z3, z1 = np.zeros((1, 3, 480, 640), np.float32), np.zeros((1, 1, 480, 640), np.float32)
    best, best_t = cores, None
    for n in sorted({c for c in (8, 16, 32, 64, cores) if c <= cores}):
        torch.set_num_threads(n)
        O.net_forward(weights, z3, z3, z1, z1)  # warm
        dt = None
        for _ in range(3):
            t = time.time()
            O.net_forward(weights, z3, z3, z1, z1)
            d = time.time() - t
            dt = d if dt is None else min(dt, d)
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_stage_split(O, synth, mesh, weights, img, pose, K, means):
    """One iteration of the restated CPU path, stage by stage (the reference logs data / net / calc_gt,
    deepim/core/tester.py:300-308): render, bbox + zoom, network, SE(3) compose; milliseconds."""
    t0 = time.time()
    r = O.render(mesh, pose[0], K, means_rgb=means)
    t1 = time.time()
    mr = r["mask"][None, None]
    mo = O.box_mask(r["bbox"], 480, 640)[None, None]
    zo, _, zr, zf, _ = O.zoom_mask(mo, mo, mr, pose.astype(np.float32), K)
    zio, zir = O.zoom_image_with_factor(zf, img, r["image"][None], np.asarray(means, np.float32))
    t2 = time.time()
    rot, trans = O.net_forward(weights, zio, zir, zo, zr)
    t3 = time.time()
    O.rt_transform(pose[0], rot[0], O.zoom_trans(zf, trans, True)[0])
    t4 = time.time()
    return {"render": round((t1 - t0) * 1e3, 2), "zoom": round((t2 - t1) * 1e3, 2), "net": round((t3 - t2) * 1e3, 2),
            "compose": round((t4 - t3) * 1e3, 3)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    K_steps, W_steps = args.steps, args.warmup
    import torch
    from deepim_b200 import synth
    from oracle import oracle as O

    mesh, weights = synth.make_blob(), synth.make_weights(0)
    cores = pick_cpu_threads(O, weights)
    K, means = synth.K_LINEMOD, synth.PIXEL_MEANS_RGB.astype(np.float32)
    n = K_steps + W_steps
    obs, ini = synth.sample_pose_pairs(max(n, 1), 4242)
    cls = np.zeros(1, np.int32)

    def step(k, n_it):
        r = O.render(mesh, obs[k], K)
        img = synth.transform_image(synth.composite_observed(r["bgr"], r["mask"], k))[None]
        O.refine(weights, [mesh], cls, img, ini[k:k + 1], K, n_it, means)

    # bounded sample per step: one instance; if K full 4-iteration refinements would not fit ~3 minutes of CPU time the
    # step is cut to 2 or 1 iteration(s) of the same instance and counted as that fraction of a refinement
    step(0, 1)  # page in the libraries / oneDNN primitives (not a timed or counted step)
    t = time.time()
    step(0, 1)
    t_iter = time.time() - t
    n_it = N_ITER
    while n_it > 1 and (K_steps + W_steps) * n_it * t_iter > 180.0:
        n_it //= 2
    for k in range(W_steps):
        step(k, n_it)
    t = time.time()
    for k in range(W_steps, n):
        step(k, n_it)
    dt = time.time() - t
    v = K_steps * (n_it / float(N_ITER)) / dt
    sample = ("each step = 1 instance x %d of the %d iterations of the C2 workload through the restated reference CPU path "
              "(counted as %g refinement)" % (n_it, N_ITER, n_it / float(N_ITER)))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": int(args.gpus),
        "steps": K_steps, "warmup": W_steps, "ms_per_step": round(dt / K_steps * 1e3, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "batch_per_step": 1, "n_iter": N_ITER,
                   "note": "MXNet/glumpy cannot be installed offline (BASELINE.md 2): the reference arm is the oracle port"},
        "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": cores, "kind": "port", "sample": sample, "cpu_model": cpu_model(), "host_cores": os.cpu_count(),
                         "stages_ms_per_iteration": cpu_stage_split(O, synth, mesh, weights, synth.transform_image(
                             synth.composite_observed(O.render(mesh, obs[0], K)["bgr"], O.render(mesh, obs[0], K)["mask"], 0))[None],
                             ini[:1], K, means)},
        "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="instances per GPU")
    ap.add_argument("--precision", default="fp16", choices=["fp16", "bf16x3", "bf16"],
                    help="fp16 = headline (single tcgen05 pass, meets 1e-4 rot / 1e-3 trans); bf16x3 = 3-pass; bf16 = fast mode")
    ap.add_argument("--step-batches", type=int, default=STEP_BATCHES, help="device batches per bench step")
    ap.add_argument("--no-fast-mode", action="store_true", help="skip the secondary bf16 fast-mode pass")
    ap.add_argument("--train-steps", type=int, default=900,
                    help="untimed set-up: train the network for this many batches (x 4 inner updates) on the bench's own input pairs so "
                         "that the ADD sanity of the line means something; 0 = random-init weights")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="label only: weak = per-GPU batch fixed (default); strong = the caller divides a fixed total over the GPUs (C5 sweep)")
    ap.add_argument("--slots", type=int, default=4, help="independent batches in flight per GPU (streams)")
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c5"],
                    help="c2 = headline config (default); c3 = 13 meshes round-robin; c5 = 50k-vert rasteriser stress mesh")
    ap.add_argument("--workload", default="refine", choices=["refine", "train"],
                    help="refine = the headline metric (default); train = config C4 training step (tools/train_bench.py)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write the refine results (poses, se3, zoom_factor, bbox) of the last timed step's "
                         "last --slots batches as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "refine" or args.impl != "b200"):
        ap.error("--dump-outputs applies to the b200 refine workload")
    if args.workload == "train":  # secondary workload: BASELINE.json configs[3]; same launch contract (torchrun for N > 1)
        sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools"))
        import train_bench
        sys.argv = [sys.argv[0], "--batch", str(4 if args.batch == 16 else args.batch), "--steps", str(args.steps or 10),
                    "--warmup", str(args.warmup or 3)]
        return train_bench.main()
    if args.impl == "reference":
        args.steps = 5 if args.steps is None else args.steps
        args.warmup = 1 if args.warmup is None else args.warmup
        run_reference(args)
    else:
        args.steps = 20 if args.steps is None else args.steps
        args.warmup = 3 if args.warmup is None else args.warmup
        run_b200(args)


if __name__ == "__main__":
    main()
