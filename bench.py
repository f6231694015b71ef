#!/usr/bin/env python
"""bench.py -- headline benchmark of the HumanRF per-ray hot path on B200 (see DESIGN.md "Measurement").

BASELINE.json's metric is "train rays/sec & render Mpix/s at 1/2/4/8 B200".  A step = one pass of the hot path over one
synthetic batch (SURVEY 8d / BASELINE.md section 2): 4096 rays x 512 samples = 2,097,152 candidate samples per GPU,
segment_sizes=(50,) (log2T=18), 8 distinct frames of 15..64:
    --mode train (default, configs[2]): jitter + prune pass (early-stop density over all candidates, keeps the composed
                  features) + MLP-only forward of the survivors + compositing + loss + backward (tensor-core MLP backward,
                  parity-slot table scatter) + gradient exchange (N > 1) + fused Adam                      [rays/s]
    --mode render (configs[1]'s kernel): the fused inference kernel, encode -> MLPs -> compositing in one launch,
                  over all 2,097,152 samples                                                               [rays/s]
    --mode image (configs[1]): full 1028x752 images, sampler -> prune -> fused render, tile-sharded over ranks       [Mpix/s]
    --mode sweep (configs[4]): the novel-view sweep, whole images of a (camera, frame) sequence dealt round-robin to the
                  ranks (actorshq/evaluation/presets.py:58-86), `--steps` images per rank, no collective          [Mpix/s]
`value` is timed with CUDA events per step (inputs resident in HBM, L2 flushed between steps); `e2e` goes through the
public API (FusedTrainer.step / volume_rendering.render) with pinned HOST buffers, H2D and D2H inside the timed region.
The default (train) line at N=1 also carries `render` and `image` (each measured in its own process right after).
`--impl reference` times the CPU oracle port of the same path (the reference's tcnn/nerfacc path is CUDA-only and not
installable here) on the box's host cores.
"""
from __future__ import annotations

import argparse
import csv
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

RAYS, SPR = 4096, 512
SEGMENTS = tuple(int(x) for x in os.environ.get("HRF_BENCH_SEGMENTS", "50").split(","))
ALG_BYTES_FWD = 3084          # SURVEY 8d: 2048 B table gathers + 1024 B vector taps + 12 B stream, per sample
ALG_BYTES_SCATTER = 6144      # SURVEY 8d backward convention: table-gradient RMW 2 x 2048 B + vector-gradient RMW 2 x 1024 B
DUMP_SAMPLE = 1 << 20        # --dump-outputs: larger outputs are written as a fixed seeded sample of this many elements
DUMP_LIMIT = 64 << 20        # bytes, all files together
METRIC = {"render": "render_rays_per_s", "train": "train_rays_per_s", "image": "render_mpix_per_s", "sweep": "render_mpix_per_s"}
UNIT = {"render": "rays/s", "train": "rays/s", "image": "Mpix/s", "sweep": "Mpix/s"}


def dist_info():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def committed_ncu(kernel_substr):
    """Per-launch figures of a kernel from the newest committed `ncu --set full` export under profiles/ that contains it
    (a measurement, not a constant in this file): DRAM bytes, L1TEX / L2 throughput %, issue-slot %."""
    unit_scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for f in sorted((ROOT / "profiles").glob("r2*_ncu_full_*_raw.csv"), key=lambda p: p.name, reverse=True):
        try:
            rows = list(csv.reader(open(f)))
        except OSError:
            continue
        if len(rows) < 3:
            continue
        h, units = rows[0], rows[1]
        for r in rows[2:]:
            d = dict(zip(h, r))
            if kernel_substr not in d.get("Kernel Name", ""):
                continue
            u = dict(zip(h, units))

            def num(k, scale=False):
                try:
                    v = float(d[k].replace(",", ""))
                except (KeyError, ValueError):
                    return None
                return v * unit_scale.get(u.get(k, ""), 1.0) if scale else v

            rd, wr = num("dram__bytes_read.sum", True), num("dram__bytes_write.sum", True)
            return {"traffic": None if rd is None or wr is None else rd + wr, "source": f"profiles/{f.name}",
                    "kernel_name": d["Kernel Name"],
                    "l1tex_pct": num("l1tex__throughput.avg.pct_of_peak_sustained_active"),
                    "l2_pct": num("lts__throughput.avg.pct_of_peak_sustained_elapsed"),
                    "dram_pct": num("gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed"),
                    "issue_slots_pct": num("smsp__issue_active.avg.pct_of_peak_sustained_active"),
                    "tensor_pipe_pct": num("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active"),
                    "ncu_duration_ms": num("gpu__time_duration.sum")}
    return None


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dump_outputs(directory, arrays):
    """Writes each output array as DIR/<name>.npy in float32 (float64 stays float64).  An array of more than DUMP_SAMPLE
    elements is flattened and reduced to the elements at DUMP_SAMPLE flat indices drawn once from a generator seeded with
    0 (sorted), the same in every run, so two builds can be compared element by element."""
    import numpy as np

    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    total = 0
    for name, x in arrays.items():
        x = x.detach()
        if x.numel() > DUMP_SAMPLE:
            idx = torch.randperm(x.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort()[0]
            x = x.reshape(-1)[idx.to(x.device)]
        a = x.cpu().numpy()
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        total += a.nbytes
        if total > DUMP_LIMIT:
            raise SystemExit(f"--dump-outputs: more than {DUMP_LIMIT >> 20} MB of outputs")
        np.save(out / f"{name}.npy", a)


def build_workload(device, seed):
    from humanrf_b200.synthetic import make_model, synthetic_rays

    model, frames = make_model(SEGMENTS, seed=123, device=device)
    batch = synthetic_rays(RAYS, SPR, frames, seed=seed)
    return model, frames, batch


def cpu_oracle_rate(mode, steps=3, warmup=1, budget_s=20.0):
    """Reference arm / cpu_baseline: the CPU oracle port of the same path on a bounded sample of the same workload, one
    single-threaded worker per host core (oracle/cpu_bench.py, run in a fresh process).  The sample is sized from a
    calibration step so that `steps + warmup` steps take about `budget_s` seconds (at least 16 rays per worker: with
    fewer, process-pool overhead dominates and the figure moves 4x between boxes)."""
    cmd = [sys.executable, str(ROOT / "oracle" / "cpu_bench.py"), "--steps", str(steps), "--warmup", str(warmup),
           "--budget-s", str(budget_s), "--samples-per-ray", str(SPR), "--mode", "train" if mode == "train" else "render",
           "--segments", *map(str, SEGMENTS)]
    out = subprocess.run(cmd, capture_output=True, text=True, check=True).stdout.strip().splitlines()[-1]
    r = json.loads(out)
    return r["rays_per_s"], r["cores"], r["sample"], r


def companion_line(mode, steps):
    """`bench.py --mode <mode>` in a fresh process; returns the headline fields of its JSON line (or the failure)."""
    cmd = [sys.executable, str(ROOT / "bench.py"), "--mode", mode, "--steps", str(steps), "--warmup", "3", "--no-cpu-baseline",
           "--no-companions"]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=200)
        full = json.loads([ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")][-1])
        keep = {k: full.get(k) for k in ("metric", "value", "unit", "steps", "warmup", "ms_per_step", "gpu_launches", "clocks")}
        keep["e2e"] = (full.get("e2e") or {}).get("value")
        keep["workload"] = (full.get("config") or {}).get("workload")
        if full.get("roofline"):
            keep["roofline"] = {k: full["roofline"].get(k) for k in ("kernel", "frac", "achieved", "kernel_ms", "traffic")}
        return keep
    except Exception as e:  # noqa: BLE001 -- the headline line must still be printed
        return {"error": f"{type(e).__name__}: {e}"[:300]}


def run_reference(args):
    rank, world, _ = dist_info()
    if rank != 0:
        return
    mode = "render" if args.mode in ("image", "sweep") else args.mode
    value, cores, sample, r = cpu_oracle_rate(mode, steps=args.steps, warmup=args.warmup, budget_s=120.0)
    line = {"impl": "reference", "metric": METRIC[mode], "value": value, "unit": "rays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{RAYS} rays x {SPR} samples, segment_sizes={SEGMENTS}, "
                                   f"{'prune + fwd + bwd + Adam' if mode == 'train' else 'render forward'}; each step = "
                                   f"{r['rays_per_step']} rays of it", "mode": mode, "note":
                       "CPU oracle port of the reference path (tcnn/nerfacc are CUDA-only and not installable offline)"},
            "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_image(args, dev, rank, world):
    """BASELINE configs[1]/[4]: full 1028x752 images through sampler -> prune -> fused render, tile-sharded over the ranks
    (contiguous pixel ranges, no collective), image assembled on the device.  Mpix/s counts every pixel of the
    image, including background pixels the sampler masks out (SURVEY 8d)."""
    import numpy as np
    import torch.distributed as dist

    from humanrf_b200.dataset.occupancy_grid_native import OccupanyGrid
    from humanrf_b200.parallel import TileShardedRenderer
    from humanrf_b200.synthetic import make_model
    from humanrf_b200.synthetic_scene import make_scene

    W, H, G = 1028, 752, 256
    model, frames = make_model(SEGMENTS, seed=123, device=dev)
    sc = make_scene(num_images=1, width=W, height=H, G=G, portrait_every=0)
    og = OccupanyGrid(G, 1)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    cam = dict(frame_numbers=t(sc["frame_numbers"]), camera_numbers=t(sc["camera_numbers"]),
               grid_handles=torch.tensor([og.add_grid(t(sc["grids"][0]))], dtype=torch.int64, device=dev),
               landscape=t(sc["landscape"]), inverse_krs=t(sc["inverse_krs"]), camera_origins=t(sc["camera_origins"]),
               aabb=t(sc["aabb"]), G=G, width=W, height=H)
    r = TileShardedRenderer(model, og, rays_per_batch=262144)
    clocks = ClockSampler(dist_info()[2])
    if args.mode == "sweep":
        return run_sweep(args, dev, rank, world, model, frames, r, clocks, W, H, G)
    for _ in range(max(args.warmup, 3)):
        r.render_image_sharded(cam, rank, world)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    host = torch.empty(((W * H + world - 1) // world + 1, 3)).pin_memory()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        s, e, img = r.render_image_sharded(cam, rank, world)
        host[: e - s].copy_(img, non_blocking=True)        # D2H of this rank's tile (the step's result)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    clk = clocks.stop()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"image_tile": img})
    if rank == 0:
        mpix = W * H * args.steps / float(dt.item()) / 1e6
        frac = float((host[: e - s].abs().sum(1) > 0).float().mean())
        cand = r.last_stats.get("candidate_samples")
        print(json.dumps({"metric": METRIC["image"], "value": mpix, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
                          "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * float(dt.item()) / args.steps,
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
                          "data": "synthetic", "config": {"workload": f"{W}x{H} image, synthetic ellipsoid occupancy G={G}, "
                                                         f"segment_sizes={SEGMENTS}, sampler + prune pass + fused MLP/composite render, "
                                                         "262144 rays/batch, wall clock incl. the sampler's host read per batch",
                                                         "object_pixel_fraction_rank0": frac, "candidate_samples_rank0": cand,
                                                         "l2": "working set (candidate arrays + features) far above the 126 MB L2"},
                          "clocks": clk, "gpu_launches": None,
                          "e2e": {"value": mpix, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": W * H * 12 // world}}))
    if world > 1:
        dist.destroy_process_group()


def run_sweep(args, dev, rank, world, model, frames, renderer, clocks, W, H, G):
    """BASELINE configs[4]: 160 cameras x 50 frames = 8000 whole images, dealt round-robin to the ranks.  A bench run renders
    `--steps` images PER RANK of that sequence (synthetic ring of 160 cameras, 2 distinct occupancy grids, frames 15..64)."""
    import numpy as np
    import torch.distributed as dist

    from humanrf_b200.parallel import deal_round_robin
    from humanrf_b200.synthetic_scene import make_scene

    n_cams, n_frames = 160, min(50, len(frames))
    sc = make_scene(num_images=n_cams, width=W, height=H, G=G, portrait_every=0)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    handles = [renderer.og.add_grid(t(sc["grids"][0]))]
    ikr, org, aabb = t(sc["inverse_krs"]), t(sc["camera_origins"]), t(sc["aabb"])
    sequence = [(c, frames[f]) for f in range(n_frames) for c in range(n_cams)]          # presets.py:58-86 order: frame-major
    mine = deal_round_robin(sequence[: (max(args.warmup, 3) + args.steps) * world], rank, world)

    def cam_of(c, f):
        return dict(frame_numbers=torch.tensor([f], dtype=torch.int32, device=dev),
                    camera_numbers=torch.tensor([c], dtype=torch.int32, device=dev),
                    grid_handles=torch.tensor(handles, dtype=torch.int64, device=dev), landscape=torch.tensor([True], device=dev),
                    inverse_krs=ikr[c:c + 1].contiguous(), camera_origins=org[c:c + 1].contiguous(), aabb=aabb, G=G, width=W, height=H)

    w = max(args.warmup, 3)
    for c, f in mine[:w]:
        renderer.render_range(cam_of(c, f), 0, W * H)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    host = torch.empty((W * H, 3)).pin_memory()
    t0 = time.perf_counter()
    for c, f in mine[w:]:
        img = renderer.render_range(cam_of(c, f), 0, W * H)
        host.copy_(img, non_blocking=True)                 # each finished image leaves the device
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    dt = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
    clk = clocks.stop()
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"image": img})
    if rank == 0:
        images = args.steps * world
        mpix = W * H * images / float(dt.item()) / 1e6
        print(json.dumps({"metric": METRIC["sweep"], "value": mpix, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
                          "warmup": w, "ms_per_step": 1e3 * float(dt.item()) / args.steps, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                          "config": {"workload": f"novel-view sweep: {images} of 160 cameras x {n_frames} frames = {n_cams * n_frames} images "
                                                 f"({W}x{H}), round-robin over {world} rank(s), segment_sizes={SEGMENTS}",
                                     "images_per_rank": args.steps, "full_sweep_estimate_s": n_cams * n_frames / images * float(dt.item())},
                          "clocks": clk, "gpu_launches": None,
                          "e2e": {"value": mpix, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": W * H * 12}}))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="train", choices=["train", "render", "image", "sweep"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-companions", action="store_true",
                    help="do not append the render / full-image numbers to the default train line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference(args)

    rank, world, local = dist_info()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the hot path has no CPU fallback (use --impl reference for the CPU oracle)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist

    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from humanrf_b200 import _lib as L
    from humanrf_b200.volume_rendering import ray_offsets, render, render_fused

    L.lib()
    if args.mode in ("image", "sweep"):
        return run_image(args, dev, rank, world)
    model, frames, b = build_workload(dev, seed=int(os.environ.get("HRF_BENCH_SEED", "123")) + rank)
    trainer = None
    if args.mode == "train":
        from humanrf_b200.dataset.input_batch import InputBatch as _IB
        from humanrf_b200.training import FusedTrainer

        # Stationary training workload: the ground truth is the initial model's own rendering ("teacher"), so the
        # model sits at a fixed point, the pruned sample count does not drift from step to step, and every step
        # still does the full work (prune pass, forward, loss, backward, gradient exchange, Adam with lr = 1e-2).
        with torch.no_grad():
            tb = {k: v.to(dev).contiguous() for k, v in b.items() if k in ("o", "d", "frames", "t", "ri")}
            out = render(_IB(ray_origins=tb["o"], ray_directions=tb["d"], frame_numbers=tb["frames"].view(-1, 1),
                             sample_distances=tb["t"].view(-1, 1), ray_indices=tb["ri"]), model, None, is_training=False)
            w = out.weights_sum.clamp(min=1e-6)
            b["rgba"] = torch.cat((out.color / w, out.weights_sum), dim=1).clamp(0, 1).cpu()
        # lr: Adam moves every touched parameter by ~lr per step whatever the size of its gradient; with the reference's 1e-2
        # the random synthetic tables (std 0.05) are rewritten within tens of steps, the densities rise and the number of
        # surviving samples -- the work per step -- drifts down during the run (round 1 measured its e2e on such a drifted
        # model).  1e-6 keeps the model at its initial statistics; the optimiser does exactly the same work for any lr.
        trainer = FusedTrainer(model, lr=float(os.environ.get("HRF_BENCH_LR", "1e-6")), world_size=world,
                               reuse=os.environ.get("HRF_TRAIN_REUSE", "feat+grid"),
                               exchange=os.environ.get("HRF_TRAIN_EXCHANGE", "p2p"),
                               overlap_exchange=os.environ.get("HRF_DP_OVERLAP", "0") == "1")
        trainer.profile = True
    g = {k: v.to(dev).contiguous() for k, v in b.items() if k in ("o", "d", "frames", "t", "ri", "rgba")}
    n = g["t"].shape[0]
    bg = torch.rand(RAYS, 3, device=dev, generator=torch.Generator(device=dev).manual_seed(7))
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    off_all = ray_offsets(g["ri"], RAYS)
    launches = {"n": 0}
    rendered = {}

    def step_render(ev=None):
        rendered["color"], rendered["weights_sum"] = render_fused(model, g["o"], g["d"], g["frames"], g["t"], g["ri"], RAYS, bg,
                                                                  ray_offsets_dev=off_all)
        if ev is not None:
            ev.record()
        launches["n"] += 2

    kept, marks_all = [], []

    def step_train(ev=None):
        launches["n"] += trainer.step(g["o"], g["d"], g["frames"], g["t"], g["ri"], g["rgba"], RAYS, kernel_event=ev)
        kept.append(trainer.last["samples"])
        marks_all.append(trainer.last["marks"])

    step = step_render if args.mode == "render" else step_train

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local)   # samples every 20 ms from the warm-up to the end of the e2e loop: the GPU is under load throughout
    for _ in range(max(args.warmup, 3)):
        flush.zero_()
        step()
    barrier()
    launches["n"] = 0
    kept.clear(), marks_all.clear()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    t_wall = time.perf_counter()
    for i in range(args.steps):
        flush.zero_()
        ev[i][0].record()
        step(ev[i][1])
        ev[i][2].record()
    barrier()
    t_wall = time.perf_counter() - t_wall
    step_ms = sum(e[0].elapsed_time(e[2]) for e in ev)
    kern_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / args.steps
    tt = torch.tensor([step_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt.item())
    gpu_launches = launches["n"]
    phases = {}
    if args.mode == "train":
        for marks in marks_all:
            for (_, e0), (name, e1) in zip(marks[:-1], marks[1:]):
                phases[name] = phases.get(name, 0.0) + e0.elapsed_time(e1) / len(marks_all)
        ph = torch.tensor([phases.get(k, 0.0) for k in sorted(phases)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ph, op=dist.ReduceOp.MAX)
        phases = {k: float(v) for k, v in zip(sorted(phases), ph.tolist())}
        trainer.profile = False
        kept_mean = sum(int(k) for k in kept) / max(len(kept), 1)
        kept_ranks = torch.tensor([kept_mean, -kept_mean], device=dev, dtype=torch.float64)
        if world > 1:   # every rank draws its own ray batch: report the spread of the per-rank work
            dist.all_reduce(kept_ranks, op=dist.ReduceOp.MAX)
        kept_max, kept_min = float(kept_ranks[0].item()), -float(kept_ranks[1].item())
    if args.dump_outputs:
        if args.mode == "render":
            outputs = dict(rendered)
        else:
            # what a caller of FusedTrainer.step gets from the last step: the loss, the surviving sample count and the
            # parameters it updated in place (with the p2p exchange, each rank's fp32 tables are current only in its shard)
            if world > 1:
                trainer.gather_master_parameters()
            names = {id(p): name for name, p in model.named_parameters()}
            outputs = {"loss": trainer.last["loss"].reshape(1), "samples_after_prune": trainer.last["samples"].reshape(1).double()}
            outputs.update({names[id(p)]: p for p in model.hot_parameters()})
        if rank == 0:
            dump_outputs(args.dump_outputs, outputs)

    # ---- e2e through the public API with pinned host buffers -------------------------------------
    host = {k: b[k].contiguous().pin_memory() for k in ("o", "d", "frames", "t", "ri", "rgba")}
    # The ray index of a sample travels as int32 (FusedTrainer.step / volume_rendering.render widen it on the device): 8
    # instead of 17 MB per step.  With int64 the 25 MB upload needs 10.8 GB/s to hide behind a 2.35 ms train step (24 GB/s
    # behind a 1.03 ms render step), which not every host of this pool sustains from pinned memory: the train e2e moved
    # 1.54-1.72 M rays/s from box to box (profiles/r2k-r2n).
    host["ri"] = b["ri"].to(torch.int32).contiguous().pin_memory()
    host_color = torch.empty(RAYS, 3).pin_memory()
    h2d = sum(host[k].numel() * host[k].element_size() for k in ("o", "d", "frames", "t", "ri"))
    d2h = host_color.numel() * 4

    from humanrf_b200.dataset.input_batch import InputBatch

    # Render: three steps in flight on three streams (one pinned->device stream sustains ~16 GB/s on this host,
    # scripts/e2e_probe.py), so step i+1's H2D copy and step i-1's D2H read overlap step i's kernels (copy engines beside
    # the SMs) -- how a renderer walks the tiles of an image.  Train: steps are sequentially dependent (Adam), so the next
    # batch's H2D copy is prefetched on a copy stream and the loss of step i is read back (pinned, asynchronously) while
    # step i+1 runs.  Every step's copies are issued, and complete, inside the timed region.
    DEPTH = 3
    streams = [torch.cuda.Stream(dev) for _ in range(DEPTH)]
    host_colors = [host_color] + [torch.empty(RAYS, 3).pin_memory() for _ in range(DEPTH - 1)]
    keys = ("o", "d", "frames", "t", "ri") if args.mode == "render" else ("o", "d", "frames", "t", "ri", "rgba")

    def upload(stream):
        with torch.cuda.stream(stream):
            bb = {k: host[k].to(dev, non_blocking=True) for k in keys}
            done = torch.cuda.Event()
            done.record(stream)
        return bb, done

    def e2e_render(k):
        for i in range(k):
            st = streams[i % DEPTH]
            bb, _ = upload(st)
            with torch.cuda.stream(st), torch.no_grad():
                ib = InputBatch(ray_origins=bb["o"], ray_directions=bb["d"], frame_numbers=bb["frames"].view(-1, 1),
                                sample_distances=bb["t"].view(-1, 1), ray_indices=bb["ri"])
                out = render(ib, model, bg, is_training=False)
                host_colors[i % DEPTH].copy_(out.color, non_blocking=True)
        torch.cuda.synchronize()

    host_loss = torch.zeros(64).pin_memory()
    e2e_kept = []
    # Train: two resident device batches; batch i+1 is copied from pinned host memory on the copy stream while step i runs
    # (the copy waits until the step that last read that buffer has finished, the step waits for its copy).
    dev_batches = [{k: torch.empty_like(host[k], device=dev) for k in keys} for _ in range(2)]
    # (the copy is split over two streams / copy engines: one pinned->device stream alone sustains 10-16 GB/s on this host,
    #  and 25 MB per step then take longer than the 2.3 ms step they hide behind)
    lanes = (("ri",), tuple(k for k in keys if k != "ri"))
    copied = [[torch.cuda.Event() for _ in lanes] for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def upload_into(slot):
        for j, ks in enumerate(lanes):
            with torch.cuda.stream(streams[j]):
                streams[j].wait_event(consumed[slot])
                for k in ks:
                    dev_batches[slot][k].copy_(host[k], non_blocking=True)
                copied[slot][j].record(streams[j])

    def e2e_train(k):
        cur = torch.cuda.current_stream()
        for c in consumed:
            c.record(cur)
        upload_into(0)
        for i in range(k):
            slot = i & 1
            for e in copied[slot]:
                cur.wait_event(e)
            if i + 1 < k:
                upload_into(slot ^ 1)
            bb = dev_batches[slot]
            trainer.step(bb["o"], bb["d"], bb["frames"], bb["t"], bb["ri"], bb["rgba"], RAYS)
            consumed[slot].record(cur)
            host_loss[i % 64:i % 64 + 1].copy_(trainer.last["loss"].reshape(1), non_blocking=True)   # the D2H read of the step's result
            e2e_kept.append(trainer.last["samples"])
        torch.cuda.synchronize()

    e2e_loop = e2e_render if args.mode == "render" else e2e_train
    e2e_loop(5)
    barrier()
    t0 = time.perf_counter()
    k_e2e = args.steps
    e2e_loop(k_e2e)
    barrier()
    e2e_s = time.perf_counter() - t0
    clk = clocks.stop()
    clk["window"] = "warm-up + timed steps + e2e loop"
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = world * RAYS * k_e2e / float(te.item())
    if args.mode == "train":
        h2d += host["rgba"].numel() * 4
        d2h = 4

    if rank == 0:
        value = world * RAYS * args.steps / (total_ms * 1e-3)
        peak, which = load_peaks()
        if args.mode == "render":
            alg_per_sample, roof_kernel = ALG_BYTES_FWD, "field_forward_kernel<composite epilogue> (+ composite_fixup_kernel)"
            achieved = alg_per_sample * n / (kern_ms * 1e-3) / 1e9
            prof = committed_ncu("field_forward_kernel")
            note = ("SURVEY 8d convention: table gathers served by L2 count as algorithmic bytes; the physical limiter is the "
                    "L1/TEX gather pipe, see l1tex_pct / issue_slots_pct")
        else:
            # dominant kernel of the train step: the table-gradient scatter over the pruned samples
            gen = os.environ.get("HRF_SCATTER", "3")      # the library's default generation (csrc/field_bwd.cu HRF_SCATTER_DEFAULT)
            gen = gen if gen in ("2", "3", "4", "5") else "3"
            alg_per_sample, roof_kernel = ALG_BYTES_SCATTER, f"grid_scatter_v{gen}_kernel"
            kern_ms = phases.get("scatter", 0.0)
            achieved = alg_per_sample * kept_mean / max(kern_ms * 1e-3, 1e-9) / 1e9
            prof = committed_ncu(roof_kernel)
            note = ("SURVEY 8d backward convention: 2 x 2048 B table-gradient RMW + 2 x 1024 B vector-gradient RMW per surviving "
                    "sample; the RMWs are L2 atomics (red.global.add.v2.f32) that run-length and warp-level combining keep off "
                    "DRAM, so the convention's bytes are not physical traffic (see traffic); physical limiters: L1TEX RED "
                    "wavefronts, L2 RED requests, issue slots (l1tex_pct / l2_pct / issue_slots_pct)")
        line = {
            "metric": METRIC[args.mode], "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"{RAYS} rays x {SPR} samples/ray = {n} samples per GPU, segment_sizes={SEGMENTS}, "
                                   f"8 frames, {'fused forward render' if args.mode == 'render' else 'prune + fwd + bwd + exchange + Adam'}",
                       "mode": args.mode, "l2": "flushed between timed steps (256 MiB memset)", "parallelism": f"dp{world}",
                       "samples_per_s": value * SPR},
            "e2e": {"value": e2e_val, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": k_e2e,
                    "api": "humanrf_b200.volume_rendering.render" if args.mode == "render" else "humanrf_b200.training.FusedTrainer.step",
                    "pipelining": "3 steps in flight on 3 streams" if args.mode == "render"
                    else "next batch's H2D prefetched on two copy streams, loss read back asynchronously"},
            "gpu_launches": gpu_launches,
            "clocks": clk,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": prof["traffic"] if prof else None, "traffic_unit": "bytes/launch",
                         "traffic_source": prof["source"] if prof else None,
                         "peak_source": which, "kernel": roof_kernel, "kernel_ms": kern_ms,
                         "algorithmic_bytes_per_sample": alg_per_sample, "note": note,
                         **({k: prof[k] for k in ("l1tex_pct", "l2_pct", "dram_pct", "issue_slots_pct", "tensor_pipe_pct")} if prof else {})},
            "wall_s_timed_loop": t_wall,
        }
        if args.mode == "train":
            line["e2e"]["samples_after_prune_mean"] = sum(int(k) for k in e2e_kept[-k_e2e:]) / k_e2e
            line["config"].update({"samples_after_prune_mean": kept_mean, "samples_after_prune_rank_min_max": [kept_min, kept_max],
                                   "reuse": trainer.reuse, "exchange": trainer.exchange,
                                   "lr": trainer.lr,
                                   "note": "prune pass over all 2,097,152 candidates, fwd+bwd+Adam over the survivors; targets are the "
                                           "initial model's own rendering so the workload is stationary"})
            line["phases_ms"] = phases          # CUDA events inside FusedTrainer.step, mean over the timed steps, max over ranks
            if world > 1:
                line["allreduce_ms"] = phases.get("exchange+adam")
                line["exchange"] = {"kind": trainer.exchange, "overlapped_with_scatter": trainer.overlap_exchange,
                                    "exposed_ms": phases.get("exchange+adam"),
                                    "note": "fused reduce-scatter/Adam/shadow all-gather kernel over NVLink peer memory between two "
                                            "barriers, one launch per hash grid on a side stream while the next grid is scattered; "
                                            "exposed_ms = what is left after the last scatter launch; replaces the single-GPU Adam "
                                            "(see phases_ms at N=1)"}
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample, _ = cpu_oracle_rate(args.mode, steps=2, warmup=1, budget_s=20.0)
            line["cpu_baseline"] = {"value": v, "unit": "rays/s", "cores": cores, "kind": "port", "sample": sample}
        if world == 1 and args.mode == "train" and not args.no_companions:
            # BASELINE.json's metric is a pair ("train rays/sec & render Mpix/s"): the other two workloads run right after
            # (each in its own process, own timed region, same rules) and are attached so one run reports all three.
            line["render"] = companion_line("render", args.steps)
            line["image"] = companion_line("image", args.steps)
            line["config"]["render_rays_per_s"] = line["render"].get("value")
            line["config"]["render_mpix_per_s"] = line["image"].get("value")
        print(json.dumps(line))
    if trainer is not None:
        trainer.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
