"""Per-kernel device times of the train step's pieces on the bench batch (4096 x 512, segment_sizes from argv), L2
flushed between repetitions, CUDA events on the launching stream.  Prints one line per piece; used to A/B variants.
    python scripts/kernel_times.py [--segments 50] [--reps 10]
"""
import argparse
import ctypes as C
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--segments", type=int, nargs="+", default=[50])
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    from humanrf_b200 import _lib as L
    from humanrf_b200.synthetic import make_model, synthetic_rays
    from humanrf_b200.volume_rendering import ray_offsets

    dev = torch.device("cuda:0")
    lib = L.lib()
    model, frames = make_model(tuple(a.segments), seed=123, device=dev)
    b = synthetic_rays(4096, 512, frames, seed=123)
    g = {k: v.to(dev).contiguous() for k, v in b.items() if k in ("o", "d", "frames", "t", "ri", "rgba")}
    nat = model.native()
    R, n0 = 4096, g["t"].shape[0]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timeit(name, fn, reps=a.reps, note="", cold=True):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(reps):
            if cold:
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        print(f"{name:44s} median {ts[len(ts) // 2]:8.4f} ms  min {ts[0]:8.4f}  {note}", flush=True)
        return ts[len(ts) // 2]

    s_all = nat.samples_rays(g["o"], g["d"], g["frames"], g["t"], g["ri"])
    off0 = ray_offsets(g["ri"], R)
    timeit("forward render (all candidates)", lambda: nat.forward(s_all, 1, False, False), note=f"{n0} samples")
    timeit("forward density-only (all candidates)", lambda: nat.forward(s_all, 0, False, False))
    timeit("forward render + save feat/egrid (all)", lambda: nat.forward(s_all, 1, False, True))
    timeit("prune pass: early-stop density", lambda: nat.density_early_stop(s_all, off0, R, 4e-4))
    timeit("prune pass + save composed features", lambda: nat.density_early_stop(s_all, off0, R, 4e-4, save="feat"))
    timeit("prune pass + save feat + per-grid feats", lambda: nat.density_early_stop(s_all, off0, R, 4e-4, save="feat+grid"))
    timeit("prune pass (L2 warm)", lambda: nat.density_early_stop(s_all, off0, R, 4e-4), cold=False)
    # survivors
    sigma0 = nat.density_early_stop(s_all, off0, R, 4e-4)
    keep = torch.empty(n0, dtype=torch.uint8, device=dev)
    kept_off = torch.empty(R + 1, dtype=torch.int32, device=dev)
    t2, ri2 = torch.empty(n0, device=dev), torch.empty(n0, dtype=torch.int64, device=dev)
    counter = torch.zeros(1, dtype=torch.int64, device=dev)

    def prune():
        L.check(lib.hrf_prune(sigma0.data_ptr(), g["t"].data_ptr(), g["ri"].data_ptr(), off0.data_ptr(), R, 4e-4, 1e-4, 1e-4,
                              keep.data_ptr(), kept_off.data_ptr(), t2.data_ptr(), ri2.data_ptr(), None, counter.data_ptr(), L.stream()))

    timeit("hrf_prune (visibility + scan + compact)", prune)
    n = int(counter.item())
    t, ri = t2[:n].contiguous(), ri2[:n].contiguous()
    s = nat.samples_rays(g["o"], g["d"], g["frames"], t, ri)
    timeit("forward render (survivors)", lambda: nat.forward(s, 1, False, False), note=f"{n} survivors")
    timeit("forward render + save (survivors)", lambda: nat.forward(s, 1, False, True))
    sigma, _, rgb, feat = nat.forward(s, 1, False, True)
    d_sigma = torch.randn(n, device=dev) * 1e-3
    d_rgb = torch.randn(n, 3, device=dev) * 1e-3
    grads = [torch.zeros_like(p) for p in model.hot_parameters()]
    import numpy as np

    sg = (L.SegmentGrads * model.num_segments)()
    for s_ in range(model.num_segments):
        for k in range(4):
            sg[s_].grid[k] = grads[5 * s_ + k].data_ptr()
        sg[s_].vectors = grads[5 * s_ + 4].data_ptr()
    sg_dev = torch.from_numpy(np.frombuffer(bytes(sg), dtype=np.uint8).copy()).to(dev)
    d_mlp = torch.zeros(model.mlp_grad_elems, device=dev)
    ws = torch.empty(n * 40, device=dev)
    egrid = feat.data_ptr() + 64 * n

    def bwd_mlp():
        L.check(lib.hrf_field_backward_mlp(C.byref(nat.field), C.byref(s), d_sigma.data_ptr(), d_rgb.data_ptr(), None, feat.data_ptr(),
                                           None, d_mlp.data_ptr(), None, ws.data_ptr(), L.stream()))

    timeit("backward MLP kernel (saved feat)", bwd_mlp)

    def bwd_mlp_noflush():   # d_mlp NULL: the weight-gradient accumulators are computed but not added to global memory
        L.check(lib.hrf_field_backward_mlp(C.byref(nat.field), C.byref(s), d_sigma.data_ptr(), d_rgb.data_ptr(), None, feat.data_ptr(),
                                           None, None, None, ws.data_ptr(), L.stream()))

    timeit("backward MLP kernel, no weight-gradient flush", bwd_mlp_noflush)

    def scatter(eg):
        L.check(lib.hrf_field_backward_tables(C.byref(nat.field), C.byref(s), sg_dev.data_ptr(), eg, None, 0, ws.data_ptr(), 0, 4, L.stream()))

    timeit("MLP-only forward from features (survivors)", lambda: nat.forward_from_features(s, feat, None))
    timeit("table scatter, saved egrid", lambda: scatter(egrid))
    timeit("table scatter, re-gather tables", lambda: scatter(None))
    timeit("table scatter, saved egrid (L2 warm)", lambda: scatter(egrid), cold=False)
    timeit("backward MLP kernel (L2 warm)", bwd_mlp, cold=False)
    tot = sum(p.numel() for p in model.hot_parameters())
    pm, pv = [torch.zeros_like(p) for p in model.hot_parameters()], [torch.zeros_like(p) for p in model.hot_parameters()]

    def adam():
        for i, p in enumerate(model.hot_parameters()):
            L.check(lib.hrf_adam_step(p.data_ptr(), pm[i].data_ptr(), pv[i].data_ptr(), grads[i].data_ptr(), None, p.numel(), 1e-9, 0.9,
                                      0.99, 1e-15, 1, 1.0, L.stream()))

    timeit("adam (one launch per tensor, no shadow)", adam, note=f"{tot} params")
    # how much of each table does one step touch?  (SURVEY 8f-2 "touched entries only")
    for gr in grads:
        gr.zero_()
    scatter(egrid)
    torch.cuda.synchronize()
    lay = model.feature_grids[0].layout
    g0 = grads[0].view(-1, 2)
    fr = [float((g0[int(lay.offset[l]):int(lay.offset[l]) + int(lay.size[l])].abs().sum(1) != 0).float().mean()) for l in range(16)]
    print("touched fraction per level (grid xyz, segment 0):", " ".join(f"{x:.3f}" for x in fr))
    print("touched fraction of all table entries:", float(sum((gr.view(-1, 2).abs().sum(1) != 0).sum() for s_ in range(model.num_segments) for gr in grads[5 * s_:5 * s_ + 4])) /
          sum(gr.numel() // 2 for s_ in range(model.num_segments) for gr in grads[5 * s_:5 * s_ + 4]))


if __name__ == "__main__":
    main()
