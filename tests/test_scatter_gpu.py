"""The table / vector gradient scatter (grid_scatter_v3_kernel; v5 behind HRF_SCATTER=5) in isolation, against float64
autograd through the oracle's hash-grid encoding and tensor composition: the kernel's only rounding is fp32 accumulation, so the bar is
1e-5 -- tight enough to catch a single dropped or doubled corner contribution (the run-length accumulation and the
shared-corner carry between neighbouring cells are exactly where such a bug would sit)."""
import ctypes as C

import numpy as np
import pytest
import torch

from helpers import make_pair, positions_of, synthetic_rays
from humanrf_b200 import _lib as L
from oracle import field as OF
from oracle import hashgrid

pytestmark = pytest.mark.gpu
GRID_AXES = ([0, 1, 2], [0, 1, 3], [1, 2, 3], [0, 2, 3])     # xyz, xyt, yzt, xzt (decomposition4d.py:126-129)
VECTOR_OF_GRID = (3, 2, 0, 1)                                 # xyz*v_t, xyt*v_z, yzt*v_x, xzt*v_y (tensor_composition.cu:49-52)


def _relnorm(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


@pytest.mark.parametrize("gen", ["5", ""], ids=["v5-lane-pairs", "v3-5ctas"])
def test_table_scatter_matches_float64_autograd(cuda, monkeypatch, gen):
    """hrf_field_backward_tables with no environment set runs v3 = csrc/scatter_v3.cu (parity-slot accumulators,
    warp-private staging, transposed vector rows); HRF_SCATTER=5 runs v5 = csrc/scatter_v5.cu (the parity slots split over a
    lane pair by the parity of the first-axis vertex, pair-wide flushes).  Two launches, grid 0 and then grids 1-3, so that
    a split launch schedule is covered too."""
    if gen:
        monkeypatch.setenv("HRF_SCATTER", gen)
    else:
        monkeypatch.delenv("HRF_SCATTER", raising=False)
    om, m, frames = make_pair((6, 6), table_std=0.5, bf16=False)
    with torch.no_grad():                                      # bf16-representable tables: the kernel re-gathers the bf16 shadows
        for s, fg in enumerate(m.feature_grids):
            for k, g in enumerate(fg.grids()):
                q = g.detach().bfloat16().float()
                g.copy_(q)
                om.segments[s].grids[k] = q.cpu().reshape(-1, 2).clone()
    nat = m.native()
    nat.refresh()
    b = synthetic_rays(96, 48, frames, ragged=True, seed=21)   # consecutive samples of a ray: neighbouring cells at the fine levels
    pos, fr = positions_of(b), b["frames"][b["ri"]]
    n = pos.shape[0]
    seg = om.f2s[fr.numpy()]
    xyzt = torch.cat((pos + 0.5, torch.from_numpy(om.f2t[fr.numpy()]).unsqueeze(1)), dim=1).float()
    g = torch.Generator().manual_seed(2)
    d_out = torch.randn(n, 32, generator=g)
    d_out[::7] = 0                                            # zero upstream gradients are skipped, not scattered

    # ---- reference: float64 autograd
    ref_tables, ref_vectors = [], []
    for s, sd in enumerate(om.segments):
        sel = torch.from_numpy(np.nonzero(seg == s)[0])
        tabs = [t.double().requires_grad_(True) for t in sd.grids]
        vec = sd.vectors.double().requires_grad_(True)
        c = xyzt[sel]
        sv = OF.lerp_vectors(vec, c)                            # fp32 tap arithmetic (exact: vec_res is a power of two), float64 blend
        out = sum(hashgrid.encode(tabs[k], c[:, GRID_AXES[k]], sd.log2T) * sv[VECTOR_OF_GRID[k]] for k in range(4))
        (out * d_out[sel].double()).sum().backward()
        ref_tables.append([t.grad.reshape(-1) for t in tabs])
        ref_vectors.append(vec.grad)

    # ---- kernel: workspace = d(features) level-major [16][n] float2 | (x,y,z,t) [n] float4 | segment [n] u8
    ws = torch.zeros(n * 40, dtype=torch.float32, device=cuda)
    ws[: 32 * n] = d_out.reshape(n, 16, 2).permute(1, 0, 2).reshape(-1).to(cuda)
    ws[32 * n: 36 * n] = xyzt.reshape(-1).to(cuda)
    ws.view(torch.uint8)[144 * n: 145 * n] = torch.from_numpy(seg.astype(np.uint8)).to(cuda)
    grads = [torch.zeros_like(p) for p in m.hot_parameters()]
    sg = (L.SegmentGrads * m.num_segments)()
    for s in range(m.num_segments):
        for k in range(4):
            sg[s].grid[k] = grads[5 * s + k].data_ptr()
        sg[s].vectors = grads[5 * s + 4].data_ptr()
    sg_dev = torch.from_numpy(np.frombuffer(bytes(sg), dtype=np.uint8).copy()).to(cuda)
    samples = nat.samples_query(pos.to(cuda).contiguous(), None, fr.to(cuda).to(torch.int32).contiguous())
    for first, count in ((0, 1), (1, 3)):                      # split launches (per-table schedule)
        L.check(L.lib().hrf_field_backward_tables(C.byref(nat.field), C.byref(samples), sg_dev.data_ptr(), None, None, 0, ws.data_ptr(),
                                                  first, count, L.stream()))
    torch.cuda.synchronize()
    for s in range(m.num_segments):
        for k in range(4):
            got, ref = grads[5 * s + k].cpu(), ref_tables[s][k]
            assert ((got != 0) & (ref == 0)).sum() == 0
            e = _relnorm(got, ref)
            worst = float((got.double() - ref).abs().max() / ref.abs().max())
            print(f"seg{s} grid{k}: relnorm {e:.2e} worst entry {worst:.2e} touched {(ref != 0).sum().item()}")
            assert e < 1e-5 and worst < 1e-5
        e = _relnorm(grads[5 * s + 4].cpu(), ref_vectors[s])
        print(f"seg{s} vectors: relnorm {e:.2e}")
        assert e < 1e-5
