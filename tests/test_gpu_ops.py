"""GPU parity of find_visited_cells / interpolate_values(+backward): vs the CPU oracle (bit-exact) and vs what the
reference's OWN kernels returned, stored in tests/golden/ref_kernels_golden.npz (few-ulp, --use_fast_math there)."""
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tetranerf.b200 import synthetic as syn

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
REF_GOLDEN = Path(__file__).resolve().parent / "golden" / "ref_kernels_golden.npz"


@pytest.fixture(scope="module")
def traced(small_mesh):
    from tetranerf import cpp

    V, C = small_mesh
    tr = cpp.TetrahedraTracer(DEV)
    tr.load_tetrahedra(torch.from_numpy(V).to(DEV), torch.from_numpy(C).to(DEV))
    o, d = syn.camera_rays(400)
    out = tr.trace_rays(torch.from_numpy(o).to(DEV), torch.from_numpy(d).to(DEV), 256)
    rng = np.random.default_rng(0)
    S = 300
    # sorted samples spanning before / inside / after the mesh, plus an unsorted set (literal pointer semantics)
    dist = np.sort(rng.uniform(0.8, 3.2, (400, S)).astype(np.float32), axis=1)
    dist[::7] = rng.uniform(0.8, 3.2, (len(dist[::7]), S)).astype(np.float32)
    return tr, out, torch.from_numpy(dist).to(DEV), V, C


def test_find_visited_cells_vs_oracle(traced):
    tr, out, dist, V, C = traced
    g = tr.find_visited_cells(out["num_visited_cells"], out["visited_cells"], out["barycentric_coordinates"], out["hit_distances"],
                              out["vertex_indices"], dist)
    c = {k: v.cpu().numpy() for k, v in out.items()}
    ref = orc.find_visited_cells(c["num_visited_cells"], c["visited_cells"], c["barycentric_coordinates"], c["hit_distances"],
                                 c["vertex_indices"], dist.cpu().numpy())
    assert g["mask"].dtype == torch.bool and g["cell_indices"].dtype == torch.int32
    assert np.array_equal(g["mask"].cpu().numpy(), ref["mask"])
    assert np.array_equal(g["cell_indices"].cpu().numpy(), ref["cell_indices"])
    assert np.array_equal(g["vertex_indices"].cpu().numpy(), ref["vertex_indices"])
    assert np.array_equal(g["barycentric_coordinates"].cpu().numpy().view(np.uint32), ref["barycentric_coordinates"].view(np.uint32))
    assert 0.2 < ref["mask"].mean() < 0.95


def test_find_visited_cells_arbitrary_segments():
    """the matcher on hand-made segment lists, including NON-monotone t_out (the warp kernel's literal fallback), empty rays,
    rays that fill M, NaN samples: bit-equal to the literal loop of the oracle (tetrahedra_tracer.cu:129-160)"""
    from tetranerf import cpp

    rng = np.random.default_rng(11)
    R, M, S = 257, 64, 101
    num = rng.integers(0, M + 1, R).astype(np.int32)
    num[:4] = (0, 1, M, M)
    t_in = np.sort(rng.uniform(0.5, 3.0, (R, M)).astype(np.float32), axis=1)
    t_out = t_in + rng.uniform(0.0, 0.08, (R, M)).astype(np.float32)   # overlapping segments, t_out mostly increasing ...
    bad = rng.random(R) < 0.5
    t_out[bad] = rng.permutation(t_out[bad].T).T                        # ... and shuffled (non-monotone) on half of the rays
    hd = np.stack([t_in, t_out], -1)
    cells = rng.integers(0, 1000, (R, M)).astype(np.int32)
    verts = rng.integers(0, 500, (R, M, 4)).astype(np.int32)
    bary = rng.random((R, M, 2, 3)).astype(np.float32)
    dist = rng.uniform(0.3, 3.3, (R, S)).astype(np.float32)
    dist[::3] = np.sort(dist[::3], axis=1)
    dist[5, 7] = np.nan
    V, C = syn.delaunay_mesh(64, seed=1)
    tr = cpp.TetrahedraTracer(DEV)
    tr.load_tetrahedra(torch.from_numpy(V).to(DEV), torch.from_numpy(C).to(DEV))
    t = lambda a: torch.from_numpy(a).to(DEV)
    g = tr.find_visited_cells(t(num), t(cells), t(bary), t(hd), t(verts), t(dist))
    ref = orc.find_visited_cells(num, cells, bary, hd, verts, dist)
    assert np.array_equal(g["mask"].cpu().numpy(), ref["mask"])
    assert np.array_equal(g["cell_indices"].cpu().numpy(), ref["cell_indices"])
    assert np.array_equal(g["vertex_indices"].cpu().numpy(), ref["vertex_indices"])
    assert np.array_equal(g["barycentric_coordinates"].cpu().numpy().view(np.uint32), ref["barycentric_coordinates"].view(np.uint32))
    assert ref["mask"].mean() > 0.05


@pytest.mark.parametrize("D,Cdim", [(4, 64), (4, 7), (3, 16), (2, 5), (6, 32)])
def test_interpolate_values_vs_oracle(traced, D, Cdim):
    from tetranerf import cpp

    tr, out, dist, V, C = traced
    rng = np.random.default_rng(D * 100 + Cdim)
    N1, N2 = 37, 53
    vi = rng.integers(0, len(V), (N1, N2, D)).astype(np.int32)
    vi[rng.random((N1, N2)) < 0.2] = -1  # unmatched samples (py_binding.cpp:191)
    vi[0, 0, 0] = -1  # a lone empty first vertex
    w = rng.random((N1, N2, D - 1)).astype(np.float32) / D
    field = syn.random_field(len(V), Cdim, seed=Cdim)
    got = cpp.interpolate_values(torch.from_numpy(vi).to(DEV), torch.from_numpy(w).to(DEV), torch.from_numpy(field).to(DEV))
    assert got.shape == (N1, N2, Cdim)
    ref = orc.interpolate_values(vi, w, field)
    assert np.array_equal(got.cpu().numpy().view(np.uint32), ref.view(np.uint32))
    gin = rng.standard_normal((N1, N2, Cdim)).astype(np.float32)
    gb = cpp.interpolate_values_backward(torch.from_numpy(vi).to(DEV), torch.from_numpy(w).to(DEV), torch.from_numpy(field).to(DEV),
                                         torch.from_numpy(gin).to(DEV))
    refb = orc.interpolate_values_backward(vi, w, field.shape, gin)
    assert gb.shape == field.shape
    np.testing.assert_allclose(gb.cpu().numpy(), refb, rtol=1e-5, atol=1e-5)  # atomics: order differs


def test_interpolate_autograd_matches_einsum(traced):
    """the reference's own test identity, tests/test_tetrahedra_tracer.py:410-416,442-453"""
    from tetranerf.utils.extension import interpolate_values

    tr, out, dist, V, C = traced
    g = tr.find_visited_cells(out["num_visited_cells"], out["visited_cells"], out["barycentric_coordinates"], out["hit_distances"],
                              out["vertex_indices"], dist)
    vi, bc = g["vertex_indices"], g["barycentric_coordinates"]
    field = torch.from_numpy(syn.random_field(len(V), 64)).to(DEV).requires_grad_(True)
    val = interpolate_values(vi, bc, field)
    safe = vi.long().clamp_min(0)
    f2 = field.detach().clone().requires_grad_(True)
    gathered = torch.where((vi >= 0)[None], f2[:, safe], torch.zeros((), device=DEV))
    full = torch.cat((1 - bc.sum(-1, keepdim=True), bc), -1)
    gt = torch.einsum("jrbi,rbi->rbj", gathered, full)
    torch.testing.assert_close(val, gt, rtol=1.3e-6, atol=1e-5)
    val.sum().backward()
    gt.sum().backward()
    torch.testing.assert_close(field.grad, f2.grad, rtol=1e-4, atol=1e-4)


def test_against_reference_kernels(traced):
    """The reference's src/tetrahedra_tracer.cu, compiled unmodified for sm_100a with the reference's flags (-O3 --use_fast_math),
    on inputs of the `traced` problem: its outputs are stored with those inputs in tests/golden/ref_kernels_golden.npz
    (tests/golden/make_ref_kernels_golden.py).  Indices exact; floats within a few ulp."""
    from tetranerf import cpp

    gold = dict(np.load(REF_GOLDEN))
    t = lambda k: torch.from_numpy(gold[k]).to(DEV)
    tr = traced[0]  # holds the mesh the stored hit lists were traced on
    g = tr.find_visited_cells(t("num_visited_cells"), t("visited_cells"), t("barycentric_coordinates"), t("hit_distances"),
                              t("vertex_indices"), t("distances"))
    assert torch.equal(t("ref_mask"), g["mask"]) and torch.equal(t("ref_cell_indices"), g["cell_indices"])
    assert torch.equal(t("ref_vertex_indices"), g["vertex_indices"])
    torch.testing.assert_close(t("ref_barycentric_coordinates"), g["barycentric_coordinates"], rtol=2e-6, atol=2e-6)
    # interpolation forward: FFMA chain -> expect bit-exact; backward: atomics -> tolerance
    vi, bc, field = t("interp_vertex_indices"), t("interp_barycentric_coordinates"), t("field")
    res = t("ref_interpolated")
    mine = cpp.interpolate_values(vi, bc, field)
    torch.testing.assert_close(mine, res, rtol=1e-6, atol=1e-6)
    frac_exact = (mine == res).float().mean().item()
    assert frac_exact > 0.99, frac_exact
    gmine = cpp.interpolate_values_backward(vi, bc, field, t("grad_interpolated"))
    torch.testing.assert_close(gmine, t("ref_field_grad"), rtol=1e-4, atol=1e-4)
