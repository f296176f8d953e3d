"""Generates tests/golden/ref_kernels_golden.npz -- run from the repo root on a GPU, after build() has compiled the reference's own
kernels into oracle/_ref/libref_kernels.so (oracle/Makefile, only where the reference sources are present):

    python tests/golden/make_ref_kernels_golden.py [OUT.npz]

The file holds inputs and what the reference's find_matched_cells, interpolate_values<4> and interpolate_values_backward<4>
(src/tetrahedra_tracer.cu, compiled unmodified for sm_100a with -O3 --use_fast_math) return for them, so that
tests/test_gpu_ops.py compares the CUDA path with the reference without the reference.  The problem is the one that test traces
(3000-point Delaunay mesh, 400 camera rays, M = 256, 300 sorted samples per ray in [0.8, 3.2]), shrunk to stay small:
  - matching: a seeded sample of 24 rays, hit lists cut to the longest of them;
  - interpolation (64 channels): all 300 samples of the first of those rays, on the reference's own matches, with vertex ids
    renumbered densely (the kernels only gather and scatter by id) so that the field and its gradient cover only those vertices."""
import ctypes
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path[:0] = [str(ROOT), str(ROOT / "tetra-nerf_b200")]
from tetranerf import cpp  # noqa: E402
from tetranerf.b200 import synthetic as syn  # noqa: E402

REF_SO = ROOT / "oracle" / "_ref" / "libref_kernels.so"
OUT = Path(__file__).parent / "ref_kernels_golden.npz"
RAYS, INTERP_RAYS, CH = 24, 1, 64


def main(out: Path):
    ref = ctypes.CDLL(str(REF_SO))
    dev = torch.device("cuda:0")
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    p = lambda x: ctypes.c_void_p(x.data_ptr())

    # the inputs of tests/test_gpu_ops.py's `traced` fixture, samples sorted
    V, C = syn.delaunay_mesh(3000, seed=0)
    tr = cpp.TetrahedraTracer(dev)
    tr.load_tetrahedra(t(V), t(C))
    o, d = syn.camera_rays(400)
    traced = {k: v.cpu().numpy() for k, v in tr.trace_rays(t(o), t(d), 256).items()}
    rng = np.random.default_rng(0)
    dist = np.sort(rng.uniform(0.8, 3.2, (400, 300)).astype(np.float32), axis=1)

    rows = np.sort(np.random.default_rng(1).choice(400, RAYS, replace=False))
    M = int(traced["num_visited_cells"][rows].max())
    inp = {k: np.ascontiguousarray(v[rows] if v.ndim == 1 else v[rows, :M]) for k, v in traced.items()}
    inp["distances"] = np.ascontiguousarray(dist[rows])
    R, S = inp["distances"].shape
    mask = torch.zeros((R, S), dtype=torch.bool, device=dev)
    cell = torch.full((R, S), -1, dtype=torch.int32, device=dev)
    bary = torch.zeros((R, S, 3), dtype=torch.float32, device=dev)
    verts = torch.full((R, S, 4), -1, dtype=torch.int32, device=dev)
    dv = {k: t(v) for k, v in inp.items()}
    torch.cuda.synchronize()
    rc = ref.ref_find_matched_cells(ctypes.c_size_t(R), ctypes.c_size_t(S), ctypes.c_size_t(M), p(t(C)), p(dv["num_visited_cells"]),
                                    p(dv["visited_cells"]), p(dv["hit_distances"]), p(dv["barycentric_coordinates"]), p(dv["distances"]),
                                    p(dv["vertex_indices"]), p(cell), p(verts), p(mask), p(bary))
    assert rc == 0, rc
    match = {"mask": mask, "cell_indices": cell, "vertex_indices": verts, "barycentric_coordinates": bary}
    match = {k: v.cpu().numpy() for k, v in match.items()}
    assert 0.2 < match["mask"].mean() < 0.95

    vi = match["vertex_indices"][:INTERP_RAYS]
    ids, dense = np.unique(vi[vi >= 0], return_inverse=True)
    vi_dense = np.full_like(vi, -1)
    vi_dense[vi >= 0] = dense
    bc = match["barycentric_coordinates"][:INTERP_RAYS]
    U, N = len(ids), vi.shape[0] * vi.shape[1]
    rng = np.random.default_rng(2)
    field = rng.standard_normal((CH, U)).astype(np.float32)
    grad = rng.standard_normal((INTERP_RAYS, S, CH)).astype(np.float32)
    res = torch.empty((CH, N), dtype=torch.float32, device=dev)
    dvi, dbc, dfield = t(vi_dense), t(bc), t(field)
    rc = ref.ref_interpolate_values4(ctypes.c_uint32(U), ctypes.c_uint32(N), ctypes.c_uint32(CH), p(dvi), p(dbc), p(dfield), p(res))
    assert rc == 0, rc
    gref = torch.zeros((CH, U), dtype=torch.float32, device=dev)
    dgrad = t(grad.reshape(N, CH).T)
    rc = ref.ref_interpolate_values_backward4(ctypes.c_uint32(U), ctypes.c_uint32(N), ctypes.c_uint32(CH), p(dvi), p(dbc), p(dgrad), p(gref))
    assert rc == 0, rc

    np.savez_compressed(
        out, **inp, **{f"ref_{k}": v for k, v in match.items()},
        interp_vertex_indices=vi_dense, interp_barycentric_coordinates=bc, field=field, grad_interpolated=grad,
        ref_interpolated=res.T.reshape(INTERP_RAYS, S, CH).cpu().numpy(), ref_field_grad=gref.cpu().numpy(),
    )
    print("wrote", out, f"({out.stat().st_size} bytes): {R} rays x {S} samples, M = {M}; interpolation {N} samples over {U} vertices")


if __name__ == "__main__":
    main(Path(sys.argv[1]) if len(sys.argv) > 1 else OUT)
