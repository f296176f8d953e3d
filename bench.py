#!/usr/bin/env python
"""bench.py -- rays/s of the Tetra-NeRF ray-sampling hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (forward render, BASELINE configs[1])
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the restated reference algorithm (oracle port)
    python bench.py --workload tetra-nerf-original ...       # 256 + 256 samples, uniform sampler (registration.py:20-46)
    python bench.py --mode train ...                         # fused training step (fwd + bwd), BASELINE configs[2] shape
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy

Workload (BASELINE.json configs[1]): 45,000 uniform random points -> scipy Delaunay -> 302,024 tetrahedra,
4096 camera-like rays per step, `tetra-nerf` config (128 + 128 samples, biased sampler, M = 512), eval-mode
forward render with random-init MLP (torch.manual_seed(0)) and N(0,1) vertex features.  A "step" = one full
pass trace -> sample -> interp+MLP -> PDF -> interp+MLP -> composite over one batch of 4096 rays per GPU.
`value` = rays/s with the rays already resident in HBM; `e2e` = the same through the plug-in call nerfstudio makes,
`TetrahedraNerf.get_outputs(RayBundle)`, with pinned HOST ray buffers (H2D + D2H inside the timed region).
Multi-GPU: rays shard across ranks (weak scaling, mesh + weights replicated); the pixels of step i are all-gathered
over NCCL on a side stream while step i+1 renders (every gather completes inside the timed region).
Both arms print the same `config`; the reference arm never imports the CUDA package.
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for p in (str(ROOT), str(ROOT / "tetra-nerf_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np
import torch

NUM_POINTS = 45_000
RAYS_PER_STEP = 4096
# SURVEY.md §8d: algorithmic FLOPs per sample (2 * MACs): coarse 41,088 MAC, fine 61,312 MAC
FLOP_COARSE, FLOP_FINE = 2 * 41_088, 2 * 61_312
WORKLOADS = {  # registration.py:20-61
    "tetra-nerf": {"num_samples": 128, "num_fine_samples": 128, "use_biased_sampler": True, "tag": "tetra-nerf(128+128,biased,M=512)"},
    "tetra-nerf-original": {"num_samples": 256, "num_fine_samples": 256, "use_biased_sampler": False, "tag": "tetra-nerf-original(256+256,uniform,M=512)"},
}
L2_CAP_BYTES_PER_CLK = 6300.0  # LTS throughput cap measured in /opt/skills/guides/B300_MICROARCH.md (same L2 design), x SM clock


def synthetic():
    """tetranerf/b200/synthetic.py loaded by path: the reference arm must not import the `tetranerf` package (that dlopens
    the CUDA library)"""
    spec = importlib.util.spec_from_file_location("tn_b200_synthetic", ROOT / "tetra-nerf_b200" / "tetranerf" / "b200" / "synthetic.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def workload_config(workload: str, mode: str, rays: int, world: int, tetrahedra: int, points: int = NUM_POINTS):
    """the `config` object: identical for both arms"""
    return {"workload": f"delaunay{points // 1000}k_{round(tetrahedra / 1000)}ktet/{rays}rays/{WORKLOADS[workload]['tag']}/{'train-fwd+bwd' if mode == 'train' else 'eval-forward'}",
            "tetrahedra": int(tetrahedra), "rays_per_step_per_gpu": int(rays),
            "parallelism": f"ray-shard x{world} (weak scaling), mesh+weights replicated, NCCL all_gather of pixels"}


def peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        d = json.loads(f.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"], "bf16_tflops_sustained": d.get("bf16_tflops_sustained"), "src": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}


class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons of one GPU every 100 ms while the timed region runs (NVML)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.stop_flag = index, [], set(), None, False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.1)

    def result(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def make_workload():
    syn = synthetic()
    V, C = syn.delaunay_mesh(NUM_POINTS, seed=0)
    field = syn.random_field(len(V), 64, seed=3, kind="normal")
    return V, C, field


def mlp_params():
    """torch default nn.Linear init under torch.manual_seed(0), in the module order of model.py:433-455."""
    g = torch.Generator().manual_seed(0)

    def lin(i, o):
        k = 1.0 / (i**0.5)
        return ((torch.rand((o, i), generator=g) * 2 - 1) * k).float(), ((torch.rand((o,), generator=g) * 2 - 1) * k).float()

    p = {}
    for name, (i, o) in (("mlp_base.layers.0", (64, 128)), ("mlp_base.layers.1", (128, 128)), ("mlp_base.layers.2", (128, 128)),
                         ("mlp_head.layers.0", (155, 128)), ("field_output_color.net", (128, 3)), ("field_output_density.net", (128, 1))):
        p[name + ".weight"], p[name + ".bias"] = lin(i, o)
    return p


def dump_outputs(directory: str, arrays: dict):
    """DIR/<name>.npy in float32 (masks as 0/1): the outputs of the last timed step, so that two builds can be compared on them.
    Each run computes them from the same seeded inputs; training gradients accumulate with atomics, so runs agree on them to rounding."""
    d = Path(directory)
    d.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(d / f"{name}.npy", torch.as_tensor(a).detach().cpu().float().numpy())


def cpu_arm(V, C, field, params, num_rays: int, seed: int, workload: str, nthreads: int = 0):
    """the restated reference algorithm on the host cores (oracle port); returns (seconds, rays, rendered outputs)"""
    from oracle import oracle as orc

    mesh = cpu_arm.mesh if getattr(cpu_arm, "mesh", None) is not None else orc.OracleMesh(V, C)
    cpu_arm.mesh = mesh
    o, d = synthetic().camera_rays(num_rays, seed=seed)
    w = WORKLOADS[workload]
    cfg = orc.RenderConfig(num_samples=w["num_samples"], num_fine_samples=w["num_fine_samples"], use_biased_sampler=w["use_biased_sampler"])
    t0 = time.perf_counter()
    img = orc.render(mesh, torch.from_numpy(field), params, o, d, cfg, nthreads=nthreads)
    return time.perf_counter() - t0, num_rays, img


def cpu_threads():
    """(oracle C++ threads, torch intra-op threads).  The C++ stages use every hardware thread; torch's fp32 GEMMs of the MLP are
    capped at 32 threads -- measured on the 128-thread host of the B200 box (profiles/r2_cpu_threads.json): 16 -> 1683, 32 -> 1918,
    64 -> 1485, 128 -> 224 rays/s.  TN_BENCH_TORCH_THREADS overrides."""
    from oracle import oracle as orc

    cores = orc.hardware_threads()
    nt = int(os.environ.get("TN_BENCH_TORCH_THREADS", "0")) or min(cores, 32)
    torch.set_num_threads(max(1, nt))
    return cores, torch.get_num_threads()


def run_reference(args, rank, world):
    if rank != 0:
        return
    V, C, field = make_workload()
    params = mlp_params()
    cores, tthreads = cpu_threads()
    sample = args.rays  # the whole batch of the named workload every step
    for i in range(args.warmup):
        cpu_arm(V, C, field, params, min(sample, 512), seed=100 + i, workload=args.workload)  # thread pools / allocator warm-up on a short batch
    tot = 0.0
    for i in range(args.steps):
        dt, _, img = cpu_arm(V, C, field, params, sample, seed=200 + i, workload=args.workload)
        tot += dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, img)
    value = sample * args.steps / tot
    line = {
        "impl": "reference", "metric": "rays/sec (4096-ray batch, 300k-tet mesh)", "value": value, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, "eval", sample, world, len(C)),
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} rays/step of the same workload (oracle: C++ trace/match/interp on {cores} threads + torch-CPU fp32 "
                                   f"MLP/compositing on {tthreads} threads); warm-up steps use 512-ray batches"},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "the reference has no CPU path (src/py_binding.cpp:30-33) and its OptiX build cannot be compiled here; this arm times the restated reference algorithm (oracle/) on the host cores",
    }
    print(json.dumps(line), flush=True)


def setup_peer_gather(lib, tracer, dist, dev, world, rank, R):
    """fused pixel gather: one gathered buffer [world*R, 6] per rank (cudaMalloc + CUDA IPC), mapped into every peer; the
    render kernels store their pixels straight into all of them (tn_render_set_gather).  Returns the local buffer as a tensor."""
    import ctypes as C

    nbytes = world * R * 6 * 4
    ptr, handle = C.c_void_p(), (C.c_ubyte * 64)()
    lib.tn_peer_alloc.argtypes = [C.c_int, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_ubyte)]
    lib.tn_peer_open.argtypes = [C.c_int, C.POINTER(C.c_ubyte), C.POINTER(C.c_void_p)]
    lib.tn_render_set_gather.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p), C.c_uint32]
    rc = lib.tn_peer_alloc(dev.index, nbytes, C.byref(ptr), handle)
    assert rc == 0, lib.tn_last_error()
    mine = torch.tensor(list(bytes(handle)), dtype=torch.uint8, device=dev)
    allh = torch.empty((world, 64), dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(allh, mine)
    allh = allh.cpu().numpy()
    ptrs = (C.c_void_p * world)()
    for k in range(world):
        if k == rank:
            ptrs[k] = ptr.value
        else:
            q = C.c_void_p()
            hb = (C.c_ubyte * 64)(*allh[k].tolist())
            rc = lib.tn_peer_open(dev.index, hb, C.byref(q))
            assert rc == 0, lib.tn_last_error()
            ptrs[k] = q.value
    rc = lib.tn_render_set_gather(tracer.handle, world, rank, ptrs, R)
    assert rc == 0, lib.tn_last_error()

    class _Buf:  # __cuda_array_interface__ view of the IPC allocation
        __cuda_array_interface__ = {"shape": (world * R, 6), "typestr": "<f4", "data": (ptr.value, False), "version": 2}

    return torch.as_tensor(_Buf(), device=dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rays", type=int, default=None, help="rays per step per GPU (default 4096; 8192 for --mode train)")
    ap.add_argument("--workload", default="tetra-nerf", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="eval", choices=["eval", "train"])
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"], help="N > 1: fused peer-store gather (default) or NCCL all_gather")
    ap.add_argument("--points", type=int, default=None, help="--mode train: points of the Delaunay mesh (default 300000 -> ~2.0 M tetrahedra)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mlp-precision", default="f16w2", choices=["f16w2", "bf16x3"],
                    help="operand precision of the inference MLP (tn_render_set_mlp_precision): f16w2 = fp16 activations x fp16 hi/lo weights, "
                         "2 MMAs per product, ~2.6e-5 abs on unit-scale density/colour (library default); bf16x3 = 3 MMAs, ~5e-7")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its last step (rank 0) as DIR/<name>.npy, float32; "
                         "--mode train adds the loss, the parameter gradients and a fixed sample of 16384 columns of the field gradient")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    if args.rays is None:
        args.rays = 8192 if args.mode == "train" else RAYS_PER_STEP
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch.distributed as dist

    from tetranerf import cpp
    from tetranerf.b200.render import RenderSettings
    from tetranerf.nerfstudio import model as tnm
    from tetranerf.utils.extension import tetranerf_cpp_extension as ext

    syn = synthetic()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    R = args.rays
    V, C, field = make_workload()
    params = mlp_params()
    w = WORKLOADS[args.workload]
    if args.mode == "train":
        return run_train(args, rank, world, dev, V, C, field, params, dist)
    # the plug-in object nerfstudio drives: TetrahedraNerf (model.py:209-662); its eval-mode get_outputs is the fused CUDA pipeline
    cfg = tnm.TetrahedraNerfConfig(num_tetrahedra_vertices=len(V), num_tetrahedra_cells=len(C), num_samples=w["num_samples"],
                                   num_fine_samples=w["num_fine_samples"], use_biased_sampler=w["use_biased_sampler"])
    model = tnm.TetrahedraNerf(cfg)
    sd = {"tetrahedra_vertices": torch.from_numpy(V), "tetrahedra_cells": torch.from_numpy(C), "tetrahedra_field": torch.from_numpy(field)}
    sd.update(params)
    model.load_state_dict(sd, strict=False)
    model = model.to(dev).eval()
    tracer = model.get_tetrahedra_tracer()
    fr = model._fused_renderer()
    fr.set_mlp_precision(2 if args.mlp_precision == "f16w2" else 3)
    st = RenderSettings(512, w["num_samples"], w["num_fine_samples"], w["use_biased_sampler"], float(model.collider.far_plane), (1.0, 1.0, 1.0))
    nsteps = args.warmup + args.steps
    # a different ray batch every step; each rank gets its own shard (weak scaling)
    host_od = []  # pinned [2,R,3] (origins | directions): one host->device copy per step on the end-to-end path
    for i in range(nsteps):
        o, d = syn.camera_rays(R, seed=1000 * (rank + 1) + i)
        host_od.append(torch.from_numpy(np.stack([o, d])).pin_memory())
    dev_od = [t.to(dev) for t in host_od]
    out = {"rgb": torch.empty((R, 3), device=dev), "accumulation": torch.empty((R, 1), device=dev), "depth": torch.empty((R, 1), device=dev),
           "ray_mask": torch.empty((R,), dtype=torch.bool, device=dev)}
    gather_mode = "none" if world == 1 else args.gather
    gathered = None
    if gather_mode == "peer":
        gathered = setup_peer_gather(ext._lib, tracer, dist, dev, world, rank, R)
    elif gather_mode == "nccl":
        pix = torch.empty((R, 5), device=dev)
        gathered = torch.empty((world * R, 5), device=dev)
    host_pix = torch.empty((R, 5), dtype=torch.float32).pin_memory()
    host_out = {k: torch.empty(v.shape, dtype=v.dtype).pin_memory() for k, v in out.items() if k != "ray_mask"}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def step(i, e2e: bool):
        if e2e:  # the call nerfstudio makes: Model.forward(RayBundle) -> collider -> TetrahedraNerf.get_outputs
            od = host_od[i].to(dev, non_blocking=True)
            with torch.no_grad():
                res = model(tnm.RayBundle(origins=od[0], directions=od[1]))
            for k, v in host_out.items():
                v.copy_(res[k], non_blocking=True)
        else:
            od = dev_od[i]
            fr.render(od[0], od[1], st, out=out)
        if gather_mode == "nccl":
            src = out if not e2e else res
            torch.cat((src["rgb"], src["accumulation"], src["depth"]), dim=1, out=pix)
            dist.all_gather_into_tensor(gathered, pix)  # final NCCL gather of rendered pixels
        # gather_mode == "peer": the render kernels already stored this rank's pixels into every rank's gathered buffer

    def timed(e2e: bool, profile: bool = False):
        fr.set_profiling(profile)  # per-kernel events only on the separate profiling pass (they feed kernel_ms / the rooflines)
        for i in range(args.warmup):
            step(i, e2e)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        kern = {}
        l0 = tracer.launch_count()
        for k in range(args.steps):
            flush.fill_(k & 0xFF)  # L2 flush between timed iterations (not timed)
            ev[k][0].record()
            step(args.warmup + k, e2e)
            ev[k][1].record()
            if profile:
                for n, v in fr.kernel_timings_ms().items():
                    kern[n] = kern.get(n, 0.0) + v
        torch.cuda.synchronize(dev)
        launches = tracer.launch_count() - l0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ms = sum(a.elapsed_time(b) for a, b in ev)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), {n: v / args.steps for n, v in kern.items()}, launches

    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_total, _, launches = timed(False)
    last = {k: v.cpu() for k, v in out.items()} if args.dump_outputs else None  # the timed runs below render into `out` again
    ms_e2e, _, _ = timed(True)
    _, kern_ms, _ = timed(False, profile=True)  # same steps again with CUDA events around every kernel of the library
    # the same timed region with the other operand precision of the MLP (reported beside the headline, never as `value`)
    other = "bf16x3" if args.mlp_precision == "f16w2" else "f16w2"
    fr.set_mlp_precision(3 if other == "bf16x3" else 2)
    ms_other, _, _ = timed(False)
    fr.set_mlp_precision(2 if args.mlp_precision == "f16w2" else 3)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    tracer.synchronize()
    n_active = int(out["ray_mask"].sum().item())
    # sum of visited tetrahedra of the last batch (SURVEY §8d traversal bytes)
    import ctypes as Ct

    bufs = fr.debug_buffers()
    numv = torch.empty((R,), dtype=torch.int32, device=dev)
    Ct.CDLL("libcudart.so").cudaMemcpy(Ct.c_void_p(numv.data_ptr()), Ct.c_void_p(bufs["num"]), Ct.c_size_t(4 * R), Ct.c_int(3))
    sum_k = int(numv.sum().item())
    if gather_mode == "peer":  # every rank's pixels of the last step landed in this rank's gathered buffer
        torch.cuda.synchronize(dev)
        dist.barrier()
        mine = gathered[rank * R:(rank + 1) * R]
        assert torch.equal(mine[:, :3], out["rgb"]) and bool((gathered[:, 3] >= 0).all()), "fused pixel gather: local block differs from the render"

    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
        pk = peaks()
        total_rays = world * R * args.steps
        value = total_rays / (ms_total * 1e-3)
        e2e = total_rays / (ms_e2e * 1e-3)
        Sc, S2 = st.num_samples, st.num_samples + st.num_fine_samples + 1
        flops = {"mlp_fine": n_active * S2 * FLOP_FINE, "mlp_coarse": n_active * Sc * FLOP_COARSE}
        traffic = {}
        prof = ROOT / "profiles" / "roofline_traffic.json"
        if prof.exists():
            try:
                traffic = json.loads(prof.read_text())
            except Exception:
                traffic = {}
        # dominant kernel: the fine interp+MLP pass (tensor-bound)
        dom = max(kern_ms, key=kern_ms.get)
        roof = {"kernel": dom, "bound": "tensor", "unit": "TFLOP/s", "peak": pk["bf16_tflops"], "peak_src": pk["src"] + " bf16 burst",
                "traffic": traffic.get(dom), "traffic_src": "ncu --set full capture committed under profiles/ (not re-measured in this run)"}
        if dom in flops:
            ach = flops[dom] / (kern_ms[dom] * 1e-3) / 1e12
            roof.update(achieved=ach, frac=ach / pk["bf16_tflops"],
                        note="algorithmic fp32-equivalent FLOPs (SURVEY §8d); the kernel issues "
                             + ("2 fp16 MMAs per algorithmic MAC (f16w2), so tensor-pipe occupancy is ~2x this fraction" if args.mlp_precision == "f16w2"
                                else "3 bf16 MMAs per algorithmic MAC (bf16x3), so tensor-pipe occupancy is ~3x this fraction"))
        # the traversal (BASELINE metric: "traversal HBM% of roofline"): SURVEY §8d algorithmic bytes / (prefetch + trace time)
        Fcount = tracer.num_faces()
        tb = 28 * R + 52 * sum_k + 12 * len(V) + 16 * len(C) + 20 * Fcount
        clk = sampler.result().get("sm_max_mhz") or pk.get("sm_max_mhz") or 1965.0
        l2_peak = L2_CAP_BYTES_PER_CLK * clk * 1e6 / 1e9
        tgb = tb / (kern_ms["trace"] * 1e-3) / 1e9
        roof_trace = {"kernel": "trace (k_l2_prefetch + k_trace / k_walk)", "bound": "hbm", "unit": "GB/s", "achieved": tgb, "peak": pk["hbm_gbs"],
                      "peak_src": pk["src"] + " HBM copy", "frac": tgb / pk["hbm_gbs"], "bytes": tb, "traffic": traffic.get("trace"),
                      "l2_peak_gbs": l2_peak, "l2_frac": tgb / l2_peak,
                      "note": "algorithmic bytes 28R + 52 sum(K) + 12V + 16T + 20F (SURVEY §8d); the ~56 MB working set is L2-resident by design, "
                              "so the L2 fraction (LTS cap 6300 B/clk x max SM clock) is reported beside the HBM fraction"}
        line = {
            "metric": "rays/sec (4096-ray batch, 300k-tet mesh)", "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (trace/interp/compositing) + " + ("f16w2 tensor-core MLP (fp16 activations x fp16 hi/lo weights, f32 accumulate; per-sample "
                                                           "density/colour within 1e-4 of the fp32 oracle, tests/test_gpu_render.py)" if args.mlp_precision == "f16w2"
                                                           else "bf16x3 tensor-core MLP with f32 accumulate"), "data": "synthetic",
            "config": workload_config(args.workload, "eval", R, world, len(C)),
            "mlp_precision": {"mode": args.mlp_precision, "other_mode": other, "other_mode_ms_per_step": ms_other / args.steps,
                              "other_mode_value": total_rays / (ms_other * 1e-3)},
            "timing": {"l2": "flushed between timed steps (256 MiB fill); a new ray batch every step", "events": "CUDA events per step on the launch stream, max over ranks",
                       "gather": {"none": "single GPU", "peer": "fused: render kernels store pixels into every rank's gathered buffer over NVLink (no collective)",
                                  "nccl": "NCCL all_gather_into_tensor inside every step"}[gather_mode]},
            "kernel_ms": kern_ms, "roofline": roof, "roofline_trace": roof_trace,
            "e2e": {"value": e2e, "unit": "rays/s", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": 2 * R * 12, "d2h_bytes_per_step": R * 20,
                    "api": "TetrahedraNerf.forward(RayBundle) -> get_outputs (the nerfstudio plug-in call), pinned host rays in, pinned host pixels out"},
            "gpu_launches": int(launches), "clocks": sampler.result(),
        }
        if world == 1 and not args.no_cpu_baseline:
            cores, tthreads = cpu_threads()
            for wi in range(2):
                cpu_arm(V, C, field, params, 256, seed=7 + wi, workload=args.workload)  # warm (thread pools, MKL)
            tot_t, tot_n, k = 0.0, 0, 0
            while tot_t < 10.0 and k < 64:  # ~10 s of CPU work
                dt, n, _ = cpu_arm(V, C, field, params, 1024, seed=300 + k, workload=args.workload)
                tot_t, tot_n, k = tot_t + dt, tot_n + n, k + 1
            line["cpu_baseline"] = {"value": tot_n / tot_t, "unit": "rays/s", "cores": cores, "kind": "port",
                                    "sample": f"{tot_n} rays ({k} batches of 1024) of the same workload through oracle/ "
                                              f"(C++ trace/match/interp on {cores} threads + torch-CPU fp32 MLP/compositing on {tthreads} threads)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


NUM_POINTS_TRAIN = 300_000  # BASELINE configs[2]: "dense 300k-point mesh" -> ~2.0 M tetrahedra


def run_train(args, rank, world, dev, V, C, field, params, dist):
    """BASELINE configs[2]: 300k-point mesh (~2.0 M tetrahedra), 8192 rays per batch, biased sampler, ONE training step = forward
    (stratified bins) + loss + backward + DDP-style gradient averaging (N > 1) + optimizer step (RAdam lr 1e-3, registration.py:37-41)
    through the plug-in API (TetrahedraNerf.forward / get_loss_dict).  `value` = rays/s with the ray batch and the target pixels
    resident in HBM, `e2e` = with pinned-host rays + targets copied in and the loss read back every step.  The same steps on the
    reference's op sequence (unfused CUDA ops + torch fp32 MLP + autograd, TETRANERF_B200_UNFUSED_TRAIN=1) are timed beside it."""
    from tetranerf.b200.distributed import average_gradients
    from tetranerf.nerfstudio import model as tnm

    syn = synthetic()
    R = args.rays
    w = WORKLOADS[args.workload]
    V, C = syn.delaunay_mesh(args.points or NUM_POINTS_TRAIN, seed=0)
    field = syn.random_field(len(V), 64, seed=3, kind="normal")

    def make_model():
        cfg = tnm.TetrahedraNerfConfig(num_tetrahedra_vertices=len(V), num_tetrahedra_cells=len(C), num_samples=w["num_samples"],
                                       num_fine_samples=w["num_fine_samples"], use_biased_sampler=w["use_biased_sampler"])
        m = tnm.TetrahedraNerf(cfg)
        sd = {"tetrahedra_vertices": torch.from_numpy(V), "tetrahedra_cells": torch.from_numpy(C), "tetrahedra_field": torch.from_numpy(field)}
        sd.update(params)
        m.load_state_dict(sd, strict=False)
        return m.to(dev).train()

    nsteps = args.warmup + args.steps
    host = []
    for i in range(nsteps):
        o, d = syn.camera_rays(R, seed=5000 * (rank + 1) + i)
        tgt = np.random.default_rng(9000 * (rank + 1) + i).random((R, 3), dtype=np.float32)
        host.append(torch.from_numpy(np.concatenate([o, d, tgt], 1)).pin_memory())  # [R, 9]
    devb = [t.to(dev) for t in host]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    host_loss = torch.empty((1,), dtype=torch.float32).pin_memory()

    def run(mode_env: str, steps: int, warmup: int, e2e: bool, capture: bool = False):
        os.environ["TETRANERF_B200_UNFUSED_TRAIN"] = mode_env
        torch.manual_seed(0)  # the stratified sampler's jitter: the same draws in every run
        model = make_model()
        opt = torch.optim.RAdam(model.parameters(), lr=1e-3)
        tracer = model.get_tetrahedra_tracer()

        def step(i):
            b = host[i].to(dev, non_blocking=True) if e2e else devb[i]
            out = model(tnm.RayBundle(origins=b[:, 0:3].contiguous(), directions=b[:, 3:6].contiguous()))
            loss = model.get_loss_dict(out, {"image": b[:, 6:9]})["rgb_loss"]
            opt.zero_grad(set_to_none=True)
            loss.backward()
            if world > 1:
                average_gradients(model.parameters())
            opt.step()
            if e2e:
                host_loss.copy_(loss.detach().reshape(1), non_blocking=True)
            return out, loss

        for i in range(warmup):
            step(i)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        l0 = tracer.launch_count()
        for k in range(steps):
            flush.fill_(k & 0xFF)
            ev[k][0].record()
            res = step(warmup + k)
            ev[k][1].record()
        torch.cuda.synchronize(dev)
        launches = tracer.launch_count() - l0
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        ms = sum(a.elapsed_time(b) for a, b in ev)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        last = None
        if capture:  # what the caller holds after the last step: outputs, loss, gradients (the field's: a fixed sample of columns)
            out, loss = res
            grads = {f"grad.{n}": p.grad for n, p in model.named_parameters() if p.grad is not None and n != "tetrahedra_field"}
            cols = torch.from_numpy(np.random.default_rng(0).choice(len(V), min(len(V), 16384), replace=False)).to(dev)
            last = {**out, "rgb_loss": loss, **grads, "grad.tetrahedra_field.sample": model.tetrahedra_field.grad[:, cols]}
            last = {k: v.detach().cpu() for k, v in last.items()}
        del model, opt
        return float(t.item()), launches, last

    sampler = ClockSampler(dev.index)
    sampler.start()
    ms_total, launches, last = run("0", args.steps, args.warmup, False, capture=bool(args.dump_outputs))
    ms_e2e, _, _ = run("0", args.steps, args.warmup, True)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    usteps = max(3, args.steps // 4)
    ms_unfused, _, _ = run("1", usteps, 3, False)
    # per-kernel breakdown of one fused step (CUDA events inside the library), plus torch-side pieces timed separately
    os.environ["TETRANERF_B200_UNFUSED_TRAIN"] = "0"
    model = make_model()
    opt = torch.optim.RAdam(model.parameters(), lr=1e-3)
    fr = model._fused_renderer()
    fr.set_profiling(True)
    kern = {}
    for i in range(4):
        b = devb[i]
        out = model(tnm.RayBundle(origins=b[:, 0:3].contiguous(), directions=b[:, 3:6].contiguous()))
        loss = model.get_loss_dict(out, {"image": b[:, 6:9]})["rgb_loss"]
        opt.zero_grad(set_to_none=True)
        loss.backward()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); opt.step(); e1.record()
        torch.cuda.synchronize(dev)
        if i >= 2:
            for n, v in {**fr.kernel_timings_ms(), **fr.backward_timings_ms(), "optimizer_radam": e0.elapsed_time(e1)}.items():
                kern[n] = kern.get(n, 0.0) + v / 2
    fr.set_profiling(False)
    del model, opt
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last)
        pk = peaks()
        total = world * R * args.steps
        S2 = w["num_samples"] + w["num_fine_samples"] + 1
        # SURVEY §8d: forward 42.03 MFLOP/ray + backward 2 x the fine pass (the coarse pass is detached)
        flop_step = R * (w["num_samples"] * FLOP_COARSE + 3 * S2 * FLOP_FINE)
        ach = world * flop_step / (ms_total / args.steps * 1e-3) / 1e12
        line = {
            "metric": "rays/sec (train step fwd+bwd+optimizer, 8192-ray batch, ~2M-tet mesh)", "value": total / (ms_total * 1e-3), "unit": "rays/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 (trace/interp/compositing/optimizer) + bf16x3 tensor-core MLP fwd+bwd with f32 accumulate",
            "data": "synthetic", "config": workload_config(args.workload, "train", R, world, len(C), int(len(V))) | {"points": int(len(V))},
            "timing": {"l2": "flushed between timed steps (256 MiB fill); a new ray batch every step", "events": "CUDA events per step on the launch stream, max over ranks",
                       "step": "TetrahedraNerf.forward (training mode) -> MSE loss -> backward -> (N>1: gradient all-reduce) -> RAdam step"},
            "roofline": {"kernel": "whole training step", "bound": "tensor", "unit": "TFLOP/s", "achieved": ach, "peak": pk["bf16_tflops_sustained"] or pk["bf16_tflops"],
                         "peak_src": pk["src"] + " bf16 sustained", "frac": ach / (pk["bf16_tflops_sustained"] or pk["bf16_tflops"]), "traffic": None,
                         "note": "algorithmic fp32-equivalent FLOPs of SURVEY §8d (fwd coarse + fine, bwd 2 x fine); bf16x3 issues 3 MMAs per MAC and the backward recomputes the fine forward"},
            "unfused_reference_sequence": {"ms_per_step": ms_unfused / usteps, "steps": usteps,
                                           "what": "same model, TETRANERF_B200_UNFUSED_TRAIN=1: the reference's op sequence on this repo's unfused CUDA ops + torch fp32 MLP + autograd"},
            "speedup_vs_unfused": (ms_unfused / usteps) / (ms_total / args.steps), "kernel_ms": kern,
            "e2e": {"value": total / (ms_e2e * 1e-3), "unit": "rays/s", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": R * 36, "d2h_bytes_per_step": 4,
                    "api": "TetrahedraNerf.forward(RayBundle) + get_loss_dict + backward + optimizer, pinned host rays/targets in, loss out"},
            "gpu_launches": int(launches), "clocks": sampler.result(),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
