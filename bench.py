#!/usr/bin/env python
"""bench.py -- rays/s of the FruitNeRF hot path (fused field + compositing, forward + backward) on
synthetic 4096-ray x 192-sample batches (BASELINE.json metric), N GPUs of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--variant small|big] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch: render forward (hash encode -> MLPs ->
composite), MSE + BCE loss, backward into the flat gradient buffer (and, for N > 1, one NCCL
all-reduce of that buffer -- the reference's DDP exchange, fruit_pipeline.py:117).  Prints ONE JSON
line on rank 0.  See DESIGN.md "Measurement" for the definitions of every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

R_RAYS, S_SAMPLES = 4096, 192
NUM_IMAGES = 100
CPU_BUDGET_S = 40.0  # wall-clock budget of the CPU arm inside the default run
HASH_BYTES_PER_POINT_FWD = 16 * 8 * 2 * 4  # L levels x 8 corners x F=2 x fp32 (SURVEY.md 8d)
HASH_BYTES_PER_POINT_BWD = 2 * HASH_BYTES_PER_POINT_FWD  # read-modify-write scatter


def _peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        j = json.loads(p.read_text())
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle-reason sampling during the timed region (B200_PROFILING.md clocks line),
    through NVML in-process (an `nvidia-smi -lms` poller next to the 256 MiB L2-flush fills stalled
    the GPU for ~10 ms per step on this pool; NVML queries from a thread do not)."""

    def __init__(self, index: int, period_s: float = 0.02):
        self.index, self.period = index, period_s
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._nv = None

    def start(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            self._nv = nv
            self._h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
        except Exception as e:  # noqa: BLE001
            self._nv = None
            self._err = repr(e)
            return
        self._thread = threading.Thread(target=self._run, daemon=True)
        self._thread.start()

    def _run(self):
        nv = self._nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
        }
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                mask = get_reasons(self._h)
                for n, bit in names.items():
                    if mask & bit:
                        self.reasons.add(n)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def stop(self):
        if self._nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"nvml unavailable: {getattr(self, '_err', '')}"]}
        self._stop.set()
        self._thread.join(timeout=2)
        sm = sorted(self.samples)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": "nvml"}


def build_field(variant: str, device, table_scale: float = 1e-1):
    """Random-init FruitField of the named variant (SURVEY.md 2.3), parameters from torch's RNG."""
    from fruitnerf_b200.fruit_field import FruitField, SceneContraction

    torch.manual_seed(0)
    kw = dict(geo_feat_dim=15, max_res=2048, log2_hashmap_size=19, num_layers_semantic=2, hidden_dim_semantics=64)
    if variant == "big":
        kw = dict(geo_feat_dim=30, max_res=4096, log2_hashmap_size=21, num_layers_semantic=3, hidden_dim_semantics=128)
    aabb = torch.tensor([[-1.0, -1, -1], [1, 1, 1]])
    f = FruitField(aabb, num_images=NUM_IMAGES, use_semantics=True, num_semantic_classes=1,
                   spatial_distortion=SceneContraction(order=float("inf")), **kw)
    with torch.no_grad():
        f.mlp_base_grid.hash_table.mul_(table_scale / 1e-3)  # U(-1,1) * table_scale
    return f.to(device).train()


def step_fn(field, batch, world, impl_id):
    """One eager step through the public op (the call FruitModel.get_outputs makes) -- used by tools/."""
    from fruitnerf_b200 import ops

    o, d, s, e, cam, img, mask = batch
    out = ops.render(field.kernel_shape(), field.kernel_params(), o, d, s, e, cam, field.position_mode(), field.appearance_mode(),
                     impl=impl_id)
    loss = torch.nn.functional.mse_loss(img, out["rgb"]) + torch.nn.functional.binary_cross_entropy_with_logits(
        out["semantics"][:, None], mask)
    return out, loss


DTYPE = "f32 (parameters, gather, compositing and accumulators fp32; MLP products on tcgen05 as bf16 hi/lo splits, 3 MMAs per product, ~2^-16)"


def _ncu_traffic(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of ``kernel`` from the committed `ncu --set full` capture
    (profiles/r2_ncu_traffic.json names the capture file of every entry); None when no capture of this kernel is committed."""
    p = ROOT / "profiles" / "r2_ncu_traffic.json"
    if not p.exists():
        return None, None
    j = json.loads(p.read_text()).get(kernel)
    return (j["dram_bytes"], j["capture"]) if j else (None, None)


DUMP_MAX_BYTES = 64_000_000
DUMP_SAMPLE_ELEMS = 1 << 20


def dump_outputs(step, field, out_dir: str) -> None:
    """Write what the last timed step handed its caller -- the loss, the render outputs and the parameter gradients -- as
    ``out_dir/<name>.npy`` (float32), so that two builds run with the same arguments can be compared array by array.  A gradient
    of more than DUMP_SAMPLE_ELEMS elements (the hash table's) is written as a sample of its rows drawn with a fixed seed, so
    every run writes the same rows."""
    import numpy as np

    names = {id(p): n for n, p in field.named_parameters()}
    arrays = {"loss": step.loss, **{f"out.{k}": v for k, v in step.outputs.items()}}
    for p in step.params:
        g = p.grad
        if g.numel() > DUMP_SAMPLE_ELEMS:
            n_rows = DUMP_SAMPLE_ELEMS * g.shape[0] // g.numel()
            rows = torch.randint(0, g.shape[0], (n_rows,), generator=torch.Generator().manual_seed(0)).unique()
            g = g[rows.to(g.device)]
        arrays[f"grad.{names[id(p)]}"] = g
    host = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_MAX_BYTES}-byte limit")
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for k, a in host.items():
        np.save(out / f"{k}.npy", a)


def kernel_names(variant: str, kernel: str):
    if kernel == "simt":
        return "simt_field_forward_kernel + simt_composite_kernel", "simt_field_backward_kernel"
    if variant == "small":
        return "tc_render_forward_ws_kernel", "tc_field_backward_kernel"
    return "tc_render_forward_big_kernel", "tc_big_backward_chain_kernel + tc_big_dw_kernel"


def _stage(msg: str) -> None:
    if os.environ.get("FNR_BENCH_DEBUG"):
        print(f"[bench {time.strftime('%H:%M:%S')}] {msg}", file=sys.stderr, flush=True)


def measure_variant(variant: str, steps: int, warmup: int, args, world: int, rank: int, dev, impl_id, with_e2e: bool = True,
                    dump_dir=None):
    """Device-timed step / forward / backward and (optionally) the end-to-end loop of one field variant; with ``dump_dir``,
    rank 0 writes the outputs of the last timed step there (dump_outputs)."""
    from fruitnerf_b200 import _lib as L
    from fruitnerf_b200 import ops
    from fruitnerf_b200 import synthetic as syn
    from fruitnerf_b200.engine import GraphedTrainStep, default_loss

    field = build_field(variant, dev)
    N_pts = R_RAYS * S_SAMPLES
    # per-rank batch (weak scaling: each rank draws its own 4096 rays, fruit_pipeline.py:97-99)
    o, d, s, e, cam = syn.ray_batch(R_RAYS, S_SAMPLES, salt=rank, num_images=NUM_IMAGES)
    img, mask = syn.targets(R_RAYS, salt=rank)
    host = [t.pin_memory() for t in (o, d, s, e, cam.to(torch.int32), img, mask)]
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    # the public training-step API: render fwd + loss + bwd captured in one CUDA graph
    exchange = None
    if world > 1:
        from fruitnerf_b200.grad_exchange import make_gradient_exchange

        # the exchange owns the flat gradient buffer (symmetric / multicast-mapped for the NVLS kernel): the backward kernels
        # accumulate straight into it
        exchange = make_gradient_exchange(ops.flat_grad_numel(field.kernel_params()), world, dev, kind=args.exchange)
    step = GraphedTrainStep(field, R_RAYS, S_SAMPLES, impl=impl_id, use_graph=not args.no_graph,
                            flat_grad=exchange.flat if exchange is not None else None)
    h2d = step.load_batch(*host)
    packed = step.pack_batch(*host)  # the same batch as one pinned byte buffer: one H2D copy per step in the e2e loop
    _stage(f"{variant}: capture")
    step.capture(warmup=max(warmup, 3))
    _stage(f"{variant}: captured, warm-up")

    def one_step():
        loss = step()
        if exchange is not None:
            exchange()  # the reference's DDP exchange: mean of the gradients over ranks (fruit_pipeline.py:117)
        return loss

    for _ in range(max(warmup, 3)):
        one_step()
    torch.cuda.synchronize()

    _stage(f"{variant}: timed loop")
    sampler = ClockSampler(dev.index) if (rank == 0 and not args.no_clocks) else None
    if sampler:
        sampler.start()  # before the barrier: host work on rank 0 between the barrier and the first timed step would show up
                         # as a long first step on the other ranks (they wait in the all-reduce)
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(steps)]
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()
    for i in range(steps):
        if not args.no_flush:
            flush.fill_(float(i))  # evict the table / weights from L2 between timed steps
        evs[i][0].record()
        one_step()
        evs[i][1].record()
    torch.cuda.synchronize()
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    clocks = sampler.stop() if sampler else None
    if dump_dir is not None and rank == 0:
        dump_outputs(step, field, dump_dir)
    step_ms = [ev[0].elapsed_time(ev[1]) for ev in evs]
    if os.environ.get("FNR_BENCH_DEBUG"):
        print(f"rank {rank} {variant} step_ms " + " ".join(f"{v:.3f}" for v in step_ms), file=sys.stderr)
    total_ms = torch.tensor([sum(step_ms)], device=dev, dtype=torch.float64)
    if world > 1:
        import torch.distributed as dist

        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms)

    # communication alone (N > 1): the exchange of the (static) flat gradient buffer, event-timed, max over ranks
    comm_ms = None
    if exchange is not None:
        import torch.distributed as dist

        cev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(10)]
        dist.barrier()
        for a_, b_ in cev:
            a_.record()
            exchange()
            b_.record()
        torch.cuda.synchronize()
        c = torch.tensor([sum(a_.elapsed_time(b_) for a_, b_ in cev) / len(cev)], device=dev, dtype=torch.float64)
        dist.all_reduce(c, op=dist.ReduceOp.MAX)
        comm_ms = float(c)

    _stage(f"{variant}: phase graphs")
    # phases, event-timed directly: graph A = forward + loss, graph B = backward (the same kernels as the one-graph step)
    st = step.static
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())

    def fwd_loss():
        out = ops.render(field.kernel_shape(), field.kernel_params(), st["origins"], st["directions"], st["starts"], st["ends"],
                         st["camera_indices"], field.position_mode(), field.appearance_mode(), impl=impl_id)
        return out, default_loss(out, st["image"], st["fruit_mask"])

    saved_grads = [p.grad for p in step.params]  # the step graph's static .grad views; restored below
    with torch.cuda.stream(side):
        for _ in range(2):
            for p in step.params:
                p.grad = None
            _, l_ = fwd_loss()
            l_.backward()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for p in step.params:
        p.grad = None
    _stage(f"{variant}: phase graphs warm, capturing")
    gA, gB = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
    # both captures on ONE stream: autograd runs a node's backward on the stream its forward ran on
    with torch.cuda.graph(gA, stream=side):
        _, loss_ab = fwd_loss()
    with torch.cuda.graph(gB, pool=gA.pool(), stream=side):
        loss_ab.backward()
    _stage(f"{variant}: phase graphs captured, replaying")
    pev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    for i in range(steps):
        if not args.no_flush:
            flush.fill_(float(i))
        pev[i][0].record()
        gA.replay()
        pev[i][1].record()
        gB.replay()
        pev[i][2].record()
    torch.cuda.synchronize()
    fwd_loss_ms = sum(ev[0].elapsed_time(ev[1]) for ev in pev) / steps
    bwd_ms = sum(ev[1].elapsed_time(ev[2]) for ev in pev) / steps
    for p, g in zip(step.params, saved_grads):
        p.grad = g

    _stage(f"{variant}: forward-only graph")
    # forward kernel alone (training forward: writes the encoding stash), for the roofline of the fused forward
    fwd_graph = torch.cuda.CUDAGraph()

    def fwd_only():
        return ops.render(field.kernel_shape(), field.kernel_params(), st["origins"], st["directions"], st["starts"], st["ends"],
                          st["camera_indices"], field.position_mode(), field.appearance_mode(), impl=impl_id)

    with torch.no_grad():
        with torch.cuda.graph(fwd_graph):
            fwd_out = fwd_only()
    fev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(steps)]
    for i in range(steps):
        if not args.no_flush:
            flush.fill_(float(i))
        fev[i][0].record()
        fwd_graph.replay()
        fev[i][1].record()
    torch.cuda.synchronize()
    fwd_ms = sum(ev[0].elapsed_time(ev[1]) for ev in fev) / steps
    del fwd_out

    # end-to-end through the public API with HOST buffers: per step H2D of the rays/targets from pinned
    # memory, one graph replay, D2H read of the loss -- all inside the timed region
    e2e = None
    _stage(f"{variant}: e2e loop")
    if with_e2e:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        step.load_packed(packed)
        pending, losses = None, []
        for i in range(steps):
            # H2D of the NEXT step's rays / bins / targets (one packed pinned buffer) overlaps this step, as a prefetching
            # data loader does; the loss of step i is copied device->host asynchronously into pinned memory and read on the host
            # one step later (no per-step drain of the GPU); every step still moves one full batch host->device and one loss
            # device->host inside the timed region, and every loss value is consumed on the host before the clock stops
            step.prefetch_packed(packed)
            one_step()
            handle = step.read_loss_async()
            step.commit_prefetched()
            if pending is not None:
                losses.append(pending.value())
            pending = handle
        losses.append(pending.value())
        torch.cuda.synchronize()
        assert len(losses) == steps and all(v == v for v in losses)
        e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world > 1:
            import torch.distributed as dist

            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
        e2e = {"value": world * R_RAYS * steps / float(e2e_s), "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
               "steps": steps}
    if world > 1:
        import torch.distributed as dist

        dist.barrier()

    _stage(f"{variant}: done")
    peak, peak_src = _peaks()
    mean_step = total_ms / steps
    fwd_bytes = N_pts * HASH_BYTES_PER_POINT_FWD
    bwd_bytes = N_pts * HASH_BYTES_PER_POINT_BWD
    fwd_kernel, bwd_kernel = kernel_names(variant, args.kernel)
    dominant_is_bwd = bwd_ms >= fwd_ms
    traffic, traffic_src = _ncu_traffic(bwd_kernel.split(" + ")[0] if dominant_is_bwd else fwd_kernel.split(" + ")[0])

    def roof(nbytes, ms, **extra):
        ach = nbytes / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "launch_ms": ms,
                "algorithmic_bytes_per_launch": nbytes, **extra}

    res = {
        "value": world * R_RAYS * steps / (total_ms * 1e-3),
        "ms_per_step": mean_step,
        "fwd_ms": fwd_ms,
        "fwd_loss_ms": fwd_loss_ms,
        "bwd_ms": bwd_ms,
        "phase_timing": "fwd_ms: forward kernel alone; fwd_loss_ms / bwd_ms: forward + loss graph and backward graph replayed back to back, "
                        "CUDA events between them (not derived by subtraction)",
        "fwd_rays_per_s": R_RAYS / (fwd_ms * 1e-3),
        "roofline": roof(bwd_bytes if dominant_is_bwd else fwd_bytes, bwd_ms if dominant_is_bwd else fwd_ms,
                         kernel=(f"render backward ({bwd_kernel} + simt_composite_backward_kernel)" if dominant_is_bwd
                                 else f"fused render forward ({fwd_kernel})"),
                         traffic=traffic, traffic_source=traffic_src, peak_source=peak_src),
        "roofline_forward": roof(fwd_bytes, fwd_ms, kernel=fwd_kernel),
        "roofline_backward": roof(bwd_bytes, bwd_ms, kernel=bwd_kernel),
        "roofline_step": roof(fwd_bytes + bwd_bytes, mean_step),
        "gpu_launches_per_step": step.launches_per_step,
        "clocks": clocks,
    }
    if comm_ms is not None:
        res["comm_ms"] = comm_ms
        res["exchange"] = exchange.describe()
    if e2e is not None:
        res["e2e"] = e2e
    del step, field, flush
    torch.cuda.empty_cache()
    return res


def measure_export(dev, n: int = 512, batch: int = 32768):
    """BASELINE.json configs[4]: uniform n^3 volume sample of the fruit_nerf field through fnr_export_forward (field + the three
    threshold selections + stream compaction per launch), batches of 32768 rays, deterministic grid.  Thresholds are taken from a
    probe batch (random weights never reach the reference constants 70 / 3) so that all three sets are populated."""
    from fruitnerf_b200 import _lib as L
    from fruitnerf_b200 import ops
    from fruitnerf_b200 import synthetic as syn
    from fruitnerf_b200.fruit_field import FruitField

    v = dict(syn.SMALL)
    sd = syn.field_state(geo=v["geo"], sem_dims=v["sem_dims"], log2_hashmap_size=v["log2_hashmap_size"], num_images=7, table_scale=2.0,
                         weight_gain=2.5)
    field = FruitField(aabb=sd["aabb"], num_images=7, geo_feat_dim=v["geo"], max_res=v["max_res"], log2_hashmap_size=v["log2_hashmap_size"],
                       num_layers_semantic=len(v["sem_dims"]) - 1, hidden_dim_semantics=v["sem_dims"][1], use_semantics=True,
                       num_semantic_classes=1, test_mode="export", spatial_distortion=None)
    field.load_state_dict(sd, strict=False)
    field = field.to(dev).eval()
    lin = torch.linspace(-1.0, 1.0, n)
    gx, gy = torch.meshgrid(lin, lin, indexing="ij")  # fruit_datamanager.py:71-121 for the cube [-1,1]^3, x-major
    pts = torch.stack([gx.reshape(-1), gy.reshape(-1), torch.full((n * n,), -1.0)], dim=-1).to(dev)
    normal, far, total = (0.0, 0.0, 1.0), 2.0, n ** 3
    bins = torch.linspace(0.0, 1.0, n + 1).to(dev)
    shape, params = field.kernel_shape(), field.kernel_params()
    mid = (n * n // 2 // 2048) * 2048
    dense = ops.export_batch(shape, params, pts[mid:mid + 2048], normal, bins, 0.0, far, ops.ExportBuffers(capacity=1, device=dev), dense_out=True)
    thr = (float(dense["semantics"].quantile(0.97)), float(dense["density"].quantile(0.97)), 0.5)
    capacity = min(total, 1 << 25)

    def run(count):
        buf = ops.ExportBuffers(capacity=capacity, device=dev)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        torch.cuda.synchronize()
        L.load().fnr_launch_count(1)
        ev[0].record()
        done = 0
        while done < count:
            o = pts[done:done + batch]
            ops.export_batch(shape, params, o, normal, bins, 0.0, far, buf, point_base=done * n, dense_out=False, thresholds=thr)
            done += o.shape[0]
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]), buf, int(L.load().fnr_launch_count(1))

    run(batch)  # warm-up
    ms, buf, launches = min((run(pts.shape[0]) for _ in range(2)), key=lambda r: r[0])
    counts = buf.counts.cpu().tolist()
    keys = [buf.keys[k][: min(counts[k], capacity)] for k in range(3)]
    ok = True
    for k in range(3):  # size-independent properties: unique global keys inside the volume, semantic sets nested in the density set
        u = torch.unique(keys[k])
        ok &= bool(u.numel() == keys[k].numel()) and (keys[k].numel() == 0 or int(u.max()) < total)
    s2 = torch.sort(keys[2]).values
    for k in (0, 1):
        if keys[k].numel():
            pos = torch.searchsorted(s2, keys[k]).clamp_(max=max(s2.numel() - 1, 0))
            ok &= bool((s2[pos] == keys[k]).all())
    peak, _ = _peaks()
    ach = total * HASH_BYTES_PER_POINT_FWD / (ms * 1e-3) / 1e9
    return {"workload": f"uniform {n}^3 volume sample of the fruit_nerf field, {batch} rays x {n} samples per launch, deterministic grid",
            "ms": ms, "points": total, "points_per_s": total / (ms * 1e-3), "counts": counts, "thresholds": thr,
            "keys_unique_and_nested": bool(ok), "gpu_launches": launches,
            "roofline": {"kernel": "tc_render_forward_ws_kernel<export>", "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "algorithmic_bytes": total * HASH_BYTES_PER_POINT_FWD}}


def run_ours(args):
    from fruitnerf_b200 import _lib as L

    L.load()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs CUDA devices (no CPU fallback in the product path)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    impl_id = {"auto": L.FNR_IMPL_AUTO, "simt": L.FNR_IMPL_SIMT, "tcgen05": L.FNR_IMPL_TCGEN05}[args.kernel]
    warm = max(args.warmup, 3)
    head = measure_variant(args.variant, args.steps, warm, args, world, rank, dev, impl_id, dump_dir=args.dump_outputs)
    variants = {}
    if args.variant == "small" and not args.no_variants:
        # BASELINE.json configs[2] / [3]: fruit_nerf_big, same batch shape, same timing rules
        try:
            b = measure_variant("big", args.steps, 3, args, world, rank, dev, impl_id)
            b["config"] = {"workload": f"fruit_nerf_big field: {R_RAYS} rays x {S_SAMPLES} samples per GPU, render fwd + MSE/BCE loss + bwd"
                                       + (" + gradient exchange" if world > 1 else ""), "steps": args.steps, "warmup": 3}
            b.pop("clocks", None)
            variants["big"] = b
        except Exception as ex:  # noqa: BLE001 -- never allowed to break the headline line
            variants["big"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
    export = None
    if world == 1 and not args.no_variants:
        try:
            export = measure_export(dev)
        except Exception as ex:  # noqa: BLE001
            export = {"error": f"{type(ex).__name__}: {ex}"[:300]}
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": "rays/sec (4096 rays x 192 samples) fused fwd+bwd",
        "value": head["value"],
        "unit": "rays/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": warm,
        "ms_per_step": head["ms_per_step"],
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": DTYPE,
        "data": "synthetic",
        "config": {
            "workload": f"fruit_nerf{'_big' if args.variant == 'big' else ''} field ({args.variant}): {R_RAYS} rays x {S_SAMPLES} samples "
                        "per GPU, render fwd + MSE/BCE loss + bwd" + (" + gradient exchange (mean over ranks)" if world > 1 else ""),
            "variant": args.variant,
            "kernel": args.kernel,
            "rays_per_gpu": R_RAYS,
            "samples_per_ray": S_SAMPLES,
            "execution": "eager" if args.no_graph else "one CUDA graph per step (fruitnerf_b200.engine.GraphedTrainStep)",
            "l2": "flushed between timed steps (256 MiB fill); per-step CUDA-event durations summed",
            "parallelism": f"dp{world}",
        },
    }
    for k in ("fwd_ms", "fwd_loss_ms", "bwd_ms", "phase_timing", "fwd_rays_per_s", "roofline", "roofline_forward", "roofline_backward", "roofline_step",
              "e2e", "comm_ms", "exchange", "clocks"):
        if k in head:
            line[k] = head[k]
    # kernels of THIS library launched inside the timed region: counted by the library itself (fnr_launch_count) while the step
    # was captured into its CUDA graph, times the replays that were timed
    line["gpu_launches"] = int(head["gpu_launches_per_step"]) * args.steps
    line["gpu_launches_per_step"] = int(head["gpu_launches_per_step"])
    if variants:
        line["variants"] = variants
    if export is not None:
        line["export_512"] = export
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(args.variant, sample_rays=args.cpu_rays, repeats=3)
    if world == 1 and not args.no_train:
        line["train_iteration"] = train_iteration_rate(args.variant, dev)
    print(json.dumps(line))


def train_iteration_rate(variant: str, dev, iterations: int = 300):
    """Supplementary number (BASELINE.json configs[1]/[2]): a WHOLE training iteration of the method on the synthetic
    apple scene -- pixel batch, proposal stage, field forward / backward, losses, Adam -- replayed as CUDA graphs by
    fruitnerf_b200.trainer.Trainer.  Never allowed to break the headline line: any failure is reported as a string."""
    try:
        from fruitnerf_b200.scripts.train import synthetic_spec
        from fruitnerf_b200.trainer import Trainer

        method = "fruit_nerf" if variant == "small" else "fruit_nerf_big"
        trainer = Trainer(synthetic_spec(method, schedule_steps=3000), device=dev, use_cuda_graph=True)
        trainer.train(40)  # warm-up: eager iterations + capture of both schedule branches
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        trainer.train(iterations)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        rays = trainer.spec.pipeline.datamanager.train_num_rays_per_batch
        return {"value": rays * iterations / dt, "unit": "rays/s", "ms_per_iteration": 1e3 * dt / iterations, "rays_per_iteration": rays,
                "iterations": iterations, "method": method,
                "what": "data + proposal sampling + field fwd/bwd + losses + optimiser, synthetic apple scene, CUDA-graph replay"}
    except Exception as ex:  # noqa: BLE001
        return {"error": f"{type(ex).__name__}: {ex}"[:300]}


def host_threads() -> int:
    """Threads of the CPU arm: every host core the process may use (torchrun sets OMP_NUM_THREADS=1, which would
    otherwise make the reference arm single-threaded at N > 1)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    return max(1, n)


def cpu_baseline(variant: str, sample_rays: int, repeats: int):
    """The oracle (a port: pure-PyTorch restatement of the reference's CPU-runnable torch path) on
    the host cores, fwd+bwd on the same workload: median of ``repeats`` passes after one warm-up pass."""
    from fruitnerf_b200 import synthetic as syn
    from oracle import fruit_ref as fr

    v = syn.SMALL if variant == "small" else syn.BIG
    sd = syn.field_state(geo=v["geo"], sem_dims=v["sem_dims"], log2_hashmap_size=v["log2_hashmap_size"], num_images=NUM_IMAGES,
                         table_scale=1e-1)
    spec = fr.FieldSpec(max_res=v["max_res"], log2_hashmap_size=v["log2_hashmap_size"], geo_feat_dim=v["geo"])
    def one_pass(rays):
        o, d, s, e, cam = syn.ray_batch(rays, S_SAMPLES, num_images=NUM_IMAGES)
        img, mask = syn.targets(rays)
        st = {k: t.clone().requires_grad_(t.is_floating_point() and k != "aabb") for k, t in sd.items()}
        t0 = time.perf_counter()
        f = fr.field_forward(st, spec, o[:, None, :], d[:, None, :], s[..., None], e[..., None], cam, True, "train")
        r = fr.render(f, s[..., None], e[..., None], training=True)
        ld = fr.loss_dict(r, img, mask)
        (ld["rgb_loss"] + ld["semantics_loss"]).backward()
        return time.perf_counter() - t0

    # thread count: all host threads is not the fastest setting for this op-by-op torch workload on a many-core host (oversubscribed
    # intra-op pools); a 256-ray probe per candidate picks the best one, and also sizes the sample so that the (repeats + 1) passes
    # fit CPU_BUDGET_S on whatever host this is (the same oracle ran at 430 .. 1900 rays/s on different boxes of this pool)
    n_all = host_threads()
    one_pass(128)  # allocator / thread-pool warm-up
    tried = {}
    for nt in sorted({min(n_all, c) for c in (8, 16, 32, 64)}):  # (all 128 threads of a pool host: 36 s for the 256-ray probe)
        torch.set_num_threads(nt)
        tried[nt] = one_pass(256)
        if tried[nt] > 4.0:  # this host is slow at this setting: do not spend the budget on the remaining candidates
            break
    best_nt = min(tried, key=tried.get)
    torch.set_num_threads(best_nt)
    # cost model t(rays) = fixed + per_ray * rays from two probes (the dense table gradient makes `fixed` large)
    t256, t1024 = tried[best_nt], one_pass(1024)
    per_ray = max(t1024 - t256, 1e-6) / 768.0
    fixed = max(t256 - 256 * per_ray, 0.0)
    requested = sample_rays
    while sample_rays > 512 and (fixed + per_ray * sample_rays) * (repeats + 1) > CPU_BUDGET_S:
        sample_rays //= 2
    o, d, s, e, cam = syn.ray_batch(sample_rays, S_SAMPLES, num_images=NUM_IMAGES)
    img, mask = syn.targets(sample_rays)
    times = []
    for _ in range(repeats + 1):  # first pass = warm-up
        st = {k: t.clone().requires_grad_(t.is_floating_point() and k != "aabb") for k, t in sd.items()}
        t0 = time.perf_counter()
        f = fr.field_forward(st, spec, o[:, None, :], d[:, None, :], s[..., None], e[..., None], cam, True, "train")
        r = fr.render(f, s[..., None], e[..., None], training=True)
        ld = fr.loss_dict(r, img, mask)
        (ld["rgb_loss"] + ld["semantics_loss"]).backward()
        times.append(time.perf_counter() - t0)
    timed = sorted(times[1:]) if repeats else times
    med = timed[len(timed) // 2]
    return {"value": sample_rays / med, "unit": "rays/s", "cores": torch.get_num_threads(), "host_cpus": os.cpu_count(), "kind": "port",
            "threads_probed_s_per_256_rays": {str(k): round(v_, 3) for k, v_ in tried.items()},
            "seconds": [round(t, 3) for t in times[1:] if repeats] or [round(times[0], 3)],
            "sample": f"{sample_rays} rays x {S_SAMPLES} samples ({'the full batch' if sample_rays == R_RAYS else f'a sample of the {requested}-ray batch: the full batch would exceed the {CPU_BUDGET_S:.0f} s budget of this arm on this host'}), "
                      f"fwd+bwd, median of {max(repeats, 1)} after 1 warm-up, torch.set_num_threads({torch.get_num_threads()})"}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path.  The reference's
    arithmetic lives in nerfstudio/tinycudann (absent, not installable: BASELINE.md section 2), so
    the arm is the oracle port on all host threads; each step = one pass over the 4096-ray batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    rays = args.cpu_rays
    n = max(1, min(args.steps, 3))
    t_all = time.perf_counter()
    base = cpu_baseline(args.variant, rays, repeats=n)
    dt = time.perf_counter() - t_all
    v = base["value"]
    line = {
        "impl": "reference",
        "metric": "rays/sec (4096 rays x 192 samples) fused fwd+bwd",
        "value": v,
        "unit": "rays/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": n,
        "warmup": 1,
        "ms_per_step": rays / v * 1e3,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"fruit_nerf field ({args.variant}): {rays} rays x {S_SAMPLES} samples, fwd+bwd, CPU oracle port "
                               f"({base['cores']} threads), median of {n} passes", "variant": args.variant, "wall_s": round(dt, 1)},
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    if os.environ.get("FNR_BENCH_DEBUG"):
        import faulthandler

        faulthandler.dump_traceback_later(int(os.environ.get("FNR_BENCH_WATCHDOG", "60")), exit=False)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of every hot-path loop (headline, phases, e2e, big variant); the export and "
                         "whole-training-iteration figures keep their fixed workloads")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--variant", default="small", choices=["small", "big"])
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel", default="auto", choices=["auto", "simt", "tcgen05"])
    ap.add_argument("--exchange", default="auto", choices=["auto", "nccl", "nvls", "nvls_bf16"],
                    help="gradient exchange at N > 1: NCCL all-reduce or the library's own multimem (NVLS) all-reduce kernel")
    ap.add_argument("--cpu-rays", type=int, default=R_RAYS)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the supplementary whole-training-iteration measurement")
    ap.add_argument("--no-variants", action="store_true", help="skip the fruit_nerf_big and 512^3 export measurements")
    ap.add_argument("--no-graph", action="store_true", help="diagnostic: eager step instead of the CUDA-graph step")
    ap.add_argument("--no-flush", action="store_true", help="diagnostic: skip the L2 flush between timed steps")
    ap.add_argument("--no-clocks", action="store_true", help="diagnostic: do not sample nvidia-smi during the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the loss, render outputs and parameter gradients of the last timed step "
                         "as DIR/<name>.npy (float32; the hash-table gradient as a fixed, seeded sample of rows)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
