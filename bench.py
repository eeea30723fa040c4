#!/usr/bin/env python
"""bench.py -- headline benchmark of the surfel-rasteriser hot path.

Workload (BASELINE.json configs[1]): 100k surfels, 512x512, 6 views, raster
forward + backward per step, synthetic inputs (SURVEY.md 8d).  One "step" is
one pass of the hot path over that batch.

  python bench.py --gpus N --steps K --warmup W            (our CUDA path)
  python bench.py --impl reference ...                     (CPU reference arm:
        the oracle port of the reference's rasteriser on all host cores)
  python bench.py ... --dump-outputs DIR                   (also writes the outputs of
        the last timed step as .npy files, to compare two builds: dump_outputs)

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the definition
of every field.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

P_SURFELS, RES, VIEWS = 100000, 512, 6
# kernels of libga_b200.so per device-timed step: preprocess, tile scan, scatter, 2 sort kernels, render fwd | render bwd,
# preprocess bwd (+ 3 memsets, not counted)
# (round 2: + tile-area pre-pass, its scan, list-walking kernel A, recompute kernel A for flagged tiles, kernel B,
# fused fallback kernel = 13 launches of our kernels per step)
LAUNCHES_PER_STEP = 13
METRIC = "512^2 views/sec @100k Gaussians (surfel raster fwd+bwd)"
UNIT = "views/s"
CONFIG = {"workload": "C2: 100k surfels, 512x512, 6 views, raster fwd+bwd",
          "surfels": P_SURFELS, "resolution": RES, "views_per_step": VIEWS,
          "l2": "256 MiB L2 flush between timed steps (outside the timed events)",
          "parallelism": "independent scenes per rank (no data-path collective)"}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_inputs(seed, P=P_SURFELS, views=VIEWS):
    """Seeded synthetic scene + look-at cameras (tools/synth.py: numpy only -- the GPU arm never loads the oracle)."""
    from tests.helpers import cameras, scene
    g = scene(P, seed)
    vs, ps, _, tf = cameras(views)
    return g, vs, ps


def pin_to_gpu_numa_node(local):
    """Binds this process to the CPUs next to its GPU (sysfs local_cpulist of the GPU's PCI function) BEFORE any
    pinned host buffer is allocated, so the staging memory of every rank is first-touched on its GPU's NUMA node
    (8 ranks uploading 24 MB per step through the wrong socket was the e2e limiter at N=8 in round 1)."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/local_cpulist" % bdf) as f:
            txt = f.read().strip()
        cpus = set()
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return {"pci": bdf, "cpus": len(cpus)}
    except Exception as ex:                                  # not fatal: report and carry on unpinned
        return {"error": repr(ex)}
    return {"cpus": 0}


DUMP_ALLMAP_SAMPLE = 1 << 22


def dump_outputs(out_dir, color, allmap, radii, grad):
    """Writes what the last timed step returned as <out_dir>/<name>.npy in float32 (43 MB in all): color [B,V,3,H,W],
    radii [B,V,P] and the surfel gradient [B,P,13] whole, and allmap_sample, the allmap [B,V,7,H,W] values at a fixed
    seeded sample of DUMP_ALLMAP_SAMPLE flat indices (sorted) -- the whole allmap alone would be 44 MB."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    idx = np.sort(np.random.default_rng(0).choice(allmap.numel(), DUMP_ALLMAP_SAMPLE, replace=False))
    sample = allmap.reshape(-1)[torch.from_numpy(idx).to(allmap.device)]
    for name, t in (("color", color), ("allmap_sample", sample), ("radii", radii), ("grad", grad)):
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy().astype(np.float32))


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def mark(self):
        """Rows sampled from now on belong to the timed region."""
        self.mark_idx = len(self.rows)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for r in self.rows if len(r) >= 7]
        timed = rows[getattr(self, "mark_idx", 0):]
        window = "timed region"
        if len(timed) < 3:      # region shorter than the sampling period: include the warm-up (same workload)
            timed, window = rows, "warm-up + timed region (timed region shorter than 3 samples)"
        sm = [float(r[1]) for r in timed if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in timed if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names)
                   if any(r[3 + k].lower().startswith("active") for r in timed)]
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm),
                "window": window}


# ---------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's rasteriser (all host threads)
# ---------------------------------------------------------------------------
def cpu_views_per_s(n_views, min_seconds, seed=40):
    from oracle import surfel_oracle as so
    from tests.helpers import oracle_view
    so.set_num_threads(os.cpu_count() or 1)            # torchrun exports OMP_NUM_THREADS=1
    g, vs, ps = make_inputs(seed)
    rng = np.random.default_rng(0)
    gc = rng.standard_normal((3, RES, RES)).astype(np.float32)
    ga = rng.standard_normal((7, RES, RES)).astype(np.float32)
    done, t0 = 0, time.perf_counter()
    while True:
        for v in range(n_views):
            o = oracle_view(g, vs[v % VIEWS], ps[v % VIEWS], [1, 1, 1], RES, RES)
            so.rasterize_backward(o, gc, ga)
            done += 1
        if time.perf_counter() - t0 >= min_seconds:
            break
    dt = time.perf_counter() - t0
    return done / dt, done, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count()
    for _ in range(args.warmup):
        cpu_views_per_s(1, 0.0)
    t0 = time.perf_counter()
    total = 0
    for _ in range(args.steps):
        _, n, _ = cpu_views_per_s(VIEWS, 0.0)
        total += n
    dt = time.perf_counter() - t0
    v = total / dt
    out = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": CONFIG,
           "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": "%d steps x %d views of the full C2 workload (oracle/surfel_oracle.c, OpenMP)"
                                      % (args.steps, VIEWS)},
           "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from gaussiananything_b200 import _lib, raster
    from gaussiananything_b200.gs_surfel import GaussianRenderer2DGS

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"          # the version banner goes to stdout, in front of the one JSON line
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib()
    lib.ga_profile_enable.argtypes = [C.c_int]
    lib.ga_profile_read.argtypes = [C.POINTER(C.c_float), C.c_int]
    lib.ga_profile_read.restype = C.c_int

    g, vs, ps = make_inputs(40 + rank)               # one independent scene per rank
    B, P, V, H, W = 1, P_SURFELS, VIEWS, RES, RES
    g13 = torch.tensor(g, device=dev)[None].contiguous()
    vm = torch.tensor(vs, device=dev).reshape(B * V, 16).contiguous()
    pm = torch.tensor(ps, device=dev).reshape(B * V, 16).contiguous()
    bg = torch.ones(3, device=dev)
    torch.manual_seed(rank)
    d_color = torch.randn(B, V, 3, H, W, device=dev)
    d_allmap = torch.randn(B, V, 7, H, W, device=dev)

    # size the workspace once (like a training loop would), outside the timed region
    _, _, _, st = raster.forward_raw(g13, vm.view(B, V, 4, 4), pm.view(B, V, 4, 4), bg, H, W)
    D = st["num_rendered"]
    max_inst = int(D * 1.25) + 1024
    LIST_K = raster.LIST_K                       # forward+backward workload: the forward records the per-pixel lists
    lib.ga_raster_forward_ex.restype = C.c_int
    L = raster.layout(B, P, V, H, W, max_inst, LIST_K)
    ws = torch.empty(L.total_bytes, device=dev, dtype=torch.uint8)
    color = torch.empty(B, V, 3, H, W, device=dev)
    allmap = torch.empty(B, V, 7, H, W, device=dev)
    radii = torch.empty(B, V, P, device=dev, dtype=torch.int32)
    nscr = lib.ga_raster_backward_scratch_bytes(B, P, V)
    scratch = torch.empty(nscr, device=dev, dtype=torch.uint8)
    grad = torch.empty(B, P, 13, device=dev)
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    p = lambda t: C.c_void_p(t.data_ptr())

    def step_device():
        rc = lib.ga_raster_forward_ex(p(g13), B, P, V, p(vm), p(pm), p(bg), H, W, 1.0, p(color), p(allmap),
                                      p(radii), p(ws), L.total_bytes, max_inst, LIST_K, None, None, stream)
        assert rc == 0, rc
        rc = lib.ga_raster_backward_ex(p(g13), B, P, V, p(vm), p(pm), p(bg), H, W, 1.0, p(radii), p(d_color),
                                       p(d_allmap), p(ws), L.total_bytes, max_inst, LIST_K, p(scratch), nscr, p(grad),
                                       stream)
        assert rc == 0, rc

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput ("value") + per-stage timing (roofline)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)                              # let nvidia-smi start sampling
    for _ in range(max(args.warmup, 3)):
        flush.zero_()
        step_device()
    torch.cuda.synchronize(dev)
    lib.ga_profile_enable(1)
    if rank == 0:
        sampler.mark()
    stage_ms = np.zeros(8)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    wall0 = time.perf_counter()
    for k in range(args.steps):
        flush.zero_()                               # L2 flush, outside the event pair
        ev[k][0].record()
        step_device()
        ev[k][1].record()
        ev[k][1].synchronize()
        buf = (C.c_float * 8)()
        n = lib.ga_profile_read(buf, 8)
        stage_ms[:n] += np.array(buf[:n])
    barrier()
    wall = time.perf_counter() - wall0
    lib.ga_profile_enable(0)
    clocks = sampler.stop() if rank == 0 else None
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    status = ws[L.status:L.status + 64].view(torch.int32).cpu()
    assert int(status[1]) == 0, "workspace overflow inside the timed region"
    assert torch.isfinite(grad).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, color, allmap, radii, grad)
    t = torch.tensor([dev_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())
    value = world * V * args.steps / (dev_ms_max * 1e-3)
    stage_ms /= args.steps

    # ---- end-to-end through the public API with host buffers ("e2e")
    rnd = GaussianRenderer2DGS(RES, 3, {})
    h_g = torch.tensor(g)[None].pin_memory()
    h_vm = torch.tensor(vs)[None].pin_memory()
    h_pm = torch.tensor(ps)[None].pin_memory()
    h_pos = torch.zeros(1, V, 3).pin_memory()
    h_target = torch.rand(1, V, 3, H, W).pin_memory()
    h2d = sum(x.numel() * x.element_size() for x in (h_g, h_vm, h_pm, h_pos, h_target))
    d2h = 4 + P * 13 * 4

    # software-pipelined like a training loop with a prefetching loader: step k's inputs are uploaded on a
    # side stream while step k-1 computes; loss + gradient come back through pinned buffers and are waited
    # for one step later.  Every step still moves h2d / d2h bytes inside the timed region.
    copy_stream = torch.cuda.Stream(dev)
    h_loss = torch.zeros(1).pin_memory()
    h_grad = torch.zeros(1, P, 13).pin_memory()

    def upload():
        with torch.cuda.stream(copy_stream):
            t = [h.to(dev, non_blocking=True) for h in (h_g, h_vm, h_pm, h_pos, h_target)]
            ev_up = torch.cuda.Event()
            ev_up.record(copy_stream)
        return t, ev_up

    state = {"pre": upload(), "done": None}

    def step_e2e():
        (gg, cv, cvp, cp, tgt), ev_up = state["pre"]
        torch.cuda.current_stream(dev).wait_event(ev_up)
        for t_ in (gg, cv, cvp, cp, tgt):
            t_.record_stream(torch.cuda.current_stream(dev))
        state["pre"] = upload()                                   # next step's inputs, overlapped
        gg.requires_grad_(True)
        out = rnd.render(gg, cv, cvp, cp, 0.36)
        loss = ((out["image"] - tgt) ** 2).mean() + 0.1 * out["dist"].mean() + 0.05 * (1 - out["alpha"]).mean() \
            + 0.01 * out["depth"].mean() + 0.01 * out["rend_normal"].abs().mean()
        loss.backward()
        if state["done"] is not None:
            state["done"].synchronize()                           # previous step's results have landed
        h_loss.copy_(loss.detach().reshape(1), non_blocking=True)
        h_grad.copy_(gg.grad, non_blocking=True)
        ev_done = torch.cuda.Event()
        ev_done.record()
        state["done"] = ev_done

    # 50 warm-up steps, then >= 500 steps AND >= 2 s (round 1 timed 20 steps = 29 ms after 3 warm-up steps: one
    # allocator / engine stall made BENCH and SCALE N=1 disagree 24x).  Per-step host times are kept: the mean gives
    # the throughput, the median / p99 / max show whether a stall was inside the window.
    E2E_WARMUP = 50
    for _ in range(E2E_WARMUP):
        step_e2e()
    state["done"].synchronize()
    torch.cuda.synchronize(dev)
    import gc
    gc.collect()
    gc.disable()                                                  # no collector pause inside the window
    barrier()
    e2e_steps, step_s = 0, []
    e0 = time.perf_counter()
    while e2e_steps < max(args.steps, 500) or (time.perf_counter() - e0) < 2.0:
        t_a = time.perf_counter()
        step_e2e()
        step_s.append(time.perf_counter() - t_a)
        e2e_steps += 1
        if e2e_steps >= 20000:
            break
    state["done"].synchronize()
    e_local = time.perf_counter() - e0
    gc.enable()
    assert bool(torch.isfinite(h_loss).all()) and bool(torch.isfinite(h_grad).all())
    barrier()
    # every rank ran for >= 2 s but not the same number of steps: whole-job rate = sum of the per-rank rates
    t = torch.tensor([V * e2e_steps / e_local], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    e2e_value = float(t.item())
    step_s = np.array(step_s)
    e2e_stats = {"steps": e2e_steps, "seconds": e_local, "warmup_steps": E2E_WARMUP,
                 "slow_step_indices": [int(i) for i in np.nonzero(step_s > 5 * np.median(step_s))[0][:12]],
                 "ms_per_step_mean": 1e3 * e_local / e2e_steps, "ms_per_step_median": 1e3 * float(np.median(step_s)),
                 "ms_per_step_p99": 1e3 * float(np.percentile(step_s, 99)), "ms_per_step_max": 1e3 * float(step_s.max()),
                 "steps_over_5x_median": int((step_s > 5 * np.median(step_s)).sum()),
                 "value_from_median": V / float(np.median(step_s)), "numa_pinning": numa}

    c5 = None
    if not args.no_c5:
        try:
            c5 = run_c5_leg(dev, world, rank, with_cascade=not args.no_dit)
        except Exception as ex:
            if world > 1:
                raise                                  # a collective leg that half the ranks abandon would hang the job
            c5 = {"error": repr(ex)}
    if rank == 0:
        hbm, peak_src = measured_peaks()
        HW = H * W
        # algorithmic bytes per launch (DESIGN.md "Kernels"): one launch covers all NV views
        bytes_k3 = 76.0 * D + 40.0 * HW * V
        bytes_k4 = 76.0 * D + 60.0 * HW * V + 72.0 * P * V
        names = ["preprocess", "binning", "render_fwd", "render_bwd", "preprocess_bwd"]
        stages = {n: float(stage_ms[i]) for i, n in enumerate(names)}
        if stages["render_bwd"] >= stages["render_fwd"]:
            dom, dom_bytes = "render_bwd", bytes_k4
        else:
            dom, dom_bytes = "render_fwd", bytes_k3
        achieved = dom_bytes / (stages[dom] * 1e-3) / 1e9
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "traffic.json")        # DRAM bytes per launch from the committed ncu capture
        if os.path.exists(tp):
            tj = json.load(open(tp))
            key = dom + "_kernel"
            if key in tj:
                traffic, traffic_src = tj[key]["dram_bytes"], tj.get("_source")
        step_bytes = V * (52.0 * P + 40.0 * HW) + 76.0 * D + V * (60.0 * HW + 104.0 * P) + 76.0 * D
        # FP32-issue view of the forward composite (SURVEY 8d): dense-equivalent pair evaluations = sum over tiles of
        # (instances in the tile x 256 pixels), ~50 flop each, against 148 SMs x 128 lanes x 2 x 1.965 GHz
        ts = ws[L.tile_start:L.tile_start + 4 * (V * ((H + 15) // 16) * ((W + 15) // 16) + 1)].view(torch.int32).cpu().numpy().astype(np.int64)
        evals = float((ts[1:] - ts[:-1]).sum() * 256)
        fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12
        fp32 = {"kernel": "render_fwd", "dense_pair_evals": evals, "flop_per_eval": 50,
                "achieved_tflops_dense_equivalent": evals * 50 / (stages["render_fwd"] * 1e-3) / 1e12, "peak_tflops": fp32_peak,
                "frac_dense_equivalent": evals * 50 / (stages["render_fwd"] * 1e-3) / 1e12 / fp32_peak,
                "note": "culling skips most of these pairs; the figure says how far the kernel is from brute force at FP32 peak"}
        cpu_v, cpu_n, cpu_dt = cpu_views_per_s(2, 10.0) if world == 1 else (None, 0, 0.0)
        dit_leg = None
        if world == 1 and not args.no_dit:
            try:
                dit_leg = run_dit_leg(dev)
                pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
                tpk = float(pk.get("bf16_tflops", 1590.0))
                for kk in dit_leg["kernels"].values():
                    kk["frac_of_bf16_peak"] = kk["tflops"] / tpk
                dit_leg["tensor_peak_tflops"] = tpk
                dit_leg["frac_of_bf16_peak_sustained"] = dit_leg["tflops"] / float(pk.get("bf16_tflops_sustained", 1400.0))
                dit_leg["deployed_L_N768"] = run_dit_deployed_leg(dev)
                dit_leg["C4_L_N4096"] = run_dit_deployed_leg(dev, nfe=10, N=4096)
                # samples/s is a throughput metric: 4 samples denoised together fill the 148 SMs far better than one
                # (M = 6144 rows instead of 1536: the D->D GEMMs go from 96 to 384 tiles)
                dit_leg["deployed_L_N768_4samples"] = run_dit_deployed_leg(dev, nfe=10, N=768, samples=4)
                try:
                    dit_leg["vae_decoder_N1"] = run_vae_decoder_leg(dev)
                except Exception as ex:                  # never let the newest leg take the DiT numbers down with it
                    dit_leg["vae_decoder_N1"] = {"error": repr(ex)}
            except Exception as ex:                      # the raster metric is the headline; report, do not hide
                dit_leg = {"error": repr(ex)}
        standin = None
        if world == 1 and not args.no_dit:
            try:
                standin = run_gpu_standin(dev)
                standin["speedup_raster_C2_vs_standin"] = value / standin["raster_C2"]["views_per_s"]
                if isinstance(dit_leg, dict) and "ms_per_nfe" in dit_leg:
                    a = standin["dit_C3_B_N2048"]
                    best = min(v for k, v in a.items() if k.endswith("ms_per_nfe"))
                    standin["speedup_C3_vs_best_standin"] = best / dit_leg["ms_per_nfe"]
                    b = standin["dit_deployed_L_N768"]
                    best = min(v for k, v in b.items() if k.endswith("ms_per_nfe"))
                    standin["speedup_deployed_L_vs_best_standin"] = best / dit_leg["deployed_L_N768"]["DiT-PixArt-PCD-CLAY-L"]["ms_per_nfe"]
            except Exception as ex:
                standin = {"error": repr(ex)}
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": dev_ms_max / args.steps,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
               "data": "synthetic", "config": CONFIG, "instances_D": D,
               "wall_s_timed_region": wall, "stage_ms": stages,
               "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": hbm, "unit": "GB/s",
                            "frac": achieved / hbm, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                            "algorithmic_bytes_per_launch": dom_bytes,
                            # what the hardware actually moved (ncu dram__bytes of the stage's kernels, profiles/traffic.json)
                            # over the live stage time: round 2's backward trades bytes (per-pixel lists, record slices)
                            # for instructions, so it moves ~4.6x the algorithmic bytes on purpose
                            "traffic_GBs": (traffic / (stages[dom] * 1e-3) / 1e9) if traffic else None,
                            "traffic_frac": (traffic / (stages[dom] * 1e-3) / 1e9 / hbm) if traffic else None,
                            "whole_step_algorithmic_GBs": step_bytes / (dev_ms_max / args.steps * 1e-3) / 1e9,
                            "whole_step_frac": step_bytes / (dev_ms_max / args.steps * 1e-3) / 1e9 / hbm, "fp32": fp32},
               "cpu_baseline": ({"value": cpu_v, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                                 "sample": "%d views fwd+bwd of the same 100k/512^2 scene in %.1f s "
                                           "(oracle/surfel_oracle.c, OpenMP)" % (cpu_n, cpu_dt)}
                                if world == 1 else None),
               "e2e": dict({"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                           **e2e_stats),
               "gpu_launches": LAUNCHES_PER_STEP * args.steps, "clocks": clocks, "dit": dit_leg, "c5": c5,
               "gpu_standin": standin}
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()



# ---------------------------------------------------------------------------
# DiT leg (BASELINE.json configs[2]: DiT-B point-latent, N=2048, 50-point Euler grid = 49 NFE, CFG, bf16)
# reported as the secondary object "dit" of the JSON line
# ---------------------------------------------------------------------------
def dit_flops_per_forward(L, N, D, M, Dc):
    """SURVEY.md 8(d): 2*L*(14 N D^2 + 2 M Dc D + 2 N M D + 2 N^2 D) per sample-forward."""
    return 2.0 * L * (14.0 * N * D * D + 2.0 * M * Dc * D + 2.0 * N * M * D + 2.0 * N * N * D)


def run_dit_leg(dev, steps_grid=50, reps=3):
    import torch
    from gaussiananything_b200 import dit, transport as tr
    torch.manual_seed(0)
    L, D, H, N, M, Dc, Cin = 12, 768, 12, 2048, 1369, 1024, 3
    m = dit.DiT_models["DiT-PixArt-PCD-CLAY-B"](input_size=32, num_classes=0, learn_sigma=False, in_channels=Cin,
                                                context_dim=Dc, roll_out=True, pooling_ctx_dim=768)
    m.randomize_zero_init_().to(dev).eval()
    B = 2                                              # one sample, CFG doubles the batch
    h_z = torch.randn(1, N, Cin).pin_memory()
    h_ctx = torch.randn(1, M, Dc).pin_memory()
    h_vec = torch.randn(1, Dc).pin_memory()
    sampler = tr.Sampler(tr.create_transport("GVP", "velocity", None, None, None, "lognorm"))
    fn = sampler.sample_ode(sampling_method="euler", num_steps=steps_grid)

    def sample_e2e():
        z = h_z.to(dev, non_blocking=True)
        c, v = h_ctx.to(dev, non_blocking=True), h_vec.to(dev, non_blocking=True)
        ctx = {"img_crossattn": torch.cat([c, torch.zeros_like(c)], 0), "img_vector": torch.cat([v, torch.zeros_like(v)], 0)}
        out = fn(torch.cat([z, z], 0), m.forward_with_cfg, context=ctx, cfg_scale=4.0)[-1]
        return out[:1].cpu()

    sample_e2e()                                       # warm-up: weight pack, K/V cache, graph capture
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for _ in range(reps):
        r = sample_e2e()
    e2e_s = (time.perf_counter() - t0) / reps
    assert torch.isfinite(r).all()
    # device-resident: NFE loop only
    z = torch.randn(B, N, Cin, device=dev)
    c = torch.randn(B, M, Dc, device=dev)
    ctx = {"img_crossattn": c, "img_vector": torch.randn(B, Dc, device=dev)}
    tt = torch.full((B,), 0.3, device=dev)
    for _ in range(3):
        m.forward_with_cfg(z, tt, ctx, 4.0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nfe = steps_grid - 1
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(nfe):
        m.forward_with_cfg(z, tt, ctx, 4.0)
    e1.record()
    e1.synchronize()
    dev_s = e0.elapsed_time(e1) * 1e-3
    flops_nfe = 2 * dit_flops_per_forward(L, N, D, M, Dc)          # x2: CFG batch
    flops_nfe_cached = flops_nfe - 2 * 2.0 * L * 2.0 * M * Dc * D   # context K/V cached across NFEs (SURVEY F11)
    # isolated kernels: self-attention and the widest GEMM at this shape
    import ctypes as C
    Lb = dit._bind()
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    eng = m._engine
    s = eng.s

    def time_kernel(launch, n=20):
        for _ in range(3):
            launch()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            launch()
        b.record()
        b.synchronize()
        return a.elapsed_time(b) * 1e-3 / n

    t_attn = time_kernel(lambda: Lb.ga_attention_bf16(dit._p(s["q"]), dit._p(s["k"]), dit._p(s["vt"]), dit._p(s["ao"]), B, H, N, N,
                                                      eng.Np, eng.Np, 0.125, eng.wb[0]["sa_bound"], st))
    wb = eng.wb[0]
    epi = eng._epi(dit.EPI_GELU_BF16, bias=wb["b1"], out=s["hid"], ld_out=4 * D)
    t_gemm = time_kernel(lambda: Lb.ga_gemm_bf16_tn(dit._p(s["h"]), D, dit._p(wb["w1"]), D, B * N, 4 * D, D, C.byref(epi), 128, st))
    fl_attn = 4.0 * N * N * 64 * B * H
    fl_gemm = 2.0 * B * N * 4 * D * D
    return {"config": "C3: DiT-PixArt-PCD-CLAY-B (L12 D768 H12), N=2048, M=1369, %d-point Euler grid (%d NFE), CFG 4.0, bf16" % (steps_grid, nfe),
            "samples_per_s": 1.0 / dev_s, "ms_per_nfe": 1e3 * dev_s / nfe,
            "tflops": flops_nfe * nfe / dev_s / 1e12, "tflops_excluding_cached_ctx_kv": flops_nfe_cached * nfe / dev_s / 1e12,
            "e2e_samples_per_s": 1.0 / e2e_s, "launches_per_nfe": eng.launches_per_forward + 1,
            "kernels": {"self_attention": {"ms": 1e3 * t_attn, "tflops": fl_attn / t_attn / 1e12},
                        "gemm_mlp1_gelu": {"ms": 1e3 * t_gemm, "tflops": fl_gemm / t_gemm / 1e12}}}


def run_vae_decoder_leg(dev, reps=5):
    """SURVEY 8f row N1 at the deployed size: 768 latent tokens -> 73 728 surfels per sample (post_quant_conv, DiT2-B,
    conv_sr, three cascaded up-samplers), random weights, batch 2.  Device time per sample and achieved TFLOP/s."""
    import torch
    from gaussiananything_b200.vae_decoder import SurfelDecoder, random_state_dict, decode_flops
    dec = SurfelDecoder(random_state_dict(768, 12, 10, seed=0), 12, 12, device=dev)
    B = 2
    lat = torch.randn(B, 768, 10, device=dev)
    xyz = (torch.rand(B, 768, 3, device=dev) - 0.5) * 0.8
    for _ in range(2):
        out = dec.decode(lat, xyz)
    assert torch.isfinite(out["gaussians_upsampled_3"]).all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(reps):
        dec.decode(lat, xyz)
    e1.record()
    e1.synchronize()
    ms = e0.elapsed_time(e1) / reps / B
    # latency of one sample alone (the C5 path decodes one sample per rank)
    for _ in range(2):
        dec.decode(lat[:1], xyz[:1])
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(reps):
        dec.decode(lat[:1], xyz[:1])
    e1.record()
    e1.synchronize()
    ms1 = e0.elapsed_time(e1) / reps
    return {"config": "N1: VAE decoder, 768 tokens x 768, DiT2-B + cascade 8*4*3 -> 73728 surfels/sample, batch 2, bf16",
            "ms_per_sample": ms, "samples_per_s": 1e3 / ms, "tflops": decode_flops(768, 12) / (ms * 1e-3) / 1e12,
            "ms_batch1": ms1, "cuda_graph": bool(dec.use_graph), "surfels_per_sample": 73728}


def run_dit_deployed_leg(dev, nfe=20, N=768, samples=1):
    """DiT-PixArt-PCD-CLAY-L (stage 1, C=3) and ...-stage2-L (C=10 + xyz PE), L24 D1024 H16, M=1369 DINO tokens, CFG
    batch 2, at N latent points: N=768 is the deployed size (SURVEY F3-F4), N=4096 is BASELINE configs[3] (C4).
    Reports ms per NFE of each stage and the DiT part of the cascade at the reference's 250-point grids
    (2 x 249 NFE) derived from it."""
    import torch
    from gaussiananything_b200 import dit
    torch.manual_seed(0)
    M, Dc, B = 1369, 1024, 2 * samples            # CFG doubles the batch: `samples` samples denoised together
    out = {}
    for name, cin, stage2 in (("DiT-PixArt-PCD-CLAY-L", 3, False), ("DiT-PixArt-PCD-CLAY-stage2-L", 10, True)):
        m = dit.DiT_models[name](input_size=32, num_classes=0, learn_sigma=False, in_channels=cin, context_dim=Dc,
                                 roll_out=True, pooling_ctx_dim=768)
        m.randomize_zero_init_().to(dev).eval()
        z = torch.randn(B, N, cin, device=dev)
        ctx = {"img_crossattn": torch.randn(B, M, Dc, device=dev), "img_vector": torch.randn(B, Dc, device=dev)}
        if stage2:
            ctx["fps-xyz"] = torch.rand(B, N, 3, device=dev) * 2 - 1
        tt = torch.full((B,), 0.4, device=dev)
        for _ in range(3):
            y = m.forward_with_cfg(z, tt, ctx, 4.0)
        assert torch.isfinite(y).all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(nfe):
            m.forward_with_cfg(z, tt, ctx, 4.0)
        e1.record()
        e1.synchronize()
        ms = e0.elapsed_time(e1) / nfe
        fl = 2 * samples * dit_flops_per_forward(24, N, 1024, M, Dc)
        out[name] = {"ms_per_nfe": ms, "tflops": fl / (ms * 1e-3) / 1e12}
        del m
        torch.cuda.empty_cache()
    tot = 249 * (out["DiT-PixArt-PCD-CLAY-L"]["ms_per_nfe"] + out["DiT-PixArt-PCD-CLAY-stage2-L"]["ms_per_nfe"]) * 1e-3
    out["samples_in_batch"] = samples
    out["derived_cascade_dit_seconds_per_batch_2x249_nfe"] = tot
    out["derived_dit_only_samples_per_s"] = samples / tot
    out["note"] = "DiT stages only (no DINOv2 conditioner, VAE decode or rendering: SURVEY 8f rows N1-N3 are not built yet)"
    return out


# ---------------------------------------------------------------------------
# C5 leg (BASELINE.json configs[4], SURVEY 8e): the cascade's multi-GPU data path, one sample per rank:
#   [DiT-L stage 1 -> stage 2 sampling] -> VAE decode (73 728 surfels) -> ONE NCCL all-gather of the decoded
#   surfels -> every rank renders its interleaved share of all (sample, view) pairs (8 views of 512^2 per sample).
# Reference hand-off being replaced: nsr/lsgm/flow_matching_trainer.py:1399-1424,1545-1567 (decode once, then a
# per-camera render loop on one GPU; scripts/gradio_app_cascaded.py:96-100 pins world size 1).
# ---------------------------------------------------------------------------
C5_VIEWS, C5_RES, C5_TOKENS = 8, 512, 768


def run_c5_leg(dev, world, rank, steps=20, cascade_samples=2, with_cascade=True):
    import torch
    import torch.distributed as dist
    from gaussiananything_b200 import dit, sharding, transport as tr
    from gaussiananything_b200.gs_surfel import GaussianRenderer2DGS
    from gaussiananything_b200.vae_decoder import SurfelDecoder, random_state_dict
    from tests.helpers import cameras
    torch.manual_seed(100 + rank)
    dec = SurfelDecoder(random_state_dict(768, 12, 10, seed=0), 12, 12, device=dev)
    rnd = GaussianRenderer2DGS(C5_RES, 3, {})
    S, V = world, C5_VIEWS
    vs, ps, cs, tf = cameras(S * V)
    cv = torch.tensor(vs, device=dev).reshape(S, V, 4, 4)
    cp = torch.tensor(ps, device=dev).reshape(S, V, 4, 4)
    pos = torch.tensor(cs, device=dev).reshape(S, V, 3)
    lat = torch.randn(1, C5_TOKENS, 10, device=dev)
    xyz = (torch.rand(1, C5_TOKENS, 3, device=dev) - 0.5) * 0.8

    def sync_max(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    ev = lambda: torch.cuda.Event(enable_timing=True)

    def decode_gather_render(latent, points):
        e = [ev() for _ in range(4)]
        e[0].record()
        surf = dec.decode(latent, points)["gaussians_upsampled_3"]            # [1, 73728, 13], the all-gather send buffer
        e[1].record()
        allg = sharding.all_gather_surfels(surf)                               # the path's only collective
        e[2].record()
        out = _render_owned(allg)
        e[3].record()
        return e, out, surf

    def _render_owned(allg):
        # surfels are already gathered: render this rank's pairs (render_sharded's body after its all-gather)
        by = sharding.group_pairs_by_sample(sharding.shard_pairs(S, V, world, rank))
        samples = list(by)
        nv = {len(v) for v in by.values()}
        assert len(nv) == 1
        bi = torch.tensor(samples, device=dev)
        vi = torch.tensor([by[b] for b in samples], device=dev)
        rows = bi[:, None].expand(-1, vi.shape[1])
        return rnd.render(allg[bi], cv[rows, vi], cp[rows, vi], pos[rows, vi], tf)

    with torch.no_grad():
        for _ in range(3):
            decode_gather_render(lat, xyz)
        barrier()
        recs = []
        w0 = ev(); w1 = ev()
        w0.record()
        for _ in range(steps):
            recs.append(decode_gather_render(lat, xyz)[0])
        w1.record()
        w1.synchronize()
        barrier()
    total_ms = sync_max(w0.elapsed_time(w1))
    dec_ms = float(np.mean([r[0].elapsed_time(r[1]) for r in recs]))
    ag_ms = float(np.mean([r[1].elapsed_time(r[2]) for r in recs]))
    ren_ms = float(np.mean([r[2].elapsed_time(r[3]) for r in recs]))
    P = 73728
    out = {"config": "C5 data path: per rank 1 sample: VAE decode (768 tokens -> 73728 surfels) -> NCCL all-gather of "
                     "[1,73728,13] f32 per rank -> render this rank's share of %d samples x %d views of %d^2 (forward)"
                     % (S, V, C5_RES),
           "n_gpus": world, "steps": steps, "views_per_step": S * V,
           "views_per_s": S * V * steps / (total_ms * 1e-3), "samples_per_s_decode_gather_render": S * steps / (total_ms * 1e-3),
           "ms_per_step": total_ms / steps,
           "stage_ms_rank0": {"vae_decode": dec_ms, "all_gather": ag_ms, "render_shard": ren_ms},
           "collective": {"op": "ncclAllGather (torch.distributed all_gather_into_tensor)" if world > 1 else "none (world 1)",
                          "bytes_per_rank": P * 13 * 4, "bytes_total": world * P * 13 * 4,
                          "us_max_over_ranks": 1e3 * sync_max(ag_ms),
                          "algbw_GBs": (world * P * 13 * 4 / 1e9) / (ag_ms * 1e-3) if world > 1 and ag_ms > 0 else None}}
    if with_cascade:
        # the whole cascade per sample (minus the DINOv2 conditioner, row N3): 2 x 249 Euler NFE with CFG on random-init
        # DiT-L weights at the deployed N = 768, then decode / gather / render as above
        M, Dc = 1369, 1024
        mk = lambda name, cin: dit.DiT_models[name](input_size=32, num_classes=0, learn_sigma=False, in_channels=cin,
                                                    context_dim=Dc, roll_out=True, pooling_ctx_dim=768).randomize_zero_init_().to(dev).eval()
        m1, m2 = mk("DiT-PixArt-PCD-CLAY-L", 3), mk("DiT-PixArt-PCD-CLAY-stage2-L", 10)
        sampler = tr.Sampler(tr.create_transport("GVP", "velocity", None, None, None, "lognorm"))
        fn = sampler.sample_ode(sampling_method="euler", num_steps=250)
        h_ctx, h_vec = torch.randn(1, M, Dc).pin_memory(), torch.randn(1, Dc).pin_memory()

        def one_sample(dedup):
            c, v = h_ctx.to(dev, non_blocking=True), h_vec.to(dev, non_blocking=True)
            ctx1 = {"img_crossattn": torch.cat([c, torch.zeros_like(c)], 0), "img_vector": torch.cat([v, torch.zeros_like(v)], 0)}
            z = torch.randn(1, C5_TOKENS, 3, device=dev)
            pts = fn(torch.cat([z, z], 0), m1.forward_with_cfg, context=ctx1, cfg_scale=4.0)[-1][:1]
            pts = (pts * 0.164).clamp(-0.45, 0.45)                               # stage-1 un-normalisation (flow_matching_trainer.py:987)
            fps = torch.cat([pts, pts], 0) / 0.45
            ctx2 = {"img_crossattn": torch.cat([c, c], 0), "img_vector": torch.cat([v, v], 0), "fps-xyz": fps}   # uc == c (SURVEY F13)
            m2.cfg_dedup = dedup
            z2 = torch.randn(1, C5_TOKENS, 10, device=dev)
            latent = fn(torch.cat([z2, z2], 0), m2.forward_with_cfg, context=ctx2, cfg_scale=4.0)[-1][:1]
            e, o, surf = decode_gather_render(latent, pts)
            return o

        res = {}
        with torch.no_grad():
            for tag, dedup in (("reference_cfg_2B_both_stages", False), ("stage2_cfg_dedup_opt_in", True)):
                one_sample(dedup)                                                # warm-up: packs, K/V, graphs
                barrier()
                t0 = time.perf_counter()
                for _ in range(cascade_samples):
                    o = one_sample(dedup)
                h_img = o["image"][:, :1, :, :8, :8].cpu()                           # a device->host read ends each timed window
                torch.cuda.synchronize(dev)
                dt = sync_max(time.perf_counter() - t0)
                barrier()
                res[tag] = {"seconds_per_sample_per_gpu": dt / cascade_samples, "samples_per_s": world * cascade_samples / dt}
        out["cascade"] = dict(res, config="DiT-PixArt-PCD-CLAY-L + ...-stage2-L (L24 D1024 H16), N=768, M=1369, 250-point Euler "
                              "grids (2 x 249 NFE), CFG 4.0, bf16 -> VAE decode -> all-gather -> %d views of %d^2; no DINOv2 "
                              "conditioner (SURVEY 8f N3 not built): context tokens are synthetic" % (V, C5_RES),
                              samples_per_step=world)
        del m1, m2
        torch.cuda.empty_cache()
    return out


def run_raster_standin(dev, steps=20):
    """The upstream rasteriser flow restated literally (baseline/raster_standin.cu): per-view launch sets with a
    device->host read of num_rendered each, cub radix sort of the whole instance list, every pixel evaluates every
    staged surfel, one atomicAdd per (pixel, surfel, gradient component).  Same C2 inputs as the headline."""
    import torch
    from baseline.raster_standin import StandinRasterizer
    g, vs, ps = make_inputs(40)
    r = StandinRasterizer(P_SURFELS, RES, RES, VIEWS, device=dev)
    g13 = torch.tensor(g, device=dev)
    vm, pm = torch.tensor(vs, device=dev), torch.tensor(ps, device=dev)
    bg = torch.ones(3, device=dev)
    torch.manual_seed(0)
    dc, da = torch.randn(VIEWS, 3, RES, RES, device=dev), torch.randn(VIEWS, 7, RES, RES, device=dev)
    flush = torch.empty(256 << 20, device=dev, dtype=torch.uint8)
    for _ in range(3):
        r.forward(g13, vm, pm, bg)
        grad = r.backward(dc, da)
    assert torch.isfinite(grad).all()
    tot = 0.0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(steps):
        flush.zero_()
        e0.record()
        r.forward(g13, vm, pm, bg)
        r.backward(dc, da)
        e1.record()
        e1.synchronize()
        tot += e0.elapsed_time(e1)
    ms = tot / steps
    return {"what": "reference-algorithm GPU baseline: per-view launches + num_rendered read-back, global cub radix sort, "
                    "dense per-tile evaluation, per-pair atomics (baseline/raster_standin.cu)",
            "ms_per_step": ms, "views_per_s": VIEWS / (ms * 1e-3)}


def run_gpu_standin(dev):
    """GPU comparison baselines on the same B200 (baseline/gpu_standin.py; BASELINE.md section 4)."""
    from baseline import gpu_standin as gs
    out = {"what": "unfused PyTorch-CUDA restatement of the reference's DiT block stack: nn.Linear under bf16 autocast (cuBLAS) + "
                   "flash_attn_func + separate norm/modulate/GELU kernels, context K/V re-projected every block, 2B CFG forward"}
    out["raster_C2"] = run_raster_standin(dev)
    out["dit_C3_B_N2048"] = gs.time_torch_dit(dev, 12, 768, 12, 2048, nfe=20)
    out["dit_deployed_L_N768"] = gs.time_torch_dit(dev, 24, 1024, 16, 768, nfe=20)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-dit", action="store_true", help="skip the secondary DiT sampling legs (DiT, cascade, stand-ins)")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 decode -> all-gather -> render leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's outputs of the last timed raster step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
