#!/usr/bin/env python
"""bench.py -- SoftRas forward+backward throughput on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c3|c2|tiny] [--dump-outputs DIR]
    (N>1: python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...)

Workload (default "c3", BASELINE.json configs[2] / the README's 39k-face row): UV sphere with
39 200 faces at 1024x1024, T=1 surface textures, renderer defaults (sigma 1e-5, gamma 1e-4,
euclidean / softmax / prod, K=16), 4 images per GPU -- B=32 at 8 GPUs, weak scaling.  One
"step" = one forward + one top-K backward over the rank's 4 images.

Prints ONE JSON line (rank 0).  `value` = frames/s over all ranks with inputs resident in
HBM; `e2e` = same through the public API with pinned HOST inputs, H2D/D2H inside the timed
region; `roofline` = the dominant kernel against the measured HBM peak; `cpu_baseline` =
the CPU oracle (restatement of the reference kernels; the reference has no CPU path,
SURVEY.md F1) on this box's host cores on a bounded sample.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree may be read-only; nothing is written into it

METRIC = "softras_fwd_bwd_frames_per_s_1024px_39k_faces"
WORKLOADS = {
    # name: (num_faces, image_size, images_per_gpu, description)
    "c3": (39200, 1024, 4, "C3: SoftRas fwd+bwd 1024x1024, UV sphere 39200 faces, 4 images/GPU (B=32 at 8 GPUs)"),
    "c2": (3280, 1024, 8, "C2: SoftRas fwd+bwd 1024x1024, UV sphere 3280 faces, 8 images/GPU"),
    "tiny": (280, 256, 2, "tiny: SoftRas fwd+bwd 256x256, UV sphere 280 faces, 2 images/GPU (smoke only)"),
    # BASELINE.json configs[3]: NMR (dr_type='n3mr') fwd+bwd, fill_back doubles the faces, texture_size 2
    # BASELINE.json configs[4]: demo2-deform silhouette fitting (reference demo2-deform.py: 120 views, Adam, IoU +
    # Laplacian + flatten losses) at 512^2; one "step" = one optimisation iteration over all views
    "c5": (3280, 512, 120, "C5: demo2-deform geometry optimisation loop, 3280-face sphere -> ellipsoid silhouettes, 512x512, 120 views/iteration"),
    "c4": (39200, 1024, 16, "C4: NMR (n3mr) fwd+bwd 1024x1024, UV sphere 39200 faces (78400 with fill_back), ts=2, 16 images/GPU"),
    # BASELINE.json configs[0] as demo1-render.py runs it: spot cow (5856 faces), texture_res 5 (T=25) baked from spot_texture.png,
    # 256x256, one view per render, forward only, image read back to the host
    "c1": (5856, 256, 1, "C1: demo1-render, spot cow 5856 faces, T=25 baked textures, 256x256, 1 view per render (forward + D2H)"),
}
ASSETS = os.path.join(ROOT, "baseline", "_ref", "assets", "data")   # staged by tools/stage_assets.py where /root/reference exists
README_39K_MS = 35.5  # BASELINE.md section 1: Jrender SoftRas 39k faces, 1024^2, hardware/batch unstated


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip the reference-CUDA-kernels-on-this-GPU leg")
    ap.add_argument("--option", action="append", default=[], metavar="NAME=VALUE",
                    help="b200r_set_option() knob for A/B runs, e.g. --option softras_exact_tail=1")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU-baseline sample time")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy")
    return ap.parse_args()


DUMP_SAMPLE = 1 << 22   # elements kept of a larger output: at most 16 MiB of float32 per array, 64 MiB for four arrays


def dump_outputs(out_dir, arrays):
    """Writes each output as out_dir/<name>.npy (float32).  An output with more than DUMP_SAMPLE elements is replaced by
    the elements at a fixed seeded sample of flat positions, so that two builds can be compared value for value."""
    assert len(arrays) <= 4
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float32)
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def build_inputs(workload, rank, world):
    from jrender_b200 import workloads as wl
    nf, H, bpg, _ = WORKLOADS[workload]
    total = bpg * world
    # global batch index -> azimuth 360*b/B (BASELINE.md section 3); this rank owns [rank*bpg, (rank+1)*bpg)
    fv_all, tex_all = wl.make_scene(nf, batch=total)
    sl = slice(rank * bpg, (rank + 1) * bpg)
    rng = np.random.default_rng(2 + rank)
    grad = rng.uniform(-1.0, 1.0, (bpg, 4, H, H)).astype(np.float32)
    return np.ascontiguousarray(fv_all[sl]), np.ascontiguousarray(tex_all[sl]), grad


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampler running DURING the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()  # exact PID we started
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- baselines (subprocesses)
def workload_config(workload, world):
    """The `config` object, identical in both arms (the driver compares them key by key)."""
    nf, H, bpg, desc = WORKLOADS[workload]
    return {"workload": desc, "images_per_gpu": bpg, "global_batch": bpg * world, "faces": nf, "image_size": H,
            "params": "T=1 sigma=1e-5 gamma=1e-4 euclidean/softmax/prod K=16 near=1 far=100 fill_back",
            "parallelism": "batch-sharded dp%d, no data-path collective" % world,
            "l2": "256 MiB buffer written between timed steps (outside the event pairs)",
            "baseline_note": "vs_baseline = value / (1000/35.5 ms): README.md:69, GPU and batch unstated"}


def _run_json(cmd, timeout):
    """Runs a baseline helper under oracle/ as a subprocess and parses the JSON object it prints."""
    env = dict(os.environ)
    for k in ("OMP_NUM_THREADS", "OMP_PROC_BIND", "OMP_PLACES"):   # torchrun exports OMP_NUM_THREADS=1
        env.pop(k, None)
    env["PYTHONDONTWRITEBYTECODE"] = "1"
    try:
        r = subprocess.run([sys.executable] + cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
        for line in reversed(r.stdout.strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line)
        return {"unavailable": "no JSON from %s (rc %d): %s" % (cmd[0], r.returncode, r.stderr.strip()[-300:])}
    except Exception as e:
        return {"unavailable": "%s: %s" % (type(e).__name__, e)}


def cpu_oracle(workload, step_seconds, steps=1, warmup=0, one_thread_seconds=4.0):
    """CPU oracle fwd+bwd on this box's host cores, pinned one thread per physical core (oracle/cpu_bench.py)."""
    nf, H, _, _ = WORKLOADS[workload]
    budget = 120 + (steps + warmup + 3) * max(step_seconds, 40.0)
    return _run_json([os.path.join("oracle", "cpu_bench.py"), "--faces", str(nf), "--image-size", str(H), "--steps", str(steps),
                      "--warmup", str(warmup), "--step-seconds", str(step_seconds), "--one-thread-seconds", str(one_thread_seconds)],
                     timeout=budget)


def cpu_baseline_object(r):
    if "unavailable" in r:
        return {"value": None, "unit": "frames/s", "cores": 0, "kind": "port", "sample": r["unavailable"]}
    o = {"value": r["frames_per_s"], "unit": "frames/s", "cores": r["threads"], "kind": "port",
         "sample": "oracle fwd+bwd: %s; %d OpenMP threads (%s)" % (r["sample"], r["threads"], r["binding"]),
         "cpu_model": r["cpu_model"], "logical_cpus": r["logical_cpus_in_mask"], "fwd_s_per_image": r["fwd_s"], "bwd_s_per_image": r["bwd_s"]}
    if "one_thread" in r:
        o["one_thread_value"] = r["one_thread"]["frames_per_s"]
        o["one_thread_note"] = r["one_thread"]["note"]
    return o


# --------------------------------------------------------------------------- reference arm
def run_reference(args, rank, world):
    """The reference has no CPU implementation (every op is CUDA-only, SURVEY.md F1) and Jittor is
    not installable here, so this arm times the CPU restatement of the reference kernels
    (oracle/, kind "port") on rank 0, one OpenMP thread per physical core.  One STEP = forward + backward of ONE
    image of the workload (a bounded sample when a whole image does not fit the per-step budget); `value` is
    images/s, `ms_per_step` the wall time each step actually took."""
    if rank != 0:
        return
    total_steps = args.steps + args.warmup
    target = max(0.5, min(15.0, 150.0 / max(1, total_steps)))
    r = cpu_oracle(args.workload, target, steps=args.steps, warmup=args.warmup, one_thread_seconds=0.0)
    if "unavailable" in r:
        print(json.dumps({"impl": "reference", "unavailable": r["unavailable"]}), flush=True)
        return
    v = r["frames_per_s"]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * float(np.mean(r["step_wall_s"])), "frames_per_step": 1,
        "higher_is_better": True, "scaling": "weak",
        "vs_baseline": v / (1000.0 / README_39K_MS) if args.workload == "c3" else None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, args.gpus),
        "note": "CPU restatement of the reference CUDA kernels (the reference ships no CPU path); one step = one image "
                "(or a bounded row sample of it); value = 1 / extrapolated seconds per whole image",
        "cpu_baseline": cpu_baseline_object(r),
        "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- our arm
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from jrender_b200 import SoftRasterizeFunction, _lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    L = _lib.lib()
    nf, H, bpg, desc = WORKLOADS[args.workload]
    fv_h, tex_h, grad_h = build_inputs(args.workload, rank, world)
    fv = torch.from_numpy(fv_h).to(dev).requires_grad_(True)
    tex = torch.from_numpy(tex_h).to(dev).requires_grad_(True)
    grad = torch.from_numpy(grad_h).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2

    def step():
        fv.grad = None
        tex.grad = None
        img = SoftRasterizeFunction(image_size=H)(fv, tex)
        img.backward(grad)
        return img

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    warmup = max(3, args.warmup)
    for _ in range(warmup):
        step()
    barrier()

    sampler = ClockSampler(local_rank if "CUDA_VISIBLE_DEVICES" not in os.environ else
                           os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank])
    if rank == 0:
        sampler.start()
    launches0 = L.b200r_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    for a, b in ev:
        flush.fill_(1.0)          # L2 flush between timed iterations (outside the event pair)
        a.record()
        img = step()
        b.record()
    barrier()
    launches = L.b200r_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    step_ms = [a.elapsed_time(b) for a, b in ev]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"soft_colors": img.detach().cpu().numpy(), "grad_face_vertices": fv.grad.cpu().numpy(),
                                         "grad_textures": tex.grad.cpu().numpy()})
    del img
    t_rank = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_rank, op=dist.ReduceOp.MAX)
    total_ms = float(t_rank.item())
    frames = bpg * world * args.steps
    value = frames / (total_ms / 1000.0)

    # ---- per-kernel device times (library event profiler, separate un-timed steps)
    import ctypes as C
    L.b200r_profile_reset()
    L.b200r_profile_enable(1)
    nprof = 5
    for _ in range(nprof):
        flush.fill_(1.0)
        step()
    torch.cuda.synchronize(dev)
    L.b200r_profile_enable(0)
    kern = {}
    for kid, name in [(0, "k_face_setup"), (1, "k_coarse_bin"), (4, "k_tile_order"), (2, "k_softras_forward"),
                      (3, "k_softras_backward"), (9, "k_softras_bwd_finalize")]:
        ms, n = C.c_double(0), C.c_longlong(0)
        L.b200r_profile_read(kid, C.byref(ms), C.byref(n))
        kern[name] = {"avg_ms": ms.value / max(1, n.value), "launches_per_step": n.value / nprof}

    # ---- end-to-end through the public API with pinned host buffers
    fv_p = torch.from_numpy(fv_h).pin_memory()
    tex_p = torch.from_numpy(tex_h).pin_memory()
    gf_p = torch.empty_like(fv_p).pin_memory()
    gt_p = torch.empty_like(tex_p).pin_memory()
    target = torch.zeros((bpg, 4, H, H), dtype=torch.float32, device=dev)

    # Software pipeline over three streams, as a training loop would run it: the H2D copy of step
    # i+1 (copy stream) and the D2H copy of step i-1's gradients and loss (second copy stream)
    # overlap the raster kernels of step i.  Every step's copies are inside the timed region;
    # the host blocks once at the end, when the last step's results have landed in pinned memory.
    s_in, s_out, s_main = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.current_stream(dev)
    d_fv = [torch.empty_like(fv_p, device=dev) for _ in range(2)]
    d_tex = [torch.empty_like(tex_p, device=dev) for _ in range(2)]
    loss_p = torch.zeros(64, dtype=torch.float32).pin_memory()
    ev_in = [torch.cuda.Event() for _ in range(2)]      # inputs of slot landed on the device
    ev_free = [torch.cuda.Event() for _ in range(2)]    # compute of the step that used the slot is done
    ev_done = [torch.cuda.Event() for _ in range(2)]
    ev_out = [torch.cuda.Event() for _ in range(2)]     # the slot's D2H copies have read their device sources
    keep = [None, None]   # device tensors the D2H stream still reads.  (Not Tensor.record_stream: recorded blocks make the
                          # caching allocator poll events on every allocation and grow the pool while they are pending.)

    def release(k, i):
        """before slot k is reused (step i >= 2): the main stream waits for the slot's D2H copies, then the tensors go
        back to the allocator (whose later main-stream users are ordered behind that wait)."""
        if i >= 2:
            s_main.wait_event(ev_out[k])
        keep[k] = None

    e2e_host = {}

    def e2e_run(n):
        t_enq0 = time.perf_counter()
        for i in range(n):
            k = i & 1
            with torch.cuda.stream(s_in):
                if i >= 2:
                    s_in.wait_event(ev_free[k])
                d_fv[k].copy_(fv_p, non_blocking=True)
                d_tex[k].copy_(tex_p, non_blocking=True)
                ev_in[k].record(s_in)
            s_main.wait_event(ev_in[k])
            release(k, i)
            a = d_fv[k].detach().requires_grad_(True)
            t = d_tex[k].detach().requires_grad_(True)
            img = SoftRasterizeFunction(image_size=H)(a, t)
            loss = torch.nn.functional.mse_loss(img, target)   # fused kernels; the loss gradient is produced on the device
            loss.backward()
            ev_free[k].record(s_main)
            ev_done[k].record(s_main)
            keep[k] = (a.grad, t.grad, loss)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_done[k])
                gf_p.copy_(a.grad, non_blocking=True)
                gt_p.copy_(t.grad, non_blocking=True)
                loss_p[i % 64].copy_(loss.detach(), non_blocking=True)   # D2H read of the step's result
                ev_out[k].record(s_out)
            del a, t, img, loss
        e2e_host["enqueue_ms"] = (time.perf_counter() - t_enq0) * 1000.0 / max(1, n)   # host time to enqueue one step
        s_out.synchronize()
        s_main.synchronize()
        keep[0] = keep[1] = None
        return float(loss_p[(n - 1) % 64])

    e2e_run(3)
    barrier()
    e2e_steps = max(3, min(args.steps, 50))   # pipeline fill and drain (one H2D, one D2H) amortised over the run
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    e0.record()
    e2e_run(e2e_steps)
    e1.record()
    e1.synchronize()
    t_host = (time.perf_counter() - t_host0) * 1000.0
    barrier()
    # device events on the main stream bracket the loop; the host wall clock (which also covers the
    # tail of the D2H stream) is taken as the e2e time when it is longer
    t_e2e = torch.tensor([max(e0.elapsed_time(e1), t_host)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = bpg * world * e2e_steps / (float(t_e2e.item()) / 1000.0)
    h2d = fv_h.nbytes + tex_h.nbytes
    d2h = fv_h.nbytes + tex_h.nbytes + 4

    # ---- render workload end to end (demo1-style: the caller wants the IMAGES): pinned host inputs -> H2D -> forward
    # only (no autograd graph) -> D2H of soft_colors [bpg,4,H,H] into pinned memory, every step, same stream pipeline
    img_p = [torch.empty((bpg, 4, H, H), dtype=torch.float32).pin_memory() for _ in range(2)]

    def render_run(n):
        for i in range(n):
            k = i & 1
            with torch.cuda.stream(s_in):
                if i >= 2:
                    s_in.wait_event(ev_free[k])
                d_fv[k].copy_(fv_p, non_blocking=True)
                d_tex[k].copy_(tex_p, non_blocking=True)
                ev_in[k].record(s_in)
            s_main.wait_event(ev_in[k])
            release(k, i)
            with torch.no_grad():
                img = SoftRasterizeFunction(image_size=H)(d_fv[k], d_tex[k])
            ev_free[k].record(s_main)
            keep[k] = img
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_free[k])
                img_p[k].copy_(img, non_blocking=True)
                ev_out[k].record(s_out)
            del img
        s_out.synchronize()
        s_main.synchronize()
        keep[0] = keep[1] = None

    render_run(3)
    barrier()
    t0 = time.perf_counter()
    render_run(e2e_steps)
    t_r = torch.tensor([(time.perf_counter() - t0) * 1000.0], dtype=torch.float64, device=dev)
    barrier()
    if world > 1:
        dist.all_reduce(t_r, op=dist.ReduceOp.MAX)
    e2e_render = {"value": bpg * world * e2e_steps / (float(t_r.item()) / 1000.0), "unit": "frames/s",
                  "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(bpg * 4 * H * H * 4),
                  "what": "forward only: pinned host inputs -> H2D -> rasterize -> D2H of the RGBA images; host wall clock"}

    # ---- optional all-gather of the output images (SURVEY.md section 8e), reported separately
    gather_ms = None
    gather_steps = None
    if world > 1:
        from jrender_b200.distributed import all_gather_images
        img = step().detach()
        for _ in range(2):
            out = all_gather_images(img, batch_size=bpg * world)
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(5):
            out = all_gather_images(img, batch_size=bpg * world)
        g1.record()
        barrier()
        tg = torch.tensor([g0.elapsed_time(g1) / 5], dtype=torch.float64, device=dev)
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
        gather_ms = float(tg.item())
        # the same step with the gather INSIDE it (every rank ends the step holding all bpg * world images):
        #   blocking   forward(all images) -> all_gather_images -> backward
        #   overlapped forward one image at a time, each image's all-gather on a side stream behind the next image's
        #              raster and the backward (jrender_b200.distributed.OverlappedImageGather)
        from jrender_b200.distributed import OverlappedImageGather

        def step_blocking():
            fv.grad = None
            tex.grad = None
            im = SoftRasterizeFunction(image_size=H)(fv, tex)
            full = all_gather_images(im.detach(), batch_size=bpg * world)
            im.backward(grad)
            return full

        def make_overlapped(chunk):
            """forward in chunks of `chunk` images; each chunk's all-gather runs on a side stream behind the next chunk's
            raster and the backward passes (chunk == bpg: one forward launch, the gather hides behind the backward)."""
            og = OverlappedImageGather(bpg, (4, H, H), dev, chunk=chunk)
            n = bpg // chunk
            fvs = [fv.detach()[i * chunk:(i + 1) * chunk].clone().requires_grad_(True) for i in range(n)]
            txs = [tex.detach()[i * chunk:(i + 1) * chunk].clone().requires_grad_(True) for i in range(n)]

            def run():
                ims = []
                for i in range(n):
                    fvs[i].grad = None
                    txs[i].grad = None
                    im = SoftRasterizeFunction(image_size=H)(fvs[i], txs[i])
                    og.push(i, im)
                    ims.append(im)
                for i in range(n):
                    ims[i].backward(grad[i * chunk:(i + 1) * chunk])
                return og.result()
            return run
        chunks = sorted({c for c in (bpg, max(1, bpg // 2), 1) if bpg % c == 0}, reverse=True)
        overlapped = {c: make_overlapped(c) for c in chunks}

        # Pipelined across steps: the gathered batch of step n is collected after step n+1's forward has been enqueued, so
        # the gather has the backward of its own step AND the raster of the next one to hide behind (a consumer that
        # logs / displays / post-processes the full batch; a loss on the gathered batch needs the variants above).
        pipe_og = [OverlappedImageGather(bpg, (4, H, H), dev, chunk=bpg) for _ in range(2)]
        pipe = {"i": 0, "pending": None}

        def step_pipelined():
            og = pipe_og[pipe["i"] & 1]
            pipe["i"] += 1
            fv.grad = None
            tex.grad = None
            im = SoftRasterizeFunction(image_size=H)(fv, tex)
            og.push(0, im)
            prev, pipe["pending"] = pipe["pending"], og
            full_prev = prev.result() if prev is not None else None
            im.backward(grad)
            return full_prev

        def timed(fn, n=10):
            for _ in range(3):
                fn()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                flush.fill_(1.0)
                fn()
            b.record()
            barrier()
            t = torch.tensor([a.elapsed_time(b) / n], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        ref_full = step_blocking().clone()
        same = all(bool(torch.equal(ref_full, f())) for f in overlapped.values())
        step_pipelined()
        same = same and bool(torch.equal(ref_full, step_pipelined()))
        t_plain = timed(lambda: step())
        gather_steps = {"images_identical": same, "step_no_gather_ms": t_plain, "step_blocking_gather_ms": timed(step_blocking),
                        "step_overlapped_gather_ms": {"chunk_%d_images" % c: timed(f) for c, f in overlapped.items()},
                        "step_pipelined_gather_ms": timed(step_pipelined),
                        "note": "each includes a 256 MiB L2 flush write per step (~0.08 ms), unlike ms_per_step; chunk = images per "
                                "forward launch (chunk == images_per_gpu: one launch, the gather hides behind the backward; smaller "
                                "chunks hide it behind the next chunk's raster too but every launch is bound by the serial chain of its pole "
                                "blocks, ~0.8 ms whatever the number of images in it); pipelined = the "
                                "batch of step n is collected during step n+1, behind its own backward and the next raster"}
        pipe["pending"].result()

    if rank != 0:
        return
    # ---- roofline of the dominant kernel.  Algorithmic bytes per launch (DESIGN.md section 5):
    #   forward : B*[ (36+12T)*nf (read fv+tex) + 16*P (write RGBA) ]
    #   backward: B*[ 32*P (read grad + RGBA) + 2*(36+12T)*nf (re-read inputs, write grads) ]
    T, P = 1, H * H
    alg = {"k_softras_forward": bpg * ((36 + 12 * T) * nf + 16 * P),
           "k_softras_backward": bpg * (32 * P + 2 * (36 + 12 * T) * nf)}
    dom = max(alg, key=lambda k: kern[k]["avg_ms"])
    peak, peak_src = peaks()
    achieved = alg[dom] / (kern[dom]["avg_ms"] / 1000.0) / 1e9
    traffic = None   # measured DRAM bytes per launch of the dominant kernel, from the committed ncu capture
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as f:
            traffic = json.load(f).get(args.workload, {}).get(dom)
    except OSError:
        pass
    # Secondary, more telling figure for this SIMT-bound path: warp instructions per launch (from the committed ncu
    # capture) over the measured kernel time, against the SM's issue ceiling (SMs x 4 schedulers x SM clock).
    issue = None
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "ncu_traffic.json")) as f:
            ninst = json.load(f).get(args.workload + "_warp_instructions", {}).get(dom)
        if ninst and clocks and clocks.get("sm_mhz"):
            import torch as _t
            sms = _t.cuda.get_device_properties(dev).multi_processor_count
            peak_i = sms * 4 * clocks["sm_mhz"] * 1e6
            ach_i = ninst / (kern[dom]["avg_ms"] / 1000.0)
            issue = {"kernel": dom, "warp_instructions_per_launch": int(ninst), "achieved_ginst_s": ach_i / 1e9,
                     "peak_ginst_s": peak_i / 1e9, "frac": ach_i / peak_i,
                     "note": "instruction count from the committed ncu capture (profiles/), time measured live"}
    except Exception:
        issue = None
    step_alg = bpg * (48 * P + 3 * (36 + 12 * T) * nf)
    line = {
        "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": value / (1000.0 / README_39K_MS) if args.workload == "c3" else None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.workload, world),
        "step_ms": {"min": float(np.min(step_ms)), "median": float(np.median(step_ms)), "max": float(np.max(step_ms))},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "what": "public API, per step: pinned host face_vertices+textures -> H2D -> forward -> on-device MSE loss -> backward -> D2H grads + loss scalar; copies of neighbouring steps overlap the kernels on two copy streams, host waits once at the end",
                "host_enqueue_ms_per_step": e2e_host.get("enqueue_ms"), "ms_per_step": float(t_e2e.item()) / e2e_steps},
        "gpu_launches": int(launches),
        "kernels": kern,
        "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": int(alg[dom]),
                     "note": "SIMT fp32 rasterization is issue-bound, not HBM-bound (SURVEY.md F9); see profiles/"},
        "roofline_step": {"algorithmic_bytes_per_step": int(step_alg),
                          "achieved_gbs": step_alg / (total_ms / args.steps / 1000.0) / 1e9,
                          "frac": step_alg / (total_ms / args.steps / 1000.0) / 1e9 / peak},
    }
    if issue is not None:
        line["roofline_issue"] = issue
    if gather_ms is not None:
        line["allgather_images_ms"] = gather_ms
        line["gather_in_step"] = gather_steps
    line["e2e_render"] = e2e_render
    if world == 1 and not args.no_cpu_baseline:
        # baselines run AFTER every timed region, in subprocesses: this process never imports oracle/
        torch.cuda.empty_cache()
        line["cpu_baseline"] = cpu_baseline_object(cpu_oracle(args.workload, args.cpu_seconds, steps=1))
        if not args.no_reference_gpu:
            line["reference_gpu"] = _run_json([os.path.join("oracle", "ref_gpu_bench.py"), "--kind", "softras", "--faces", str(nf),
                                               "--image-size", str(H), "--batch", str(bpg)], timeout=300)
    print(json.dumps(line), flush=True)


def run_nmr(args, rank, world, local_rank):
    """Secondary workload (not the headline metric): NMR forward + backward, BASELINE config C4."""
    import ctypes as C
    import torch
    from jrender_b200 import _lib
    from jrender_b200.n3mr import RasterizeFunction
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    L = _lib.lib()
    nf, H, bpg, desc = WORKLOADS[args.workload]
    from jrender_b200 import workloads as wl
    faces_h, tex_h = wl.nmr_scene(nf, batch=1, ts=2)
    # one mesh, bpg cameras: rotate the azimuth per image like build_inputs does for SoftRas
    v, f = wl.sphere_by_faces(nf)
    eyes = np.asarray([wl.get_points_from_angles(2.732, 30.0, 360.0 * (rank * bpg + b) / (bpg * world)) for b in range(bpg)], np.float32)
    cam = wl.perspective(wl.look_at(np.repeat(v[None], bpg, 0), eyes), 30.0)
    fv = wl.face_vertices(cam, f)
    faces_h = np.ascontiguousarray(np.concatenate([fv, fv[:, :, ::-1]], 1))
    tex_h = np.ascontiguousarray(np.repeat(tex_h, bpg, 0))
    faces = torch.from_numpy(faces_h).to(dev).requires_grad_(True)
    tex = torch.from_numpy(tex_h).to(dev).requires_grad_(True)
    g = torch.from_numpy(np.random.default_rng(3 + rank).uniform(-1.0, 1.0, (bpg, H, H, 3)).astype(np.float32)).to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def step():
        faces.grad = None
        tex.grad = None
        rgb, _, _ = RasterizeFunction(H, 0.1, 100.0, 1e-3, (0, 0, 0), True, False, False)(faces, tex)
        rgb.backward(g)
        return rgb
    for _ in range(max(3, args.warmup)):
        step()
    torch.cuda.synchronize(dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    l0 = L.b200r_launch_count()
    for a, b in ev:
        flush.fill_(1.0)
        a.record(); rgb = step(); b.record()
    torch.cuda.synchronize(dev)
    launches = L.b200r_launch_count() - l0
    ms = [a.elapsed_time(b) for a, b in ev]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"rgb": rgb.detach().cpu().numpy(), "grad_faces": faces.grad.cpu().numpy(),
                                         "grad_textures": tex.grad.cpu().numpy()})
    del rgb
    L.b200r_profile_reset(); L.b200r_profile_enable(1)
    for _ in range(3):
        flush.fill_(1.0); step()
    torch.cuda.synchronize(dev); L.b200r_profile_enable(0)
    kern = {}
    for kid, name in [(5, "k_nmr_zbuffer"), (6, "k_nmr_resolve"),
                      (10, "k_nmr_pack"), (7, "k_nmr_backward_pixel_map"), (8, "k_nmr_backward_maps")]:
        t, n = C.c_double(0), C.c_longlong(0)
        L.b200r_profile_read(kid, C.byref(t), C.byref(n))
        kern[name] = {"avg_ms": t.value / max(1, n.value), "launches_per_step": n.value / 3}
    if rank != 0:
        return
    nf2, ts, P = 2 * nf, 2, H * H
    alg = bpg * (36 * P + 2 * (36 + 12 * ts ** 3) * nf2)   # BASELINE.md section 4
    peak, src = peaks()
    tot = float(np.sum(ms))
    ref_gpu = None
    if world == 1 and not args.no_reference_gpu:
        torch.cuda.empty_cache()
        ref_gpu = _run_json([os.path.join("oracle", "ref_gpu_bench.py"), "--kind", "nmr", "--faces", str(nf), "--image-size", str(H),
                             "--batch", str(bpg), "--reps", "3"], timeout=600)
    print(json.dumps({
        "metric": "nmr_fwd_bwd_frames_per_s_1024px_39k_faces", "value": bpg * args.steps / (tot / 1000.0), "unit": "frames/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": tot / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "mode": "rgb", "texture_size": ts, "l2": "256 MiB flush between steps"},
        "step_ms": {"min": float(np.min(ms)), "median": float(np.median(ms)), "max": float(np.max(ms))},
        "gpu_launches": int(launches), "kernels": kern, "reference_gpu": ref_gpu,
        "roofline_step": {"algorithmic_bytes_per_step": int(alg), "achieved_gbs": alg / (tot / args.steps / 1000.0) / 1e9,
                          "frac": alg / (tot / args.steps / 1000.0) / 1e9 / peak, "peak_source": src}}), flush=True)


def run_deform(args, rank, world, local_rank):
    """Secondary workload: BASELINE config C5, the whole demo2 optimisation iteration (model -> fused pre-raster
    stage -> SoftRas silhouette forward -> losses -> backward -> Adam), eager and as one replayed CUDA graph."""
    import torch
    from jrender_b200 import _lib
    from examples import demo2_deform
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    L = _lib.lib()
    nf, H, views, desc = WORKLOADS["c5"]
    iters = max(8, args.steps)
    out = {}
    src = {}
    staged = all(os.path.exists(os.path.join(ASSETS, f)) for f in ("source.npy", "camera.npy", "obj/sphere/sphere_1352.obj"))
    if staged:   # demo2-deform.py:50-55 literally: sphere_1352.obj template, data/source.npy silhouettes (64^2, nearest-upsampled), data/camera.npy
        src = dict(filename_input=os.path.join(ASSETS, "source.npy"), camera_input=os.path.join(ASSETS, "camera.npy"),
                   template_mesh=os.path.join(ASSETS, "obj/sphere/sphere_1352.obj"))
        desc = "C5: demo2-deform as configured (sphere_1352.obj -> data/source.npy silhouettes, data/camera.npy), 512x512, 120 views/iteration"
    for mode in ("eager", "cuda_graph"):
        l0 = L.b200r_launch_count()
        r = demo2_deform.run(iters=iters, image_size=H, batch_size=views, verbose=False, cuda_graph=(mode == "cuda_graph"),
                             device=str(dev), **src)
        out[mode] = {"ms_per_iter": r["device_ms_per_iter"], "host_ms_per_iter": r["ms_per_iter"], "first_iou": r["first_iou"],
                     "final_iou": r["final_iou"], "library_launches": int(L.b200r_launch_count() - l0),
                     "iou_history": [[int(i), round(float(v), 4)] for i, _, v in r["history"]]}
    if rank != 0:
        return
    best = min(out.values(), key=lambda d: d["ms_per_iter"])
    print(json.dumps({
        "metric": "demo2_deform_views_per_s_512px", "value": views * 1000.0 / best["ms_per_iter"], "unit": "frames/s",
        "n_gpus": world, "steps": iters, "warmup": 3, "ms_per_step": best["ms_per_iter"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "reference assets (baseline/_ref/assets)" if staged else "synthetic",
        "config": {"workload": desc, "optimizer": "Adam(0.01, betas=(0.5, 0.99))", "sigma_val": 1e-4, "mode": "silhouettes"},
        "modes": out, "gpu_launches": out["eager"]["library_launches"]}), flush=True)


def run_render(args, rank, world, local_rank):
    """Secondary workload: BASELINE config C1, demo1-render.py:21-45 -- load the spot cow with texture_res 5 (GPU texture bake),
    render one view per call while the camera orbits (azimuth += 4 degrees), read every image back to the host."""
    import ctypes as C
    import torch
    import jrender_b200 as jr
    from jrender_b200 import _lib
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    L = _lib.lib()
    nf, H, bpg, desc = WORKLOADS["c1"]
    obj = os.path.join(ASSETS, "obj", "spot", "spot_triangulated.obj")
    if not os.path.exists(obj):
        if rank == 0:
            print(json.dumps({"metric": "demo1_render_frames_per_s_256px", "unavailable": "reference assets not staged (tools/stage_assets.py needs /root/reference)"}))
        return
    t0 = time.perf_counter()
    mesh = jr.Mesh.from_obj(obj, load_texture=True, texture_res=5, texture_type='surface', dr_type='softras').to(dev)
    load_s = time.perf_counter() - t0
    renderer = jr.Renderer(dr_type='softras')
    host = torch.empty((1, 3, H, H), dtype=torch.float32).pin_memory()   # mode='rgb' returns images[:, :3]

    def frame(az):
        mesh.reset_()
        renderer.transform.set_eyes_from_angles(2.732, 30, az)
        with torch.no_grad():
            rgb = renderer.render_mesh(mesh, mode='rgb')
        host.copy_(rgb, non_blocking=True)
    for k in range(max(3, args.warmup)):
        frame(4.0 * k)
    torch.cuda.synchronize(dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    l0 = L.b200r_launch_count()
    t0 = time.perf_counter()
    for k, (a, b) in enumerate(ev):
        a.record(); frame(4.0 * k); b.record()
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - t0
    launches = L.b200r_launch_count() - l0
    ms = [a.elapsed_time(b) for a, b in ev]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"rgb": host.numpy()})
    L.b200r_profile_reset(); L.b200r_profile_enable(1)
    for k in range(5):
        frame(4.0 * k)
    torch.cuda.synchronize(dev); L.b200r_profile_enable(0)
    kern = {}
    for kid, name in [(15, "k_surface_lighting"), (11, "k_project_faces"), (0, "k_face_setup"), (1, "k_coarse_bin"), (4, "k_tile_order"), (2, "k_softras_forward")]:
        t, n = C.c_double(0), C.c_longlong(0)
        L.b200r_profile_read(kid, C.byref(t), C.byref(n))
        kern[name] = {"avg_ms": t.value / max(1, n.value), "launches_per_step": n.value / 5}
    if rank != 0:
        return
    cover = float((host[0].sum(0) > 0.05).float().mean())
    print(json.dumps({
        "metric": "demo1_render_frames_per_s_256px", "value": args.steps / wall, "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": 1000.0 * wall / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "reference assets (baseline/_ref/assets)",
        "config": {"workload": desc, "params": "Renderer(dr_type='softras') defaults: sigma 1e-5, gamma 1e-4, ambient 0.5 + directional 0.5, fill_back"},
        "device_ms_per_frame": {"min": float(np.min(ms)), "median": float(np.median(ms)), "max": float(np.max(ms))},
        "what": "host wall clock over the loop: mesh.reset_ + set_eyes + lighting + transform + rasterize (forward) + D2H of the image, one view per call",
        "load_and_bake_s": load_s, "lit_pixel_fraction": cover, "gpu_launches": int(launches), "kernels": kern,
        "e2e": {"value": args.steps / wall, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 3 * H * H * 4}}), flush=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (args.impl == "reference" or args.workload == "c5"):
        raise SystemExit("bench.py: --dump-outputs covers --impl ours on every workload but c5 (its loop runs inside "
                         "examples/demo2_deform.py)")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    for kv in args.option:
        from jrender_b200 import _lib
        name, value = kv.split("=")
        _lib.set_option(name, int(value))
    try:
        if args.workload == "c4":
            run_nmr(args, rank, world, local_rank)
        elif args.workload == "c1":
            run_render(args, rank, world, local_rank)
        elif args.workload == "c5":
            run_deform(args, rank, world, local_rank)
        else:
            run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
