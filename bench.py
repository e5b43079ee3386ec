#!/usr/bin/env python
"""bench.py -- Mrays/s of the NeuMan ray-marching hot path at 128+128 samples on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): render_vanilla -- background NeRF, 1280x720 = 921 600 rays, 128 coarse +
128 importance samples (the fine net evaluates 256), seeded default-init weights, synthetic camera:
BASELINE.json configs[1]'s frame at the sample counts its `metric` is quoted on.  One step = one frame.
N > 1: the frame's pixels are dealt to the ranks as interleaved 16x16 tiles (SURVEY.md §8e; no data-path collective
while rendering), one NCCL all_gather of equal shards + one un-permute kernel reassemble the frame -- total work is
fixed, so scaling is "strong".

`value`   : device-resident throughput (rays generated on device, outputs left in HBM).
`e2e`     : the same metric through the public API that hands back host arrays: camera (host struct) in,
            frame copied device->host inside the timed region.
`roofline`: the dominant kernel (k_mlp_tc, tcgen05 fp16xfp16->fp32) timed per launch with CUDA events on
            its own stream inside the timed region (nm_profile_*), algorithmic FLOPs = evals x 1 186 816.
`--dump-outputs DIR`: after the timed steps, the frame the last timed step computed -- what the device-resident call
            hands back -- is written as DIR/rgb.npy (float32 [921600, 3]) and DIR/depth.npy (float32 [921600]), 14.7 MB
            in all.  Weights and camera are seeded, so the same arguments give the same inputs on every run and two
            builds can be compared output for output.
`configs` : BASELINE.json configs 2-5 at their stated sizes (device-resident, 1 warm + 2 timed frames each):
            Mrays/s, MLP evaluations, hit rays, MLP TFLOP/s.
`cpu_baseline` / `--impl reference`: the UNMODIFIED reference's own render_vanilla (baseline/_ref, installed by
            tools/install_reference.py) on the host cores, on a 64x64-pixel block (4096 rays) of the same frame:
            1 warm-up + 3 timed runs, median, thread count picked by a short sweep (BASELINE.md §3).  Falls back to the
            oracle port (kind "port") only when the reference copy is absent.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 720, 1280
S, N = 128, 128
FLOP_PER_EVAL = 1186816            # SURVEY.md §8(d)
EVALS_PER_RAY = S + (S + N)        # 384
METRIC = "Mrays/sec @128+128 samples"
WORKLOAD = "render_vanilla background NeRF 1280x720 (921600 rays), 128 coarse + 128 importance samples, random default-init weights"
CPU_WINDOW = (608, 328)            # pixel block of the frame the CPU arm renders (64x64 = 4096 rays)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return {"tflops_burst": j.get("bf16_tflops"), "tflops_sustained": j.get("bf16_tflops_sustained"),
                "hbm_gbs": j.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops_burst": 1590.0, "tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# -------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own functions on the host cores (test infrastructure: oracle/, baseline/_ref)
# -------------------------------------------------------------------------------------------------------------
def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class CpuArm:
    """render_vanilla of the frame's pixel block [x0, x0+w) x [y0, y0+h) on the CPU: the unmodified reference when its copy
    is importable (kind "reference"), else the oracle port (kind "port")."""

    def __init__(self):
        from neuman_b200 import synthetic
        from oracle import ref_import
        self.synthetic = synthetic
        self.K, self.c2w = synthetic.camera(H, W, seed=1)
        self.kind = "port"
        self.ref = None
        if ref_import.available():
            try:
                self.ref = ref_import.load()
                self.kind = "reference"
            except Exception as e:                                   # pragma: no cover
                print(f"bench.py: reference import failed ({e}); timing the oracle port", file=sys.stderr)
        if self.ref is not None:
            from oracle import ref_opts
            self.coarse, self.fine = synthetic.seed_nets(self.ref.vanilla.build_nerf, ref_opts.default_opt(), 1)
        else:
            import neuman_b200 as nb
            from oracle import neuman_oracle as no
            coarse, fine = synthetic.seed_nets(nb.build_nerf, nb.default_opt(use_cuda=False), 1)
            self.cp, self.fp = no.net_params_from_joiner(coarse), no.net_params_from_joiner(fine)

    def render(self, x0, y0, w, h):
        """-> (seconds, rgb [h*w,3], depth [h*w])"""
        Kw = self.synthetic.window_camera(self.K, x0, y0)
        torch.set_grad_enabled(False)
        t0 = time.perf_counter()
        if self.ref is not None:
            import contextlib
            import io
            ref = self.ref
            cam = ref.pinhole_camera.PinholeCamera(w, h, Kw[0, 0], Kw[1, 1], Kw[0, 2], Kw[1, 2])
            pose = ref.camera_pose.CameraPose.from_camera_to_world(self.c2w.astype(np.float64))
            cap = ref.captures.BasePinholeCapture(cam, pose)
            cap.near, cap.far = {"bkg": 0.0}, {"bkg": 3.14}
            with contextlib.redirect_stdout(io.StringIO()):
                rgb, dep = ref.render_utils.render_vanilla(self.coarse, cap, fine_net=self.fine, rays_per_batch=2048,
                                                           samples_per_ray=S, importance_samples_per_ray=N, return_depth=True)
            rgb, dep = rgb.reshape(-1, 3), dep.reshape(-1)
        else:
            from oracle import neuman_oracle as no
            rgb, dep = no.render_vanilla(self.cp, self.fp, Kw, self.c2w, h, w, 0.0, 3.14, rays_per_batch=2048,
                                         samples_per_ray=S, importance_samples_per_ray=N)
        return time.perf_counter() - t0, rgb, dep

    def pick_threads(self):
        """Short sweep on a 16x16 block: the thread count with the best throughput (oversubscribing both sockets' SMT
        siblings with 2048-ray batches is several times slower than one socket's cores)."""
        n = os.cpu_count() or 1
        cands = sorted({c for c in (8, 16, 32, 64, n // 2, n) if 1 <= c <= n})
        best, best_t = cands[0], None
        sweep = {}
        for c in cands:
            torch.set_num_threads(c)
            self.render(CPU_WINDOW[0], CPU_WINDOW[1], 16, 16)        # warm
            dt, _, _ = self.render(CPU_WINDOW[0], CPU_WINDOW[1], 16, 16)
            sweep[c] = round(dt, 3)
            if best_t is None or dt < best_t:
                best, best_t = c, dt
        torch.set_num_threads(best)
        return best, sweep

    def measure(self, runs=3, warm=1, side=64, budget_s=150.0):
        threads, sweep = self.pick_threads()
        x0, y0 = CPU_WINDOW
        dt, rgb, dep = self.render(x0, y0, side, side)               # warm-up (also sizes the sample)
        while side > 16 and dt * (runs + warm) > budget_s:
            side //= 2
            dt, rgb, dep = self.render(x0, y0, side, side)
        times = []
        for _ in range(runs):
            dt, rgb, dep = self.render(x0, y0, side, side)
            times.append(dt)
        med = float(np.median(times))
        n_rays = side * side
        return {"value": n_rays / med / 1e6, "unit": "Mrays/s", "cores": threads, "kind": self.kind,
                "sample": (f"{side}x{side} pixel block at ({x0},{y0}) of the same 1280x720 frame = {n_rays} rays, 128+128, "
                           f"{'unmodified reference render_vanilla (baseline/_ref)' if self.kind == 'reference' else 'torch-CPU oracle port'}, "
                           f"1 warm-up + {runs} runs, median {med:.2f} s; {threads} threads of {os.cpu_count()} logical CPUs "
                           f"({cpu_model()}), 16x16-block thread sweep s: {sweep}"),
                "cpu_model": cpu_model(), "times_s": [round(t, 3) for t in times]}, (x0, y0, side), rgb, dep


def run_reference(args, rank):
    if rank != 0:
        return
    arm = CpuArm()
    runs = max(1, min(args.steps, 5))
    cb, _, _, _ = arm.measure(runs=runs, warm=max(1, min(args.warmup, 2)))
    ms = 1e3 * float(np.median(cb["times_s"]))
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "Mrays/s", "n_gpus": args.gpus, "steps": runs,
            "warmup": max(1, min(args.warmup, 2)), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "sample": cb["sample"], "timing": "median of the timed steps (BASELINE.md §3)"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# -------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the cfg2-5 side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's rgb / depth as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    assert world == args.gpus or world == 1, f"WORLD_SIZE={world} but --gpus {args.gpus}"
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    import neuman_b200 as nb
    from neuman_b200 import render, sharding
    from neuman_b200._lib import Context
    from neuman_b200 import synthetic as scenes     # seeded synthetic inputs (camera, weight seeds)
    coarse, fine = scenes.seed_nets(nb.build_nerf, nb.default_opt(use_cuda=False), 1)
    coarse, fine = coarse.to(dev), fine.to(dev)
    K, c2w = scenes.camera(H, W, seed=1)
    cap = nb.SimpleCapture(K, c2w, H, W, 0.0, 3.14)
    n_pix = H * W
    ctx = Context.get(local)
    part = sharding.TilePartition(H, W, rank, world, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        rgb, depth, _ = part.buffers(with_acc=False)
        render.render_vanilla_range(coarse, cap, fine, S, N, pixels=part.pixels, host_out=False, out=(rgb, depth))
        return part.gather()                        # (rgb [H*W,3], depth [H*W], None) on every rank

    def step_e2e():
        if world == 1:
            # the reference-signature public call: camera in (host), numpy H x W x 3 / H x W frames out
            rgb, depth = nb.render_vanilla(coarse, cap, fine_net=fine, samples_per_ray=S, importance_samples_per_ray=N,
                                           return_depth=True)
            return rgb
        rgb, depth, _ = step_device()
        host = (rgb.cpu(), depth.cpu()) if rank == 0 else None
        return host

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), out

    # warm-up: at least W (>= 3) frames, and -- the board runs into its power cap within a few seconds of this
    # workload -- at least 3 s, so that the device-resident and the end-to-end measurements below see the same
    # steady-state clocks (bounded to 12 frames)
    t_w, n_w, go = time.time(), 0, True
    while go:
        step_device()
        torch.cuda.synchronize()
        n_w += 1
        go = n_w < max(args.warmup, 3) or (time.time() - t_w < 3.0 and n_w < 12 * world)
        if world > 1:                                   # every rank must run the same number of frames (collective inside)
            flag = torch.tensor([1 if go else 0], device=dev)
            dist.broadcast(flag, 0)
            go = bool(flag.item())
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    ctx.profile(True)
    l0 = ctx.launch_count()
    ms_total, frame = timed(step_device, args.steps)
    launches = ctx.launch_count() - l0
    prof = ctx.profile_read()
    ctx.profile(False)
    clocks = sampler.stop() if sampler else None
    ms_step = ms_total / args.steps
    value = n_pix / (ms_step * 1e3)
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in (("rgb", frame[0]), ("depth", frame[1])):
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), t.float().cpu().numpy())
    for _ in range(2):
        step_e2e()
    ms_e2e, host = timed(step_e2e, args.steps)
    e2e_val = n_pix / (ms_e2e / args.steps * 1e3)
    ctx.range_check()                                   # raises if any launch saturated an fp16 operand

    pk = peaks()
    side = {}
    if not args.no_configs:
        side = side_configs(nb, render, sharding, scenes, ctx, dev, rank, world, dist, pk)
    train = train_step_ms(nb, dev) if (world == 1 and not args.no_configs) else None
    human_train = None
    if world == 1 and not args.no_configs:
        try:
            human_train = human_train_step_ms(nb, dev)
        except Exception as e:                         # a side measurement must never cost the line
            human_train = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0:
        mlp_ms_per_launch = prof["mlp_ms"] / max(prof["mlp_launches"], 1)
        flops_per_launch = prof["mlp_evals"] / max(prof["mlp_launches"], 1) * FLOP_PER_EVAL
        achieved = flops_per_launch / (mlp_ms_per_launch * 1e-3) / 1e12 if prof["mlp_ms"] > 0 else None
        peak = pk["tflops_sustained"]
        traffic = None
        tp = os.path.join(ROOT, "profiles", "mlp_tc_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic = tj.get("dram_bytes_per_launch_bench")       # ncu capture of THIS workload's launches (mean of S=128 and S=256)
        line = {
            "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16 operands x f32 accumulate (tcgen05 kind::f16); f32 elsewhere", "data": "synthetic",
            "config": {"workload": WORKLOAD, "global_rays_per_step": n_pix, "mlp_evals_per_ray": EVALS_PER_RAY,
                       "parallelism": f"ray-shard x{world}: interleaved 16x16 pixel tiles + 1 all_gather + un-permute kernel", "warmup_frames_run": n_w,
                       "l2": "per-step working set (raw [32768x256x4] f32 chunks, 3.8 GB/frame) >> 126 MB L2; no flush needed"},
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": (achieved / peak) if achieved else None,
                         "traffic": traffic, "traffic_unit": "DRAM bytes per launch: ncu dram__bytes_read+write of this workload's two launch shapes (32768 rays x 128 / x 256 samples), mean; algorithmic 20 B/eval mostly stays in L2",
                         "kernel": "k_mlp_tc<2>", "peak_source": pk["source"] + " bf16_tflops_sustained (fp16 runs at the bf16 rate)",
                         "mlp_launches": prof["mlp_launches"], "mlp_ms_per_step": prof["mlp_ms"] / args.steps,
                         "mlp_share_of_step": prof["mlp_ms"] / ms_total},
            "e2e": {"value": e2e_val, "unit": "Mrays/s", "h2d_bytes_per_step": 208, "d2h_bytes_per_step": n_pix * 4 * 4,
                    "api": "neuman_b200.render_vanilla(coarse, cap, fine_net=fine, ...) -> numpy rgb [720,1280,3] + depth (reference signature); "
                           "inputs = the capture's K / camera_to_world (208 B host struct), rays are generated on the device"},
            "gpu_launches": int(launches), "clocks": clocks, "configs": side, "train_step": train,
            "human_train_step": human_train,
        }
        if not args.no_cpu_baseline and world == 1:
            arm = CpuArm()
            cb, (x0, y0, sd), rgb_cpu, dep_cpu = arm.measure()
            line["cpu_baseline"] = cb
            fr = frame[0].reshape(H, W, 3)[y0:y0 + sd, x0:x0 + sd].reshape(-1, 3).cpu().numpy()
            fd = frame[1].reshape(H, W)[y0:y0 + sd, x0:x0 + sd].reshape(-1).cpu().numpy()
            line["parity_vs_cpu_sample"] = {"rays": int(sd * sd), "max_abs_rgb": float(np.abs(fr - rgb_cpu).max()),
                                            "max_abs_depth": float(np.abs(fd - dep_cpu).max()),
                                            "note": "depth gate = max(1e-4, 1.5 x the 11-bit-operand floor of the oracle on the same rays), tests/test_gpu_fullsize.py"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def train_step_ms(nb, dev, R=2048, steps=20):
    """SURVEY.md §8f-1: one optimiser step of the background-NeRF trainer (trainers/vanilla_nerf_trainer.py:206-223: loss_func
    + backward + Adam) on the CUDA path at the reference's defaults (2048 rays, 128 + 128 samples, perturb 1, raw_noise_std 1)."""
    import torch.nn.functional as F
    from neuman_b200 import synthetic, train as nt
    opt = nb.default_opt(perturb=1.0, raw_noise_std=1.0)
    coarse, fine = synthetic.seed_nets(nb.build_nerf, nb.default_opt(use_cuda=False), 3)
    coarse, fine = coarse.to(dev), fine.to(dev)
    optim = torch.optim.Adam(list(coarse.parameters()) + list(fine.parameters()), lr=5e-4)
    g = torch.Generator(device=dev).manual_seed(0)
    batch = dict(origin=torch.randn(R, 3, device=dev, generator=g) * 0.1,
                 direction=F.normalize(torch.randn(R, 3, device=dev, generator=g), dim=-1),
                 near=torch.full((R,), 0.5, device=dev), far=torch.full((R,), 4.0, device=dev),
                 color=torch.rand(R, 3, device=dev, generator=g))
    for _ in range(5):
        nt.train_batch(coarse, fine, optim, batch, opt, check_bad_weights=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = nt.train_batch(coarse, fine, optim, batch, opt, check_bad_weights=False)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"ms_per_step": ms, "rays_per_s": R / ms * 1e3, "rays_per_batch": R, "samples": "128+128", "mlp_evals_per_step": R * 384,
            "loss_finite": bool(torch.isfinite(loss)), "what": "neuman_b200.train.train_batch: CUDA forward/backward kernels + torch.optim.Adam"}


def human_train_step_ms(nb, dev, R=2048, S=128, steps=10):
    """SURVEY.md §8f-1: the human branch of one HumanNeRFTrainer step (trainers/human_nerf_trainer.py:241-278,
    `_eval_human_samples`, then backward + Adam) on the CUDA path at the reference's defaults (2048 rays x 128 samples):
    ray_to_samples, offset network (tensor-core kernels), SMPL vertex_forward (training kernels), closest-face query,
    fused blend / inverse / apply / directions, canonical human network -- and the adjoint of each, down to the human and
    offset networks' weights and the per-frame poses / betas / alignments."""
    from neuman_b200 import train as nt
    from neuman_b200.synthetic import make_model
    rng = np.random.RandomState(0)
    pose, betas = rng.normal(0, 0.3, (1, 72)).astype(np.float32), rng.normal(0, 1.0, (1, 10)).astype(np.float32)
    align = np.eye(4, dtype=np.float32)
    align[3, :3] = (0.3, -0.1, 2.0)
    opt = nb.default_opt(use_cuda=True, num_offset_nets=1, offset_scale=0.02, offset_scale_type='tanh', samples_per_ray=S)
    torch.manual_seed(0)
    model = make_model(0)
    net = nb.HumanNeRF(opt, poses=pose, betas=betas, alignments=align[None], scale=0.4, smpl_model=model)
    faces = np.ascontiguousarray(model["f"][:, :3].astype(np.int64))
    with torch.no_grad():
        V0 = net.vertex_forward(0)[0][0]
    g = torch.Generator(device=dev).manual_seed(0)
    eye = V0.mean(0) + torch.tensor([0.0, 0.0, -2.0], device=dev)
    d = V0[torch.randint(0, V0.shape[0], (R,), device=dev, generator=g)] + 0.02 * torch.randn(R, 3, device=dev, generator=g) - eye
    dist = d.norm(dim=1, keepdim=True)
    batch = {'origin': eye[None].repeat(R, 1), 'direction': d / dist, 'human_near': dist - 0.2, 'human_far': dist + 0.2,
             'cur_view_f': 3 / 11, 'cap_id': 0}
    params = (list(net.coarse_human_net.parameters()) + list(net.offset_nets.parameters())
              + [net.poses, net.betas, net.alignments])
    optim = torch.optim.Adam(params, lr=1e-4)

    def step():
        optim.zero_grad()
        out = nt.eval_human_samples(net, batch, opt, faces, offset_net=net.offset_nets[0])
        loss = out[5].square().mean()
        loss.backward()
        optim.step()
        return loss
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    ok = bool(torch.isfinite(loss)) and all(bool(torch.isfinite(p).all()) for p in (net.poses, net.betas, net.alignments))
    return {"ms_per_step": ms, "rays_per_s": R / ms * 1e3, "rays_per_batch": R, "samples": S, "mlp_evals_per_step": 2 * R * S,
            "finite": ok, "what": "neuman_b200.train.eval_human_samples (offset net + SMPL + warp + human net on the CUDA kernels) "
                                  "+ backward + torch.optim.Adam over the nets and poses / betas / alignments"}


def side_configs(nb, render, sharding, scenes, ctx, dev, rank, world, dist, pk):
    """BASELINE.json configs 2-5 at their stated sizes, device-resident, sharded like the main workload.  Bodies come from
    the device SMPL kernels (ops.smpl_scene_transforms) on the synthetic SMPL-shaped model."""
    from neuman_b200 import ops
    torch.manual_seed(1)
    model = nb.HumanNeRF(nb.default_opt(use_cuda=False))
    scenes.boost_density(model.coarse_human_net)
    model = model.to(dev)
    sm = scenes.make_model(0)
    par = sm["kintree_table"][0].astype(np.int64)
    smpl = ops.SmplModelDevice(sm["v_template"], sm["shapedirs"], sm["J_regressor"], sm["weights"], par, device=dev)
    faces = torch.from_numpy(sm["f"].astype(np.int32)).to(dev)
    out = {}

    def bodies_of(cfg):
        bs = []
        for a in cfg["actors"]:
            pose, betas, align = scenes.actor_pose(a)
            verts, joints, T = ops.smpl_scene_transforms(smpl, pose, betas, align, a["scale"])
            bs.append({"verts": verts.contiguous(), "T": T, "geo": float(torch.linalg.norm(joints[3] - joints[0]))})
        return bs

    for name in ("cfg2", "cfg3_can", "cfg3", "cfg4", "cfg5"):
        cfg = scenes.FULLSIZE[name.split("_")[0]]
        Hc, Wc, Sc, Nc = cfg["H"], cfg["W"], cfg["S"], cfg["N"]
        K, c2w = scenes.fullsize_camera(name.split("_")[0])
        cap = nb.SimpleCapture(K, c2w, Hc, Wc, cfg["near"], cfg["far"])
        part = sharding.TilePartition(Hc, Wc, rank, world, device=dev)
        bs = bodies_of(cfg)
        geo = bs[0]["geo"] if bs else 0.2
        if name == "cfg2":
            cn, fn_ = model.coarse_bkg_net, model.fine_bkg_net

            def fn(ev=None):
                rgb, depth, _ = part.buffers(with_acc=False)
                render.render_vanilla_range(cn, cap, fn_, Sc, Nc, pixels=part.pixels, host_out=False, out=(rgb, depth))
                if ev is not None:
                    ev.record()
                return part.gather()
        elif name.startswith("cfg3"):
            can = name.endswith("_can")

            def fn(ev=None):
                bufs = part.buffers()
                render.render_smpl_nerf_range(model, cap, bs[0]["verts"], faces, bs[0]["T"], Sc, True, can, geo, 1.0,
                                              pixels=part.pixels, host_out=False, out=bufs)
                if ev is not None:
                    ev.record()
                return part.gather()
        elif name == "cfg4":
            def fn(ev=None):
                bufs = part.buffers()
                render.render_hybrid_nerf_range(model, cap, bs[0]["verts"], faces, bs[0]["T"], Sc, Nc, True, geo,
                                                pixels=part.pixels, host_out=False, out=bufs)
                if ev is not None:
                    ev.record()
                return part.gather()
        else:
            def fn(ev=None):
                bufs = part.buffers()
                render._hybrid(model, [model] * len(bs), cap, [b["verts"] for b in bs], [faces] * len(bs), [b["T"] for b in bs],
                               Sc, Nc, True, geo, True, 0, None, False, render.CHUNK, pixels=part.pixels, out=bufs)
                if ev is not None:
                    ev.record()
                return part.gather()
        fn()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ctx.profile(True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        reps = 2
        fn()
        eb, em = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        eb.record()
        fn(em)                                      # second frame: also stamp the end of this rank's own rendering
        e1.record()
        torch.cuda.synchronize()
        busy_ms = eb.elapsed_time(em)
        prof = ctx.profile_read()
        ctx.profile(False)
        st = ctx.render_stats()
        t = torch.tensor([e0.elapsed_time(e1) / reps, prof["mlp_ms"] / reps, float(st["mlp_evals"]), float(st["hit_rays"]), busy_ms],
                         device=dev, dtype=torch.float64)
        if world > 1:
            tmax, tsum = t.clone(), t.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
            ms, mlp_ms, evals, hits = float(tmax[0]), float(tmax[1]), float(tsum[2]), float(tsum[3])
            busy = [float(x) for x in _gather_scalars(dist, t[4], world, dev)]
            hit_per_rank = [int(x) for x in _gather_scalars(dist, t[3], world, dev)]
        else:
            ms, mlp_ms, evals, hits = (float(x) for x in t[:4])
            busy, hit_per_rank = [busy_ms], [int(hits)]
        tf = evals / world * FLOP_PER_EVAL / (mlp_ms * 1e-3) / 1e12 if mlp_ms > 0 else None
        out[name] = {"driver": cfg["driver"] + (" render_can=True" if name.endswith("_can") else ""), "frame": f"{Wc}x{Hc}",
                     "samples": f"{Sc}+{Nc}", "ms_per_frame": ms, "Mrays_s": Hc * Wc / ms / 1e3, "mlp_evals": int(evals),
                     "hit_rays": int(hits), "mlp_ms": mlp_ms, "mlp_tflops_per_gpu": tf,
                     "mlp_frac_of_peak": tf / pk["tflops_sustained"] if tf else None,
                     "non_mlp_share": 1.0 - mlp_ms / ms if ms > 0 else None,
                     "per_rank_render_ms": busy, "per_rank_hit_rays": hit_per_rank}
    return out


def _gather_scalars(dist, x, world, dev):
    buf = torch.zeros(world, device=dev, dtype=torch.float64)
    dist.all_gather_into_tensor(buf, x.reshape(1).to(torch.float64))
    return buf.tolist()


if __name__ == "__main__":
    main()
