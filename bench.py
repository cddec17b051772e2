#!/usr/bin/env python
"""bench.py — SCNeRF hot-path training step on B200 (BASELINE.json metric: rays/sec at 4096 rays x (64c+128f)
samples, 8x256 MLP; % of tensor-core roofline).

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c2|c3|c4|c5]
                  [--scaling weak|strong] [--precision bf16x3|bf16|fp32] [--no-cpu-baseline] [--dump-outputs DIR]

A "step" = one pass of the hot path over one synthetic batch.  Workloads (BASELINE.json `configs`, 0-based):
  c2 (default) configs[1]: pixel indices -> learnable-camera rays -> NDC -> stratified + importance sampling -> coarse +
               fine PE/MLP -> composite -> loss -> gradients of both MLPs and all camera parameters
               (NeRF/run_nerf.py:385-506,600; no optimiser), 4096 rays x (64c+128f) per GPU.
  c3           configs[2]: c2 + the PRD loss on 512 sub-pixel matches of an image pair + CustomAdamOptimizer.step + lr
               decay inside the step (NeRF/run_nerf.py:482-621).
  c4           configs[3]: NeRF++ inverted-sphere fg/bg, 4096 rays x cascade (64,128), one fused C-ABI call
               (nerfplusplus/ddp_train_nerf.py:421-488,552).
  c5           configs[4]: NeRF++ 8192 rays x cascade (128,256), distortion camera.
Scaling: weak (default; every rank renders its own batch, as the reference's DDP trainer) or strong (the batch is split
over the ranks).  One all-reduce of the flat gradient buffer per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

FLOP_PER_SAMPLE = 1_186_816            # SURVEY.md §8(d): 593,408 MAC per NeRF/ MLP evaluation (fg MLPNet: the same)
FLOP_PER_SAMPLE_BG = 2 * 604_160       # NeRF++ background MLPNet (84-channel PE)
IMG_ELEMS_WGRAD = 4960                 # DESIGN §4.4: bf16 elements per sample the wgrad pass reads (x 2 B x hi,lo)

WORKLOADS = {
    "c2": dict(cfg=1, rays=4096, Nc=64, Nf=128, kind="nerf",
               text="configs[1]: LLFF fern full, 4096 rays x (64c+128f), learnable intrinsics+extrinsics "
                    "(+ray_o/ray_d residual grids), fwd+bwd"),
    "c3": dict(cfg=2, rays=4096, Nc=64, Nf=128, kind="nerf", prd_matches=512,
               text="configs[2]: full SCNeRF camera + PRD loss (512 sub-pixel matches) + custom Adam step, "
                    "4096 rays x (64c+128f), fwd+bwd+optimiser"),
    "c4": dict(cfg=3, rays=4096, Nc=64, Nf=128, kind="nerfpp", distortion=False,
               text="configs[3]: NeRF++ inverted-sphere fg/bg, 4096 rays x cascade (64,128), fwd+bwd"),
    "c5": dict(cfg=4, rays=8192, Nc=128, Nf=256, kind="nerfpp", distortion=True,
               text="configs[4]: NeRF++ fg/bg, 8192 rays x cascade (128,256), distortion camera, fwd+bwd"),
}


def evals_flop_per_ray(w):
    """Algorithmic forward FLOP per ray: coarse/level-0 on Nc samples, fine/level-1 on Nc+Nf."""
    n = w["Nc"] + (w["Nc"] + w["Nf"])
    per = FLOP_PER_SAMPLE + (FLOP_PER_SAMPLE_BG if w["kind"] == "nerfpp" else 0)
    return n * per


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["bf16_tflops"], d.get("bf16_tflops_sustained", d["bf16_tflops"]), d["hbm_gbs"], "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"          # B200_PROFILING.md fallback


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            self.t.join(2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# =====================================================================================================================
# reference arm / cpu_baseline: the reference's algorithm (CPU PyTorch restatement, oracle/, pinned by the golden
# vectors) on the host cores, on the FULL batch of the workload, fixed thread count.
# =====================================================================================================================
def cpu_threads():
    return min(32, os.cpu_count() or 1)       # eager CPU PyTorch oversubscribes beyond ~32 threads on the 128-core box


class CpuReference:
    """One full-batch step of the workload on the CPU oracle (chunked over rays: the loss is a mean over rays, so the
    chunk losses are weighted and the gradients accumulate; the reference's activation graph of 4096 x 192 samples
    does not fit a sane amount of host memory in one piece)."""

    def __init__(self, wname, chunk=512):
        self.w, self.wname, self.chunk = WORKLOADS[wname], wname, chunk
        from scnerf_b200 import synth
        self.synth = synth
        w = self.w
        T = torch.from_numpy
        if w["kind"] == "nerf":
            from oracle import scnerf_oracle as O
            self.O = O
            H, W = synth.FERN_H, synth.FERN_W
            self.cam = O.Camera(synth.intrinsic_init(), synth.camera_poses(0), synth.camera_args(), H, W)
            self.cam.load(synth.camera_noise_state(0), True)
            self.Pc = O.state_to_tensors(synth.mlp_state(0), requires_grad=True)
            self.Pf = O.state_to_tensors(synth.mlp_state(1), requires_grad=True)
            kps, idx, target = synth.pixel_batch(1000, w["rays"])
            self.inputs = (T(kps), T(idx), T(target))
            self.params = list(self.Pc.values()) + list(self.Pf.values()) + self.cam.learnables()
            if wname == "c3":
                k0, k1 = synth.c3_matches(1000, N=w["prd_matches"], pose_seed=0)
                self.matches = (T(k0), T(k1))
                self.adam = dict(m=[torch.zeros_like(p) for p in self.params], v=[torch.zeros_like(p) for p in self.params], t=0)
        else:
            from oracle import scnerf_pp_oracle as OP
            self.OP = OP
            H, W = synth.PP_H, synth.PP_W
            args = synth.pp_camera_args() if w["distortion"] else synth.pp_camera_args(camera_model="pinhole_rot_noise_10k_rayo_rayd")
            self.cam = OP.CameraPP(synth.intrinsic_init(H, W, synth.PP_FOCAL), synth.pp_camera_poses(0), args, H, W,
                                   k=(-0.05, 0.01) if w["distortion"] else None)
            self.cam.load(synth.camera_noise_state(0, n_cams=synth.PP_NCAM, H=H, W=W, with_distortion=w["distortion"]), True)
            cv = lambda st: {k: T(v).clone().requires_grad_(True) for k, v in st.items()}     # noqa: E731
            self.nets = [(cv(synth.pp_mlp_state(10 + 2 * m, 63)), cv(synth.pp_mlp_state(11 + 2 * m, 84))) for m in range(2)]
            sel, self.cam_idx, target = synth.pp_pixel_batch(1000, w["rays"])
            self.inputs = (T(sel), T(target))
            self.params = [t for f, b in self.nets for t in list(f.values()) + list(b.values())]
            self.params += [getattr(self.cam, k) for k in OP.CameraPP.LEARNABLE if getattr(self.cam, k, None) is not None]

    def step(self):
        w, N = self.w, self.w["rays"]
        for p in self.params:
            p.grad = None
        total = 0.0
        for s in range(0, N, self.chunk):
            e = min(N, s + self.chunk)
            n = e - s
            if w["kind"] == "nerf":
                kps, idx, target = (t[s:e] for t in self.inputs)
                loss, _, _ = self.O.train_step(self.cam, self.Pc, self.Pf, kps, idx, target, self.synth.FERN_H,
                                               self.synth.FERN_W, w["Nc"], w["Nf"], t_rand=torch.rand(n, w["Nc"]),
                                               u=torch.rand(n, w["Nf"]), noise0=torch.randn(n, w["Nc"]),
                                               noise1=torch.randn(n, w["Nc"] + w["Nf"]))
            else:
                sel, target = (t[s:e] for t in self.inputs)
                rand = dict(t_fg=torch.rand(n, w["Nc"]), t_bg=torch.rand(n, w["Nc"]), u_fg=torch.rand(n, w["Nf"]),
                            u_bg=torch.rand(n, w["Nf"]))
                loss, _, _ = self.OP.train_step(self.cam, self.cam_idx, sel, target, self.nets, [w["Nc"], w["Nf"]], rand)
            (loss * (n / N)).backward()
            total += float(loss.detach()) * n / N
        if self.wname == "c3":
            O, C = self.O, self.synth.c3_case()
            i, j = C["pair"]
            k0, k1 = self.matches
            ri, rj = O.rays_pixels_camera(self.synth.FERN_H, self.synth.FERN_W, self.cam, k0, idx=i), \
                O.rays_pixels_camera(self.synth.FERN_H, self.synth.FERN_W, self.cam, k1, idx=j)
            prd, _ = O.proj_ray_dist_loss(k0, k1, ri, rj, self.cam.intrinsic(), self.cam.extrinsic()[[i, j]], C["threshold"])
            (C["prd_weight"] * prd).backward()
            a = self.adam
            a["t"] += 1
            live = [k for k, p in enumerate(self.params) if p.grad is not None]
            new = O.custom_adam_step([self.params[k].detach() for k in live], [self.params[k].grad for k in live],
                                     [a["m"][k] for k in live], [a["v"][k] for k in live], [None] * len(live),
                                     [a["t"]] * len(live), self.synth.camera_args().camera_model, amsgrad=False, beta1=0.9,
                                     beta2=0.999, lr=C["lrate"], weight_decay=C["weight_decay"], eps=1e-8)
            with torch.no_grad():
                for k, p_new in zip(live, new):
                    self.params[k].copy_(p_new)
        return total


def time_cpu_reference(wname, steps, warmup, budget_s):
    """-> (rays/s, seconds per step, steps actually timed).  Stops early when `budget_s` of wall time is used up."""
    torch.set_num_threads(cpu_threads())
    ref = CpuReference(wname)
    t_start = time.perf_counter()
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        ref.step()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
        if time.perf_counter() - t_start + dt > budget_s:      # the next step would overrun the budget
            if not times:
                times.append(dt)          # budget used up during warm-up: the last warm-up step is the sample
            break
    sec = sum(times) / len(times)
    return WORKLOADS[wname]["rays"] / sec, sec, len(times)


def run_reference(args, rank):
    if rank != 0:
        return
    w = WORKLOADS[args.workload]
    rps, sec, done = time_cpu_reference(args.workload, args.steps, args.warmup, budget_s=240.0)
    th = cpu_threads()
    line = {
        "impl": "reference", "metric": "rays/sec", "value": rps, "unit": "rays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "steps_timed": done, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["text"], "rays_per_step": w["rays"], "N_samples": w["Nc"], "N_importance": w["Nf"],
                   "note": "every step = the FULL batch on the host CPU (chunked over rays, gradients accumulated); "
                           "timing stops after 240 s of wall time if --steps would take longer"},
        "cpu_baseline": {"value": rps, "unit": "rays/s", "cores": th, "kind": "port",
                         "sample": f"full {w['rays']}-ray batch per step, fwd+bwd, {sec:.1f} s/step, {done} step(s) timed; "
                                   f"CPU PyTorch restatement of the reference (oracle/, pinned by tests/golden); "
                                   f"{th} of {os.cpu_count()} host threads (fixed)"},
        "e2e": {"value": rps, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# =====================================================================================================================
# B200 arm
# =====================================================================================================================
class NerfWorkload:
    """c2 / c3 on scnerf_train_step (+ PRD + fused Adam for c3)."""

    def __init__(self, wname, rays, rank, dev, precision):
        from scnerf_b200 import synth
        from scnerf_b200.engine import TrainStep
        self.w, self.wname, self.N, self.precision = WORKLOADS[wname], wname, rays, precision
        w = self.w
        self.mods = synth.build_modules(0, dev)                           # identical replicas on every rank
        kps, idx, target = synth.pixel_batch(1000 + rank, rays)           # each rank draws its own rays
        m = self.mods
        self.eng = eng = TrainStep(m["cam"], m["coarse"], m["fine"], rays, w["Nc"], w["Nf"], perturb=1.0,
                                   raw_noise_std=1.0, precision=precision, seed=rank)
        T = torch.from_numpy
        eng.kps_dev.copy_(T(kps)); eng.idx_dev.copy_(T(idx)); eng.target_dev.copy_(T(target))
        eng.kps_host.copy_(T(kps)); eng.idx_host.copy_(T(idx)); eng.target_host.copy_(T(target))
        self.grads = eng.grads
        self.h2d, self.d2h = eng.h2d_bytes, eng.d2h_bytes
        self.api = "scnerf_train_step(inputs_on_host=1): pinned host pixel/target buffers in, loss out"
        if wname == "c3":
            import types
            from scnerf_b200.custom_optim import CustomAdamOptimizer
            self.C = C = synth.c3_case()
            k0, k1 = synth.c3_matches(1000 + rank, N=w["prd_matches"], pose_seed=0)
            self.kps0_host, self.kps1_host = T(k0).pin_memory(), T(k1).pin_memory()
            self.kps0, self.kps1 = T(k0).to(dev), T(k1).to(dev)
            self.args = types.SimpleNamespace(camera_model=synth.camera_args().camera_model,
                                              proj_ray_dist_threshold=C["threshold"])
            eng.assign_grads()
            grad_vars = list(m["coarse"].parameters()) + list(m["fine"].parameters()) + list(m["cam"].parameters())
            self.opt = CustomAdamOptimizer(params=grad_vars, lr=C["lrate"], betas=(0.9, 0.999),
                                           weight_decay=C["weight_decay"], H=synth.FERN_H, W=synth.FERN_W, args=self.args)
            self.global_step = C["global_step0"]
            self.h2d += 2 * self.kps0.numel() * 4
            self.api = ("scnerf_train_step(host buffers) + get_rays_kps_use_camera / proj_ray_dist_loss_single on pinned-host "
                        "matches + CustomAdamOptimizer.step (scnerf_adam_step)")
        self.loss_host = eng.loss_host

    def inference_step(self):
        """Forward only, as `render_path` calls it (no_grad `batchify_rays`, NeRF/render.py:398-413): ray packing done once,
        then coarse + hierarchical sampling + fine with the alpha-composite fused into the field kernel's epilogue."""
        from scnerf_b200 import synth
        from scnerf_b200.render import batchify_rays
        if not hasattr(self, "inf_rays"):
            from scnerf_b200.get_rays import get_rays_kps_use_camera
            from scnerf_b200.render import _pack_rays
            cam, eng, H, W = self.mods["cam"], self.eng, synth.FERN_H, synth.FERN_W
            with torch.no_grad():
                o, d = get_rays_kps_use_camera(H=H, W=W, camera_model=cam, idx_in_camera_param=eng.idx_dev, kps_list=eng.kps_dev)
                self.inf_rays = _pack_rays(H, W, o, d, cam, None, True, True, 0., 1.)
            self.inf_kw = dict(network_fn=self.mods["coarse"], network_query_fn=None, N_samples=self.w["Nc"],
                               N_importance=self.w["Nf"], network_fine=self.mods["fine"], perturb=0., raw_noise_std=0.,
                               precision=self.precision)
        with torch.no_grad():
            return batchify_rays(self.inf_rays, self.N, **self.inf_kw)

    def step(self, on_host):
        from scnerf_b200 import synth
        eng = self.eng
        if self.wname != "c3":
            eng.step_host() if on_host else eng.step_device()
            self.grads.all_reduce_mean()
            return
        # configs[2]: the PRD term goes FIRST (its host-side asserts / n_match read synchronise the stream, as the
        # reference's do: better while the GPU holds a few microseconds of work than behind the 12 ms render step);
        # its camera gradients land in the flat buffer, the fused step accumulates on top, then all-reduce + Adam.
        from scnerf_b200.custom_optim import update_lrate
        from scnerf_b200.get_rays import get_rays_kps_use_camera
        from scnerf_b200.ray_dist_loss import proj_ray_dist_loss_single
        C, cam = self.C, self.mods["cam"]
        H, W = synth.FERN_H, synth.FERN_W
        self.grads.zero_()
        if on_host:
            self.kps0.copy_(self.kps0_host, non_blocking=True); self.kps1.copy_(self.kps1_host, non_blocking=True)
        i, j = C["pair"]
        ri = get_rays_kps_use_camera(H=H, W=W, camera_model=cam, idx_in_camera_param=i, kps_list=self.kps0)
        rj = get_rays_kps_use_camera(H=H, W=W, camera_model=cam, idx_in_camera_param=j, kps_list=self.kps1)
        prd, _ = proj_ray_dist_loss_single(kps0_list=self.kps0, kps1_list=self.kps1, img_idx0=i, img_idx1=j, rays0=ri,
                                           rays1=rj, mode="train", device=self.kps0.device, H=H, W=W, args=self.args,
                                           camera_model=cam, method="NeRF", i_map=np.arange(synth.FERN_NCAM))
        self.prd = prd.detach()
        (C["prd_weight"] * prd).backward()                 # accumulates into the flat buffer (assign_grads)
        eng.step_host(zero=False) if on_host else eng.step_device(zero=False)
        self.grads.all_reduce_mean()
        self.opt.step()
        update_lrate(self.opt, C["lrate"], C["lrate_decay"], self.global_step)
        self.global_step += 1


class NerfppWorkload:
    """c4 / c5 on scnerf_pp_train_step."""

    def __init__(self, wname, rays, rank, dev, precision):
        from scnerf_b200 import synth
        from scnerf_b200.nerfplusplus.engine import PPTrainStep
        self.w, self.wname, self.N = WORKLOADS[wname], wname, rays
        w = self.w
        self.mods = synth.build_pp_modules(0, dev, levels=2, precision=precision, distortion=w["distortion"])
        sel, cam_idx, target = synth.pp_pixel_batch(1000 + rank, rays)
        self.eng = eng = PPTrainStep(self.mods["cam"], self.mods["nets"], rays, [w["Nc"], w["Nf"]], camera_idx=cam_idx,
                                     precision=precision, seed=rank)
        T = torch.from_numpy
        eng.sel_dev.copy_(T(sel)); eng.target_dev.copy_(T(target))
        eng.sel_host.copy_(T(sel)); eng.target_host.copy_(T(target))
        self.grads = eng.grads
        self.h2d, self.d2h = eng.h2d_bytes, eng.d2h_bytes
        self.api = "scnerf_pp_train_step(inputs_on_host=1): pinned host pixel-index/target buffers in, loss out"
        self.loss_host = eng.loss_host

    def step(self, on_host):
        self.eng.step_host() if on_host else self.eng.step_device()
        self.grads.all_reduce_mean()


# launch sites of the three tensor-core kernel classes (names as SCNERF_LAUNCH stringifies them)
KCLASS = (("fwd", ("field_fwd_pipe_kernel",)),
          ("dgrad", ("field_dgrad_pipe_kernel",)),
          ("wgrad", ("field_wgrad_kernel",)))


def kernel_breakdown(lib, wl, steps, w, burst, sustained, hbm, src):
    """Per-kernel share of the step, measured with CUDA events on the launching stream in a separate short pass
    (scnerf_kernel_timing: one event pair per launch; the headline timed region carries none)."""
    from scnerf_b200 import _lib
    torch.cuda.synchronize()
    lib.scnerf_kernel_timing(1)
    for _ in range(steps):
        wl.step(False)
    torch.cuda.synchronize()
    recs = _lib.kernel_times()
    lib.scnerf_kernel_timing(0)
    agg, other = {}, 0.0
    for name, grid, ms in recs:
        for cls, pats in KCLASS:
            if any(p in name for p in pats):
                agg[cls] = agg.get(cls, 0.0) + ms
                break
        else:
            other += ms
    samples = wl.N * (w["Nc"] + w["Nc"] + w["Nf"]) * (2 if w["kind"] == "nerfpp" else 1)      # MLP evaluations per step
    flop = wl.N * evals_flop_per_ray(w)                                                          # one pass (fwd = dgrad = wgrad)
    tj = {}
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
    out = []
    for cls, _ in KCLASS:
        if cls not in agg:
            continue
        ms = agg[cls] / steps
        tf = flop / (ms * 1e-3) / 1e12
        e = {"kernel": cls, "ms_per_step": ms, "algorithmic_tflops": tf, "frac_of_burst": tf / burst,
             "frac_of_3mma_ceiling": 3.0 * tf / burst}
        if cls == "wgrad":         # HBM-bound: the tile images are its algorithmic bytes (DESIGN §4.4)
            gbs = samples * IMG_ELEMS_WGRAD * 4 / (ms * 1e-3) / 1e9
            e.update(bound="hbm", achieved_gbs=gbs, frac_of_hbm=gbs / hbm)
        else:
            e.update(bound="tensor")
        out.append(e)
    out.sort(key=lambda e: -e["ms_per_step"])
    return out, other / steps, tj


def dump_outputs(wl, out_dir):
    """Write what a caller of the timed step holds after its last call, one ``<name>.npy`` (float32) per array: the
    loss (for c3 also ``loss.prd``, the PRD term), every parameter gradient after the all-reduce as
    ``grad.<module>.<parameter>`` and, for c3, whose step ends in the optimiser, the updated parameters as
    ``param.<module>.<parameter>``.  The inputs are seeded, so two builds run with the same arguments can be compared
    array for array.  c2, c4 and c5 start every step from the same parameters, so round-off does not accumulate (c2 on
    a B200: 4e-7 of each tensor's max after 20 steps); c3 feeds each step's round-off back
    through the optimiser and the threshold-masked PRD loss, so its dumps drift apart step by step (on a B200, camera
    parameters 2e-10 apart after the first step, 7e-4 after the seventh): compare c3 with few steps."""
    m = wl.mods
    if "nets" in m:
        nets = {f"net{k}.{s}": getattr(net, s + "_net") for k, net in enumerate(m["nets"]) for s in ("fg", "bg")}
    else:
        nets = {"coarse": m["coarse"], "fine": m["fine"]}
    out = {"loss": wl.eng.loss_dev}
    if wl.wname == "c3":
        out["loss.prd"] = wl.prd
    for key, g in wl.grads.views.items():          # flat-buffer keys: "<module>.<field tensor index>", "camera.<name>"
        prefix, _, i = key.rpartition(".")
        if prefix == "camera":
            name, p = key, getattr(m["cam"], i)
        else:
            p = nets[prefix].field_tensors()[int(i)]
            name = prefix + "." + next(n for n, q in nets[prefix].named_parameters() if q is p)
        out["grad." + name] = g
        if wl.wname == "c3":
            out["param." + name] = p
    out = {k: v.detach().float().cpu().numpy() for k, v in out.items()}
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100,
                    help="timed steps; --impl reference stops early once 240 s of wall time are used (its JSON line "
                         "reports the steps it timed as steps_timed)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--precision", default=os.environ.get("SCNERF_PRECISION", "bf16x3"),
                    help="bf16x3 (default: split-bf16 tensor-core path, the parity-grade mode) | bf16 | fp32")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-inference", action="store_true", help="skip the forward-only section (ncu launch lists of the timed step)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss and gradients of the last one (and, for c3, the updated "
                         "parameters) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 step (--impl b200)")
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch.distributed as dist
    from scnerf_b200 import _lib
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU path)"
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))
    lib = _lib.load()
    w = WORKLOADS[args.workload]
    rays = w["rays"] if args.scaling == "weak" else w["rays"] // world
    wl = (NerfWorkload if w["kind"] == "nerf" else NerfppWorkload)(args.workload, rays, rank, dev, args.precision)
    warmup = max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(on_host, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            wl.step(on_host)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps

    for _ in range(warmup):
        wl.step(False)
    lib.scnerf_launch_count(1)
    with ClockSampler(local) as clk:
        ms_dev = timed(False, args.steps)
    launches = int(lib.scnerf_launch_count(1))
    if args.dump_outputs and rank == 0:
        dump_outputs(wl, args.dump_outputs)
    for _ in range(2):
        wl.step(True)
    ms_e2e = timed(True, args.steps)
    loss = float(wl.loss_host)

    # forward-only (inference) throughput of the same batch (SURVEY 8d asks for it next to the training metric): outside
    # the timed training region, device-resident rays
    ms_inf = None
    if hasattr(wl, "inference_step") and not args.no_inference:
        for _ in range(3):
            wl.inference_step()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n_inf = max(10, min(args.steps, 50))
        for _ in range(n_inf):
            wl.inference_step()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_inf = float(t) / n_inf

    burst, sustained, hbm, src = measured_peaks()
    kernels, other_ms, tj = kernel_breakdown(lib, wl, 5, w, burst, sustained, hbm, src)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    rays_total = rays * world
    train_flop_per_ray = 3 * evals_flop_per_ray(w)       # fwd + dgrad + wgrad (activations kept as tile images, no recompute)
    step_tf = train_flop_per_ray * rays / (ms_dev * 1e-3) / 1e12
    top = kernels[0] if kernels else None
    roof = None
    if top is not None:
        tkey = {"fwd": "field_fwd_pipe_kernel", "dgrad": "field_dgrad_pipe_kernel", "wgrad": "field_wgrad_kernel"}[top["kernel"]]
        traffic = tj.get(f"{tkey}/{args.precision}/train", {}).get("dram_bytes")
        if top["bound"] == "hbm":
            roof = {"bound": "hbm", "achieved": top["achieved_gbs"], "peak": hbm, "unit": "GB/s", "frac": top["frac_of_hbm"]}
        else:
            roof = {"bound": "tensor", "achieved": top["algorithmic_tflops"], "peak": burst, "unit": "TFLOP/s",
                    "frac": top["frac_of_burst"]}
        roof.update({
            "traffic": traffic,
            "traffic_note": "dram bytes of the fine-pass launch of this kernel from the committed ncu --set full capture "
                            "(profiles/traffic.json, tools/ncu_traffic.py); per step it launches twice (fine + coarse)",
            "peak_source": f"{src} ({'copy bandwidth' if top['bound'] == 'hbm' else 'cuBLAS bf16 burst'})",
            "kernel": f"{top['kernel']} (training mode, {args.precision}; ms and rates summed over its fine + coarse launches "
                      f"of one step, CUDA events on the launching stream)",
            "ms": top["ms_per_step"],
            "kernels": kernels,
            "other_kernels_ms_per_step": other_ms,
            "step": {"algorithmic_tflops": step_tf, "frac_of_burst": step_tf / burst, "frac_of_sustained": step_tf / sustained,
                     "frac_of_3mma_ceiling_burst": 3.0 * step_tf / burst,
                     "note": "bf16x3 issues 3 tensor-core MACs per algorithmic MAC (hi*hi + lo*hi + hi*lo): the algorithmic "
                             "fraction is capped at 1/3 of the bf16 peak by construction (DESIGN.md §3)"},
        })
    line = {
        "metric": "rays/sec", "value": rays_total / (ms_dev * 1e-3), "unit": "rays/s", "n_gpus": world,
        "steps": args.steps, "warmup": warmup, "ms_per_step": ms_dev, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None,
        "dtype": {"fp32": "f32", "bf16x3": "bf16x3", "bf16": "bf16"}[args.precision], "data": "synthetic",
        "config": {"workload": w["text"] + (", per GPU" if args.scaling == "weak" else f", split over {world} GPU(s)"),
                   "baseline_config_index": w["cfg"], "rays_per_gpu": rays, "N_samples": w["Nc"], "N_importance": w["Nf"],
                   "mlp": "8x256 coarse + 8x256 fine" if w["kind"] == "nerf" else "2 cascade levels x (fg + bg) 8x256",
                   "parallelism": f"dp{world}", "precision": args.precision, "perturb": 1,
                   "raw_noise_std": 1.0 if w["kind"] == "nerf" else None,
                   "l2": "no flush: per-step working set (bf16 tile images of every layer input and dZ, ~20 GB) >> 126 MB L2",
                   "train_flop_per_ray": train_flop_per_ray},
        "e2e": {"value": rays_total / (ms_e2e * 1e-3), "unit": "rays/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": wl.h2d, "d2h_bytes_per_step": wl.d2h, "api": wl.api},
        "gpu_launches": launches,
        "loss": loss,
        "clocks": clk.summary(),
        "roofline": roof,
    }
    if ms_inf is not None:
        fwd_tf = evals_flop_per_ray(w) * rays / (ms_inf * 1e-3) / 1e12
        line["inference"] = {"value": rays_total / (ms_inf * 1e-3), "unit": "rays/s", "ms_per_batch": ms_inf,
                             "algorithmic_tflops": fwd_tf, "frac_of_burst": fwd_tf / burst,
                             "frac_of_3mma_ceiling_burst": 3.0 * fwd_tf / burst,
                             "api": "no_grad batchify_rays (render_path's call), perturb=0, raw_noise_std=0, device-resident rays; "
                                    "coarse + sample_pdf + fine, alpha-composite fused into the field kernel"}
    if world == 1 and not args.no_cpu_baseline:
        rps, sec, done = time_cpu_reference(args.workload, 1, 1, budget_s=25.0)
        th = cpu_threads()
        line["cpu_baseline"] = {"value": rps, "unit": "rays/s", "cores": th, "kind": "port",
                                "sample": f"full {w['rays']}-ray batch, fwd+bwd, {sec:.1f} s/step ({done} step timed), CPU PyTorch "
                                          f"restatement of the reference (oracle/); {th} of {os.cpu_count()} host threads (fixed)"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
