#!/usr/bin/env python
"""bench.py -- fwd+bwd throughput of the Gaussian feature rasterizer on BASELINE.json's headline config.

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference] [--dump-outputs DIR]

* workload (config.workload): BASELINE.json configs[1] = synthetic 1M Gaussians, 1080x1920, K=32, one
  camera per GPU per step (SYN(P,H,W,K,cam) of BASELINE.md section 2.2; camera index = rank).
* a "step" = one forward + backward of the rasterizer over one camera on every rank, plus (N>1) ONE all-reduce of the
  per-Gaussian feature gradient dL_dcolors [P,K].  Weak scaling: per-GPU work is fixed.
* metric = Gaussians*pixels/s = (sum over ranks of P*H*W) * K_steps / time; time = CUDA events on the launching
  stream, barrier + synchronize on both sides, max over ranks.
* `value`  : Gaussian parameters, upstream gradient and camera resident in HBM, operator called directly; nothing but the
             steps (and three NVML clock samples taken while the GPU is busy) runs between the two events.
* `e2e`    : the same step through the reference-shaped public API as a user drives it -- per step the camera
             (view / projection / centre / background: the only host-side inputs the reference API has; the
             Gaussian parameters are resident model state exactly as in train_contrastive_feature.py) is copied
             from pinned host memory, the loss (sum(image * dL)) is read back to the host.
* `roofline`: HBM roofline of the dominant kernel.  Its average launch duration comes from per-stage CUDA-event timings
             taken by the library on its launch stream in a SEPARATE pass of the same steps (the instrumentation costs
             ~18 event records per step, so it stays out of the `value` region); algorithmic bytes per launch as in DESIGN.md.
* `c4`     : BASELINE.json configs[3] (3M Gaussians, 8 cameras, STRONG scaling: 8 / N cameras per rank, one all-reduce of
             the 384 MB feature gradient per 8-camera batch), measured in the same run after the headline numbers, over
             --steps batches like the headline; --no-c4 skips it (with --impl reference, whose batches are far slower, this leg
             dominates the run time at the default --steps).
* `cpu_baseline`: the CPU oracle port (oracle/sagars_oracle.c, OpenMP over tiles) timed on the host cores on the
             same workload (rank 0, N=1 only).
* `--impl reference`: the UNMODIFIED reference extension (oracle/_ref, rebuilt for sm_100a from the reference's sources by
             oracle/build_ref.py) through its own GaussianRasterizer API on the same inputs.  NOTE: the reference has
             no CPU implementation of this path -- its implementation IS the CUDA extension, and the north star's
             ">= 3x the reference CUDA rasterizer" is a ratio against exactly this arm.  If oracle/_ref is absent the
             arm falls back to the CPU oracle port and says so.
* `--dump-outputs DIR`: after the timed steps, what the last step of the `value` region computed on rank 0 -- the image and
             radii the forward returned for rank 0's last camera and the gradients of the six inputs it differentiates -- as
             DIR/<name>.npy (float32).  The gradients are those the step leaves on the leaves: summed over all of rank 0's
             cameras and, with N > 1, dL_dcolors all-reduced over the ranks; compare dumps of runs with the same workload and
             the same number of GPUs only.  An array of more than DUMP_MAX_ELEMENTS elements is stored as a fixed, seeded
             sample of that many elements (the same positions in every run), so two builds can be compared output for output:
             the inputs are seeded as well.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

WORKLOADS = {
    # BASELINE.json configs[1]
    "c2": dict(P=1_000_000, H=1080, W=1920, K=32, cameras=None,
               desc="synthetic 1M Gaussians, 1080x1920, K=32 affinity features, 1 camera/GPU, fwd+bwd"),
    # BASELINE.json configs[3]: strong scaling of an 8-camera batch
    "c4": dict(P=3_000_000, H=1080, W=1920, K=32, cameras=8,
               desc="synthetic 3M Gaussians, 1080x1920, K=32, batch of 8 cameras sharded over the GPUs, fwd+bwd + feature-gradient all-reduce"),
    # BASELINE.json configs[2]-like (parity-test case, not the bench line): 5M Gaussians
    "c3": dict(P=5_000_000, H=1036, W=1600, K=32, cameras=None,
               desc="synthetic 5M Gaussians, 1036x1600, K=32 (garden-like), 1 camera/GPU, fwd+bwd"),
    # configs[1] at K=3 (the BASE variant's channel count; developer A/B of the forward kernels, never a bench line)
    "c2_k3": dict(P=1_000_000, H=1080, W=1920, K=3, cameras=None, desc="synthetic 1M Gaussians, 1080x1920, K=3, 1 camera/GPU, fwd+bwd"),
    # small variant for quick local checks (never a bench line)
    "tiny": dict(P=20_000, H=270, W=480, K=32, cameras=None, desc="tiny smoke workload"),
}
DUMP_MAX_ELEMENTS = 1 << 20       # 8 arrays of at most 4 MB each


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed steps of each measured region (value, e2e) and timed batches of the c4 leg (8 cameras each); "
                         "the per-stage profiling pass runs min(steps, 20)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c4", action="store_true", help="skip the BASELINE configs[3] strong-scaling leg")
    ap.add_argument("--fwd-kernel", default="default", choices=["default", "tile", "warp_any"], help="developer A/B switch (rasterizer.set_blend_kernels)")
    ap.add_argument("--bwd-kernel", default="default", choices=["default", "tile", "tc"], help="developer A/B switch (default = the warp-per-block mma.sync kernel)")
    ap.add_argument("--allreduce-mode", default="overlap", choices=["overlap", "sync"],
                    help="N > 1: 'overlap' = the all-reduce runs on a side stream and gates only the next forward's blend stage (its "
                         "geometry stages overlap the exchange); 'sync' = the all-reduce serialises with the step")
    ap.add_argument("--allreduce", default="nccl", choices=["nccl", "multimem"],
                    help="N > 1, developer switch: 'multimem' = the library's own all-reduce over the NVSwitch multicast mapping")
    ap.add_argument("--binning", default="default", choices=["default", "radix", "tile_sort", "depth_first"], help="developer A/B switch (rasterizer.set_binning)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32; large arrays as a fixed, seeded sample)")
    return ap.parse_args()


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region, read through NVML (the quantities
    `nvidia-smi --query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.*` prints; B200_PROFILING.md recipe).
    Samples are taken explicitly from the launching thread right after the last timed step has been launched, while the GPU
    is still executing the last two timed steps (the launch loop keeps a two-step lead), so the read costs no GPU time.
    A polling child / thread is deliberately NOT used: `nvidia-smi -lms 50` was measured to slow this launch-heavy step 3x
    and a 100 ms NVML thread still added up to ~1 ms/step of jitter, which would falsify the number it guards."""

    def __init__(self, index: int):
        self.index, self.rows, self.ok = index, [], False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")   # CUDA ordinal -> NVML index
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].strip().isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:   # pragma: no cover
            self.err = repr(e)

    def sample(self):
        if not self.ok:
            return
        nv = self.nv
        try:
            sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
            rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.rows.append((sm, int(rs)))
        except Exception:
            pass

    def result(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")]}
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        reasons = sorted(n for n, bit in names.items() if any(r[1] & bit for r in self.rows))
        sm = [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(self.max_sm), "reasons": reasons,
                "samples": len(sm), "source": "nvml, sampled while the timed steps execute"}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def algorithmic_bytes(P, R, HW, T, C):
    """DESIGN.md section 'algorithmic bytes' (SURVEY.md Appendix C): each datum crosses HBM once."""
    binning = P * 20 + R * 12 + R * 24 + R * 8 + T * 8          # key emission + one sort's worth of traffic + range detection
    per_stage = {
        "preprocess": P * (44 + 60),
        "scan_block_sums": P * 8,
        "duplicate_keys": P * 20 + R * 12,
        "radix_sort": R * 24,
        "tile_ranges": R * 8 + T * 8,
        "render_forward": R * (28 + 4 * C) + HW * (4 * C + 8),
        "render_backward": R * (28 + 4 * C) + HW * (4 * C + 8) + P * (4 * C + 24),
        "geom_backward": P * (96 + 64),
    }
    return per_stage, P * (44 + 60) + P * 8 + binning + per_stage["render_forward"] + per_stage["render_backward"] + per_stage["geom_backward"]


class Runner:
    """One rank's share of a workload: resident Gaussian parameters, the cameras this rank renders per step, the step functions."""

    def __init__(self, a, wl, world, rank, dev, use_dist, Settings, Rast, R):
        from seganygaussians_b200 import synthetic
        self.a, self.wl, self.world, self.rank, self.dev, self.use_dist, self.R = a, wl, world, rank, dev, use_dist, R
        P, H, W, K = wl["P"], wl["H"], wl["W"], wl["K"]
        n_used = world if use_dist else 1
        if wl["cameras"] is None:
            self.cams = [rank % 8]                                   # weak scaling: one camera per rank
            self.cameras_per_step = n_used
        else:
            self.cams = list(range(rank if use_dist else 0, wl["cameras"], n_used))     # strong scaling: camera i -> rank i mod N
            self.cameras_per_step = wl["cameras"]
        sc = synthetic.scene(P, H, W, K, cam=self.cams[0] if self.cams else 0)
        self.sc = sc
        g = sc.gauss
        self.means3D = g.means3D.to(dev).requires_grad_(True)
        self.means2D = torch.zeros(P, 3, device=dev, requires_grad=True)
        self.opac = g.opacities.to(dev).requires_grad_(True)
        self.scales = g.scales.to(dev).requires_grad_(True)
        self.rots = g.rotations.to(dev).requires_grad_(True)
        self.colors = g.colors.to(dev).requires_grad_(True)
        self.leaves = (self.means3D, self.means2D, self.opac, self.scales, self.rots, self.colors)
        self.dL = sc.dL_dout.to(dev)
        self.Settings, self.Rast = Settings, Rast
        self.host_cams, self.rasts = [], []
        self.h2d_bytes = 0
        for ci in self.cams:
            c = synthetic.make_camera(H, W, ci)
            dev_t = [t.to(dev) for t in (c.world_view_transform, c.full_proj_transform, c.camera_center, torch.zeros(K))]
            self.rasts.append(Rast(raster_settings=self._settings(c, *dev_t)))
            # the camera as ONE pinned buffer (view 16 | projection 16 | background K | centre 3 floats; every part 16-byte aligned):
            # one host -> device copy per step
            pinned = torch.cat([c.world_view_transform.reshape(-1), c.full_proj_transform.reshape(-1), torch.zeros(K),
                                c.camera_center.reshape(-1)]).float().pin_memory()
            self.host_cams.append((c, pinned))
            self.h2d_bytes += pinned.numel() * 4
        self.reducer = None
        self.own_allreduce = None
        if use_dist and a.impl == "ours":
            from seganygaussians_b200.data_parallel import FeatureGradReducer, MulticastAllReduce
            if a.allreduce == "multimem":
                self.own_allreduce = MulticastAllReduce(P * K, dev)
            if a.allreduce_mode == "overlap":
                self.reducer = FeatureGradReducer(side_stream=True, reduce_fn=self.own_allreduce.all_reduce_ if self.own_allreduce else None)
        self.last = {}
        self.keep_color = False                                      # outputs() needs the last step's image

    def _settings(self, c, view, proj, campos, bg):
        wl = self.wl
        return self.Settings(image_height=wl["H"], image_width=wl["W"], tanfovx=c.tanfovx, tanfovy=c.tanfovy, bg=bg, scale_modifier=1.0,
                             viewmatrix=view, projmatrix=proj, sh_degree=0, campos=campos, prefiltered=False, debug=False)

    def _render(self, rast):
        return rast(means3D=self.means3D, means2D=self.means2D, opacities=self.opac, shs=None, colors_precomp=self.colors,
                    scales=self.scales, rotations=self.rots, cov3D_precomp=None)

    def _reduce(self):
        import torch.distributed as dist
        if self.colors.grad is None:                               # a rank without a camera still joins the collective
            self.colors.grad = torch.zeros_like(self.colors)
        if self.reducer is not None:
            self.reducer.wait()                                    # at most one exchange in flight
            self.reducer.reduce_async(self.colors.grad)            # side stream, behind everything queued so far
            self.R.set_blend_wait_event(self.reducer.ready_event())  # next forward: geometry stages run ahead, the blend waits
        elif self.own_allreduce is not None:
            self.own_allreduce.all_reduce_(self.colors.grad)
        else:
            dist.all_reduce(self.colors.grad)

    def step_resident(self):
        for t in self.leaves:
            t.grad = None
        for rast in self.rasts:
            color, radii = self._render(rast)
            self.last["grad_fn"], self.last["radii"] = color.grad_fn, radii
            if self.keep_color:
                self.last["color"] = color.detach()
            color.backward(self.dL)
        if self.use_dist:
            self._reduce()

    def step_e2e(self):
        for t in self.leaves:
            t.grad = None
        total = None
        for (c, pinned) in self.host_cams:
            cam = pinned.to(self.dev, non_blocking=True)
            K_ = self.wl["K"]
            view, proj, bg, campos = cam[0:16].view(4, 4), cam[16:32].view(4, 4), cam[32:32 + K_], cam[32 + K_:35 + K_]
            rast = self.Rast(raster_settings=self._settings(c, view, proj, campos, bg))
            color, radii = self._render(rast)
            loss = torch.dot(color.reshape(-1), self.dL.reshape(-1))   # = (color * dL).sum(), one reduction instead of two kernels
            loss.backward()
            total = loss.detach() if total is None else total + loss.detach()
        if self.use_dist:
            self._reduce()
        return float(total.item()) if total is not None else 0.0   # device -> host read of the step's result

    def barrier(self):
        if self.use_dist:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize(self.dev)

    def timed(self, fn, steps, sampler=None):
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        # The launching thread may run at most two steps ahead of the GPU: far enough that the GPU never waits for a launch, close
        # enough that the caching allocator keeps recycling the same scratch blocks.  NVML is read AFTER the last launch, while the
        # GPU still executes the last two timed steps (an NVML call takes milliseconds: in the middle of the loop it drained the
        # two-step lead and idled the GPU -- measured as `value` > `e2e`).
        lead = []
        e0.record()
        for i in range(steps):
            fn()
            ev = torch.cuda.Event()
            ev.record()
            lead.append(ev)
            if len(lead) > 2:
                lead.pop(0).synchronize()
        if self.reducer is not None:
            self.reducer.wait()           # the last exchange belongs to the timed region
        e1.record()
        if sampler is not None:
            sampler.sample()              # the GPU is still executing timed steps
            sampler.sample()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.use_dist:
            import torch.distributed as dist
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def outputs(self):
        """The last resident step's outputs as float32 host arrays, large ones sampled: image and radii of this rank's last
        camera; the leaves' gradients, i.e. summed over this rank's cameras and, under torchrun, with dL_dcolors all-reduced."""
        named = {"color": self.last["color"], "radii": self.last["radii"], "dL_dmeans3D": self.means3D.grad,
                 "dL_dmeans2D": self.means2D.grad, "dL_dopacities": self.opac.grad, "dL_dscales": self.scales.grad,
                 "dL_drotations": self.rots.grad, "dL_dcolors": self.colors.grad}
        out = {}
        for name, t in named.items():
            flat = t.detach().reshape(-1)
            if flat.numel() > DUMP_MAX_ELEMENTS:
                idx = np.sort(np.random.default_rng(0).choice(flat.numel(), DUMP_MAX_ELEMENTS, replace=False))
                flat = flat[torch.from_numpy(idx).to(flat.device)]
            out[name] = flat.float().cpu().numpy()
        return out

    def counters(self, ours: bool):
        """Work counters of this rank's last camera (SURVEY.md section 8(d)), decoded from the last call's scratch."""
        wl = self.wl
        H, W = wl["H"], wl["W"]
        gf = self.last["grad_fn"]
        R_inst = int(gf.num_rendered)
        vis = int((self.last["radii"] > 0).sum().item())
        pairs = None
        try:
            img_state = gf.saved_tensors[-1]                       # both implementations save the image-state bytes last
            if ours:
                from seganygaussians_b200 import _lib
                off = _lib.image_layout(W, H).n_contrib
            else:
                off = (4 * H * W + 127) // 128 * 128               # reference layout: accum_alpha f32[N] | n_contrib u32[N] (SURVEY.md Appendix B)
            pairs = int(img_state[off: off + 4 * H * W].view(torch.int32).sum(dtype=torch.int64).item())
        except Exception:
            pairs = None
        return R_inst, vis, pairs


def kernel_names(a, K):
    fwd = {"default": "mma.sync warp kernel at K=32, fp32 tile kernel otherwise", "tile": "tcgen05 tile kernel",
           "warp_any": "mma.sync warp kernel for every K"}[a.fwd_kernel]
    bwd = {"default": "mma.sync warp-per-block kernel", "tile": "mma.sync tile kernel",
           "tc": "tcgen05 / TMEM pixel-group kernel"}[a.bwd_kernel]
    return {"forward": fwd, "backward": bwd, "binning": a.binning}


def main():
    a = parse()
    wl = WORKLOADS[a.workload]
    P, H, W, K = wl["P"], wl["H"], wl["W"], wl["K"]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # Reference arm under torchrun: the reference's rasterizer is a CUDA extension, so it gets the same treatment as ours
    # (one camera per rank + the all-reduce of dL_dcolors, i.e. what train_contrastive_feature.py would do under DDP).
    # Only the CPU-port fallback (no oracle/_ref on this box) runs on rank 0 alone.
    ref_is_cuda = False
    if a.impl == "reference":
        from tests import common as _c
        ref_is_cuda = _c.have_ref("cf") and K == 32
        if world > 1 and rank != 0 and not ref_is_cuda:
            return 0
    import torch.distributed as dist
    use_dist = world > 1 and (a.impl == "ours" or ref_is_cuda)
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if use_dist:
        opts = None
        if a.allreduce_mode == "overlap":
            # the exchange runs beside the next forward's geometry kernels: give its CTAs priority over their queued blocks
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)

    # ---------------- implementation under test ----------------
    ref_kind = None
    R = None
    if a.impl == "ours":
        from seganygaussians_b200 import rasterizer as R, _lib
        _lib.load()
        R.set_blend_kernels(forward=a.fwd_kernel, backward=a.bwd_kernel)
        if a.binning != "default":
            R.set_binning(a.binning)
        Settings, Rast = R.GaussianRasterizationSettings, R.GaussianRasterizerContrastiveF
    else:
        from tests import common
        if common.have_ref("cf") and K == 32:
            mod = common.ref_module("cf")
            Settings, Rast = mod.GaussianRasterizationSettings, mod.GaussianRasterizer
            ref_kind = "reference-cuda-ext"
        else:
            if a.dump_outputs is not None:
                raise SystemExit("--dump-outputs needs a CUDA implementation; the CPU fallback of --impl reference has no timed steps")
            from seganygaussians_b200 import synthetic
            return reference_cpu_arm(a, wl, synthetic.scene(P, H, W, K))

    run = Runner(a, wl, world, rank, dev, use_dist, Settings, Rast, R)
    run.keep_color = a.dump_outputs is not None

    # ---------------- warm-up, then the timed regions ----------------
    sampler = ClockSampler(local_rank) if rank == 0 else None
    warm = max(a.warmup, 3)
    for _ in range(warm):
        run.step_resident()
    run.step_e2e()
    run.barrier()
    if a.impl == "ours":
        _lib.reset_launch_count()
    ms_total = run.timed(run.step_resident, a.steps, sampler)
    launches = _lib.launch_count() if a.impl == "ours" else None
    dumped = run.outputs() if a.dump_outputs is not None and rank == 0 else None    # before the e2e pass replaces the gradients
    ms_e2e = run.timed(run.step_e2e, a.steps)
    clocks = sampler.result() if sampler else None
    stage, stage_steps = None, min(a.steps, 20)
    if a.impl == "ours":           # per-stage CUDA-event times: a separate pass, the instrumentation stays out of the numbers above
        _lib.profile_read(reset=True)
        _lib.profile_enable(True)
        run.timed(run.step_resident, stage_steps)
        _lib.profile_enable(False)
        stage = _lib.profile_read(reset=True)

    n_used = world if use_dist else 1
    gp_per_step = float(P) * H * W * run.cameras_per_step
    value = gp_per_step * a.steps / (ms_total * 1e-3)
    e2e_value = gp_per_step * a.steps / (ms_e2e * 1e-3)
    R_inst, radii_vis, pairs_to_last = run.counters(a.impl == "ours")

    # ---------------- BASELINE configs[3]: 8-camera batch, strong scaling ----------------
    c4 = None
    if not a.no_c4 and a.workload == "c2":
        del run
        torch.cuda.empty_cache()
        c4 = c4_leg(a, world, rank, dev, use_dist, Settings, Rast, R)

    if rank != 0:
        if use_dist:
            dist.destroy_process_group()
        return 0
    if dumped is not None:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in dumped.items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)

    T_tiles = ((W + 15) // 16) * ((H + 15) // 16)
    strong = wl["cameras"] is not None
    line = {
        "metric": f"fwd+bwd Gaussians*pixels/s @K={K}", "value": value, "unit": "Gaussian*pixel/s",
        "n_gpus": world if (use_dist or a.impl != "ours") else a.gpus, "steps": a.steps, "warmup": warm,
        "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "impl": a.impl,
        "config": {"workload": wl["desc"], "P": P, "H": H, "W": W, "K": K, "cameras_per_step": gp_per_step / (float(P) * H * W),
                   "parallelism": f"camera-dp{n_used}" + ("+allreduce(dL_dcolors)" if use_dist else ""),
                   "l2": "inputs_exceed_l2 (features 128 MB + upstream gradient 265 MB + image 265 MB >> 126 MB L2)",
                   "P_visible": radii_vis, "R_instances": R_inst,
                   # work-proportional counters (SURVEY.md section 8(d)): S = pair tests a tile-per-CTA traversal would make at
                   # most (256 threads x every instance of the tile); n_contrib summed = pairs up to each pixel's last contributor
                   "S_pair_tests_upper_bound": 256 * R_inst, "pairs_up_to_last_contributor": pairs_to_last},
        "e2e": {"value": e2e_value, "unit": "Gaussian*pixel/s", "ms_per_step": ms_e2e / a.steps,
                "h2d_bytes_per_step": run_h2d(wl, n_used), "d2h_bytes_per_step": 8,
                "note": "camera from pinned host memory each step; loss scalar + num_rendered read back"},
        "clocks": clocks,
    }
    if a.impl == "ours":
        line["kernels"] = kernel_names(a, K)
        line["allreduce"] = None if not use_dist else (
            ("own multimem all-reduce" if a.allreduce == "multimem" else "ncclAllReduce") +
            (" on a side stream, gating only the next forward's blend stage" if a.allreduce_mode == "overlap" else ", serialised"))
        peak, peak_src = load_peaks()
        per_stage_bytes, step_bytes = algorithmic_bytes(P, R_inst, H * W, T_tiles, K)
        dom_name, (dom_ms, dom_n) = max(stage.items(), key=lambda kv: kv[1][0])
        dom_avg_ms = dom_ms / max(dom_n, 1)
        achieved = per_stage_bytes[dom_name] / (dom_avg_ms * 1e-3) / 1e9
        traffic = inst = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp) and a.workload == "c2":      # the committed capture is of the c2 workload
            try:
                prof = json.load(open(tp))
                traffic = prof.get(dom_name)
                inst = prof.get("inst_executed", {}).get(dom_name)
            except Exception:
                traffic = None
        step_ms = ms_total / a.steps
        line["roofline"] = {"bound": "hbm", "kernel": dom_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                            "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                            "algorithmic_bytes_per_launch": per_stage_bytes[dom_name], "avg_launch_ms": dom_avg_ms,
                            "share_of_step": dom_avg_ms * len(run_cams(wl, n_used)) / step_ms,
                            "timing": f"library stage events over a separate pass of {stage_steps} steps (instrumentation off in the value / e2e regions)"}
        if inst is not None and clocks and clocks.get("sm_mhz") and dom_avg_ms > 0:
            # the bound that actually holds for the blend kernels: warp instructions issued per second against the issue-slot
            # peak at the SM clock measured during the run (instruction count from the committed ncu capture, time live)
            peak_issue = 148 * 4 * clocks["sm_mhz"] * 1e6
            line["roofline"]["issue"] = {"warp_inst_per_launch": inst, "achieved_per_s": inst / (dom_avg_ms * 1e-3),
                                         "peak_per_s": peak_issue, "frac": inst / (dom_avg_ms * 1e-3) / peak_issue,
                                         "note": "issue-bound kernel: HBM frac is low by construction (DESIGN.md section 5)"}
        line["roofline_step"] = {"algorithmic_bytes_per_step": step_bytes,
                                 "achieved": step_bytes / (step_ms * 1e-3) / 1e9, "unit": "GB/s",
                                 "frac": step_bytes / (step_ms * 1e-3) / 1e9 / peak}
        line["stage_ms_per_step"] = {k: v[0] / stage_steps for k, v in stage.items()}
        line["gpu_launches"] = launches
    else:
        line["reference_kind"] = ref_kind
        line["gpu_launches"] = None
    if c4 is not None:
        line["c4"] = c4
    if world == 1 and not a.no_cpu_baseline:
        from seganygaussians_b200 import synthetic
        line["cpu_baseline"] = cpu_baseline(synthetic.scene(P, H, W, K), K)
        line["cpu_autograd_c1"] = cpu_autograd_c1()
    print(json.dumps(line))
    if use_dist:
        dist.destroy_process_group()
    return 0


def run_cams(wl, n_used):
    return [0] if wl["cameras"] is None else list(range(0, wl["cameras"], n_used))


def run_h2d(wl, n_used):
    return len(run_cams(wl, n_used)) * (16 + 16 + 3 + wl["K"]) * 4


def c4_leg(a, world, rank, dev, use_dist, Settings, Rast, R):
    """BASELINE.json configs[3]: SYN(3M, 1080x1920, K=32) x 8 cameras, camera i on rank i mod N, local accumulation of the
    feature gradient over a rank's cameras, ONE all-reduce of dL_dcolors [3M, 32] (384 MB) per batch.  Strong scaling: the
    batch is fixed, `value` = 8 * P * H * W * steps / time (max over ranks)."""
    wl = WORKLOADS["c4"]
    n_used = world if use_dist else 1
    steps = a.steps
    try:
        run = Runner(a, wl, world, rank, dev, use_dist, Settings, Rast, R)
        for _ in range(2):
            run.step_resident()
        run.step_e2e()
        ms = run.timed(run.step_resident, steps)
        ms_e2e = run.timed(run.step_e2e, steps)
        gp = float(wl["P"]) * wl["H"] * wl["W"] * wl["cameras"]
        R_inst, vis, pairs = run.counters(a.impl == "ours")
        out = {"workload": wl["desc"], "scaling": "strong", "cameras_per_batch": wl["cameras"], "cameras_per_rank": len(run.cams),
               "steps": steps, "ms_per_batch": ms / steps, "value": gp * steps / (ms * 1e-3), "unit": "Gaussian*pixel/s",
               "e2e": {"ms_per_batch": ms_e2e / steps, "value": gp * steps / (ms_e2e * 1e-3), "h2d_bytes_per_step": run.h2d_bytes, "d2h_bytes_per_step": 8},
               "allreduce_bytes": (wl["P"] * wl["K"] * 4) if use_dist else 0, "R_instances_last_camera": R_inst, "P_visible_last_camera": vis,
               "parallelism": f"camera-dp{n_used}: camera i -> rank i mod {n_used}" + ("; one all-reduce(dL_dcolors) per batch" if use_dist else "")}
        del run
        torch.cuda.empty_cache()
        return out
    except Exception as e:   # the headline line must not die with the secondary leg
        return {"workload": wl["desc"], "error": repr(e)}


def cpu_baseline(sc, K, max_seconds=40.0):
    """The CPU oracle port on the host cores.  Sample: the largest top-left crop of the SAME workload whose
    fwd+bwd is estimated to fit ~10-30 s (same Gaussians, same camera intrinsics, fewer pixel rows)."""
    from tests import common
    from oracle import oracle
    nthreads = oracle.max_threads()
    P, H, W = sc.P, sc.H, sc.W
    # the whole c2 frame takes ~15-30 s on 8 cores; keep full frame unless the box is small
    t0 = time.time()
    orc = common.run_oracle(sc, K, backward=True, nthreads=nthreads)
    dt = time.time() - t0
    return {"value": float(P) * H * W / dt, "unit": "Gaussian*pixel/s", "cores": nthreads, "kind": "port",
            "seconds": dt,
            "sample": f"1 fwd+bwd step of the full workload (P={P}, {H}x{W}, K={K}) with the C oracle port, {nthreads} OpenMP threads"}


def cpu_autograd_c1():
    """BASELINE.json configs[0]: SYN(10k, 256x256, K=3) forward + backward on the host through the PyTorch-autograd
    restatement (oracle/autograd_oracle.py, float64, one thread).  Reported beside the C port; not the headline."""
    try:
        from oracle import autograd_oracle
        from seganygaussians_b200 import synthetic
        P1, H1, W1, K1 = 10_000, 256, 256, 3
        sc1 = synthetic.scene(P1, H1, W1, K1)
        t0 = time.time()
        out = autograd_oracle.run_scene(sc1, K1)
        dt = time.time() - t0
        return {"value": float(P1) * H1 * W1 / dt, "unit": "Gaussian*pixel/s", "cores": 1, "kind": "port", "seconds": dt,
                "sample": f"1 fwd+bwd of SYN({P1}, {H1}x{W1}, K={K1}) (BASELINE configs[0]), torch.autograd float64, R={out.num_rendered}"}
    except Exception as e:   # pragma: no cover
        return {"value": None, "error": repr(e)}


def reference_cpu_arm(a, wl, sc):
    """Fallback of --impl reference when oracle/_ref is absent: the CPU oracle port as the reference arm."""
    cb = cpu_baseline(sc, wl["K"])
    line = {"metric": "fwd+bwd Gaussians*pixels/s @K=32", "value": cb["value"], "unit": "Gaussian*pixel/s", "n_gpus": a.gpus,
            "steps": 1, "warmup": 0, "ms_per_step": cb["seconds"] * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference", "reference_kind": "cpu-oracle-port",
            "config": {"workload": wl["desc"]}, "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "Gaussian*pixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    sys.exit(main())
