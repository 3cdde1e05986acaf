#!/usr/bin/env python
"""bench.py -- denoise-steps/sec of the FRESCO hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl fresco|reference] [--workload ...] [--dump-outputs DIR]

A "step" is one UNet forward of an SD-1.5-shaped random-init fp16 UNet with the FRESCO hooks installed through the
reference's own plug-in surface (apply_FRESCO_attn / apply_FRESCO_opt -> pipe.unet(...)):
  * FRESCO attention on the 6 decoder self-attention layers of up_blocks.2/3
    (cross-frame always; spatial-guided on schedule step 0; temporal-guided while t >= 350),
  * warp_tensor background fusion on the 4 decoder features on the optimisation steps.
Steps walk the reference's 15-step schedule (SURVEY Appendix A) cyclically.

  --gpus 1 (default)   BASELINE configs[1]: ONE batch of N=8 keyframes at 512x512 (CFG => 16 samples).  The headline.
  --gpus G > 1         BASELINE configs[3] (north_star's partition): ONE batch of N=16 keyframes FRAME-SHARDED over the
                       G ranks -- K/V all-gather per FRESCO layer, trajectory-sharded temporal attention (two
                       all-to-alls per layer while it is on) -- strong scaling of a fixed batch.  `value` counts
                       8-keyframe batch-steps (one step of the 16-frame batch = 2) so that it is the same unit as the
                       1-GPU line; the step is replayed from CUDA graphs (the per-rank batch is small enough to be
                       launch-bound in eager mode).  --workload replicas gives the round-1 independent-replica run.
  --workload config3   adds optimize_feature (20 Adam iterations, temporal + Gram-L1) on 10 of 15 steps, GMFlow's
                       correlation kernel on a per-batch preparation call inside the timed region.

Output: ONE JSON line (rank 0).  `value` = device-resident inputs; `e2e` = same call with pinned-host inputs/outputs
copied inside the timed region; `roofline` = the dominant kernel timed per launch with CUDA events; `kernels` = every
kernel of the hot path with algorithmic work (SURVEY 8d), CUDA-event time and fraction of the measured peak;
`gpu_eager_baseline` = the reference's math in PyTorch eager on the same GPU; `cpu_baseline` = the CPU oracle on a
bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_FRAMES = 8
N_FRAMES_SHARDED = 16
RES = 512
CHUNKS = 2
TIMESTEPS = [950 - 50 * i for i in range(20)]          # DDPMScheduler.set_timesteps(20), "leading"
WARMUP_STEPS = 5                                        # SDEdit warm-up: run timesteps[5:]
SCHEDULE = TIMESTEPS[WARMUP_STEPS:]                     # 15 steps: 700 .. 0
OPT_STEPS = TIMESTEPS[WARMUP_STEPS:15]                  # optimisation / warp active on t in 700..250
METRIC = "denoise-steps/sec"
UNIT = "steps/s"
CPU_THREADS_CAP = 32                                    # one policy for both CPU legs: min(host cores, 32)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"tflops": float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))),
                "tflops_burst": float(d.get("bf16_tflops", 1590.0)), "hbm_gbs": float(d.get("hbm_gbs", 6650.0)),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def load_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, per launch, from the committed
    `ncu --set full` capture of this same workload (profiles/r02_attn_traffic.json, else round 1's); None if absent."""
    for name in ("r02_attn_traffic.json", "r01_attn_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                d = json.load(f)
            return {"bytes_per_launch": d["traffic_bytes_per_launch"], "unit": "B", "source": d["source"]}
        except Exception:
            continue
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.lines = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------
# workload construction (fresco arm)
# --------------------------------------------------------------------------------------------
def schedule_state(i):
    """(spatial-guided on, temporal-guided on, optimisation / warp step) of schedule step i (src/pipe_FRESCO.py:171-174,
    run_fresco.py:232)"""
    return (i == 0, SCHEDULE[i] >= 350, SCHEDULE[i] in OPT_STEPS)


class Workload:
    def __init__(self, device, seed=0, n_frames=N_FRAMES, res=RES, optimise=False, shard=None, with_gmflow=False,
                 controlnet=False, warp=None):
        """shard = (world, rank): frame-sharded batch (config 4); n_frames is then the GLOBAL frame count and this
        rank feeds frames [rank*n/world, (rank+1)*n/world) of both CFG chunks through the UNet."""
        from fresco_b200 import diffusion_hacked as dh
        from fresco_b200 import flow_utils as fu
        from fresco_b200.harness import synth
        from fresco_b200.harness.sd15_unet import FakePipe, SD15UNet
        self.dh = dh
        self.device = device
        self.n = n_frames
        self.res = res
        torch.manual_seed(seed)
        unet = SD15UNet().to(device=device, dtype=torch.float16).eval()
        self.pipe = FakePipe(unet)
        self.shard = shard
        if shard is not None:
            world, rk = shard
            self.lo, self.hi = rk * n_frames // world, (rk + 1) * n_frames // world
        else:
            self.lo, self.hi = 0, n_frames
        n_local = self.hi - self.lo
        self.proc = dh.apply_FRESCO_attn(self.pipe, shard=None if shard is None else (shard[0], shard[1], None))
        ctrl = self.proc.controller
        ctrl.disable_controller()
        dh.disable_FRESCO_opt(self.pipe)
        lat = res // 8
        g = torch.Generator().manual_seed(seed + 1)
        self.latents_host = torch.randn(n_frames, 4, lat, lat, generator=g)[self.lo:self.hi].half().pin_memory()
        prompt_full = torch.randn(CHUNKS, n_frames, 77, 768, generator=g)
        self.prompt_host = prompt_full[:, self.lo:self.hi].reshape(CHUNKS * n_local, 77, 768).half().pin_memory()
        self.out_host = torch.empty(CHUNKS * n_local, 4, lat, lat, dtype=torch.float16).pin_memory()
        self.latents = self.latents_host.to(device)
        self.prompt = self.prompt_host.to(device)
        # per-batch FRESCO parameters (what get_flow_and_interframe_paras produces, with synthetic flow)
        self.flows, self.occs = synth.smooth_flows(n_frames, res, res, device, seed=seed + 2)
        self.imgs = synth.frames(n_frames, res, res, device, seed + 3)
        self.saliency = synth.saliency(n_frames, device, seed + 4)
        self.attn_mask = dh.cross_frame_attn_masks(self.occs[1])
        fm, bm, im = [], [], []
        for scale in (8.0, 16.0):
            f, b, m = fu.get_mapping_ind(self.flows[1], self.occs[1], self.imgs, scale=scale)
            fm.append(f), bm.append(b), im.append(m)
        self.interattn_paras = {"fwd_mappings": fm, "bwd_mappings": bm, "interattn_masks": im}
        self.kv_len = {int(m.shape[1]): int(m.sum().item()) for m in self.attn_mask}
        # reference pass: store the 6 decoder self-attention inputs (get_intraframe_paras, store=True)
        ctrl.clear_store()
        ctrl.enable_store()
        with torch.no_grad():
            self.pipe.unet(torch.cat([self.latents] * 2), TIMESTEPS[-1], encoder_hidden_states=self.prompt,
                           return_dict=False)
        ctrl.disable_store()
        self.gmflow_feats = None
        if with_gmflow:
            # GMFlow's 1/8-resolution features of the N frame pairs (random, LayerNorm scale): the operand of G1
            gg = torch.Generator().manual_seed(seed + 5)
            f0 = torch.randn(n_frames, 128, lat, lat, generator=gg).to(device)
            self.gmflow_feats = (f0, torch.roll(f0, (1, -2), (2, 3)) + 0.3 * torch.randn(f0.shape, generator=gg).to(device))
        self.graphs = None
        self.residuals = None
        if controlnet:
            # ControlNet-HED residuals (BASELINE configs[4]): random tensors with the shapes of SD1.5's 12 down-block
            # residuals + the mid-block residual, added inside the UNet forward exactly as diffusers does
            gg = torch.Generator().manual_seed(seed + 6)
            shapes = [(320, lat)] * 3 + [(320, lat // 2)] + [(640, lat // 2)] * 2 + [(640, lat // 4)] + \
                     [(1280, lat // 4)] * 2 + [(1280, lat // 8)] * 3
            mk = lambda c, s: (0.1 * torch.randn(CHUNKS * n_local, c, s, s, generator=gg)).half().to(device)
            self.residuals = (tuple(mk(c, s) for c, s in shapes), mk(1280, lat // 8))
        if shard is not None:
            # frame-sharded batch: FRESCO attention (K/V all-gather, trajectory all-to-alls) + the warp_tensor fusion of
            # config 2 with the chain re-sharded by channel (two all-to-alls per decoder feature)
            gram = []
            if optimise:
                # + config 3's work on the sharded batch: Gram targets of this rank's frames, temporal term through the
                # ring-halo exchange (one boundary frame per Adam iteration to each neighbour)
                with torch.no_grad():
                    feats = self.pipe.unet(torch.cat([self.latents] * 2), TIMESTEPS[-1], encoder_hidden_states=self.prompt,
                                           return_dict=False)[1:]
                gram = dh.gram_targets(feats)
            dh.apply_FRESCO_opt(self.pipe, steps=OPT_STEPS, flows=self.flows, occs=self.occs, correlation_matrix=gram,
                                intra_weight=1e2, iters=20, optimize_temporal=optimise, saliency=self.saliency,
                                shard=(shard[0], shard[1], None))
            return
        if optimise:
            # BASELINE configs[2]: FRESCO feature optimisation (20 Adam iterations, temporal + Gram-L1 loss) on the 4
            # decoder features on the optimisation steps, Gram targets from the reference pass (get_intraframe_paras)
            with torch.no_grad():
                feats = self.pipe.unet(torch.cat([self.latents] * 2), TIMESTEPS[-1], encoder_hidden_states=self.prompt,
                                       return_dict=False)[1:]
            self.gram = dh.gram_targets(feats)
            dh.apply_FRESCO_opt(self.pipe, steps=OPT_STEPS, flows=self.flows, occs=self.occs,
                                correlation_matrix=self.gram, intra_weight=1e2, iters=20, optimize_temporal=True,
                                saliency=self.saliency)
        else:
            # BASELINE configs[1]: warp-only decoder fusion on the optimisation steps (optimize_feature early-outs:
            # no Gram targets, optimize_temporal=False)
            dh.apply_FRESCO_opt(self.pipe, steps=OPT_STEPS, flows=self.flows, occs=self.occs, correlation_matrix=[],
                                optimize_temporal=False, saliency=self.saliency)

    def set_state(self, i):
        """absolute flag state of schedule step i (what the incremental toggles of pipe_FRESCO.inference add up to)"""
        ctrl = self.proc.controller
        intra, inter, _ = schedule_state(i)
        if i == 0 or self.graphs is not None:
            ctrl.enable_controller(interattn_paras=self.interattn_paras, attn_mask=self.attn_mask)
        if not intra:
            ctrl.disable_intraattn()
        if not inter:
            ctrl.disable_interattn()

    def _forward(self, i, lat, prompt):
        if self.gmflow_feats is not None and i == 0:
            # per-batch preparation inside the timed region of config 3: the all-pairs correlation of GMFlow
            from fresco_b200 import gmflow_matching
            gmflow_matching.global_correlation_softmax(self.gmflow_feats[0], self.gmflow_feats[1], pred_bidir_flow=True)
        kw = {}
        if self.residuals is not None:
            kw = {"down_block_additional_residuals": self.residuals[0], "mid_block_additional_residual": self.residuals[1]}
        return self.pipe.unet(torch.cat([lat] * 2), SCHEDULE[i], encoder_hidden_states=prompt, return_dict=False, **kw)[0]

    @torch.no_grad()
    def build_graphs(self):
        """one CUDA graph per distinct flag state of the schedule (4 of them), static input / output buffers"""
        self.graphs = {}
        self.lat_static = self.latents.clone()
        self.prompt_static = self.prompt.clone()
        side = torch.cuda.Stream()
        for i in range(len(SCHEDULE)):
            key = schedule_state(i)
            if key in self.graphs:
                continue
            self.set_state(i)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                      # warm-up on a side stream (plans, caches, autotune)
                for _ in range(2):
                    self._forward(i, self.lat_static, self.prompt_static)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            if key[0]:
                self.proc.controller.enable_intraattn()        # ring index of the stored reference features back to 0
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self._forward(i, self.lat_static, self.prompt_static)
            self.graphs[key] = (g, out)

    @torch.no_grad()
    def step(self, k, host_io=False):
        i = k % len(SCHEDULE)
        if self.graphs is not None:
            if host_io:
                self.lat_static.copy_(self.latents_host, non_blocking=True)
                self.prompt_static.copy_(self.prompt_host, non_blocking=True)
            g, out = self.graphs[schedule_state(i)]
            g.replay()
        else:
            self.set_state(i)
            if host_io:
                lat = self.latents_host.to(self.device, non_blocking=True)
                prompt = self.prompt_host.to(self.device, non_blocking=True)
            else:
                lat, prompt = self.latents, self.prompt
            out = self._forward(i, lat, prompt)
        if host_io:
            self.out_host.copy_(out, non_blocking=True)
        return out


@torch.no_grad()
def sharded_selfcheck(wl, world, rank):
    """Every N>1 run: one level-A FRESCO layer (all three guidance modes) on this rank's frame shard -- K/V all-gather,
    trajectory all-to-alls -- must be BIT-identical to the same layer computed unsharded on the full batch."""
    from fresco_b200 import diffusion_hacked as dh
    from fresco_b200.dist import ShardedFRESCOAttention
    N, dev = wl.n, wl.device
    L, C, heads = (wl.res // 16) ** 2, 640, 8
    g = torch.Generator().manual_seed(99)                       # same tensors on every rank
    q, k, v, rq, rk = ((torch.randn(CHUNKS * N, L, C, generator=g) * (2.0 if i == 1 else 1.0)).half().to(dev) for i in range(5))
    ctrl = dh.AttentionControl()
    ctrl.stored_attn["decoder_attn"] = [q]                       # only switches use_intraattn on; ref_q / ref_k are passed in
    ctrl.enable_controller(interattn_paras=wl.interattn_paras, attn_mask=wl.attn_mask)
    full = ShardedFRESCOAttention(ctrl, 1, 0, CHUNKS)(q, k, v, heads, ref_q=rq, ref_k=rk)
    sel = torch.cat([torch.arange(c * N + wl.lo, c * N + wl.hi) for c in range(CHUNKS)]).to(dev)
    mine = ShardedFRESCOAttention(ctrl, world, rank, CHUNKS)(q[sel].contiguous(), k[sel].contiguous(), v[sel].contiguous(),
                                                           heads, ref_q=rq[sel].contiguous(), ref_k=rk[sel].contiguous())
    same = bool(torch.equal(mine, full[sel]))
    t = torch.tensor([1 if same else 0], device=dev)
    import torch.distributed as dist
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return {"bit_identical_to_unsharded": bool(t.item() == 1), "layer": "level A: [%d,%d,%d], %d heads, spatial + cross-frame "
            "(Lk=%d) + temporal" % (CHUNKS * N, L, C, heads, wl.kv_len[L])}


def dist_setup():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        else:
            dist.init_process_group("gloo")
    return world, rank, local


def timed_region(wl, steps, warmup, host_io, world):
    """(ms of the `steps` timed steps, the output of the last one)"""
    import torch.distributed as dist
    for k in range(warmup):
        wl.step(k, host_io)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    out = None
    for k in range(steps):
        out = wl.step(k, host_io)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms, out


def dump_outputs(directory, arrays):
    """--dump-outputs: every array as <directory>/<name>.npy in float32, so that two builds can be compared output for
    output on the same seeded inputs"""
    import numpy as np
    os.makedirs(directory, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), t.detach().float().cpu().numpy())


# --------------------------------------------------------------------------------------------
# per-kernel table
# --------------------------------------------------------------------------------------------
def summarise_profile(prof, peaks):
    """ops.PROFILE entries -> {tag: {bound, work, ms (mean of launches), achieved, peak, frac, launches}}"""
    by_tag = {}
    for tag, work, a, b, bound in prof:
        by_tag.setdefault(tag, []).append((work, a.elapsed_time(b), bound))
    table = {}
    for tag, ent in sorted(by_tag.items()):
        ms = sum(t for _, t, _ in ent) / len(ent)
        work, bound = ent[0][0], ent[0][2]
        if bound == "tensor":
            ach, peak, unit = work / (ms * 1e-3) / 1e12, peaks["tflops"], "TFLOP/s"
        else:
            ach, peak, unit = work / (ms * 1e-3) / 1e9, peaks["hbm_gbs"], "GB/s"
        table[tag] = {"bound": bound, "work": work, "ms": round(ms, 4), "achieved": round(ach, 1), "peak": peak,
                      "unit": unit, "frac": round(ach / peak, 4), "launches": len(ent),
                      "total_ms": round(sum(t for _, t, _ in ent), 3)}
    return table


@torch.no_grad()
def side_pass_kernels(wl, peaks):
    """The kernels config 2 does not launch (optimize_feature at the 4 decoder shapes of config 3, GMFlow's correlation),
    each timed with CUDA events through ops.PROFILE -- outside the timed region, after it."""
    from fresco_b200 import diffusion_hacked as dh, gmflow_matching, ops
    dev = wl.device
    N = wl.n
    g = torch.Generator().manual_seed(123)
    ops.PROFILE = []
    for C, h in [(1280, 8), (1280, 16), (1280, 32), (640, 64)]:
        sample = torch.randn(2 * N, C, h, h, generator=g).half().to(dev)
        ref = (sample.float() + 0.5 * torch.randn(2 * N, C, h, h, generator=g).to(dev)).half()
        target = dh.gram_targets([ref])[0]
        for _ in range(2):                                             # first call warms caches (adjoint lists, attributes)
            keep = len(ops.PROFILE)
            dh.optimize_feature(sample, wl.flows, wl.occs, correlation_matrix=[target], iters=4)
            if _ == 0:
                del ops.PROFILE[keep:]
        del target
    lat = wl.res // 8
    f0 = torch.randn(N, 128, lat, lat, generator=g).to(dev)
    f1 = torch.roll(f0, (1, -2), (2, 3)) + 0.3 * torch.randn(f0.shape, generator=g).to(dev)
    for _ in range(3):
        keep = len(ops.PROFILE)
        gmflow_matching.global_correlation_softmax(f0, f1, pred_bidir_flow=True)
        if _ == 0:
            del ops.PROFILE[keep:]
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    return summarise_profile(prof, peaks)


def gpu_eager_baseline(wl, ours):
    """The reference's math in PyTorch eager on this GPU (oracle/ref_gpu.py) for one level-B FRESCO layer, warp_tensor on
    the layer-3 decoder feature and optimize_feature at layer 3, next to the same calls through libfresco_b200.so."""
    from fresco_b200 import diffusion_hacked as dh, flow_utils as fu
    from oracle import ref_gpu
    dev, N = wl.device, wl.n
    g = torch.Generator().manual_seed(7)
    res = {}

    def timeit(fn, iters):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    # ---- one level-B FRESCO layer (all three guidance modes on: schedule step 0)
    L, C, heads = (wl.res // 8) ** 2, 320, 8
    x = torch.randn(2 * N, L, C, generator=g).half().to(dev)
    refh = torch.randn(2 * N, L, C, generator=g).half().to(dev)
    w = [(torch.randn(C, C, generator=g) / C ** 0.5).half().to(dev) for _ in range(4)]
    bo = torch.zeros(C, dtype=torch.float16, device=dev)
    mask = [m for m in wl.attn_mask if m.shape[1] == L][0]
    idx = [i for i, f in enumerate(wl.interattn_paras["fwd_mappings"]) if f.shape[2] == L][0]
    fm, bm, im = (wl.interattn_paras[k][idx] for k in ("fwd_mappings", "bwd_mappings", "interattn_masks"))
    t_ref = timeit(lambda: ref_gpu.fresco_layer(x, *w, bo, heads, mask, refh, fm, bm, im), 3)

    class _Attn(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.heads = heads
            self.spatial_norm = self.group_norm = None
            self.norm_cross = self.residual_connection = False
            self.rescale_output_factor = 1.0
            self.to_q, self.to_k, self.to_v = (torch.nn.Linear(C, C, bias=False) for _ in range(3))
            self.to_out = torch.nn.ModuleList([torch.nn.Linear(C, C), torch.nn.Dropout(0.0)])
    attn = _Attn().to(dev).half()
    with torch.no_grad():
        for lin, ww in zip((attn.to_q, attn.to_k, attn.to_v, attn.to_out[0]), w):
            lin.weight.copy_(ww)
        attn.to_out[0].bias.zero_()
    ctrl = dh.AttentionControl()
    proc = dh.FRESCOAttnProcessor2_0(2, ctrl)
    ctrl.stored_attn["decoder_attn"] = [refh]

    ctrl.enable_controller(interattn_paras=wl.interattn_paras, attn_mask=wl.attn_mask)

    def ours_layer():
        ctrl.enable_intraattn()                                # ring index of the stored reference feature back to 0
        with torch.no_grad():
            return proc(attn, x)
    t_ours = timeit(ours_layer, 5)
    with torch.no_grad():
        err = (ours_layer().float() - ref_gpu.fresco_layer(x, *w, bo, heads, mask, refh, fm, bm, im).float()).abs().max().item()
    res["fresco_layer_level_B"] = {"reference_eager_ms": round(t_ref, 3), "fresco_b200_ms": round(t_ours, 3),
                                   "speedup": round(t_ref / t_ours, 2), "max_abs_diff": round(err, 5),
                                   "shape": "[%d,%d,%d] fp16, Lk=%d, spatial + cross-frame + temporal" % (2 * N, L, C, wl.kv_len[L])}
    # ---- warp_tensor on the layer-3 decoder feature
    feat = torch.randn(2 * N, 640, 64, 64, generator=g).half().to(dev)
    t_ref = timeit(lambda: ref_gpu.warp_tensor(feat, wl.flows, wl.occs, wl.saliency, 2), 3)
    t_ours = timeit(lambda: fu.warp_tensor(feat, wl.flows, wl.occs, wl.saliency, 2), 5)
    res["warp_tensor_layer3"] = {"reference_eager_ms": round(t_ref, 3), "fresco_b200_ms": round(t_ours, 3),
                                 "speedup": round(t_ref / t_ours, 2), "shape": "[16,640,64,64] fp16"}
    # ---- optimize_feature at layer 3 (20 Adam iterations, temporal + Gram-L1)
    reff = (feat.float() + 0.5 * torch.randn(feat.shape, generator=g).to(dev)).half()
    target = dh.gram_targets([reff])[0]
    dense = target.dense()                       # what the reference stores and reads back every iteration
    t_ref = timeit(lambda: ref_gpu.optimize_feature(feat, wl.flows, wl.occs, dense, iters=20), 1)
    del dense
    t_ours = timeit(lambda: dh.optimize_feature(feat, wl.flows, wl.occs, correlation_matrix=[target], iters=20), 2)
    res["optimize_feature_layer3"] = {"reference_eager_ms": round(t_ref, 2), "fresco_b200_ms": round(t_ours, 2),
                                      "speedup": round(t_ref / t_ours, 2), "shape": "[16,640,64,64], 20 Adam iterations"}
    res["note"] = ("reference math restated with the reference's own torch calls (oracle/ref_gpu.py: F.scaled_dot_product_"
                   "attention, mask indexing + repeat, gather, grid_sample, fp32 bmm + autograd + torch.optim.Adam), eager, "
                   "same GPU, same inputs; CUDA events")
    return res


# --------------------------------------------------------------------------------------------
# CPU baseline / reference arm (oracle port; see oracle/ref_step.py)
# --------------------------------------------------------------------------------------------
def cpu_reference_line(args, as_reference_arm):
    from oracle import ref_step
    cores = min(os.cpu_count() or 1, CPU_THREADS_CAP)
    torch.set_num_threads(cores)
    steps = args.steps if as_reference_arm else 1
    warm = args.warmup if as_reference_arm else 0
    res = ref_step.run(n_full=N_FRAMES, n_sample=args.cpu_sample_frames, res=RES, schedule=SCHEDULE,
                       opt_steps=OPT_STEPS, steps=steps, warmup=warm, max_seconds=args.cpu_budget_s)
    cb = {"value": res["steps_per_s"], "unit": UNIT, "cores": cores, "kind": "port", "sample": res["sample"]}
    return cb, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=15)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="fresco", choices=["fresco", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the kernels side pass and the GPU eager baseline")
    ap.add_argument("--cpu-sample-frames", type=int, default=2)
    ap.add_argument("--cpu-budget-s", type=float, default=150.0)
    ap.add_argument("--workload", default="auto", choices=["auto", "config2", "config3", "config4", "config4opt", "config5", "replicas"],
                    help="auto: config2 on one GPU, config4 (ONE N=16 batch frame-sharded) on several; config3: + feature "
                         "optimisation and GMFlow's correlation kernel; replicas: one independent N=8 batch per GPU")
    ap.add_argument("--graphs", default="auto", choices=["auto", "on", "off"],
                    help="replay the step from CUDA graphs (auto: on for the frame-sharded workload)")
    ap.add_argument("--profile-mode", action="store_true",
                    help="for ncu captures only: 1 warm-up + --steps, no e2e / cpu baseline; never a bench value")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last timed step's output to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "fresco" and not args.profile_mode:
        args.warmup = max(args.warmup, 3)

    if args.impl == "reference" and int(os.environ.get("RANK", "0")) != 0:
        return                                   # under torchrun only rank 0 runs (and prints) the CPU arm
    world, rank, local = (1, 0, 0) if args.impl == "reference" else dist_setup()
    workload = args.workload
    if workload == "auto":
        workload = "config2" if world == 1 else "config4"
    if workload == "replicas":
        workload = "config2"
        replicas = True
    else:
        replicas = world > 1 and workload not in ("config4", "config4opt", "config5")
    config = {"workload": "N=8 keyframes 512x512 (CFG batch 16), SD1.5-shaped random-init fp16 UNet, FRESCO "
                          "attention (cross-frame + spatial step 0 + temporal t>=350) on 6 decoder layers + "
                          "warp_tensor fusion on 4 decoder features; 15-step DDPM schedule t=700..0 walked cyclically",
              "frames": N_FRAMES, "resolution": RES,
              "parallelism": "one GPU" if world == 1 else "replicas x%d (one 8-keyframe batch per GPU)" % world,
              "l2": "working set (1.7 GB weights + activations) >> 126 MB L2, no explicit flush"}

    if args.impl == "reference":
        config["parallelism"] = "host cores only (rank 0); n_gpus echoes --gpus"
        cb, res = cpu_reference_line(args, True)
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
                "steps": res["steps"], "warmup": res["warmup"], "ms_per_step": round(res["raw_ms_per_step"], 1),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "ms_per_step is the measured time of one bounded-sample step; value is that sample scaled to the full "
                        "N=8 step by algorithmic work (see cpu_baseline.sample): full-step ms = %.0f" % (1000.0 / cb["value"]),
                "detail": res["detail"]}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl fresco needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    from fresco_b200 import _lib, ops
    _lib.lib()
    n_frames = N_FRAMES
    res = RES
    if workload == "config5":
        # BASELINE configs[4]: N=8 keyframes at 768x768 + ControlNet residuals, frame-sharded over the ranks (1 GPU: all 8)
        res = 768
        wl = Workload(device, seed=0, n_frames=n_frames, res=res, shard=(world, rank) if world > 1 else None, controlnet=True)
        config.update({"workload": "N=8 keyframes 768x768 (CFG batch 16) + ControlNet-shaped down/mid residuals, SD1.5-shaped "
                       "random-init fp16 UNet, FRESCO attention on 6 decoder layers (L = 9216 / 2304)" +
                       " + warp_tensor fusion on 4 decoder features" + (", frame-sharded over the ranks" if world > 1 else ""),
                       "resolution": res,
                       "parallelism": "one GPU" if world == 1 else "frame-sharded x%d (strong scaling of one batch)" % world})
    elif workload in ("config4", "config4opt"):
        # every rank must build the same per-batch parameters (same seed); only the frame slice differs
        n_frames = N_FRAMES_SHARDED
        wl = Workload(device, seed=0, n_frames=n_frames, shard=(world, rank), optimise=workload == "config4opt")
        config.update({"workload": "ONE batch of N=16 keyframes 512x512 (CFG batch 32) frame-sharded over the ranks, SD1.5-"
                       "shaped random-init fp16 UNet, FRESCO attention on 6 decoder layers: one NCCL all-gather of the "
                       "compacted K/V per layer + trajectory-sharded temporal attention (two all-to-alls per layer while "
                       "it is on) + warp_tensor fusion on 4 decoder features re-sharded by channel (two all-to-alls each); "
                       "value counts 8-keyframe batch-steps (one step of this batch = 2)",
                       "frames": n_frames, "parallelism": "frame-sharded x%d (strong scaling of one batch)" % world})
        if workload == "config4opt":
            config["workload"] += ("; + optimize_feature (20 Adam iterations, temporal + Gram-L1) on the 4 decoder features "
                                   "on 10 of 15 steps, sharded by frames: ring halo of one boundary frame per iteration")
    else:
        wl = Workload(device, seed=rank, optimise=workload == "config3", with_gmflow=workload == "config3")
    if workload == "config3":
        config["workload"] += ("; + optimize_feature (20 Adam iters, temporal + Gram-L1) on 4 decoder features, 10 of 15 "
                               "steps; + GMFlow global correlation (8 pairs, 128 x 64 x 64, bidirectional) once per cycle")
    shard_check = sharded_selfcheck(wl, world, rank) if (world > 1 and workload in ("config4", "config4opt", "config5")) else None
    if shard_check is not None and not shard_check["bit_identical_to_unsharded"]:
        raise SystemExit("config 4: the frame-sharded layer is not bit-identical to the unsharded one")
    sharded = world > 1 and workload in ("config4", "config4opt", "config5")
    use_graphs = args.graphs == "on" or (args.graphs == "auto" and sharded)
    graph_note = None
    if use_graphs:
        try:
            wl.build_graphs()
        except Exception as e:                        # never hide the number: fall back to eager and say why
            wl.graphs = None
            graph_note = "graph capture failed, eager: %r" % (e,)
            torch.cuda.synchronize()
    config["execution"] = "CUDA graphs (one per flag state of the schedule)" if wl.graphs is not None else "eager"
    if graph_note:
        config["execution"] += " (" + graph_note + ")"

    # ---- value: inputs resident in HBM
    peaks = load_peaks()
    sampler = ClockSampler(local)
    ops.PROFILE = [] if wl.graphs is None else None
    launches0 = _lib.launch_count()
    sampler.start()
    ms, last_out = timed_region(wl, args.steps, args.warmup, False, world)
    clocks = sampler.stop()
    launches = _lib.launch_count() - launches0
    prof = ops.PROFILE
    ops.PROFILE = None
    if args.dump_outputs:
        # the noise prediction of the last timed step (a rank's frame shard when sharded); saved before any further step
        # can overwrite a graph's static output buffer
        dump_outputs(args.dump_outputs, {"noise_pred" if world == 1 else "noise_pred_rank%d" % rank: last_out})
    prof_steps = args.steps + args.warmup
    if wl.graphs is not None:
        # launches inside a replayed graph are not seen by the library's counter: count one eager cycle instead, and
        # take the per-kernel CUDA-event times from it (events cannot be recorded inside a captured graph)
        graphs, wl.graphs = wl.graphs, None
        for k in range(2):
            wl.step(k)
        ops.PROFILE = []
        launches0 = _lib.launch_count()
        for k in range(len(SCHEDULE)):
            wl.step(k)
        torch.cuda.synchronize()
        launches = (_lib.launch_count() - launches0) * (args.steps + args.warmup) / float(len(SCHEDULE))
        prof, ops.PROFILE = ops.PROFILE, None
        prof_steps = len(SCHEDULE)
        wl.graphs = graphs
    # launches counted above include the warm-up steps: rescale to the timed steps only
    gpu_launches = int(round(launches * args.steps / float(args.steps + args.warmup)))
    if args.profile_mode:
        print(json.dumps({"profile_mode": True, "ms_per_step": ms / args.steps, "note": "not a bench value"}))
        return
    # ---- e2e: pinned-host inputs / outputs copied inside the timed region
    ms_e2e, _ = timed_region(wl, args.steps, 1, True, world)

    units = (n_frames / float(N_FRAMES)) if workload in ("config4", "config4opt", "config5") else (world if replicas else 1)
    value = units * args.steps / (ms / 1000.0)
    e2e_value = units * args.steps / (ms_e2e / 1000.0)
    h2d = wl.latents_host.numel() * 2 + wl.prompt_host.numel() * 2
    d2h = wl.out_host.numel() * 2

    # ---- per-kernel table + roofline of the dominant kernel: cross-frame attention at level B (L=4096, d=40)
    kernels = summarise_profile(prof, peaks)
    L_b = (res // 8) ** 2
    n_q = 2 * (wl.hi - wl.lo)
    dom_tag = "attn_d40_L%d_Lk%d" % (L_b, wl.kv_len[L_b])
    roof = None
    if dom_tag in kernels:
        kd = kernels[dom_tag]
        attn_ms = sum(v["total_ms"] for t, v in kernels.items() if t.startswith("attn_"))
        ours_ms = sum(v["total_ms"] for v in kernels.values())
        roof = {"kernel": "%s (cross-frame, L=%d, Lk=%d, B=%d, 8 heads)" % (_lib.lib().fresco_attn_variant(40).decode(), L_b,
                                                                                wl.kv_len[L_b], n_q),
                "bound": "tensor", "achieved": kd["achieved"], "peak": peaks["tflops"], "unit": "TFLOP/s",
                "frac": kd["frac"], "traffic": load_traffic(), "peak_source": peaks["source"],
                "algorithmic_flops_per_launch": kd["work"], "avg_launch_ms": kd["ms"], "launches_timed": kd["launches"],
                "share_of_step_time": round(kd["total_ms"] / (prof_steps / float(args.steps) * ms), 4)
                if wl.graphs is None else None,
                "all_attention_ms_per_step": round(attn_ms / prof_steps, 3),
                "fresco_kernels_ms_per_step": round(ours_ms / prof_steps, 3),
                "timed": "live in the timed region" if wl.graphs is None else "one eager cycle right after the graph-replayed timed region"}

    line = {"metric": METRIC, "value": round(value, 4), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True,
            "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic", "config": config, "clocks": clocks,
            "e2e": {"value": round(e2e_value, 4), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": round(ms_e2e / args.steps, 3)},
            "gpu_launches": gpu_launches, "roofline": roof, "kernels": kernels, "kv_len": wl.kv_len}
    if sharded:
        line["batch_steps_per_s"] = round(args.steps / (ms / 1000.0), 4)        # steps of the 16-frame batch itself
        line["sharded_check"] = shard_check
    if rank == 0:
        if world == 1 and not args.no_extras and workload in ("config2", "config3"):
            try:
                line["kernels"].update(side_pass_kernels(wl, peaks))
            except Exception as e:
                line["kernels_side_pass_error"] = repr(e)
            try:
                line["gpu_eager_baseline"] = gpu_eager_baseline(wl, kernels)
            except Exception as e:
                line["gpu_eager_baseline"] = {"error": repr(e)}
        if not args.no_cpu_baseline and world == 1:
            try:
                cb, _ = cpu_reference_line(args, False)
                line["cpu_baseline"] = cb
            except Exception as e:  # the baseline is a reported extra; never hide the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                                        "sample": "failed: %r" % (e,)}
        print(json.dumps(line), flush=True)
    if world > 1:
        # Leave without tearing NCCL down: destroying a process group whose collectives live in captured CUDA graphs
        # hung for the full timeout on the 2-GPU box (profiles/README.md); everything is printed and flushed by now.
        import torch.distributed as dist
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
