"""Generate golden vectors by running the REAL reference (the original FRESCO project) on CPU.

Only regenerating the fixtures needs the original project; the tests read the committed .npz files:

    FRESCO_REFERENCE_DIR=<checkout of FRESCO> python tests/golden/make_golden.py [--set b | --set control]

The reference imports two diffusers names and matplotlib at module top
(src/diffusion_hacked.py:7-8, src/utils.py:5); neither is used on the path we
exercise, so they are stubbed in ``sys.modules``.  Outputs: small ``.npz``
fixtures next to this script, consumed by tests/test_oracle_golden.py (oracle
vs reference) and by the ``-m gpu`` parity tests.
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get("FRESCO_REFERENCE_DIR", "")


def import_reference():
    for name, attrs in (
        ("diffusers", {}),
        ("diffusers.models", {}),
        ("diffusers.models.unet_2d_condition", {"UNet2DConditionOutput": object}),
        ("diffusers.models.attention_processor", {"AttnProcessor2_0": object}),
        ("matplotlib", {}),
        ("matplotlib.pyplot", {}),
    ):
        if name not in sys.modules:
            m = types.ModuleType(name)
            for k, v in attrs.items():
                setattr(m, k, v)
            sys.modules[name] = m
    if not os.path.isdir(REF):
        raise SystemExit("set FRESCO_REFERENCE_DIR to a checkout of the original FRESCO project")
    os.chdir(REF)
    sys.path.insert(0, REF)
    import src.diffusion_hacked as dh   # noqa
    import src.flow_utils as fu         # noqa
    from gmflow import geometry, matching  # noqa  (path appended by the reference itself)
    import src.utils as ut              # noqa
    return dh, fu, geometry, matching, ut


class FakeAttn(torch.nn.Module):
    """The attributes FRESCOAttnProcessor2_0 reads from diffusers' Attention."""

    def __init__(self, c, heads, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.heads = heads
        self.spatial_norm = None
        self.group_norm = None
        self.norm_cross = False
        self.residual_connection = False
        self.rescale_output_factor = 1.0
        self.to_q = torch.nn.Linear(c, c, bias=False)
        self.to_k = torch.nn.Linear(c, c, bias=False)
        self.to_v = torch.nn.Linear(c, c, bias=False)
        self.to_out = torch.nn.ModuleList([torch.nn.Linear(c, c), torch.nn.Dropout(0.0)])
        with torch.no_grad():
            for p in self.parameters():
                p.copy_(torch.randn(p.shape, generator=g) * (2.0 / c ** 0.5 if p.ndim == 2 else 0.1))


def smooth_flows(n, H, W, seed, mag):
    g = torch.Generator().manual_seed(seed)
    coarse = torch.randn(n, 2, 4, 4, generator=g) * mag
    fwd = F.interpolate(coarse, size=(H, W), mode="bicubic", align_corners=False)
    bwd = -fwd + 0.5 * F.interpolate(torch.randn(n, 2, 4, 4, generator=g), size=(H, W), mode="bicubic")
    return fwd, bwd


def scenario_b(dh, fu, geometry, matching, ut):
    """Second fixture set (``python tests/golden/make_golden.py --set b``): an ODD number of frames, a NON-SQUARE
    plane and head_dim 80 (SD1.5 level A), so that nothing in the oracle or the kernels can silently rely on
    N being even, h == w or d == 40.  Same reference entry points as set A."""
    torch.manual_seed(1)
    torch.set_grad_enabled(False)
    N, H, W = 3, 64, 96
    fwd, bwd = smooth_flows(N, H, W, 21, 4.0)
    fo, bo = geometry.forward_backward_consistency_check(fwd, bwd)
    imgs = torch.rand(N, 3, H, W) * 2 - 1
    bocc = torch.clamp(bo + (torch.rand(N, H, W) > 0.85).float(), 0, 1)
    res = {"fwd": fwd.numpy(), "bwd": bwd.numpy(), "fwd_occ": fo.numpy(), "bwd_occ": bocc.numpy(), "imgs": imgs.numpy()}

    # mapping at scale 8 (8 x 12 tokens)
    fm, bm, im = fu.get_mapping_ind(bwd, bocc, imgs, scale=8.0)
    res.update(fwd_map=fm.numpy(), bwd_map=bm.numpy(), inter_mask=im.numpy())

    # attention, all 8 flag combinations, C = 160 / 2 heads => head_dim 80
    C, heads, chunks = 160, 2, 2
    L = (H // 8) * (W // 8)
    attn = FakeAttn(C, heads, 5)
    x = torch.randn(chunks * N, L, C)
    ref_hidden = torch.randn(chunks * N, L, C)
    attn_mask = []
    for scale in [8.0, 16.0, 32.0]:
        o_ = F.interpolate(bocc[:-1].unsqueeze(1), scale_factor=1. / scale, mode='bilinear')
        attn_mask += [torch.cat((o_[0:1].reshape(1, -1) > -1, o_.reshape(o_.shape[0], -1) > 0.5), dim=0)]
    paras = {"fwd_mappings": [fm], "bwd_mappings": [bm], "interattn_masks": [im]}
    res.update(x=x.numpy(), ref_hidden=ref_hidden.numpy(), heads=np.int64(heads), wq=attn.to_q.weight.numpy(),
               wk=attn.to_k.weight.numpy(), wv=attn.to_v.weight.numpy(), wo=attn.to_out[0].weight.numpy(),
               bo=attn.to_out[0].bias.numpy())
    for i, m in enumerate(attn_mask):
        res[f"attn_mask{i}"] = m.numpy()
    for flags in (0, 1, 6, 7):     # set A holds all eight; here: none, cross-frame only, intra+inter, all
        cf, intra, inter = bool(flags & 1), bool(flags & 2), bool(flags & 4)
        ctrl = dh.AttentionControl()
        proc = dh.FRESCOAttnProcessor2_0(chunks, ctrl)
        if intra:
            ctrl.stored_attn['decoder_attn'] = [ref_hidden.clone()]
            ctrl.enable_intraattn()
        if inter:
            ctrl.enable_interattn(paras)
        if cf:
            ctrl.enable_cfattn(attn_mask)
        res[f"out_{flags}"] = proc(attn, x.clone()).numpy()

    # warp_tensor: decoder feature (2 chunks) and image (Dilate(13) path)
    sal = torch.rand(N, 1, 32, 48)
    s_feat = torch.randn(2 * N, 6, 8, 12)
    s_img = torch.randn(N, 3, H, W)
    res.update(saliency=sal.numpy(), sample_feat=s_feat.numpy(), sample_img=s_img.numpy(),
               out_feat=fu.warp_tensor(s_feat.clone(), [fwd, bwd], [fo, bocc], sal, 2).numpy(),
               out_img=fu.warp_tensor(s_img.clone(), [fwd, bwd], [fo, bocc], sal, 1).numpy())

    # optimize_feature, 2 iterations, on an 8 x 12 plane
    Cc, h, w = 16, 8, 12
    sample = torch.randn(2 * N, Cc, h, w)
    other = sample + 0.5 * torch.randn(2 * N, Cc, h, w)
    lv = other.reshape(2 * N, Cc, h * w).transpose(1, 2)
    lv = lv / ((lv ** 2).sum(dim=2, keepdim=True) ** 0.5)
    target = torch.bmm(lv, lv.transpose(-1, -2))
    losses = []
    orig_step = torch.optim.Adam.step

    def rec_step(self, closure=None):
        r = orig_step(self, closure)
        losses.append(float(r))
        return r

    torch.optim.Adam.step = rec_step
    try:
        for tag, kw in {"full1": dict(iters=1), "full3": dict(iters=3)}.items():
            losses.clear()
            o = dh.optimize_feature(sample.clone(), [fwd, bwd], [fo, bocc], correlation_matrix=[target],
                                    intra_weight=1e2, **kw)
            res[f"opt_{tag}_out"] = o.detach().numpy()
            res[f"opt_{tag}_losses"] = np.array(losses, dtype=np.float64)
    finally:
        torch.optim.Adam.step = orig_step
    res.update(opt_sample=sample.numpy(), opt_target=target.numpy())
    np.savez_compressed(os.path.join(HERE, "set_b.npz"), **res)
    print("golden fixture set B written to", HERE)


def control_sequence():
    """The operations AttentionControl is driven through: store, replay of the stored features with wrap-around of the
    ring index, every enable / disable, re-enabling with and without new parameters, clear_store."""
    t = [torch.full((1,), float(i)) for i in range(6)]
    return [("enable_controller", ()), ("enable_store", ()), ("call", (t[0],)), ("call", (t[1],)), ("call", (t[2],)),
            ("disable_store", ()), ("enable_intraattn", ()), ("call", (None,)), ("call", (None,)), ("call", (None,)),
            ("call", (None,)), ("enable_cfattn", ([torch.ones(2, 4, dtype=torch.bool)],)),
            ("enable_interattn", ({"fwd_mappings": [1]},)), ("disable_interattn", ()), ("enable_interattn", ()),
            ("disable_controller", ()), ("enable_controller", ()), ("clear_store", ()), ("enable_intraattn", ()),
            ("call", (t[3],))]


def control_trace(ctrl):
    """control_sequence() applied to `ctrl`: the operation names; after every operation (store, index, use_intraattn,
    use_interattn, use_cfattn, number of stored features); what each call returned (NaN for None); and the bias / scale
    attributes at the end."""
    ops, states, returned = [], [], []
    for name, args in control_sequence():
        if name == "call":
            r = ctrl(*args)
            returned.append(float("nan") if r is None else r.item())
        else:
            getattr(ctrl, name)(*args)
        ops.append(name)
        states.append((ctrl.store, ctrl.index, ctrl.use_intraattn, ctrl.use_interattn, ctrl.use_cfattn,
                       len(ctrl.stored_attn["decoder_attn"])))
    attrs = (ctrl.intraattn_bias, ctrl.intraattn_scale_factor, ctrl.interattn_scale_factor)
    return {"ops": np.array(ops), "states": np.array(states, dtype=np.int64),
            "returned": np.array(returned, dtype=np.float64), "attrs": np.array(attrs, dtype=np.float64)}


def scenario_control(dh):
    """The reference's AttentionControl (src/diffusion_hacked.py:23-137) through control_sequence()."""
    np.savez_compressed(os.path.join(HERE, "attention_control.npz"), **control_trace(dh.AttentionControl()))
    print("golden AttentionControl trace written to", HERE)


def main():
    dh, fu, geometry, matching, ut = import_reference()
    which = sys.argv[sys.argv.index("--set") + 1] if "--set" in sys.argv else "a"
    if which == "b":
        return scenario_b(dh, fu, geometry, matching, ut)
    if which == "control":
        return scenario_control(dh)
    torch.manual_seed(0)
    torch.set_grad_enabled(False)

    # ---------------- geometry ----------------
    N, H, W = 4, 64, 64
    fwd, bwd = smooth_flows(N, H, W, 1, 3.0)
    fo, bo = geometry.forward_backward_consistency_check(fwd, bwd)
    feat = torch.randn(N, 5, H, W)
    np.savez_compressed(os.path.join(HERE, "geometry.npz"),
                        fwd=fwd.numpy(), bwd=bwd.numpy(), fwd_occ=fo.numpy(), bwd_occ=bo.numpy(),
                        feat=feat.numpy(), warped=geometry.flow_warp(feat, bwd).numpy())

    # ---------------- mapping (integer path) ----------------
    imgs = torch.rand(N, 3, H, W) * 2 - 1
    out = {}
    for tag, (hh, mag, sc) in {"a": (64, 3.0, 8.0), "b": (128, 10.0, 8.0), "c": (128, 14.0, 16.0)}.items():
        f_, b_ = smooth_flows(N, hh, hh, 7 + hh, mag)
        _, bo_ = geometry.forward_backward_consistency_check(f_, b_)
        im_ = torch.rand(N, 3, hh, hh) * 2 - 1
        fm, bm, im = fu.get_mapping_ind(b_, bo_, im_, scale=sc)
        mp, unl = fu.get_single_mapping_ind(b_[0:1], bo_[0:1], im_[0:2], scale=sc)
        out.update({f"{tag}_bwd_flows": b_.numpy(), f"{tag}_bwd_occs": bo_.numpy(), f"{tag}_imgs": im_.numpy(),
                    f"{tag}_scale": np.float32(sc), f"{tag}_fwd_map": fm.numpy(), f"{tag}_bwd_map": bm.numpy(),
                    f"{tag}_mask": im.numpy(), f"{tag}_single_map": mp.numpy(), f"{tag}_single_unl": unl.numpy()})
    np.savez_compressed(os.path.join(HERE, "mapping.npz"), **out)

    # ---------------- attention, all 8 flag combinations ----------------
    C, heads, chunks = 80, 2, 2
    L = (H // 8) * (W // 8)
    attn = FakeAttn(C, heads, 3)
    x = torch.randn(chunks * N, L, C)
    ref_hidden = torch.randn(chunks * N, L, C)
    bocc = torch.clamp(bo + (torch.rand(N, H, W) > 0.8).float(), 0, 1)      # denser occlusion
    attn_mask = []
    for scale in [8.0, 16.0, 32.0]:   # formula of diffusion_hacked.py:935-938 evaluated by the reference's own ops
        o_ = F.interpolate(bocc[:-1].unsqueeze(1), scale_factor=1. / scale, mode='bilinear')
        attn_mask += [torch.cat((o_[0:1].reshape(1, -1) > -1, o_.reshape(o_.shape[0], -1) > 0.5), dim=0)]
    fm, bm, im = fu.get_mapping_ind(bwd, bocc, imgs, scale=8.0)
    paras = {"fwd_mappings": [fm], "bwd_mappings": [bm], "interattn_masks": [im]}
    res = {"x": x.numpy(), "ref_hidden": ref_hidden.numpy(), "heads": np.int64(heads),
           "wq": attn.to_q.weight.numpy(), "wk": attn.to_k.weight.numpy(), "wv": attn.to_v.weight.numpy(),
           "wo": attn.to_out[0].weight.numpy(), "bo": attn.to_out[0].bias.numpy(),
           "fwd_map": fm.numpy(), "bwd_map": bm.numpy(), "inter_mask": im.numpy()}
    for i, m in enumerate(attn_mask):
        res[f"attn_mask{i}"] = m.numpy()
    for flags in range(8):
        cf, intra, inter = bool(flags & 1), bool(flags & 2), bool(flags & 4)
        ctrl = dh.AttentionControl()
        proc = dh.FRESCOAttnProcessor2_0(chunks, ctrl)
        if intra:
            ctrl.stored_attn['decoder_attn'] = [ref_hidden.clone()]
            ctrl.enable_intraattn()
        if inter:
            ctrl.enable_interattn(paras)
        if cf:
            ctrl.enable_cfattn(attn_mask)
        res[f"out_{flags}"] = proc(attn, x.clone()).numpy()
    # cross-frame without a matching mask => frame-0 K/V (:236-237)
    ctrl = dh.AttentionControl()
    proc = dh.FRESCOAttnProcessor2_0(chunks, ctrl)
    ctrl.enable_cfattn([attn_mask[1]])
    res["out_cf_nomask"] = proc(attn, x.clone()).numpy()
    np.savez_compressed(os.path.join(HERE, "attention.npz"), **res)

    # ---------------- warp_tensor ----------------
    sal = torch.rand(N, 1, 32, 32)
    s_feat = torch.randn(2 * N, 6, 8, 8)
    s_img = torch.randn(N, 3, H, W)
    np.savez_compressed(
        os.path.join(HERE, "warp_tensor.npz"), fwd=fwd.numpy(), bwd=bwd.numpy(), fwd_occ=fo.numpy(),
        bwd_occ=bocc.numpy(), saliency=sal.numpy(), sample_feat=s_feat.numpy(), sample_img=s_img.numpy(),
        out_feat=fu.warp_tensor(s_feat.clone(), [fwd, bwd], [fo, bocc], sal, 2).numpy(),
        out_img=fu.warp_tensor(s_img.clone(), [fwd, bwd], [fo, bocc], sal, 1).numpy())

    # ---------------- optimize_feature (losses captured through Adam.step's return value) ----------------
    Cc, h, w = 16, 8, 8
    sample = torch.randn(2 * N, Cc, h, w)
    other = sample + 0.5 * torch.randn(2 * N, Cc, h, w)
    lv = other.reshape(2 * N, Cc, h * w).transpose(1, 2)
    lv = lv / ((lv ** 2).sum(dim=2, keepdim=True) ** 0.5)
    target = torch.bmm(lv, lv.transpose(-1, -2))
    losses = []
    orig_step = torch.optim.Adam.step

    def rec_step(self, closure=None):
        r = orig_step(self, closure)
        losses.append(float(r))
        return r

    torch.optim.Adam.step = rec_step
    opt = {"sample": sample.numpy(), "target": target.numpy(), "fwd": fwd.numpy(), "bwd": bwd.numpy(),
           "fwd_occ": fo.numpy(), "bwd_occ": bocc.numpy()}
    with torch.enable_grad():
        pass
    for tag, kw in {"full1": dict(iters=1), "full5": dict(iters=5),
                    "temporal3": dict(iters=3, correlation_matrix=[]),
                    "spatial3": dict(iters=3, optimize_temporal=False)}.items():
        losses.clear()
        kwargs = dict(correlation_matrix=[target], intra_weight=1e2)
        kwargs.update(kw)
        o = dh.optimize_feature(sample.clone(), [fwd, bwd], [fo, bocc], **kwargs)
        opt[f"{tag}_out"] = o.detach().numpy()
        opt[f"{tag}_losses"] = np.array(losses, dtype=np.float64)
    torch.optim.Adam.step = orig_step
    opt["adain_out"] = ut.adaptive_instance_normalization(other, sample).numpy()
    opt["adain_content"] = other.numpy()
    np.savez_compressed(os.path.join(HERE, "optimize.npz"), **opt)

    # ---------------- GMFlow global correlation ----------------
    f0 = torch.randn(2, 16, 6, 8)
    f1 = torch.roll(f0, shifts=(1, -2), dims=(2, 3)) * 3 + 0.3 * torch.randn(2, 16, 6, 8)
    flow_b, prob_b = matching.global_correlation_softmax(f0, f1, pred_bidir_flow=True)
    flow_u, _ = matching.global_correlation_softmax(f0, f1, pred_bidir_flow=False)
    np.savez_compressed(os.path.join(HERE, "gmflow_corr.npz"), f0=f0.numpy(), f1=f1.numpy(),
                        flow_bidir=flow_b.numpy(), flow_uni=flow_u.numpy(), prob_bidir=prob_b.numpy())
    scenario_gmflow_attention()
    scenario_ddpm_step()
    print("golden fixtures written to", HERE)


def scenario_ddpm_step():
    """src/pipe_FRESCO.py step() (no background smoothing) on a DDPM-1000 scaled-linear table, incl. repeat_noise, and
    the classifier-free-guidance combine of inference() (:212-215); Dilate(5) and Dilate(13) of src/utils.py:81-93."""
    import src.pipe_FRESCO as pf
    import src.utils as ut

    class Sched:
        def __init__(self):
            betas = torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=torch.float32) ** 2
            self.alphas_cumprod = torch.cumprod(1.0 - betas, dim=0)
            self.one = torch.tensor(1.0)

        def previous_timestep(self, t):
            return t - 50

    class Pipe:
        scheduler = Sched()

    g = torch.Generator().manual_seed(77)
    N = 3
    raw = torch.randn(2 * N, 4, 16, 24, generator=g)
    sample = torch.randn(N, 4, 16, 24, generator=g)
    res = {"raw": raw.numpy(), "sample": sample.numpy(), "alphas_cumprod": Pipe.scheduler.alphas_cumprod.numpy()}
    u, t = raw.chunk(2)
    guided = u + 7.5 * (t - u)
    for tag, ts, rep in (("a", 700, False), ("b", 0, False), ("c", 350, True)):
        gen = torch.Generator().manual_seed(5)
        prev, x0 = pf.step(Pipe, guided, ts, sample, gen, repeat_noise=rep)
        noise = torch.randn(guided.shape, generator=torch.Generator().manual_seed(5))
        res.update({f"{tag}_t": ts, f"{tag}_prev": prev.numpy(), f"{tag}_x0": x0.numpy(), f"{tag}_noise": noise.numpy(),
                    f"{tag}_repeat": rep})
    m = (torch.rand(3, 1, 40, 56, generator=g) > 0.9).float()
    res.update(dil_in=m.numpy(), dil5=ut.Dilate(kernel_size=5, device="cpu")(m).numpy(),
               dil13=ut.Dilate(kernel_size=13, device="cpu")(m).numpy())
    np.savez_compressed(os.path.join(HERE, "ddpm_step.npz"), **res)


def scenario_gmflow_attention():
    """GMFlow transformer attention (gmflow/transformer.py): plain, 2 x 2 windows, shifted 2 x 2 windows, and the
    flow-propagation attention, at C = 128 on a 32 x 32 grid (inputs are fp16-representable so that the fp16 kernels
    see exactly these operands)."""
    from gmflow import transformer as T
    g = torch.Generator().manual_seed(2024)
    b, h, w, c = 1, 32, 32, 128
    q = (torch.randn(b, h * w, c, generator=g) * 1.5).half().float()
    k = torch.randn(b, h * w, c, generator=g).half().float()
    v = torch.randn(b, h * w, c, generator=g).half().float()
    res = {"q": q.half().numpy(), "k": k.half().numpy(), "v": v.half().numpy(), "h": h, "w": w}
    res["out_full"] = T.single_head_full_attention(q, k, v).numpy()
    res["out_split"] = T.single_head_split_window_attention(q, k, v, num_splits=2, with_shift=False, h=h, w=w).numpy()
    mask = T.generate_shift_window_attn_mask((h, w), h // 2, w // 2, h // 4, w // 4, device=torch.device("cpu"))
    res["out_shift"] = T.single_head_split_window_attention(q, k, v, num_splits=2, with_shift=True, h=h, w=w,
                                                            attn_mask=mask).numpy()
    torch.manual_seed(7)
    ffa = T.FeatureFlowAttention(in_channels=c)
    with torch.no_grad():
        for prm in ffa.parameters():
            prm.copy_(prm.half().float())
        f0 = torch.randn(2, c, h, w, generator=g).half().float()
        flow = torch.randn(2, 2, h, w, generator=g) * 4
        res.update(ffa_f0=f0.half().numpy(), ffa_flow=flow.numpy(), ffa_out=ffa(f0, flow).numpy(),
                   ffa_wq=ffa.q_proj.weight.numpy(), ffa_bq=ffa.q_proj.bias.numpy(), ffa_wk=ffa.k_proj.weight.numpy(),
                   ffa_bk=ffa.k_proj.bias.numpy())
    np.savez_compressed(os.path.join(HERE, "gmflow_attn.npz"), **res)


if __name__ == "__main__":
    main()
