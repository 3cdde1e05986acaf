"""CPU-only tests: the C-ABI library loads and exports every symbol the header declares,
the host-side mirror of the reference's hook surface behaves like the reference, and the
product path refuses to run without CUDA (no silent fallback)."""
import ctypes
import importlib.util
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built_lib():
    sys.path.insert(0, ROOT)
    import __graft_entry__ as g
    g.build()
    from fresco_b200 import _lib
    return _lib


def test_library_exports_every_header_symbol(built_lib):
    hdr = open(os.path.join(ROOT, "include", "fresco_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b((?:fresco|gmflow)_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 18
    l = ctypes.CDLL(built_lib.LIB_PATH)
    for n in sorted(names):
        assert hasattr(l, n), f"libfresco_b200.so does not export {n}"
    assert names == set(built_lib.EXPORTED_SYMBOLS), names ^ set(built_lib.EXPORTED_SYMBOLS)
    assert l.fresco_abi_version() == 1


def test_argument_errors_do_not_touch_the_gpu(built_lib):
    l = built_lib.lib()
    rc = l.fresco_attn_fwd(None, None, None, None, 1, 1, 1, 1, 40, 1, 1.0, 0.0, None)
    assert rc == -1 and b"null pointer" in l.fresco_last_error()
    rc = l.fresco_kv_compact(None, None, None, None, None, 2, 8, 4, 320, None)
    assert rc == -1


def test_default_attention_kernel_per_head_dim(built_lib):
    """Host-side kernel selection through the C ABI (no launch): the measured-best kernel per head_dim is the default,
    the options select the other parity-tested variants, negative values restore the defaults, unknown names fail."""
    l = built_lib.lib()
    names = ("FRESCO_ATTN_WIDE", "FRESCO_ATTN_POLY")
    for n in names:
        assert l.fresco_set_option(n.encode(), -1) == 0
    v = lambda d: l.fresco_attn_variant(d).decode()
    assert v(40) == "fresco_attn_twin_kernel<40,poly8,2>"          # two threads per row at the dominant FRESCO shape
    assert v(80) == "fresco_attn_twin_kernel<80,poly4,1>"
    assert v(64).startswith("fresco_attn_kernel<64,poly0>") and v(128).startswith("fresco_attn_kernel<128,poly0>")
    try:
        assert l.fresco_set_option(b"FRESCO_ATTN_WIDE", 1) == 0 and l.fresco_set_option(b"FRESCO_ATTN_POLY", 0) == 0
        assert v(40) == "fresco_attn_twin_kernel<40,poly0,1>" and v(64) == "fresco_attn_twin_kernel<64,poly0,1>"
        assert v(128).startswith("fresco_attn_kernel<128")          # the twin kernel stops at head_dim 80
        assert l.fresco_set_option(b"FRESCO_ATTN_WIDE", 0) == 0
        assert v(40).startswith("fresco_attn_kernel<40,poly0>")
        assert l.fresco_set_option(b"FRESCO_NO_SUCH_OPTION", 1) == -1
    finally:
        for n in names:
            l.fresco_set_option(n.encode(), -1)
    assert v(40) == "fresco_attn_twin_kernel<40,poly8,2>"


def test_no_cpu_fallback(built_lib):
    from fresco_b200 import ops
    from fresco_b200._lib import FrescoError
    q = torch.zeros(2, 128, 80, dtype=torch.float16)
    with pytest.raises(FrescoError):
        ops.attn_fwd(q, q, q, 2)
    from fresco_b200 import flow_utils
    with pytest.raises(FrescoError):
        flow_utils.flow_warp(torch.zeros(1, 1, 4, 4), torch.zeros(1, 2, 4, 4))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "fresco_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, os.path.join(dp, f)


def test_attention_control_state_machine_matches_reference(golden):
    """drive our AttentionControl through the call sequence the reference's was driven through to make the fixture
    (tests/golden/make_golden.py --set control) and compare the state after every operation"""
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(ROOT, "tests", "golden", "make_golden.py"))
    make_golden = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(make_golden)
    from fresco_b200 import diffusion_hacked as my_dh
    want, got = golden("attention_control"), make_golden.control_trace(my_dh.AttentionControl())
    assert want["ops"].tolist() == got["ops"].tolist()
    for i, name in enumerate(got["ops"]):
        assert want["states"][i].tolist() == got["states"][i].tolist(), (i, name, want["states"][i], got["states"][i])
    assert np.array_equal(want["returned"], got["returned"], equal_nan=True), (want["returned"], got["returned"])
    assert want["attrs"].tolist() == got["attrs"].tolist()


def test_hook_surface_on_harness_unet():
    """apply_FRESCO_attn installs the shared processor on the 12 up_blocks.2/3 attentions;
    apply_FRESCO_opt's forward returns (sample, *4 decoder features) with return_dict=False."""
    from fresco_b200 import diffusion_hacked as dh
    from fresco_b200.harness.sd15_unet import FakePipe, SD15UNet
    torch.manual_seed(0)
    unet = SD15UNet(block_out=(32, 64, 128, 128), heads=8, cross_dim=24)
    pipe = FakePipe(unet)
    keys = list(unet.attn_processors.keys())
    assert len(keys) == 32 and "up_blocks.3.attentions.2.transformer_blocks.0.attn1.processor" in keys
    x, e = torch.randn(2, 4, 16, 16), torch.randn(2, 7, 24)
    with torch.no_grad():
        plain = unet(x, 500, e).sample
    dh.apply_FRESCO_opt(pipe)            # == disable_FRESCO_opt: hooks record only
    with torch.no_grad():
        out = unet(x, torch.tensor(500), e, return_dict=False)
    assert len(out) == 5 and torch.equal(out[0], plain)
    assert [tuple(o.shape) for o in out[1:]] == [(2, 128, 2, 2), (2, 128, 4, 4), (2, 128, 8, 8), (2, 64, 16, 16)]
    proc = dh.apply_FRESCO_attn(pipe)
    table = unet.attn_processors
    assert sum(1 for v in table.values() if v is proc) == 12
    assert all(k.startswith(("up_blocks.2", "up_blocks.3")) for k, v in table.items() if v is proc)
    # cross-attention (encoder_hidden_states given) must behave as plain SDPA even with the FRESCO processor
    attn2 = unet.up_blocks[3].attentions[0].transformer_blocks[0].attn2
    h = torch.randn(2, 256, 32)
    from fresco_b200.harness.sd15_unet import PlainProcessor
    with torch.no_grad():
        assert torch.allclose(proc(attn2, h, encoder_hidden_states=e), PlainProcessor()(attn2, h, e), atol=1e-6)


class _TorchOps:
    """fp32 torch stand-ins for the three kernels the processor calls (same signatures as fresco_b200.ops); the
    results are rounded to fp16 like the kernels' outputs.  Lets the processor's HOST logic run without a GPU."""

    @staticmethod
    def kv_compact(k, v, idx, chunks):
        B, L, C = k.shape
        rows = (B // chunks) * L
        return k.reshape(chunks, rows, C)[:, idx.long()].contiguous(), v.reshape(chunks, rows, C)[:, idx.long()].contiguous()

    @staticmethod
    def attn_fwd(q, k, v, heads, q_per_kv=1, softmax_scale=None, diag_bias=0.0, out=None):
        B, L, C = q.shape
        d = C // heads
        qf, kf, vf = q.float(), k.float().repeat_interleave(q_per_kv, 0), v.float().repeat_interleave(q_per_kv, 0)
        qh, kh, vh = (t.view(t.shape[0], -1, heads, d).transpose(1, 2) for t in (qf, kf, vf))
        s = qh @ kh.transpose(-1, -2) * (softmax_scale if softmax_scale is not None else d ** -0.5)
        if diag_bias:
            s = s + torch.eye(L, kh.shape[2]) * diag_bias
        return (torch.softmax(s, -1) @ vh).transpose(1, 2).reshape(B, L, C).to(q.dtype)

    @staticmethod
    def temporal_attn_fwd(q, k, v, fwd_map, traj_mask, chunks, heads, scale):
        B, L, C = q.shape
        N, d = B // chunks, C // heads
        gi = fwd_map[None, :, :, None, None].expand(chunks, N, L, heads, d)
        qt, kt, vt = (torch.gather(t.float().view(chunks, N, L, heads, d), 2, gi) for t in (q, k, v))
        s = torch.einsum("bfphd,bgphd->bphfg", qt, kt) * scale
        s = s.masked_fill(~traj_mask.bool()[None, :, None], float("-inf"))
        o = torch.einsum("bphfg,bgphd->bfphd", torch.softmax(s, -1), vt)
        out = torch.empty_like(o)
        out.scatter_(2, gi, o)
        return out.reshape(B, L, C).to(v.dtype)


class _GoldenAttn(torch.nn.Module):
    def __init__(self, g):
        super().__init__()
        c = g["wq"].shape[0]
        self.heads = int(g["heads"])
        self.spatial_norm = self.group_norm = None
        self.norm_cross = self.residual_connection = False
        self.rescale_output_factor = 1.0
        self.to_q, self.to_k, self.to_v = (torch.nn.Linear(c, c, bias=False) for _ in range(3))
        self.to_out = torch.nn.ModuleList([torch.nn.Linear(c, c), torch.nn.Dropout(0.0)])
        with torch.no_grad():
            for lin, key in ((self.to_q, "wq"), (self.to_k, "wk"), (self.to_v, "wv"), (self.to_out[0], "wo")):
                lin.weight.copy_(torch.from_numpy(g[key]))
            self.to_out[0].bias.copy_(torch.from_numpy(g["bo"]))


@pytest.mark.parametrize("fixture,flag_sets", [("attention", range(8)), ("set_b", (0, 1, 6, 7))])
def test_processor_host_logic_against_reference_outputs(golden, monkeypatch, fixture, flag_sets):
    """The product processor (mask -> K/V row indices, frame-0 fallback, query replacement by the spatial-guided
    pass, trajectory tables, scale factors, chunk / frame layout) reproduces the REFERENCE's outputs when its three
    kernel calls are served by fp32 torch stand-ins: set A (N=4, 64 tokens, head_dim 40, all 8 mode combinations) and
    set B (N=3 frames, 8 x 12 tokens, head_dim 80).  Bound: fp16 rounding of q / k / v / attention output, as in the
    -m gpu test of the same fixtures."""
    from fresco_b200 import diffusion_hacked as dh
    monkeypatch.setattr(dh, "ops", _TorchOps)
    g = golden(fixture)
    attn = _GoldenAttn(g)
    x, ref_hidden = torch.from_numpy(g["x"]), torch.from_numpy(g["ref_hidden"])
    masks = [torch.from_numpy(g[f"attn_mask{i}"]) for i in range(3)]
    paras = {"fwd_mappings": [torch.from_numpy(g["fwd_map"])], "bwd_mappings": [torch.from_numpy(g["bwd_map"])],
             "interattn_masks": [torch.from_numpy(g["inter_mask"])]}
    for flags in flag_sets:
        ctrl = dh.AttentionControl()
        proc = dh.FRESCOAttnProcessor2_0(2, ctrl)
        if flags & 2:
            ctrl.stored_attn["decoder_attn"] = [ref_hidden.clone()]
            ctrl.enable_intraattn()
        if flags & 4:
            ctrl.enable_interattn(paras)
        if flags & 1:
            ctrl.enable_cfattn(masks)
        with torch.no_grad():
            out = proc(attn, x.clone())
        ref = torch.from_numpy(g[f"out_{flags}"])
        assert (out - ref).abs().max().item() < 1e-2 * ref.abs().max().item(), (fixture, flags)
    if fixture == "attention":          # cross-frame attention without a mask of this resolution: frame-0 K/V
        ctrl = dh.AttentionControl()
        proc = dh.FRESCOAttnProcessor2_0(2, ctrl)
        ctrl.enable_cfattn([masks[1]])
        with torch.no_grad():
            out = proc(attn, x.clone())
        ref = torch.from_numpy(g["out_cf_nomask"])
        assert (out - ref).abs().max().item() < 1e-2 * ref.abs().max().item()


class _TorchWarpOps:
    """fp32 stand-ins (built on the oracle's flow_warp / single_mapping_ind, test-side only) for the kernels that
    flow_utils.warp_tensor and get_mapping_ind call, so that their HOST code (flow / occlusion / saliency resizing,
    dilation, blend weights, cache keys, mapping chain and trajectory cuts) runs on CPU."""

    @staticmethod
    def flow_warp(src, flow):
        from oracle import fresco_oracle as O
        return O.flow_warp(src, flow[torch.arange(src.shape[0]) % flow.shape[0]])

    @staticmethod
    def warp_fuse_chain(sample, bwd_flow, fwd_flow_last, blend, chunks, out=None):
        from oracle import fresco_oracle as O
        z = sample.float().clone()
        n = sample.shape[0] // chunks
        for j in range(chunks):
            base = n * j
            for ii in range(n - 1):
                m = blend[ii:ii + 1]
                z[base + ii + 1] = (z[base + ii + 1:base + ii + 2] * (1 - m) + O.flow_warp(z[base + ii:base + ii + 1], bwd_flow[ii:ii + 1]) * m)[0]
            m = blend[n - 1:n]
            z[base + n - 1] = (z[base + n - 1:base + n] * (1 - m) + O.flow_warp(z[base:base + 1], fwd_flow_last[None]) * m)[0]
        return z.to(sample.dtype)

    @staticmethod
    def mapping_single(bwd_flow, bwd_occ, imgs, scale):
        from oracle import fresco_oracle as O
        return O.single_mapping_ind(bwd_flow, bwd_occ, imgs, float(scale))

    @staticmethod
    def dilate(x, k):
        from oracle import fresco_oracle as O
        return O.dilate(x, k)


@pytest.mark.parametrize("fixture", ["set_a", "set_b"])
def test_warp_tensor_and_mapping_host_logic_against_reference_outputs(golden, monkeypatch, fixture):
    """flow_utils.warp_tensor / get_mapping_ind with their kernel calls served by CPU stand-ins reproduce the
    REFERENCE's outputs: square N=4 fixtures (set A) and the N=3, 64 x 96 fixture (set B)."""
    from fresco_b200 import flow_utils as fu
    monkeypatch.setattr(fu, "ops", _TorchWarpOps)
    fu._PREP_CACHE.clear()
    T = torch.from_numpy
    if fixture == "set_a":
        g = golden("warp_tensor")
        flows, occs, sal = [T(g["fwd"]), T(g["bwd"])], [T(g["fwd_occ"]), T(g["bwd_occ"])], T(g["saliency"])
    else:
        g = golden("set_b")
        flows, occs, sal = [T(g["fwd"]), T(g["bwd"])], [T(g["fwd_occ"]), T(g["bwd_occ"])], T(g["saliency"])
    feat = T(g["sample_feat"])
    keep = feat.clone()
    o = fu.warp_tensor(feat, flows, occs, sal, 2)
    assert torch.equal(feat, keep)                                   # never mutates its input
    assert (o - T(g["out_feat"])).abs().max().item() < 1e-5
    o = fu.warp_tensor(T(g["sample_img"]), flows, occs, sal, 1)     # image resolution: Dilate(13) path
    assert (o - T(g["out_img"])).abs().max().item() < 1e-5
    if fixture == "set_a":
        m = golden("mapping")
        for tag in "abc":
            fm, bm, mask = fu.get_mapping_ind(T(m[f"{tag}_bwd_flows"]), T(m[f"{tag}_bwd_occs"]), T(m[f"{tag}_imgs"]),
                                              scale=float(m[f"{tag}_scale"]))
            assert torch.equal(fm, T(m[f"{tag}_fwd_map"])) and torch.equal(bm, T(m[f"{tag}_bwd_map"]))
            assert torch.equal(mask, T(m[f"{tag}_mask"]))
    else:
        fm, bm, mask = fu.get_mapping_ind(flows[1], occs[1], T(g["imgs"]), scale=8.0)
        assert torch.equal(fm, T(g["fwd_map"])) and torch.equal(bm, T(g["bwd_map"])) and torch.equal(mask, T(g["inter_mask"]))
    fu._PREP_CACHE.clear()


def test_prep_cache_never_serves_another_batch(monkeypatch):
    """ADVICE r1 (high): per-batch preparation was keyed on (data_ptr, version, shape); the allocator hands the same
    address to the next batch's flows, so batch k could silently get batch j's resized flows.  Entries are now keyed on
    tensor identity and hold a reference: two same-shape batches, the first one freed before the second is made."""
    from fresco_b200 import flow_utils as fu
    from oracle import fresco_oracle as O
    monkeypatch.setattr(fu, "ops", _TorchWarpOps)
    fu.clear_prep_cache()
    outs, wants = [], []
    for seed in (1, 2, 3, 4, 5, 6):
        flows, occs = O.synth_flows(3, 64, 64, seed=seed, mag=6.0)
        sal = torch.rand(3, 1, 32, 32, generator=torch.Generator().manual_seed(seed))
        feat = torch.randn(6, 4, 8, 8, generator=torch.Generator().manual_seed(100 + seed))
        outs.append(fu.warp_tensor(feat, flows, occs, sal, 2))
        outs.append(fu.warp_tensor(feat, flows, occs, sal, 2))          # second call of the batch: served from the cache
        fu_fresh = O.warp_tensor(feat.clone(), flows, occs, sal, 2)
        wants += [fu_fresh, fu_fresh]
        del flows, occs, sal                                             # the next batch may reuse these addresses
    for o, w in zip(outs, wants):
        assert (o - w).abs().max().item() < 1e-5
    assert len(fu._PREP_CACHE) <= fu._PREP_CACHE_MAX
    fu.clear_prep_cache()


def test_sharded_plan_follows_the_mask_tensor():
    """ADVICE r1 (medium): the sharded K/V exchange plan was cached per token count forever; it must be rebuilt when
    enable_cfattn installs the next batch's mask."""
    from fresco_b200 import diffusion_hacked as dh
    from fresco_b200.dist import ShardedFRESCOAttention
    ctrl = dh.AttentionControl()
    sh = ShardedFRESCOAttention(ctrl, world=1, rank=0, backend=object())
    m1 = torch.zeros(4, 64, dtype=torch.bool)
    m1[0] = True
    m1[1, :5] = True
    ctrl.enable_cfattn([m1])
    p1 = sh._plan(64)
    assert p1.total == 64 + 5 and sh._plan(64) is p1
    m2 = m1.clone()
    m2[2, :7] = True
    ctrl.enable_cfattn([m2])
    p2 = sh._plan(64)
    assert p2 is not p1 and p2.total == 64 + 5 + 7


class _TorchAttnOps:
    """fp32 stand-ins for the kernels fresco_b200.gmflow_transformer calls (host-logic test only)"""

    @staticmethod
    def attn_fwd(q, k, v, heads, q_per_kv=1, softmax_scale=None, diag_bias=0.0, out=None):
        q, k, v = q.float(), k.float(), v.float()
        return (torch.softmax(q @ k.transpose(1, 2) * softmax_scale, -1) @ v).half()

    @staticmethod
    def rows_gather(src, idx, dst, dst_col=0):
        dst[:, dst_col:dst_col + src.shape[-1]] = src[idx.long()]
        return dst

    @staticmethod
    def rows_scatter(src, idx, dst):
        dst[idx.long()] = src
        return dst

    @staticmethod
    def gmflow_flow_attention(q, k, values, scale):
        p = torch.softmax(q.float() @ k.float().transpose(1, 2) * scale, -1)
        return (p @ values).transpose(1, 2).contiguous()


def test_gmflow_transformer_attention_host_logic(golden, monkeypatch):
    """SURVEY 8(f)-1: the window / shifted-window decomposition and the flow-propagation attention of
    fresco_b200.gmflow_transformer reproduce the REFERENCE's outputs (gmflow/transformer.py) with their kernel calls
    served by torch stand-ins."""
    from fresco_b200 import gmflow_transformer as gt
    monkeypatch.setattr(gt, "ops", _TorchAttnOps)
    g = golden("gmflow_attn")
    T = torch.from_numpy
    q, k, v = (T(g[n]).float() for n in "qkv")
    h, w = int(g["h"]), int(g["w"])
    tol = 2e-3 * float(abs(g["out_full"]).max())
    assert (gt.single_head_full_attention(q, k, v) - T(g["out_full"])).abs().max().item() < tol
    o = gt.single_head_split_window_attention(q, k, v, num_splits=2, with_shift=False, h=h, w=w)
    assert (o - T(g["out_split"])).abs().max().item() < tol
    o = gt.single_head_split_window_attention(q, k, v, num_splits=2, with_shift=True, h=h, w=w, attn_mask=None)
    assert (o - T(g["out_shift"])).abs().max().item() < tol

    class FFA(torch.nn.Module):
        def __init__(self):
            super().__init__()
            c = g["ffa_wq"].shape[0]
            self.q_proj, self.k_proj = torch.nn.Linear(c, c), torch.nn.Linear(c, c)
            with torch.no_grad():
                self.q_proj.weight.copy_(T(g["ffa_wq"])), self.q_proj.bias.copy_(T(g["ffa_bq"]))
                self.k_proj.weight.copy_(T(g["ffa_wk"])), self.k_proj.bias.copy_(T(g["ffa_bk"]))
    out = gt.feature_flow_attention(FFA(), T(g["ffa_f0"]).float(), T(g["ffa_flow"]))
    assert (out - T(g["ffa_out"])).abs().max().item() < 2e-2            # flow units (pixels), fp16 projections


class _TorchStepOps:
    """stand-ins for fresco_cfg_pred_x0 / fresco_ddpm_prev (host-logic tests of fresco_b200.pipe_FRESCO)"""

    @staticmethod
    def cfg_pred_x0(noise_pred, sample, guidance_scale, alpha_prod_t, do_cfg=True):
        if do_cfg:
            u, t = noise_pred.chunk(2)
            eps = u + guidance_scale * (t - u)
        else:
            eps = noise_pred
        return (sample - (1 - alpha_prod_t) ** 0.5 * eps) / alpha_prod_t ** 0.5

    @staticmethod
    def ddpm_prev(x0, sample, noise, c_x0, c_xt, sigma, repeat_noise=False):
        z = noise[0:1].expand_as(noise) if repeat_noise else noise
        return c_x0 * x0 + c_xt * sample + sigma * z


class _Sched:
    def __init__(self, ac):
        self.alphas_cumprod = ac
        self.one = torch.tensor(1.0)
        self.order = 1

    def previous_timestep(self, t):
        return t - 50

    def add_noise(self, x0, noise, t):
        a = self.alphas_cumprod[t]
        return a ** 0.5 * x0 + (1 - a) ** 0.5 * noise


def test_pipe_step_host_logic_against_reference(golden, monkeypatch):
    """fresco_b200.pipe_FRESCO.step: coefficient arithmetic + noise draw reproduce the reference's step() outputs, with
    the guidance fused (raw [2N] UNet output) or applied by the caller as in the reference."""
    from fresco_b200 import pipe_FRESCO as pf
    monkeypatch.setattr(pf, "ops", _TorchStepOps)
    g = golden("ddpm_step")
    T = torch.from_numpy

    class Pipe:
        scheduler = _Sched(T(g["alphas_cumprod"]))
    raw, sample = T(g["raw"]), T(g["sample"])
    u, t = raw.chunk(2)
    guided = u + 7.5 * (t - u)
    for tag in "abc":
        ts, rep = int(g[f"{tag}_t"]), bool(g[f"{tag}_repeat"])
        prev, x0 = pf.step(Pipe, guided, ts, sample, torch.Generator().manual_seed(5), repeat_noise=rep)
        assert (prev - T(g[f"{tag}_prev"])).abs().max() < 1e-5 and (x0 - T(g[f"{tag}_x0"])).abs().max() < 1e-5
        prev, x0 = pf.step(Pipe, raw, ts, sample, torch.Generator().manual_seed(5), repeat_noise=rep, guidance_scale=7.5)
        assert (prev - T(g[f"{tag}_prev"])).abs().max() < 1e-5 and (x0 - T(g[f"{tag}_x0"])).abs().max() < 1e-5


def test_get_intraframe_paras_host_logic_on_harness_unet(monkeypatch):
    """P2 (src/diffusion_hacked.py:843-901) end to end on CPU: stub scheduler / VAE, the harness UNet with the hook surface
    installed, torch stand-ins for the kernels.  The store pass must leave the six decoder self-attention inputs in the
    controller (in call order, store switched off again, guidance flags off), and the returned targets must be the
    reference's formula -- bmm of the row-normalised decoder features, fp32 [2N, hw, hw] -- on the four decoder features
    of that same pass."""
    from fresco_b200 import diffusion_hacked as dh
    from fresco_b200.harness.sd15_unet import FakePipe, SD15UNet
    monkeypatch.setattr(dh, "ops", _TorchOps)
    torch.manual_seed(1)
    unet = SD15UNet(block_out=(32, 64, 128, 128), heads=8, cross_dim=24)
    pipe = FakePipe(unet)
    ac = torch.linspace(0.999, 0.01, 1000)

    class Sched(_Sched):
        timesteps = torch.arange(950, -1, -50)

    class VAE:
        class config:
            scaling_factor = 0.5

        @staticmethod
        def encode(x):
            class D:
                latent_dist = None

            d = D()
            d.latent_dist = d
            d.sample = lambda: torch.nn.functional.avg_pool2d(x, 8)[:, :1].repeat(1, 4, 1, 1)
            return d

    pipe.scheduler, pipe.vae, pipe._execution_device = Sched(ac), VAE(), torch.device("cpu")
    pipe.prepare_latents = lambda B, C, H, W, dtype, device, generator, latents=None: torch.randn(
        B, C, H // 8, W // 8, generator=generator, dtype=dtype)
    proc = dh.apply_FRESCO_attn(pipe)
    N = 2
    imgs = torch.rand(N, 3, 128, 128) * 2 - 1
    pe = torch.randn(2 * N, 7, 24)
    corr = dh.get_intraframe_paras(pipe, imgs, proc, pe, seed=3)
    ctrl = proc.controller
    assert not ctrl.store and not ctrl.use_cfattn and not ctrl.use_intraattn and not ctrl.use_interattn
    stored = ctrl.stored_attn["decoder_attn"]
    assert [tuple(t.shape) for t in stored] == [(2 * N, 64, 64)] * 3 + [(2 * N, 256, 32)] * 3   # up_blocks.2 then .3
    # the same pass again, by hand: identical noise (same seed), hooks recording the decoder features
    g = torch.Generator().manual_seed(3)
    lat = pipe.prepare_latents(N, 4, 128, 128, pe.dtype, torch.device("cpu"), g)
    x0 = 0.5 * VAE.encode(imgs).latent_dist.sample()
    lat = pipe.scheduler.add_noise(x0, lat, Sched.timesteps[-1])
    with torch.no_grad():
        out = pipe.unet(torch.cat([lat] * 2), Sched.timesteps[-1], encoder_hidden_states=pe, return_dict=False)
    assert len(out) == 5 and len(corr) == 4
    for tgt, feat in zip(corr, out[1:]):
        v = feat.reshape(feat.shape[0], feat.shape[1], -1).transpose(1, 2)
        v = v / ((v ** 2).sum(dim=2, keepdim=True) ** 0.5)
        want = torch.bmm(v, v.transpose(-1, -2)).to(torch.float32)
        assert tgt.dtype == torch.float32 and tuple(tgt.shape) == tuple(want.shape)
        assert torch.allclose(tgt, want, atol=1e-6)
        assert torch.allclose(torch.diagonal(tgt, dim1=1, dim2=2), torch.ones(tgt.shape[0], tgt.shape[1]), atol=1e-5)
