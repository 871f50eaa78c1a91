"""CPU: the C-ABI library loads and exports every symbol include/*.h declares, the host-side
modules mirror the reference's interface (state_dict keys and shapes from the fixtures), and the
product path fails loudly -- never falls back -- without a CUDA device."""
import copy
import ctypes
import glob
import os
import pickle
import re
import types

import pytest
import torch

import galerkin_transformer_b200 as G
from galerkin_transformer_b200 import _lib, build as B
from helpers import golden_names, load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_symbols():
    names = set()
    for h in glob.glob(os.path.join(ROOT, "include", "*.h")):
        src = open(h).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names |= set(re.findall(r"\b(gb200_[a-z0-9_]+)\s*\(", src))
    return names


def test_library_builds_and_exports_every_declared_symbol():
    B.build()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    declared = _declared_symbols()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/ but not exported"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert _lib.load().gb200_version() >= 100


def test_error_reporting_without_gpu():
    lib = _lib.load()
    rc = lib.gb200_gemm(0, None, 1, 0, None, 1, 0, None, 1, 4, 4, 4, 1, 0, 0, 0, 1.0, None, 0, None, 0, 0.0,
                        0, None, 0, 1.0, 0, 1, None, 0, None)
    assert rc != 0
    assert b"null operand" in lib.gb200_last_error()
    with pytest.raises(RuntimeError, match="null operand"):
        _lib.check(rc, "gb200_gemm")


def build_module(fix):
    name, cfg = fix["name"], fix["config"]
    for prefix, cls in (("attn_", G.SimpleAttention), ("enc_", G.SimpleTransformerEncoderLayer),
                        ("sc1d_", G.SpectralConv1d), ("sc2d_", G.SpectralConv2d),
                        ("model_ft2dlite_", G.FourierTransformer2DLite),
                        ("model_ft2d_", G.FourierTransformer2D), ("model_simple_", G.SimpleTransformer)):
        if name.startswith(prefix):
            return cls(**cfg)
    raise KeyError(name)


@pytest.mark.parametrize("name", golden_names())
def test_state_dict_layout_matches_reference(name):
    fix = load_golden(name)
    mod = build_module(fix)
    sd, ref = mod.state_dict(), fix["state_dict"]
    assert list(sd.keys()) == list(ref.keys())
    for k in sd:
        assert sd[k].shape == ref[k].shape, k
    mod.load_state_dict(ref)                       # reference checkpoints load unchanged
    clone = copy.deepcopy(mod)                     # model.py:896, 1153 deepcopy the layer
    blob = pickle.dumps(mod)                       # utils_ft.py:804 pickles whole models
    assert list(pickle.loads(blob).state_dict().keys()) == list(clone.state_dict().keys())


def test_dropin_patch_rebinds_module_namespaces():
    """dropin.patch rebinds the hot-path classes in stand-ins for the reference's `layers` / `model` modules, whose
    assembly code looks its classes up in the module namespace at call time; assembly classes stay untouched."""
    from galerkin_transformer_b200.dropin import LAYER_CLASSES, MODEL_CLASSES, patch
    layers, model = types.ModuleType("layers"), types.ModuleType("model")
    for n in LAYER_CLASSES:
        setattr(layers, n, type(n, (torch.nn.Module,), {}))
    for n in MODEL_CLASSES + ("FourierTransformer2D",):
        setattr(model, n, type(n, (torch.nn.Module,), {}))
    model.SimpleAttention = layers.SimpleAttention          # what `from layers import *` leaves in libs/model.py
    assembly = model.FourierTransformer2D
    exec("def encoder_layer(**kw):\n    return SimpleTransformerEncoderLayer(**kw)\n", vars(model))

    done = patch(layers, model)
    assert done == {"layers": list(LAYER_CLASSES), "model": ["SimpleAttention", *MODEL_CLASSES]}
    for ns, names in ((layers, LAYER_CLASSES), (model, MODEL_CLASSES + ("SimpleAttention",))):
        for n in names:
            assert getattr(ns, n) is getattr(G, n), n
    assert model.FourierTransformer2D is assembly
    fix = load_golden("enc_galerkin_attnnorm")
    layer = model.encoder_layer(**fix["config"])
    assert isinstance(layer, G.SimpleTransformerEncoderLayer) and isinstance(layer.attn, G.SimpleAttention)
    assert list(layer.state_dict().keys()) == list(fix["state_dict"].keys())
    layer.load_state_dict(fix["state_dict"])


def test_no_cpu_fallback():
    attn = G.SimpleAttention(n_head=2, d_model=16, pos_dim=1, attention_type="galerkin", norm=True)
    x = torch.randn(2, 8, 16)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        attn(x, x, x, pos=torch.rand(2, 8, 1))
    conv = G.SpectralConv2d(4, 4, 2)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        conv(torch.randn(1, 8, 8, 4))


def test_unsupported_arguments_raise():
    with pytest.raises(NotImplementedError):
        G.SimpleAttention(n_head=2, d_model=16, attention_type="softmax")
    with pytest.raises(AssertionError):
        G.SimpleAttention(n_head=3, d_model=16)
    attn = G.SimpleAttention(n_head=2, d_model=16, attention_type="galerkin")
    x = torch.randn(1, 4, 16)
    with pytest.raises(RuntimeError, match="casual mask"):
        attn(x, x, x, mask=torch.ones(1, 4, 4))
    with pytest.raises(ValueError, match="Dimension not implemented"):
        G.SpectralConv2d(4, 4, 2)(torch.randn(8, 4))


def test_initialisation_statistics_follow_reference():
    torch.manual_seed(0)
    a = G.SimpleAttention(n_head=4, d_model=64, xavier_init=1e-2, diagonal_weight=1e-2, norm=True,
                          attention_type="galerkin", pos_dim=2)
    w = a.linears[0].weight
    off = w - torch.diag(torch.diag(w))
    bound = 1e-2 * (6 / 128) ** 0.5
    assert off.abs().max() <= bound + 1e-7
    assert abs(torch.diag(w).mean().item() - 1e-2) < 5e-3
    assert a.linears[1].bias.abs().max() == 0
    assert a.fc.weight.shape == (64, 64 + 4 * 2)
    s = G.SpectralConv2d(8, 8, 3)
    assert s.fourier_weight[0].shape == (8, 8, 3, 3, 2)


def test_scaler_sizes():
    assert G.scaler_sizes(141, 43) == ((0.555, 0.555), ((77, 77), (141, 141)))
    down, up = G.scaler_sizes(211, 71)
    assert up[1] == (211, 211)
    assert G.scaler_sizes(141, 43, scale_factor=False)[0] == ((77, 77), (43, 43))


@pytest.mark.parametrize("attention_type,norm", [("galerkin", True), ("fourier", True), ("galerkin", False)])
def test_packed_attention_parameter_layout(attention_type, norm):
    """The one-launch parameter pack (gb200_pack) and the slices the kernels / the flat gradient use must agree:
    concat(_packed_parts()) unpacks to W_qkv = [W_q; W_k; W_v], b_qkv and the (H, d_k) LayerNorm tables."""
    from galerkin_transformer_b200.functional import _unpack_attention_params
    H, dk = 3, 8
    dm = H * dk
    a = G.SimpleAttention(n_head=H, d_model=dm, pos_dim=2, attention_type=attention_type, norm=norm)
    with torch.no_grad():
        for p in a.parameters():
            p.copy_(torch.randn_like(p))
    flat = torch.cat([p.detach().reshape(-1) for p in a._packed_parts()])
    w, b, g1, b1, g2, b2 = _unpack_attention_params(flat, dm, H, dk, norm)
    assert torch.equal(w, torch.cat([l.weight for l in a.linears], 0))
    assert torch.equal(b, torch.cat([l.bias for l in a.linears], 0))
    if not norm:
        assert g1 is None and b2 is None and flat.numel() == 3 * dm * dm + 3 * dm
        return
    second = a.norm_V if attention_type == "galerkin" else a.norm_Q
    assert torch.equal(g1, torch.stack([m.weight for m in a.norm_K])) and torch.equal(b1, torch.stack([m.bias for m in a.norm_K]))
    assert torch.equal(g2, torch.stack([m.weight for m in second])) and torch.equal(b2, torch.stack([m.bias for m in second]))
    assert flat.numel() == 3 * dm * dm + 3 * dm + 4 * dm


def _resize_restated(x, Hout, Wout, backward_of=None):
    """csrc/interp.cu restated in numpy float32: forward taps / weights, and the GATHER backward with its candidate
    ranges (dst_range) -- the algorithm, not the kernel."""
    import math
    import numpy as np
    f32 = np.float32
    B_, Hin, Win, C = x.shape if backward_of is None else backward_of

    def axis(nin, nout):
        scale = f32(nin - 1) / f32(nout - 1) if nout > 1 else f32(0)
        s = (scale * np.arange(nout, dtype=f32)).astype(f32)
        i0 = np.minimum(s.astype(np.int64), nin - 1)
        i1 = i0 + (i0 < nin - 1)
        l = (s - i0.astype(f32)).astype(f32)
        return scale, i0, i1, l
    sy, y0, y1, ly = axis(Hin, Hout)
    sx, x0, x1, lx = axis(Win, Wout)
    if backward_of is None:
        v = x.astype(f32)
        top = v[:, y0][:, :, x0] * (1 - lx)[None, None, :, None] + v[:, y0][:, :, x1] * lx[None, None, :, None]
        bot = v[:, y1][:, :, x0] * (1 - lx)[None, None, :, None] + v[:, y1][:, :, x1] * lx[None, None, :, None]
        return top * (1 - ly)[None, :, None, None] + bot * ly[None, :, None, None]

    def ranges_and_weights(scale, nin, nout, i0, i1, l):
        out = []
        for i in range(nin):
            if scale <= 0:
                lo, hi = 0, nout - 1
            else:
                lo = max(0, int(math.floor(float(f32(i - 1) / scale))))
                hi = min(nout - 1, int(math.ceil(float(f32(i + 1) / scale))) + 1)
            w = [(d, (1 - l[d] if i0[d] == i else 0.0) + (l[d] if i1[d] == i else 0.0)) for d in range(lo, hi + 1)]
            touched = {d for d in range(nout) if i0[d] == i or i1[d] == i}
            assert touched <= set(range(lo, hi + 1)), "candidate range misses a contributing output index"
            out.append([(d, wd) for d, wd in w if wd != 0.0])
        return out
    wy = ranges_and_weights(sy, Hin, Hout, y0, y1, ly)
    wx = ranges_and_weights(sx, Win, Wout, x0, x1, lx)
    g = x.astype(f32)                                   # d_out (B, Hout, Wout, C)
    din = np.zeros((B_, Hin, Win, C), dtype=f32)
    for iy in range(Hin):
        for ix in range(Win):
            for oy, a_ in wy[iy]:
                for ox, b_ in wx[ix]:
                    din[:, iy, ix] += f32(a_ * b_) * g[:, oy, ox]
    return din


@pytest.mark.parametrize("Hin,Win,Hout,Wout", [(15, 15, 9, 9), (9, 9, 15, 15), (10, 7, 29, 31), (13, 11, 5, 4), (6, 6, 1, 1),
                                               (1, 1, 4, 5), (8, 8, 8, 8)])
def test_resize_algorithm_restated_on_cpu(Hin, Win, Hout, Wout):
    """The algorithm of csrc/interp.cu (taps, fp32 source indices, gather backward over dst_range candidates) equals
    F.interpolate(mode='bilinear', align_corners=True) and its autograd adjoint (libs/layers.py:493, 506, 660, 668)."""
    import numpy as np
    torch.manual_seed(0)
    x = torch.randn(2, Hin, Win, 3, dtype=torch.float64, requires_grad=True)
    y = torch.nn.functional.interpolate(x.permute(0, 3, 1, 2), size=(Hout, Wout), mode="bilinear", align_corners=True)
    cot = torch.randn(2, Hout, Wout, 3, dtype=torch.float64)
    (gx,) = torch.autograd.grad((y * cot.permute(0, 3, 1, 2)).sum(), [x])
    yr = _resize_restated(x.detach().numpy(), Hout, Wout)
    gr = _resize_restated(cot.numpy(), Hout, Wout, backward_of=(2, Hin, Win, 3))
    assert np.abs(yr - y.detach().permute(0, 2, 3, 1).numpy()).max() < 1e-5
    assert np.abs(gr - gx.numpy()).max() < 1e-5


def test_single_use_tracking_decides_when_side_stream_joins_may_be_deferred():
    """functional._note_use / _single_use: a parameter-gradient side stream may stay unjoined until the end of backward only
    if autograd will ADOPT the gradient tensor -- leaf parameter, used by exactly one node of the graph, no existing .grad."""
    import torch
    from galerkin_transformer_b200 import functional as GF
    w, b = torch.nn.Parameter(torch.zeros(3)), torch.nn.Parameter(torch.zeros(3))
    GF._note_use(w, b, None)
    assert GF._single_use((w, b, None))                       # one forward use each, grads empty
    assert GF._single_use((w,)) and w._gb200_total == 0       # counters are back to rest (a stray second call stays safe)
    # a rollout: the same weight feeds three nodes; none of the three backward nodes may defer
    for _ in range(3):
        GF._note_use(w)
    assert [GF._single_use((w,)) for _ in range(3)] == [False, False, False]
    GF._note_use(w)
    assert GF._single_use((w,))                               # next step: single use again
    # an existing gradient means accumulation on the launching stream
    w.grad = torch.ones(3)
    GF._note_use(w)
    assert not GF._single_use((w,))
    w.grad = None
    # non-leaf "parameters" (packed weights) are consumed by the next backward node right away
    packed = torch.cat([w, b]) * 1.0
    GF._note_use(packed)
    assert not GF._single_use((packed,))
    # no bookkeeping without grad mode (inference must not poison the counters)
    with torch.no_grad():
        GF._note_use(b)
    assert getattr(b, "_gb200_pending", 0) == 0
