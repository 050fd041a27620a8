# -*- coding: utf-8 -*-
"""CPU checks of the fp8 weight-only numerics contract (include/pia_b200.h, DESIGN §3): ops.quantize_fp8 element for
element, the tiled e4m3 layout of the GEMM plans, the ABI surface, and the shapes quantize_weights() refuses."""
import os
import re

import numpy as np
import pytest
import torch

from painlessinferenceacceleration_b200.common import ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _e4m3_grid():
    """every finite non-negative e4m3fn value, ascending"""
    codes = torch.arange(0, 0x7F, dtype=torch.uint8)   # 0x7F is NaN
    return codes.view(torch.float8_e4m3fn).float()


def _rne_reference(x):
    """round-to-nearest-even onto the e4m3 grid, saturating at 448, computed independently of torch's cast"""
    grid = _e4m3_grid().double().numpy()
    a = np.minimum(np.abs(x.double().numpy()), 448.0)
    i = np.clip(np.searchsorted(grid, a), 1, len(grid) - 1)
    lo, hi = grid[i - 1], grid[i]
    pick_hi = (a - lo > hi - a) | ((a - lo == hi - a) & ((i % 2) == 0))   # tie: even code (codes are i-1, i)
    out = np.where(a >= grid[-1], grid[-1], np.where(pick_hi, hi, lo))
    out = np.where(a <= 0, 0.0, out)
    return torch.from_numpy(np.copysign(out, x.double().numpy()))


def test_quantize_matches_formula():
    g = torch.Generator().manual_seed(0)
    w = (torch.randn(256, 384, generator=g) * 0.05).to(torch.bfloat16)
    w[3] = 0                                    # all-zero row: s = 1
    w[7, 11] = -3.0                             # a row dominated by one element
    w[9] = w[9] * 1e-4                          # tiny row: most of it lands in the subnormal range after scaling
    wq, s = ops.quantize_fp8(w)
    assert wq.dtype == torch.float8_e4m3fn and s.dtype == torch.float32 and s.shape == (256,)
    amax = w.float().abs().amax(dim=1)
    want_s = torch.where(amax == 0, torch.ones_like(amax), amax / 448.0)
    assert torch.equal(s, want_s)
    assert s[3] == 1.0 and torch.all(wq[3].float() == 0)
    scaled = w.float() / want_s[:, None]
    assert torch.equal(wq.float().double(), _rne_reference(scaled))
    # the row maximum maps to +-448 exactly
    assert torch.equal(wq.float().abs().amax(dim=1)[amax > 0], torch.full_like(amax[amax > 0], 448.0))


def test_quantize_error_bounds():
    g = torch.Generator().manual_seed(1)
    w = (torch.randn(128, 512, generator=g) * torch.logspace(-3, 0, 512)[None]).to(torch.bfloat16)
    wq, s = ops.quantize_fp8(w)
    x = w.float() / s[:, None]
    q = wq.float()
    normal = x.abs() >= 2.0 ** -6
    rel = ((q - x).abs() / x.abs())[normal]
    assert normal.sum() > 1000 and rel.max() <= 2.0 ** -4
    sub = ~normal
    assert sub.sum() > 100
    # half the subnormal step 2^-9, i.e. 2^-10 * s in the weight's own units
    assert ((q - x).abs()[sub]).max() <= 2.0 ** -10
    deq = q * s[:, None]
    assert (((deq - w.float()).abs())[sub] <= 2.0 ** -10 * s[:, None].expand_as(deq)[sub] * (1 + 1e-6)).all()


def test_quantize_saturates_and_ties_to_even():
    # scale fixed by a 448 element in each row; the other elements probe ties and the top of the range
    probe = torch.tensor([448.0, 17.0, 19.0, 0.5 * (1 + 1.125) * 2 ** -6, 2 ** -10, 3 * 2 ** -10, -17.0, 464.0, -464.0])
    w = probe[None].repeat(128, 1).to(torch.float32)
    w = torch.cat([w, torch.zeros(128, 128 - probe.numel())], dim=1)
    # +-464 set the scale; every element is compared with the independent RNE restatement
    s_want = w.abs().amax(dim=1) / 448.0
    wq, s = ops.quantize_fp8(w)
    assert torch.equal(s, s_want)
    x = w / s[:, None]
    assert torch.equal(wq.float().double(), _rne_reference(x))
    row = wq[0].float()
    assert row.abs().max() == 448.0                     # saturation, never NaN
    assert not torch.isnan(row).any()
    # direct ties at scale 1: 17 = between 16 and 18 -> 16 (even mantissa), 19 -> 20
    one = torch.tensor([[17.0, 19.0, 2 ** -10, 3 * 2 ** -10, 448.0] + [0.0] * 123])
    q1, s1 = ops.quantize_fp8(one)
    assert s1.item() == 1.0
    assert q1[0, :4].float().tolist() == [16.0, 20.0, 0.0, 2.0 ** -8]


def test_quantize_leading_dims():
    w = torch.randn(3, 128, 256).to(torch.bfloat16)
    wq, s = ops.quantize_fp8(w)
    assert wq.shape == (3, 128, 256) and s.shape == (3, 128)
    for e in range(3):
        q1, s1 = ops.quantize_fp8(w[e])
        assert torch.equal(q1.view(torch.uint8), wq[e].view(torch.uint8)) and torch.equal(s1, s[e])


def test_tile_weight_fp8_layout():
    w = torch.randint(0, 0x7E, (384, 256), dtype=torch.uint8).view(torch.float8_e4m3fn)
    t = ops.tile_weight_fp8(w)
    assert t.shape == (3, 2, 128, 128) and t.is_contiguous() and t.pia_shape == (384, 256)
    u8, t8 = w.view(torch.uint8), t.view(torch.uint8)
    for nt in range(3):
        for kt in range(2):
            assert torch.equal(t8[nt, kt], u8[nt * 128:(nt + 1) * 128, kt * 128:(kt + 1) * 128])
    assert torch.equal(ops.untile_weight_fp8(t).view(torch.uint8), u8)
    stacked = torch.stack([w, w]).contiguous()
    ts = ops.tile_weight_fp8(stacked)
    assert ts.shape == (2, 3, 2, 128, 128)
    assert torch.equal(ts[1].view(torch.uint8), t8)
    with pytest.raises(ValueError):
        ops.tile_weight_fp8(w[:, :192])


def _declared():
    hdr = open(os.path.join(ROOT, 'include', 'pia_b200.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    return set(re.findall(r'\b(pia_[a-z0-9_]+)\s*\(', hdr))


def test_fp8_symbols_declared_bound_and_exported():
    import ctypes
    from painlessinferenceacceleration_b200 import _lib
    from painlessinferenceacceleration_b200.build import build_library
    names = {'pia_gemm_plan_create_fp8', 'pia_gemm_plan_create_grouped_fp8'}
    assert names <= _declared()
    assert names <= set(_lib.SYMBOLS)
    assert len(_lib.SYMBOLS['pia_gemm_plan_create_fp8'][1]) == 9
    assert len(_lib.SYMBOLS['pia_gemm_plan_create_grouped_fp8'][1]) == 8
    lib = ctypes.CDLL(build_library())
    assert all(hasattr(lib, n) for n in names)


def _meta_llama(**over):
    from tests.tiny_models import tiny_config
    from painlessinferenceacceleration_b200.models.llama.modeling_llama import LlamaForCausalLM
    return LlamaForCausalLM(tiny_config('llama', **over), device=torch.device('meta'))


def test_quantize_weights_rejects_gpt2_and_unaligned_shapes():
    from tests.tiny_models import tiny_config
    from painlessinferenceacceleration_b200.models.gpt2.modeling_gpt2 import GPT2LMHeadModel
    g = GPT2LMHeadModel(tiny_config('gpt2'), device=torch.device('meta'))
    with pytest.raises(ValueError):
        g.quantize_weights(torch.float8_e4m3fn)
    # K % 128 != 0: hidden 192 (o / gate_up / qkv have K = 192)
    m = _meta_llama(hidden_size=192, num_attention_heads=1, num_key_value_heads=1, head_dim=192)
    with pytest.raises(ValueError, match='multiples of 128'):
        m.quantize_weights()
    assert not m.quantized and hasattr(m.model.layers[0].self_attn, 'q_proj')   # nothing was changed
    # intermediate 320: down has K = 320
    m = _meta_llama(intermediate_size=320)
    with pytest.raises(ValueError, match='multiples of 128'):
        m.quantize_weights()
    with pytest.raises(ValueError):
        _meta_llama().quantize_weights(torch.float8_e5m2)


def test_prequantised_checkpoints_are_rejected():
    m = _meta_llama(quantization_config={'quant_method': 'gptq', 'bits': 4})
    with pytest.raises(ValueError, match='pre-quantised'):
        m.quantize_weights()
