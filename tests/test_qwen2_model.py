# -*- coding: utf-8 -*-
"""Qwen2ForCausalLM's module tree and the shapes it accepts (no device needed: the model is built on the CPU)."""
import pytest
import torch

from tests.tiny_qwen2 import qwen2_config, qwen2_hf_model


@pytest.mark.parametrize('shape', ['g7', 'g6_tied'])
def test_parameter_names_are_hf_qwen2s(shape):
    from painlessinferenceacceleration_b200.models.qwen2.modeling_qwen2 import Qwen2ForCausalLM
    hf = qwen2_hf_model(shape, dtype=torch.bfloat16, vocab=96)
    ours = Qwen2ForCausalLM(hf.config, device='cpu')
    assert set(ours.state_dict()) == set(hf.state_dict())
    ours.load_state_dict(hf.state_dict(), strict=True)
    ours.fuse()   # the biases become views of one fused qkv bias, in q, k, v order
    a, h = ours.model.layers[1].self_attn, hf.model.layers[1].self_attn
    assert torch.equal(a.qkv_bias, torch.cat([h.q_proj.bias, h.k_proj.bias, h.v_proj.bias]))
    assert a.v_proj.bias.data_ptr() == a.qkv_bias[-a.v_proj.bias.numel():].data_ptr()
    g = ours.geometry()
    assert (g['n_q_heads'], g['n_kv_heads'], g['head_dim']) == (hf.config.num_attention_heads, 1, 128)


def test_head_dim_other_than_128_is_refused():
    from painlessinferenceacceleration_b200.models.qwen2.modeling_qwen2 import Qwen2ForCausalLM
    cfg = qwen2_config('g7', hidden_size=896, num_attention_heads=14, num_key_value_heads=2)   # Qwen2-0.5B: 64
    with pytest.raises(ValueError, match='Qwen2ForCausalLM: head_dim 64'):
        Qwen2ForCausalLM(cfg, device='meta')


def test_sliding_window_is_reported():
    from painlessinferenceacceleration_b200.models.qwen2.modeling_qwen2 import Qwen2ForCausalLM
    cfg = qwen2_config('g7', use_sliding_window=True, sliding_window=16)
    m = Qwen2ForCausalLM(cfg, device='cpu')
    with pytest.warns(UserWarning, match='sliding_window=16 is ignored'):
        m.rope_tables(64)
