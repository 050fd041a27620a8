# -*- coding: utf-8 -*-
"""Qwen2 (Qwen1.5 / Qwen2 / Qwen2.5 checkpoints, HF `Qwen2ForCausalLM`) with the lookahead patch.

Reference: models/qwen2/modeling_qwen2.py - the patch :997-1000 is Llama's (position_ids = rowsum - 1, additive
finfo.min mask), attention :234-236 adds a bias to the q/k/v projections.  Everything else is the Llama decoder:
RMSNorm, SiLU MLP, RoPE (rope_theta 1e6 on the published checkpoints), GQA.  The verify forward is
LlamaForCausalLM's; the fused qkv projection runs as one cuBLASLt GEMM with a bias epilogue.  On the main
checkpoints G = 28 / 4 = 7 query heads per KV head: the tree attention packs head pairs within a KV head (the last
group of each KV head holds its leftover head alone)."""
from torch import nn

from ..llama.modeling_llama import LlamaAttention, LlamaDecoderLayer, LlamaForCausalLM, LlamaModel
from ..mistral.modeling_mistral import warn_sliding_window


def _head_dim(cfg):
    hd = getattr(cfg, 'head_dim', None) or cfg.hidden_size // cfg.num_attention_heads
    if hd != 128:
        raise ValueError(f'Qwen2ForCausalLM: head_dim {hd} is not supported (the tree attention kernel is built for '
                         f'head_dim 128; Qwen2-0.5B-sized models with head_dim 64 are not)')
    return hd


class Qwen2Attention(LlamaAttention):
    """HF's parameter names; q/k/v carry a bias, o does not (reference :234-237)"""

    def __init__(self, cfg, device, dtype):
        nn.Module.__init__(self)
        hd = _head_dim(cfg)
        kv = getattr(cfg, 'num_key_value_heads', None) or cfg.num_attention_heads
        kw = dict(device=device, dtype=dtype)
        self.q_proj = nn.Linear(cfg.hidden_size, cfg.num_attention_heads * hd, bias=True, **kw)
        self.k_proj = nn.Linear(cfg.hidden_size, kv * hd, bias=True, **kw)
        self.v_proj = nn.Linear(cfg.hidden_size, kv * hd, bias=True, **kw)
        self.o_proj = nn.Linear(cfg.num_attention_heads * hd, cfg.hidden_size, bias=False, **kw)


class Qwen2DecoderLayer(LlamaDecoderLayer):
    def _make_attn(self, cfg, device, dtype):
        return Qwen2Attention(cfg, device, dtype)


class Qwen2Model(LlamaModel):
    layer_cls = Qwen2DecoderLayer


class Qwen2ForCausalLM(LlamaForCausalLM):
    model_cls = Qwen2Model

    def geometry(self):
        g = super().geometry()
        g['head_dim'] = _head_dim(self.config)
        return g

    def rope_tables(self, max_pos):
        # use_sliding_window=True: the reference's lookahead branch ignores the window as Mistral's does
        if getattr(self.config, 'use_sliding_window', False):
            warn_sliding_window(self.config, max_pos)
        return super().rope_tables(max_pos)
