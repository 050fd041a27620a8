# -*- coding: utf-8 -*-
"""GPT-2 with the lookahead patch, B200-native.

Reference: /root/reference/lookahead/lookahead/models/gpt2/modeling_gpt2.py - patch :805-809 (rank-4 mask ->
position_ids = rowsum - 1, additive mask), attention `_attn` :183-221 (its own causal bias AND the tree mask; a tree
mask is a subset of the causal one, so one visibility test suffices), Conv1D projections, LayerNorm, gelu_new MLP,
tied lm_head.  The module tree and parameter names are HF's (`transformer.wte/wpe/h.N.{ln_1,attn.c_attn,attn.c_proj,
ln_2,mlp.c_fc,mlp.c_proj}/ln_f`), so checkpoints load unchanged.

GPT-2's heads are 64 wide (any width <= 128 works): they run on the SAME tcgen05 tree-attention kernel as the Llama
family by zero-padding every head to the kernel's 128-wide tile - the fused c_attn weight is re-laid out once so that
the projection writes padded q | k | v heads, K/V are appended to the cache through k_rope_kv_append with an identity
rotation table (cos = 1, sin = 0: GPT-2 has learned absolute positions, added to the embedding), the kernel's softmax
scale 1/sqrt(128) is corrected by scale_mul = sqrt(128 / head_dim), and c_proj ignores the padding columns.  The
projections are plain library GEMMs with bias (torch.addmm), LayerNorm / GELU are torch ops: the model is 124 M
parameters - the hot, non-library ops are the trie, the tree attention and the accept path, shared with every family."""
import math

import torch
from torch import nn
from torch.nn import functional as F

from ...common import ops
from ...common.pretrained_model import LookaheadPreTrainedModel

PAD_D = 128


class Conv1D(nn.Module):
    """HF's Conv1D: y = x @ weight + bias with weight [in, out]"""

    def __init__(self, nf, nx, device, dtype):
        super().__init__()
        self.weight = nn.Parameter(torch.empty((nx, nf), device=device, dtype=dtype))
        self.bias = nn.Parameter(torch.zeros((nf,), device=device, dtype=dtype))


class GPT2Attention(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        self.c_attn = Conv1D(3 * cfg.n_embd, cfg.n_embd, device, dtype)
        self.c_proj = Conv1D(cfg.n_embd, cfg.n_embd, device, dtype)


class GPT2MLP(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        inner = cfg.n_inner if getattr(cfg, 'n_inner', None) else 4 * cfg.n_embd
        self.c_fc = Conv1D(inner, cfg.n_embd, device, dtype)
        self.c_proj = Conv1D(cfg.n_embd, inner, device, dtype)


class GPT2Block(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        kw = dict(eps=cfg.layer_norm_epsilon, device=device, dtype=dtype)
        self.ln_1 = nn.LayerNorm(cfg.n_embd, **kw)
        self.attn = GPT2Attention(cfg, device, dtype)
        self.ln_2 = nn.LayerNorm(cfg.n_embd, **kw)
        self.mlp = GPT2MLP(cfg, device, dtype)


class GPT2Model(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        self.wte = nn.Embedding(cfg.vocab_size, cfg.n_embd, device=device, dtype=dtype)
        self.wpe = nn.Embedding(cfg.n_positions, cfg.n_embd, device=device, dtype=dtype)
        self.h = nn.ModuleList([GPT2Block(cfg, device, dtype) for _ in range(cfg.n_layer)])
        self.ln_f = nn.LayerNorm(cfg.n_embd, eps=cfg.layer_norm_epsilon, device=device, dtype=dtype)


class GPT2LMHeadModel(LookaheadPreTrainedModel):
    def __init__(self, config, device=None, dtype=torch.bfloat16):
        super().__init__(config)
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device()) if torch.cuda.is_available() else 'meta'
        assert dtype == torch.bfloat16, 'the B200 path computes in bf16'
        assert config.n_embd % config.n_head == 0 and config.n_embd // config.n_head <= PAD_D
        self.transformer = GPT2Model(config, device, dtype)
        self.lm_head = nn.Linear(config.n_embd, config.vocab_size, bias=False, device=device, dtype=dtype)
        self.lm_head.weight = self.transformer.wte.weight  # tied (reference :1000)
        self._fused = False
        for p_ in self.parameters():
            p_.requires_grad_(False)

    @torch.no_grad()
    def init_weights(self, seed=0, std=0.02):
        gen = torch.Generator(device=self.device)
        gen.manual_seed(seed)
        for name, p in self.named_parameters():
            if '.ln_' in name or name.endswith('ln_f.weight') or name.endswith('ln_f.bias'):
                p.fill_(1.0 if name.endswith('weight') else 0.0)
            elif name.endswith('bias'):
                p.zero_()
            else:
                p.normal_(0.0, std, generator=gen)
        return self

    # ------------------------------------------------------------------ geometry / tables
    def geometry(self):
        c = self.config
        return dict(n_layers=c.n_layer, hidden=c.n_embd, n_q_heads=c.n_head, n_kv_heads=c.n_head, head_dim=PAD_D,
                    inter=c.n_inner if getattr(c, 'n_inner', None) else 4 * c.n_embd, vocab=c.vocab_size)

    def rope_tables(self, max_pos):
        """identity rotation: k_rope_kv_append then only copies q and appends K / V (x * 1 + rot(x) * 0, exact)"""
        dev = self.device
        return (torch.ones((max_pos, PAD_D // 2), dtype=torch.bfloat16, device=dev),
                torch.zeros((max_pos, PAD_D // 2), dtype=torch.bfloat16, device=dev))

    @torch.no_grad()
    def quantize_weights(self, dtype=None):
        raise ValueError('fp8 weights are not built for GPT-2: its Conv1D projections run through torch, not the '
                         'weight-streaming GEMM')

    def fuse(self):
        """c_attn / c_proj re-laid out for 128-wide (zero padded) heads; done once, outside any captured graph"""
        if self._fused:
            return
        c = self.config
        H, E = c.n_head, c.n_embd
        d = E // H
        for blk in self.transformer.h:
            a = blk.attn
            w = a.c_attn.weight.data            # [E, 3E]: q | k | v, each H heads of d
            wp = torch.zeros((E, 3 * H * PAD_D), dtype=w.dtype, device=w.device)
            bp = torch.zeros((3 * H * PAD_D,), dtype=w.dtype, device=w.device)
            wp.view(E, 3 * H, PAD_D)[:, :, :d] = w.view(E, 3 * H, d)
            bp.view(3 * H, PAD_D)[:, :d] = a.c_attn.bias.data.view(3 * H, d)
            a.qkv_weight_padded, a.qkv_bias_padded = wp.contiguous(), bp
            wo = torch.zeros((H * PAD_D, E), dtype=w.dtype, device=w.device)
            wo.view(H, PAD_D, E)[:, :d] = a.c_proj.weight.data.view(H, d, E)
            a.o_weight_padded = wo.contiguous()
        self._fused = True

    # ------------------------------------------------------------------ the verify forward on static buffers
    def _positions(self, rt, b):
        """position_ids = rowsum(attention_mask) - 1 (reference :807): visible prefix of the row's slot + tree depth"""
        rows, rps = b.slots.rows, b.slots.rows_per_slot
        key = ('gpt2_pos', rows, rps)
        aux = rt.__dict__.setdefault('_aux', {})
        if key not in aux:
            aux[key] = (torch.arange(rows, device=rt.device) // rps, torch.arange(64, device=rt.device))
        slot_of_row, shifts = aux[key]
        depth = ((b.mask[:rows].unsqueeze(-1) >> shifts) & 1).sum(dim=(1, 2)) - 1
        P = b.slots.prefix_len[:b.slots.batch].long()[slot_of_row]
        pad = b.slots.pad_len[:b.slots.batch].long()[slot_of_row] if b.slots.pad_len is not None else 0
        return ((P - pad).clamp(min=0) + depth).clamp(min=0, max=self.config.n_positions - 1)

    def _verify_layers(self, rt, bufs=None, last_only=False):
        self.fuse()
        b = bufs if bufs is not None else rt.decode_bufs
        c = self.config
        H = c.n_head
        rows = b.slots.rows
        eps = c.layer_norm_epsilon
        tr = self.transformer
        scale_mul = math.sqrt(PAD_D / (c.n_embd // H))
        ids = b.ids[:rows].long().clamp(min=0, max=c.vocab_size - 1)
        x = tr.wte.weight[ids] + tr.wpe.weight[self._positions(rt, b)]
        for li, blk in enumerate(tr.h):
            a = blk.attn
            y = F.layer_norm(x, (c.n_embd,), blk.ln_1.weight, blk.ln_1.bias, eps)
            torch.addmm(a.qkv_bias_padded, y, a.qkv_weight_padded, out=b.qkv[:rows])
            ops.rope_kv_append(b.qkv, b.mask, b.slots, H, H, PAD_D, rt.rope_cos, rt.rope_sin, b.q,
                               rt.k_layer(li, b.kv_slot), rt.v_layer(li, b.kv_slot), rt.max_seq)
            rt.plan.forward(li, b.q, b.mask, b.slots, b.attn, scale_mul=scale_mul)
            x = x + torch.addmm(a.c_proj.bias, b.attn[:rows], a.o_weight_padded)
            y = F.layer_norm(x, (c.n_embd,), blk.ln_2.weight, blk.ln_2.bias, eps)
            h = F.gelu(torch.addmm(blk.mlp.c_fc.bias, y, blk.mlp.c_fc.weight), approximate='tanh')   # gelu_new
            x = x + torch.addmm(blk.mlp.c_proj.bias, h, blk.mlp.c_proj.weight)
        if last_only:
            return
        x = F.layer_norm(x, (c.n_embd,), tr.ln_f.weight, tr.ln_f.bias, eps)
        b.y[:rows].copy_(x)
        if b.logits is not None:
            torch.mm(x, self.lm_head.weight.t(), out=b.logits[:rows])

