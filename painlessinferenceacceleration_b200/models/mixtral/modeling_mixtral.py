# -*- coding: utf-8 -*-
"""Mixtral with the lookahead patch (reference: models/mixtral/modeling_mixtral.py, patch :1032-1036, attention
:302-381, MixtralSparseMoeBlock :692-759, expert MLP :668-683).

Attention / norms / RoPE are the Llama-family kernels (GQA packed into the UMMA tile).  The MoE block: at n = 64
draft nodes with top-2 of 8 routing practically every expert is hit, so the verify step reads all expert weights
either way (SURVEY.md 8d: >= 90 GB per step); the block therefore evaluates every expert on all n rows with
static-shape GEMMs (CUDA-graph friendly, no host-side routing) and combines with the routing weights, zero for
unselected experts.  Rounding follows the reference: fp32 softmax -> top-k -> renormalise -> cast to bf16 (:723-727);
per token the two selected expert outputs are scaled in bf16 and accumulated in expert-index order, exactly what
`index_add_` into a zero tensor produces (:729-757); adding an unselected expert's 0 is exact."""
import torch
from torch import nn

from ...common import ops
from ..llama.modeling_llama import LlamaDecoderLayer, LlamaForCausalLM, LlamaModel
from ..mistral.modeling_mistral import warn_sliding_window


class MixtralRouter(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        self.weight = nn.Parameter(torch.empty((cfg.num_local_experts, cfg.hidden_size), device=device, dtype=dtype))


class MixtralExperts(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        E, H, I = cfg.num_local_experts, cfg.hidden_size, cfg.intermediate_size
        self.gate_up_proj = nn.Parameter(torch.empty((E, 2 * I, H), device=device, dtype=dtype))
        self.down_proj = nn.Parameter(torch.empty((E, H, I), device=device, dtype=dtype))


class MixtralSparseMoeBlock(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        self.top_k = cfg.num_experts_per_tok
        self.num_experts = cfg.num_local_experts
        self.gate = MixtralRouter(cfg, device, dtype)
        self.experts = MixtralExperts(cfg, device, dtype)


class MixtralDecoderLayer(LlamaDecoderLayer):
    def _make_mlp(self, cfg, device, dtype):
        return MixtralSparseMoeBlock(cfg, device, dtype)


class MixtralModel(LlamaModel):
    layer_cls = MixtralDecoderLayer


class MixtralForCausalLM(LlamaForCausalLM):
    model_cls = MixtralModel

    def _fuse_mlp(self, layer):
        pass  # experts are stored fused ([E, 2I, H]) already

    def rope_tables(self, max_pos):
        warn_sliding_window(self.config, max_pos)  # mixtral/modeling_mixtral.py:1032-1036: no window on the lookahead branch
        return super().rope_tables(max_pos)

    def _convert_checkpoint_keys(self, sd):
        """published Mixtral checkpoints (and the reference, mixtral/modeling_mixtral.py:692-759) name the MoE block
        `block_sparse_moe` with per-expert `experts.N.w1 / w3 / w2` Linear weights; this module tree keeps the experts
        stacked: gate_up_proj[e] = [w1; w3] ([2I, H]), down_proj[e] = w2 ([H, I]), router = `mlp.gate.weight`.  Tensors
        of one layer's experts may arrive in different shards: partial stacks are kept until complete."""
        import re
        out = {}
        pend = self.__dict__.setdefault('_pending_experts', {})
        E = self.config.num_local_experts
        pat = re.compile(r'^(model\.layers\.\d+)\.block_sparse_moe\.experts\.(\d+)\.(w1|w2|w3)\.weight$')
        for k, v in sd.items():
            m = pat.match(k)
            if m:
                pend.setdefault(m.group(1), {})[(int(m.group(2)), m.group(3))] = v
            elif '.block_sparse_moe.gate.weight' in k:
                out[k.replace('.block_sparse_moe.gate.weight', '.mlp.gate.weight')] = v
            else:
                out[k] = v
        for layer in list(pend):
            parts = pend[layer]
            if len(parts) == 3 * E:
                out[layer + '.mlp.experts.gate_up_proj'] = torch.stack(
                    [torch.cat([parts[(e, 'w1')], parts[(e, 'w3')]], dim=0) for e in range(E)], dim=0)
                out[layer + '.mlp.experts.down_proj'] = torch.stack([parts[(e, 'w2')] for e in range(E)], dim=0)
                del pend[layer]
        return out

    def geometry(self):
        g = super().geometry()
        g['n_experts'] = self.config.num_local_experts
        return g

    def _layer_gemm_plans(self, layer, b):
        """decode steps (64-row buffers): all experts' gate_up as ONE k_gemm_ws launch over the stacked [E*2I, H] weight,
        SiLU*up over the [64*E, 2I] view, all experts' down projections as one grouped launch, then the routing-weighted
        sum in expert order.  Dense over experts like the cuBLAS path below: at n = 64 draft rows every expert is hit
        (SURVEY 8d), and the step is bound by the expert weight bytes either way.  PIA_MOE_GEMM=0 keeps cuBLAS."""
        import os
        moe = layer.mlp
        E, two_i, H = moe.experts.gate_up_proj.shape
        inter = two_i // 2
        if os.environ.get('PIA_MOE_GEMM', '1') == '0' or H % 128 or H % 64 or inter % 64 or (E * two_i) % 128:
            return {}
        self._moe_bufs(b, E, inter, H)
        return {'moe_gate_up': ops.Gemm(moe.experts.gate_up_proj.data.view(E * two_i, H), b.y),
                'moe_down': ops.Gemm.grouped(moe.experts.down_proj.data, b.moe_act)}

    @staticmethod
    def _moe_bufs(b, E, inter, H):
        if not hasattr(b, 'moe_gu'):
            dev = b.y.device
            b.moe_gu = torch.zeros((b.rows, E * 2 * inter), dtype=torch.bfloat16, device=dev)
            b.moe_act = torch.zeros((b.rows, E * inter), dtype=torch.bfloat16, device=dev)
            b.moe_out = torch.zeros((b.rows, H), dtype=torch.bfloat16, device=dev)
            b.moe_dense = torch.zeros((b.rows, E), dtype=torch.bfloat16, device=dev)

    def _quantize_mlp(self, layer):
        """stacked experts: gate_up [E, 2I, H] -> one fp8 weight [E*2I, H] (one plan over all experts, as the bf16
        path), down [E, H, I] -> per-expert tiles + scales [E, H] for the grouped plan"""
        ex = layer.mlp.experts
        E, two_i, H = ex.gate_up_proj.shape
        wq, s = ops.quantize_fp8(ex.gate_up_proj.data)
        ex.register_buffer('gate_up_fp8', ops.tile_weight_fp8(wq.view(E * two_i, H)))
        ex.register_buffer('gate_up_scale', s.reshape(E * two_i).contiguous())
        del wq
        wq, s = ops.quantize_fp8(ex.down_proj.data)
        ex.register_buffer('down_fp8', ops.tile_weight_fp8(wq))
        ex.register_buffer('down_scale', s.contiguous())
        del ex.gate_up_proj, ex.down_proj

    def _fp8_mlp_plans(self, layer, b):
        moe, c = layer.mlp, self.config
        self._moe_bufs(b, moe.num_experts, c.intermediate_size, c.hidden_size)
        return {'moe_gate_up': ops.Gemm.fp8(moe.experts.gate_up_fp8, moe.experts.gate_up_scale, b.y),
                'moe_down': ops.Gemm.grouped_fp8(moe.experts.down_fp8, moe.experts.down_scale, b.moe_act)}

    def _mlp(self, rt, layer, y, plans=None, pf=None, b=None):
        moe = layer.mlp
        if plans:
            b = b if b is not None else rt.decode_bufs
            E = moe.num_experts
            inter = self.config.intermediate_size
            ops.moe_router(y, moe.gate.weight, moe.top_k, b.moe_dense)              # :721-727 in one kernel
            plans['moe_gate_up'].run(b.rows, out=b.moe_gu)
            ops.silu_mul(b.moe_gu.view(b.rows * E, 2 * inter), b.moe_act.view(b.rows * E, inter))
            ye = plans['moe_down'].run(b.rows)                                      # [E, rows, H]
            ops.moe_combine(ye, b.moe_dense, b.moe_out)
            return b.moe_out, None
        dense = torch.empty((y.shape[0], moe.num_experts), dtype=y.dtype, device=y.device)
        ops.moe_router(y, moe.gate.weight, moe.top_k, dense)                        # :721-727
        out = torch.zeros_like(y)
        inter = moe.experts.down_proj.shape[2]
        act = torch.empty((y.shape[0], inter), dtype=y.dtype, device=y.device)
        for e in range(moe.num_experts):                                            # expert-index order (:734)
            gu = torch.mm(y, moe.experts.gate_up_proj[e].t())
            ops.silu_mul(gu, act)
            ye = torch.mm(act, moe.experts.down_proj[e].t())
            out += ye * dense[:, e:e + 1]                                           # bf16 scale, bf16 accumulate
        return out, None
