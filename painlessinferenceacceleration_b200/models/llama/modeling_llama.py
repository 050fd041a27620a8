# -*- coding: utf-8 -*-
"""Llama with the lookahead patch, B200-native.

Reference: /root/reference/lookahead/lookahead/models/llama/modeling_llama.py
  patch :584-588 (rank-4 mask -> position_ids = rowsum-1, additive mask), attention :243-308, RoPE :93-169,
  RMSNorm :76-90, MLP :172-186, LM head :768-769.
The module tree and parameter names are HF's (so checkpoints load unchanged); the forward over a draft of
<= 64/128 tree nodes runs on static buffers:  fused QKV / gate-up cuBLAS GEMMs + libpia_b200 kernels
(rmsnorm+residual, rope+kv-append into a preallocated cache, tcgen05 tree attention, silu*mul).  The rank-4 mask
is never built: `mask` is the per-node ancestor bit set, the prefix is implicit."""
import glob
import json
import os

import torch
from torch import nn

from ...common import ops
from ...common.pretrained_model import LookaheadPreTrainedModel


class LlamaRMSNorm(nn.Module):
    def __init__(self, hidden_size, eps=1e-6, device=None, dtype=None):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(hidden_size, device=device, dtype=dtype))
        self.variance_epsilon = eps


class LlamaAttention(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        hd = cfg.hidden_size // cfg.num_attention_heads
        kv = getattr(cfg, 'num_key_value_heads', None) or cfg.num_attention_heads
        kw = dict(bias=False, device=device, dtype=dtype)
        self.q_proj = nn.Linear(cfg.hidden_size, cfg.num_attention_heads * hd, **kw)
        self.k_proj = nn.Linear(cfg.hidden_size, kv * hd, **kw)
        self.v_proj = nn.Linear(cfg.hidden_size, kv * hd, **kw)
        self.o_proj = nn.Linear(cfg.num_attention_heads * hd, cfg.hidden_size, **kw)


class LlamaMLP(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        kw = dict(bias=False, device=device, dtype=dtype)
        self.gate_proj = nn.Linear(cfg.hidden_size, cfg.intermediate_size, **kw)
        self.up_proj = nn.Linear(cfg.hidden_size, cfg.intermediate_size, **kw)
        self.down_proj = nn.Linear(cfg.intermediate_size, cfg.hidden_size, **kw)


class LlamaDecoderLayer(nn.Module):
    def __init__(self, cfg, device, dtype):
        super().__init__()
        self.self_attn = self._make_attn(cfg, device, dtype)
        self.mlp = self._make_mlp(cfg, device, dtype)
        self.input_layernorm = LlamaRMSNorm(cfg.hidden_size, cfg.rms_norm_eps, device, dtype)
        self.post_attention_layernorm = LlamaRMSNorm(cfg.hidden_size, cfg.rms_norm_eps, device, dtype)

    def _make_attn(self, cfg, device, dtype):
        return LlamaAttention(cfg, device, dtype)

    def _make_mlp(self, cfg, device, dtype):
        return LlamaMLP(cfg, device, dtype)


class LlamaModel(nn.Module):
    layer_cls = LlamaDecoderLayer

    def __init__(self, cfg, device, dtype):
        super().__init__()
        self.embed_tokens = nn.Embedding(cfg.vocab_size, cfg.hidden_size, device=device, dtype=dtype)
        self.layers = nn.ModuleList([self.layer_cls(cfg, device, dtype) for _ in range(cfg.num_hidden_layers)])
        self.norm = LlamaRMSNorm(cfg.hidden_size, cfg.rms_norm_eps, device, dtype)


class LlamaForCausalLM(LookaheadPreTrainedModel):
    model_cls = LlamaModel

    def __init__(self, config, device=None, dtype=torch.bfloat16):
        super().__init__(config)
        if device is None:
            device = torch.device('cuda', torch.cuda.current_device()) if torch.cuda.is_available() else 'meta'
        assert dtype == torch.bfloat16, 'the B200 path computes in bf16'
        self.model = self.model_cls(config, device, dtype)
        self.lm_head = nn.Linear(config.hidden_size, config.vocab_size, bias=False, device=device, dtype=dtype)
        self._fused = False
        for p_ in self.parameters():  # inference only: no autograd state on the hot path
            p_.requires_grad_(False)

    # ------------------------------------------------------------------ weights
    @torch.no_grad()
    def init_weights(self, seed=0, std=0.02):
        """random-init weights of the configured shape (there are no checkpoints offline)"""
        gen = torch.Generator(device=self.device)
        gen.manual_seed(seed)
        for name, p in self.named_parameters():
            if name.endswith('layernorm.weight') or name.endswith('norm.weight'):
                p.fill_(1.0)
            else:
                p.normal_(0.0, std, generator=gen)
        return self

    @classmethod
    def from_pretrained(cls, path, torch_dtype=torch.bfloat16, device=None, weight_dtype=None, **kwargs):
        """HF checkpoint directory (config.json + *.safetensors / pytorch_model*.bin) -> model on the GPU.
        weight_dtype=torch.float8_e4m3fn: load the bf16 checkpoint, then quantize_weights() (fp8 projections)"""
        from transformers import AutoConfig
        config = AutoConfig.from_pretrained(path)
        _reject_prequantised(config)
        if weight_dtype not in (None, torch_dtype, torch.float8_e4m3fn):
            raise ValueError(f'weight_dtype {weight_dtype} is not built (bf16 or torch.float8_e4m3fn)')
        model = cls(config, device=device, dtype=torch_dtype)
        files = sorted(glob.glob(os.path.join(path, '*.safetensors')))
        own = dict(model.named_parameters())
        seen = set()
        if files:
            from safetensors.torch import load_file
            shards = (load_file(f) for f in files)
        else:
            shards = (torch.load(f, map_location='cpu') for f in sorted(glob.glob(os.path.join(path, 'pytorch_model*.bin'))))
        with torch.no_grad():
            for sd in shards:
                for k, v in model._convert_checkpoint_keys(sd).items():
                    if k in own:
                        own[k].copy_(v.to(torch_dtype))
                        seen.add(k)
        if 'lm_head.weight' not in seen and getattr(config, 'tie_word_embeddings', False):
            with torch.no_grad():
                model.lm_head.weight.copy_(model.model.embed_tokens.weight)
            seen.add('lm_head.weight')
        missing = [k for k in own if k not in seen]
        if missing:
            raise RuntimeError(f'checkpoint is missing {len(missing)} tensors, e.g. {missing[:4]}')
        if weight_dtype == torch.float8_e4m3fn:
            model.quantize_weights(weight_dtype)
        return model

    def _convert_checkpoint_keys(self, sd):
        """checkpoint tensor names -> this module tree's names (identity for Llama / Mistral)"""
        return sd

    def fuse(self):
        """QKV and gate/up weights (and q/k/v biases, where the family has them) into single GEMM operands; the
        HF-named parameters become views of them"""
        if self._fused:
            return
        for layer in self.model.layers:
            a = layer.self_attn
            w = torch.cat([a.q_proj.weight.data, a.k_proj.weight.data, a.v_proj.weight.data], dim=0).contiguous()
            nq, nk = a.q_proj.weight.shape[0], a.k_proj.weight.shape[0]
            a.q_proj.weight.data, a.k_proj.weight.data, a.v_proj.weight.data = w[:nq], w[nq:nq + nk], w[nq + nk:]
            a.qkv_weight = w
            a.qkv_bias = None
            if a.q_proj.bias is not None:
                bias = torch.cat([a.q_proj.bias.data, a.k_proj.bias.data, a.v_proj.bias.data]).contiguous()
                a.q_proj.bias.data, a.k_proj.bias.data, a.v_proj.bias.data = bias[:nq], bias[nq:nq + nk], bias[nq + nk:]
                a.qkv_bias = bias
            self._fuse_mlp(layer)
        self._fused = True

    def _fuse_mlp(self, layer):
        m = layer.mlp
        w = torch.cat([m.gate_proj.weight.data, m.up_proj.weight.data], dim=0).contiguous()
        ni = m.gate_proj.weight.shape[0]
        m.gate_proj.weight.data, m.up_proj.weight.data = w[:ni], w[ni:]
        m.gate_up_weight = w

    # ------------------------------------------------------------------ fp8 weight-only quantisation
    @property
    def quantized(self):
        return self.__dict__.get('_fp8', False)

    def _fp8_targets(self, layer):
        """(module, name, [N, K]) of the projections quantize_weights() replaces in one layer (after fuse())"""
        c = self.config
        hd = self.geometry()['head_dim']
        kv = getattr(c, 'num_key_value_heads', None) or c.num_attention_heads
        H, nq = c.hidden_size, c.num_attention_heads * hd
        a, m = layer.self_attn, layer.mlp
        return [(a, 'qkv', (nq + 2 * kv * hd, H)), (a, 'o', (H, nq)),
                (m, 'gate_up', (2 * c.intermediate_size, H)), (m, 'down', (H, c.intermediate_size))]

    @torch.no_grad()
    def quantize_weights(self, dtype=torch.float8_e4m3fn):
        """Weight-only FP8: every decoder projection (fused qkv, o, fused gate/up, down; Mixtral's stacked experts)
        becomes e4m3 tiles plus one fp32 scale per output channel (ops.quantize_fp8, include/pia_b200.h) and from then
        on runs on the fp8 GEMM plans; the embedding, the norms, the MoE router and lm_head stay bf16.  Layer by layer,
        so that peak memory is the model plus one layer's bf16 projections; the bf16 storage is freed (the HF-named
        q/k/v/o/gate/up/down parameters are removed).  Irreversible; lookahead decoding stays lossless with respect to
        the quantised model."""
        if dtype != torch.float8_e4m3fn:
            raise ValueError(f'quantize_weights: {dtype} is not built (torch.float8_e4m3fn)')
        if self.quantized:
            return self
        _reject_prequantised(self.config)
        for mod, name, (N, K) in self._fp8_targets(self.model.layers[0]):
            if N % 128 or K % 128:
                raise ValueError(f'quantize_weights: the {name} projection is [{N}, {K}]; fp8 weights need both '
                                 'dimensions to be multiples of 128')
        self.fuse()
        self._rt = None                              # its GEMM plans hold the bf16 operands
        self.__dict__.pop('_tiled_weights', None)
        for layer in self.model.layers:
            self._quantize_layer(layer)
        self._fp8 = True
        if torch.cuda.is_available() and self.device.type == 'cuda':
            torch.cuda.empty_cache()
        return self

    @staticmethod
    def _put_fp8(mod, name, w):
        wq, s = ops.quantize_fp8(w)
        mod.register_buffer(name + '_fp8', ops.tile_weight_fp8(wq))
        mod.register_buffer(name + '_scale', s.contiguous())

    def _quantize_layer(self, layer):
        a = layer.self_attn
        self._put_fp8(a, 'qkv', a.qkv_weight)
        self._put_fp8(a, 'o', a.o_proj.weight)
        bias = a.qkv_bias
        del a.q_proj, a.k_proj, a.v_proj, a.o_proj, a.qkv_bias
        a.qkv_weight = None
        a.register_buffer('qkv_bias', bias)     # None for Llama / Mistral / Mixtral
        self._quantize_mlp(layer)

    def _quantize_mlp(self, layer):
        m = layer.mlp
        self._put_fp8(m, 'gate_up', m.gate_up_weight)
        self._put_fp8(m, 'down', m.down_proj.weight)
        del m.gate_proj, m.up_proj, m.down_proj
        m.gate_up_weight = None

    # ------------------------------------------------------------------ geometry / tables
    def geometry(self):
        c = self.config
        hd = c.hidden_size // c.num_attention_heads
        return dict(n_layers=c.num_hidden_layers, hidden=c.hidden_size, n_q_heads=c.num_attention_heads,
                    n_kv_heads=getattr(c, 'num_key_value_heads', None) or c.num_attention_heads, head_dim=hd,
                    inter=c.intermediate_size, vocab=c.vocab_size)

    def rope_tables(self, max_pos):
        """cos/sin exactly as LlamaRotaryEmbedding.forward returns them (reference :100, :111-127): fp32 angles,
        then cast to the model dtype"""
        c = self.config
        hd = self.geometry()['head_dim']
        rp = getattr(c, 'rope_parameters', None) or {}
        theta = float(getattr(c, 'rope_theta', None) or rp.get('rope_theta', 10000.0))
        scaling = getattr(c, 'rope_scaling', None) or ({k: v for k, v in rp.items() if k != 'rope_theta'} if rp else None)
        rtype = (scaling or {}).get('rope_type', (scaling or {}).get('type', 'default')) if scaling else 'default'
        dev = self.device
        inv_freq = 1.0 / (theta ** (torch.arange(0, hd, 2, dtype=torch.int64).float().to(dev) / hd))
        pos = torch.arange(max_pos, device=dev).float()
        if rtype in (None, 'default'):
            pass
        elif rtype == 'linear':      # LlamaLinearScalingRotaryEmbedding (reference :130-146): t / factor
            pos = pos / float(scaling['factor'])
        elif rtype == 'dynamic':     # LlamaDynamicNTKScalingRotaryEmbedding (reference :149-169): base grows with seq_len
            factor, mpe = float(scaling['factor']), int(c.max_position_embeddings)
            if max_pos > mpe:
                base = theta * ((factor * max_pos / mpe) - (factor - 1)) ** (hd / (hd - 2))
                inv_freq = 1.0 / (base ** (torch.arange(0, hd, 2, dtype=torch.int64).float().to(dev) / hd))
        else:                        # the reference raises on unknown types as well (:241 `Unknown RoPE scaling type`)
            raise ValueError(f'Unknown RoPE scaling type {rtype}')
        freqs = pos[:, None] * inv_freq[None, :]
        return freqs.cos().to(torch.bfloat16).contiguous(), freqs.sin().to(torch.bfloat16).contiguous()

    # ------------------------------------------------------------------ weight-streaming GEMM plans (decode rows)
    def _gemm_plans(self, rt):
        """tcgen05 weight-streaming GEMMs (csrc/gemm_ws.cu) for the 64-row decode buffers: HBM-tiled copies of the
        fused weights, one plan per (weight, activation buffer).  Prefill passes (256 rows) stay on cuBLAS."""
        plans = getattr(rt, 'gemm_plans', None)
        if plans is not None:
            return plans
        if self.quantized:
            return self._fp8_gemm_plans(rt)
        import os
        if os.environ.get('PIA_GEMM', '1') == '0' or rt.max_nodes != 64:
            rt.gemm_plans = False
            return False
        b = rt.decode_bufs
        g = rt.g
        dev = b.y.device
        b.gu = torch.zeros((b.rows, 2 * g['inter']), dtype=torch.bfloat16, device=dev)
        b.act = torch.zeros((b.rows, g['inter']), dtype=torch.bfloat16, device=dev)
        plans = {'layers': []}
        for layer in self.model.layers:
            plans['layers'].append(self._layer_gemm_plans(layer, b))
        plans['lm_head'] = self._mk_gemm(self.lm_head.weight.data, b.y)
        rt.gemm_plans = plans
        return plans

    def _layer_gemm_plans(self, layer, b):
        """Which projections go through k_gemm_ws is decided by measurement (Llama-2-7B shapes; whole verify forward
        as one CUDA graph, scripts/microbench.py --forward-only, us per forward): gate_up only 3453; + down as a
        4-CTA cluster split-K (fp32 partials reduced through DSMEM) 3421; + o (cluster 4) 3527; + qkv (cluster 2)
        3482; everything 3740 - a k_gemm_ws launched behind the 200 KB-per-SM attention kernel cannot use its early
        weight streaming, and cuBLAS' 64x32 tiles win on the 32/96-tile projections.  Per launch (scripts/gemm_bench.py):
        gate_up 31.5 us vs cuBLAS 34.6, lm_head 42.3 vs 46.6.  PIA_GEMM_SET overrides the set, except that a biased qkv
        projection (Qwen2) always stays on cuBLAS: k_gemm_ws has no bias epilogue, and adding the bias after a bf16
        output would round twice where the reference's F.linear rounds once."""
        import os
        want = os.environ.get('PIA_GEMM_SET', 'gate_up,down').split(',')
        plans = {}
        if 'gate_up_silu' in want and layer.mlp.gate_up_weight.shape[0] % 256 == 0:
            # SiLU(gate) * up in the GEMM epilogue: every 128-row weight tile holds 64 gate rows + the 64 up rows of the same
            # columns (ops.interleave_gate_up), the plan writes act [rows, inter] directly
            cache = self.__dict__.setdefault('_tiled_weights', {})
            key = ('gate_up_silu', layer.mlp.gate_up_weight.data_ptr())
            if key not in cache:
                cache[key] = ops.tile_weight(ops.interleave_gate_up(layer.mlp.gate_up_weight))
            plans['gate_up_silu'] = ops.Gemm(cache[key], b.y, tiled=True).set_silu()
        elif 'gate_up' in want or 'gate_up_silu' in want:
            plans['gate_up'] = self._mk_gemm(layer.mlp.gate_up_weight, b.y)
        biased = layer.self_attn.qkv_bias is not None
        if 'qkv' in want and not biased:
            plans['qkv'] = self._mk_gemm(layer.self_attn.qkv_weight, b.y)
        sk = int(os.environ.get('PIA_GEMM_SPLIT', '-4'))   # > 1: fp32 slices summed by the next rmsnorm; < -1: cluster
        if 'qkv2' in want and not biased:
            plans['qkv'] = self._mk_gemm(layer.self_attn.qkv_weight, b.y, split_k=-2)
        if 'o' in want:
            plans['o'] = self._mk_gemm(layer.self_attn.o_proj.weight.data, b.attn, split_k=sk)
        if 'down' in want and layer.mlp.down_proj.weight.shape[1] % 64 == 0 and layer.mlp.down_proj.weight.shape[1] >= 64 * abs(sk):
            plans['down'] = self._mk_gemm(layer.mlp.down_proj.weight.data, b.act, split_k=sk)
        for name in os.environ.get('PIA_GEMM_NOPDL', '').split(','):   # experiment knob: plain kernel boundaries
            if name in plans:
                plans[name].set_pdl(False)
        return plans

    # split-K of the narrow fp8 projections (1: none, 4: fp32 slices summed by the next rmsnorm, -2 / -4: 2 / 4 K
    # splits as one cluster reducing through DSMEM).  Chosen in the whole verify forward (64 rows, one CUDA graph) at
    # the Llama-2-7B shape, one choice changed at a time (scripts/bench_fp8.py, B200 at 1000 W / 1965 MHz, us):
    #   qkv -2, o -4, down -4: 4285 | qkv 1: 4414, qkv -4: 4385 | o 1: 4831, o 4: 4305, o -2: 4459 |
    #   down 1: 5951, down 4: 4325, down -2: 4863
    FP8_SPLIT = dict(qkv=-2, o=-4, down=-4)

    def _fp8_gemm_plans(self, rt):
        """every projection of a quantised model on fp8 plans: the decode buffers (64 or 128 rows) and the 256-row
        prefill buffers; lm_head stays bf16 (k_gemm_ws plan at 64 rows, as for bf16 models)"""
        g = rt.g
        plans = {}
        for b in (rt.decode_bufs, rt.prefill_bufs):
            dev = b.y.device
            b.gu = torch.zeros((b.rows, 2 * g['inter']), dtype=torch.bfloat16, device=dev)
            b.act = torch.zeros((b.rows, g['inter']), dtype=torch.bfloat16, device=dev)
            b.fp8_plans = {'layers': [self._fp8_layer_plans(layer, b) for layer in self.model.layers]}
        plans = rt.decode_bufs.fp8_plans
        if rt.max_nodes == 64:
            plans['lm_head'] = self._mk_gemm(self.lm_head.weight.data, rt.decode_bufs.y)
        rt.gemm_plans = plans
        return plans

    @staticmethod
    def _fp8_split(split_k, w):
        """the configured split for a tiled fp8 weight, halved while its K (in 128-wide chunks) cannot give every CTA of
        a cluster split a share (small models)"""
        chunks = w.shape[-3]
        c = -split_k
        while c > 1 and -(-chunks // -(-chunks // c)) != c:
            c //= 2
        return split_k if split_k >= 1 else (-c if c > 1 else 1)

    def _fp8_layer_plans(self, layer, b):
        a, sk = layer.self_attn, self.FP8_SPLIT
        plans = {'qkv': ops.Gemm.fp8(a.qkv_fp8, a.qkv_scale, b.y, bias=a.qkv_bias,
                                     split_k=self._fp8_split(sk['qkv'], a.qkv_fp8)),
                 'o': ops.Gemm.fp8(a.o_fp8, a.o_scale, b.attn, split_k=self._fp8_split(sk['o'], a.o_fp8))}
        plans.update(self._fp8_mlp_plans(layer, b))
        return plans

    def _fp8_mlp_plans(self, layer, b):
        m = layer.mlp
        return {'gate_up': ops.Gemm.fp8(m.gate_up_fp8, m.gate_up_scale, b.y),
                'down': ops.Gemm.fp8(m.down_fp8, m.down_scale, b.act,
                                     split_k=self._fp8_split(self.FP8_SPLIT['down'], m.down_fp8))}

    def _mk_gemm(self, w, x, split_k=1):
        """HBM-tiled copy of the weight when its row count allows it (N % 128 == 0), else the row-major tensor.
        The tiled copies belong to the model (one per weight), not to a runtime: rebuilding the runtime for a longer
        max_seq or another slot count must not duplicate 9 GB of weights"""
        if w.shape[0] % 128 == 0:
            cache = self.__dict__.setdefault('_tiled_weights', {})
            key = (w.data_ptr(), tuple(w.shape))
            if key not in cache:
                cache[key] = ops.tile_weight(w)
            return ops.Gemm(cache[key], x, split_k=split_k, tiled=True)
        return ops.Gemm(w.contiguous(), x, split_k=split_k)

    # ------------------------------------------------------------------ weight prefetch beside the small kernels
    def _prefetch_cfg(self, rt):
        """PIA_PREFETCH="o_frac,gate_up_frac,down_frac,gbytes_per_s" (0 disables): which share of the next
        projections' weights is pulled into L2 on a side stream while RoPE + tree attention (o, gate_up) and
        SiLU*up (down) keep HBM idle; the step is weight-streaming bound, so HBM time hidden here comes straight
        off the step.  Decode steps only."""
        cfg = getattr(rt, 'prefetch_cfg', None)
        if cfg is None:
            import os
            spec = os.environ.get('PIA_PREFETCH', '0')
            v = [float(t) for t in spec.split(',')] if spec not in ('', '0') else []
            cfg = False
            if v and torch.cuda.is_available():
                v = (v + [0.0] * 4)[:4]
                cfg = dict(o=v[0], gate_up=v[1], down=v[2], rate=v[3], side=torch.cuda.Stream(device=self.device))
            rt.prefetch_cfg = cfg
        return cfg

    @staticmethod
    def _prefetch(pf, jobs):
        """fork: the side stream picks up after the kernels launched so far and issues the prefetch jobs"""
        main = torch.cuda.current_stream()
        pf['side'].wait_stream(main)
        with torch.cuda.stream(pf['side']):
            for (t, frac, tile_bytes) in jobs:
                if frac <= 0:
                    continue
                total = t.numel() * t.element_size()
                if tile_bytes:   # HBM-tiled weight: the first share of every tile (= its first k chunks)
                    rb = max(16384, int(tile_bytes * min(frac, 1.0)) // 16384 * 16384)
                    ops.l2_prefetch(t, n_ranges=total // tile_bytes, stride_bytes=tile_bytes, range_bytes=min(rb, tile_bytes),
                                    gbytes_per_s=pf['rate'])
                else:
                    ops.l2_prefetch(t, range_bytes=int(total * min(frac, 1.0)) // 16 * 16, gbytes_per_s=pf['rate'])
        pf['dirty'] = True

    # ------------------------------------------------------------------ the verify forward on static buffers
    def _mlp(self, rt, layer, y, plans=None, pf=None, b=None):
        """returns (x, parts): the MLP output as a bf16 tensor or as fp32 split-K slices for the next rmsnorm"""
        m = layer.mlp
        if plans:
            b = b if b is not None else rt.decode_bufs
            if 'gate_up_silu' in plans:
                plans['gate_up_silu'].run(b.rows, out=b.act)
            else:
                if 'gate_up' in plans:
                    plans['gate_up'].run(b.rows, out=b.gu)
                else:
                    torch.mm(y, m.gate_up_weight.t(), out=b.gu)
                if pf:
                    self._prefetch(pf, [(m.down_proj.weight, pf['down'], 0)])
                ops.silu_mul(b.gu, b.act)
            if 'down' in plans:
                o = plans['down'].run(b.rows)
                return (o, None) if plans['down'].splits == 1 else (None, o)
            return torch.mm(b.act, m.down_proj.weight.t()), None
        gu = torch.mm(y, m.gate_up_weight.t())
        act = torch.empty((gu.shape[0], gu.shape[1] // 2), dtype=gu.dtype, device=gu.device)
        ops.silu_mul(gu, act)
        return torch.mm(act, m.down_proj.weight.t()), None

    def _verify_layers(self, rt, bufs=None, last_only=False):
        """embed -> decoder layers -> final norm -> lm_head over the rows described by `bufs` (default: the decode
        buffers = the drafts of the request slots in rt.ids / rt.mask / rt.n on top of rt.prefix_len cached tokens;
        bufs.slots says which slot owns which rows).  A prefill pass uses wider buffers holding several 64-row chain
        chunks (one table slot each): the GEMMs run once over all rows.  Writes bufs.logits (skipped when
        last_only)."""
        self.fuse()
        b = bufs if bufs is not None else rt.decode_bufs
        g = rt.g
        eps = self.config.rms_norm_eps
        ops.embed_gather(self.model.embed_tokens.weight, b.ids, b.n_total, b.h)
        if self.quantized:   # every projection on fp8 plans, prefill passes included
            plans = self._gemm_plans(rt) if b is rt.decode_bufs else b.fp8_plans
            pf = False
        else:
            plans = self._gemm_plans(rt) if b is rt.decode_bufs else False
            pf = self._prefetch_cfg(rt) if plans else False
        fused_attn = b is rt.decode_bufs and os.environ.get('PIA_ATTN_FUSED', '0') != '0' and \
            (b.slots.batch == 1 or b.slots.kv_slot_stride != 0)
        x, parts, resid_in = b.h, None, None  # norm(x | parts, resid_in) -> (resid = x + resid_in, y = norm(resid))

        def norm(w):
            if parts is not None:
                ops.rmsnorm_partials(parts, resid_in, w, eps, b.resid, b.y)
            else:
                ops.rmsnorm(x, resid_in, w, eps, b.resid, b.y)

        for li, layer in enumerate(self.model.layers):
            lp = plans['layers'][li] if plans else None
            norm(layer.input_layernorm.weight)
            a = layer.self_attn
            if lp and 'qkv' in lp:
                lp['qkv'].run(b.rows, out=b.qkv)
            elif a.qkv_bias is not None:   # Qwen2: cuBLASLt bias epilogue, one rounding of the fp32 xW^T + b
                torch.addmm(a.qkv_bias, b.y, a.qkv_weight.t(), out=b.qkv)
            else:
                torch.mm(b.y, a.qkv_weight.t(), out=b.qkv)
            if pf and lp and 'gate_up' in lp:
                gw = lp['gate_up'].weight
                self._prefetch(pf, [(a.o_proj.weight, pf['o'], 0),
                                    (gw, pf['gate_up'], gw.shape[1] * gw.shape[2] * gw.shape[3] * 2 if gw.dim() == 4 else 0)])
            # every request slot / prefill chunk of the table in one launch each (pia_slots_t)
            if fused_attn:   # decode steps: RoPE + KV append happen inside the attention kernel
                rt.plan.forward_fused(li, b.qkv, b.mask, b.slots, rt.rope_cos, rt.rope_sin, b.attn)
            else:            # prefill chunks share one cache: append first, then attend
                ops.rope_kv_append(b.qkv, b.mask, b.slots, g['n_q_heads'], g['n_kv_heads'], g['head_dim'], rt.rope_cos,
                                   rt.rope_sin, b.q, rt.k_layer(li, b.kv_slot), rt.v_layer(li, b.kv_slot), rt.max_seq)
                rt.plan.forward(li, b.q, b.mask, b.slots, b.attn)
            if lp and 'o' in lp:
                o = lp['o'].run(b.rows)
                x, parts, resid_in = (o, None, b.resid) if lp['o'].splits == 1 else (None, o, b.resid)
            else:
                x, parts, resid_in = torch.mm(b.attn, a.o_proj.weight.t()), None, b.resid
            norm(layer.post_attention_layernorm.weight)
            x, parts = self._mlp(rt, layer, b.y, lp, pf, b)
        if pf and pf.pop('dirty', False):  # join the side stream (required before a capture ends)
            torch.cuda.current_stream().wait_stream(pf['side'])
        if last_only:
            return
        norm(self.model.norm.weight)
        if b.logits is not None:
            if plans and 'lm_head' in plans:
                plans['lm_head'].run(b.rows, out=b.logits)
            else:
                torch.mm(b.y, self.lm_head.weight.t(), out=b.logits)


def _reject_prequantised(config):
    q = getattr(config, 'quantization_config', None)
    if q:
        method = q.get('quant_method', '?') if isinstance(q, dict) else getattr(q, 'quant_method', '?')
        raise ValueError(f'pre-quantised checkpoints ({method}) are not built: load the bf16 checkpoint with '
                         'weight_dtype=torch.float8_e4m3fn to serve fp8 weights')


class LlamaPreTrainedModel(LookaheadPreTrainedModel):
    pass
