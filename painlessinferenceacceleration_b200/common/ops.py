# -*- coding: utf-8 -*-
"""Thin typed wrappers over the C ABI (include/pia_b200.h) for torch tensors: raw device pointers + the current
torch stream, nothing else. Every call is asynchronous and CUDA-graph capturable."""
import ctypes as C

import torch

from .. import _lib as L


def _s():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return t.data_ptr() if t is not None else None


def rmsnorm(x, residual_in, weight, eps, residual_out, y):
    rows, hidden = x.shape
    L.check(L.load().pia_rmsnorm(_p(x), _p(residual_in), _p(weight), float(eps), rows, hidden, _p(residual_out),
                                 _p(y), _s()))


def rmsnorm_partials(parts, residual_in, weight, eps, residual_out, y):
    """parts: fp32 [n_parts, 64, hidden] split-K slices of a Gemm"""
    n_parts, prow, hidden = parts.shape
    rows = y.shape[0]
    L.check(L.load().pia_rmsnorm_partials(_p(parts), n_parts, prow * hidden, _p(residual_in), _p(weight), float(eps),
                                          rows, hidden, _p(residual_out), _p(y), _s()))


def tile_weight(w):
    """[N, K] -> [N/128, K/64, 128, 64] contiguous: one 16 KB block per (128-row tile, 64-wide k chunk), the unit the
    GEMM kernel's TMA box moves, so each CTA reads one contiguous slab of HBM"""
    N, K = w.shape
    assert N % 128 == 0 and K % 64 == 0
    t = w.view(N // 128, 128, K // 64, 64).permute(0, 2, 1, 3).contiguous()
    t.pia_shape = (N, K)
    return t


FP8_MAX = 448.0


def quantize_fp8(w):
    """weight-only e4m3 quantisation with one fp32 scale per output channel (include/pia_b200.h, DESIGN §3):
    s[n] = max_k |W[n, k]| / 448 (1 for an all-zero row), Wq = e4m3(W / s) rounded to nearest even and saturated at
    +-448.  w: [..., N, K] on any device -> (Wq float8_e4m3fn [..., N, K], s float32 [..., N])"""
    wf = w.float()
    s = wf.abs().amax(dim=-1) / FP8_MAX
    s = torch.where(s == 0, torch.ones_like(s), s)
    wq = (wf / s.unsqueeze(-1)).clamp_(-FP8_MAX, FP8_MAX).to(torch.float8_e4m3fn)
    return wq, s


def tile_weight_fp8(wq):
    """e4m3 [N, K] (or [G, N, K]) -> [(G,) N/128, K/128, 128, 128]: one contiguous 16 KB block per (128-row tile,
    128-wide k chunk), the TMA box of the fp8 GEMM plans"""
    *lead, N, K = wq.shape
    if N % 128 or K % 128:
        raise ValueError(f'fp8 weights need N % 128 == 0 and K % 128 == 0, got [{N}, {K}]')
    t = wq.reshape(*lead, N // 128, 128, K // 128, 128).transpose(-3, -2).contiguous()
    t.pia_shape = (N, K)
    return t


def untile_weight_fp8(t):
    """inverse of tile_weight_fp8"""
    *lead, nt, kt, _, _ = t.shape
    return t.transpose(-3, -2).reshape(*lead, nt * 128, kt * 128)


def interleave_gate_up(w_gate_up):
    """[gate (I rows); up (I rows)] -> per 128-row tile: 64 gate rows then the 64 up rows of the same columns, the
    layout the fused SiLU*up epilogue of the GEMM expects"""
    two_i, K = w_gate_up.shape
    inter = two_i // 2
    assert inter % 64 == 0
    g = w_gate_up[:inter].view(inter // 64, 64, K)
    u = w_gate_up[inter:].view(inter // 64, 64, K)
    return torch.cat([g, u], dim=1).reshape(two_i, K).contiguous()


def _tok(rows):
    return 64 if rows <= 64 else 128 if rows <= 128 else 256


class Gemm(object):
    """pia_gemm_plan_t: Y = X @ W^T for one (weight, activation buffer) pair; `out` is bf16 [rows, N] when the plan
    has one K split, else fp32 [splits, 64, N]"""

    def __init__(self, weight, x, split_k=1, tiled=False):
        """weight: [N, K] row-major, or (tiled=True) the output of tile_weight() with its logical shape in .pia_shape"""
        N, K = weight.pia_shape if tiled else weight.shape
        assert x.shape[1] == K and x.is_contiguous() and weight.is_contiguous()
        self.lib = L.load()
        self.h = L.vp()
        with torch.cuda.device(weight.device):
            L.check(self.lib.pia_gemm_plan_create(_p(weight), N, K, _p(x), x.shape[0], split_k, int(tiled),
                                                  C.byref(self.h)))
        self.splits = self.lib.pia_gemm_plan_splits(self.h)
        self.N = N
        self._keep = (weight, x)
        self.weight = weight
        if self.splits == 1:
            self.out = torch.empty((x.shape[0], N), dtype=torch.bfloat16, device=weight.device)
        else:
            self.out = torch.empty((self.splits, 64, N), dtype=torch.float32, device=weight.device)

    @classmethod
    def grouped(cls, weight, x):
        """one launch for all experts: weight [G, N, K] (stacked, contiguous), x [rows >= 64, G * K];
        out [G, 64, N] bf16 (pia_gemm_plan_create_grouped)"""
        G, N, K = weight.shape
        assert weight.is_contiguous() and x.is_contiguous() and x.shape[1] == G * K
        self = cls.__new__(cls)
        self.lib = L.load()
        self.h = L.vp()
        with torch.cuda.device(weight.device):
            L.check(self.lib.pia_gemm_plan_create_grouped(_p(weight), G, N, K, _p(x), x.shape[0], C.byref(self.h)))
        self.splits, self.N, self.weight, self._keep = 1, N, weight, (weight, x)
        self.out = torch.empty((G, 64, N), dtype=torch.bfloat16, device=weight.device)
        return self

    @classmethod
    def fp8(cls, weight, scale, x, bias=None, split_k=1):
        """fp8 weight-only plan (pia_gemm_plan_create_fp8): weight = tile_weight_fp8(Wq) [N/128, K/128, 128, 128],
        scale fp32 [N], bias bf16 [N] or None, x bf16 [rows <= 256, K].  out: bf16 [x.shape[0], N], or fp32
        [splits, tok, N] slices with tok = 64 / 128 / 256 (the smallest that covers x's rows)"""
        N, K = weight.shape[-4] * 128, weight.shape[-3] * 128
        assert weight.dim() == 4 and weight.dtype == torch.float8_e4m3fn and weight.is_contiguous()
        assert scale.dtype == torch.float32 and scale.shape == (N,) and scale.is_contiguous()
        assert bias is None or (bias.dtype == torch.bfloat16 and bias.shape == (N,) and bias.is_contiguous())
        assert x.dtype == torch.bfloat16 and x.shape[1] == K and x.is_contiguous()
        self = cls.__new__(cls)
        self.lib = L.load()
        self.h = L.vp()
        with torch.cuda.device(weight.device):
            L.check(self.lib.pia_gemm_plan_create_fp8(_p(weight), _p(scale), _p(bias), N, K, _p(x), x.shape[0],
                                                      int(split_k), C.byref(self.h)))
        self.splits = self.lib.pia_gemm_plan_splits(self.h)
        self.N, self.weight, self._keep = N, weight, (weight, scale, bias, x)
        self.tok = _tok(x.shape[0])
        if self.splits == 1:
            self.out = torch.empty((x.shape[0], N), dtype=torch.bfloat16, device=weight.device)
        else:
            self.out = torch.empty((self.splits, self.tok, N), dtype=torch.float32, device=weight.device)
        return self

    @classmethod
    def grouped_fp8(cls, weight, scale, x):
        """all experts in one launch (pia_gemm_plan_create_grouped_fp8): weight = tile_weight_fp8 of the stacked
        [G, N, K] e4m3 weights ([G, N/128, K/128, 128, 128]), scale fp32 [G, N], x bf16 [rows <= 256, G * K];
        out bf16 [G, tok, N]"""
        G, N, K = weight.shape[0], weight.shape[1] * 128, weight.shape[2] * 128
        assert weight.dim() == 5 and weight.dtype == torch.float8_e4m3fn and weight.is_contiguous()
        assert scale.dtype == torch.float32 and scale.shape == (G, N) and scale.is_contiguous()
        assert x.dtype == torch.bfloat16 and x.shape[1] == G * K and x.is_contiguous()
        self = cls.__new__(cls)
        self.lib = L.load()
        self.h = L.vp()
        with torch.cuda.device(weight.device):
            L.check(self.lib.pia_gemm_plan_create_grouped_fp8(_p(weight), _p(scale), G, N, K, _p(x), x.shape[0],
                                                              C.byref(self.h)))
        self.splits, self.N, self.weight, self._keep = 1, N, weight, (weight, scale, x)
        self.tok = _tok(x.shape[0])
        self.out = torch.empty((G, self.tok, N), dtype=torch.bfloat16, device=weight.device)
        return self

    def set_pdl(self, on=True):
        L.check(self.lib.pia_gemm_plan_set_pdl(self.h, int(on)))
        return self

    def set_silu(self, on=True):
        L.check(self.lib.pia_gemm_plan_set_silu(self.h, int(on)))
        return self

    def run(self, rows=64, out=None):
        o = out if out is not None else self.out
        L.check(self.lib.pia_gemm_run(self.h, rows, _p(o), _s()))
        return o

    def __del__(self):
        try:
            if self.h:
                self.lib.pia_gemm_plan_destroy(self.h)
                self.h = None
        except Exception:
            pass


class Slots(object):
    """pia_slots_t: the request slots of one verify step.  `n`, `prefix_len`, `pad_len` are int32 DEVICE tensors of
    `batch` entries read when the kernels run (so one CUDA graph serves every length / padding); slot s owns rows
    [s * rows_per_slot, (s + 1) * rows_per_slot) of the activation and draft buffers and the KV cache that starts
    kv_slot_stride elements after slot s-1's (0: all slots share one cache, e.g. the chain chunks of a prefill pass)."""

    def __init__(self, n, prefix_len, pad_len=None, rows_per_slot=64, kv_slot_stride=0, batch=None, kv_first_slot=0):
        batch = int(batch if batch is not None else n.numel())
        assert n.dtype == torch.int32 and prefix_len.dtype == torch.int32 and n.numel() >= batch <= prefix_len.numel()
        assert pad_len is None or (pad_len.dtype == torch.int32 and pad_len.numel() >= batch)
        self.batch, self.rows_per_slot, self.kv_slot_stride = batch, int(rows_per_slot), int(kv_slot_stride)
        self.n, self.prefix_len, self.pad_len = n, prefix_len, pad_len
        self.kv_first_slot = int(kv_first_slot)
        self.c = L.Slots(batch, int(rows_per_slot), _p(n), _p(prefix_len), _p(pad_len), int(kv_slot_stride),
                         int(kv_first_slot))

    @property
    def rows(self):
        return self.batch * self.rows_per_slot

    def ref(self):
        return C.byref(self.c)


def rope_kv_append(qkv, mask, slots, n_q_heads, n_kv_heads, head_dim, cos, sin, q_out, k_layer, v_layer, max_seq):
    """qkv / q_out: >= slots.rows rows; mask: [>= slots.rows, W] int64 ancestor rows; k_layer / v_layer: the layer's
    [n_kv_heads, max_seq, head_dim] planes of slot 0"""
    assert qkv.shape[0] >= slots.rows and mask.shape[0] >= slots.rows
    L.check(L.load().pia_rope_kv_append(_p(qkv), _p(mask), mask.shape[-1], slots.ref(), n_q_heads, n_kv_heads,
                                        head_dim, _p(cos), _p(sin), cos.shape[0], _p(q_out), _p(k_layer), _p(v_layer),
                                        max_seq, _s()))


def silu_mul(gate_up, out):
    rows, two_inter = gate_up.shape
    L.check(L.load().pia_silu_mul(_p(gate_up), rows, two_inter // 2, _p(out), _s()))


def moe_combine(expert_out, weights, out):
    """out[t] = sum_e expert_out[e, t] * weights[t, e] in expert order, bf16 rounding per step (pia_moe_combine)"""
    E, rows_cap, hidden = expert_out.shape
    rows = weights.shape[0]
    assert weights.shape[1] == E and weights.is_contiguous() and expert_out.is_contiguous() and out.shape[0] >= rows
    L.check(L.load().pia_moe_combine(_p(expert_out), _p(weights), E, rows, rows_cap, hidden, _p(out), _s()))


def moe_router(y, gate_weight, top_k, dense_out):
    """dense routing weights [rows, E] (0 for unselected experts) of the rows of y (pia_moe_router)"""
    rows, hidden = y.shape
    E = gate_weight.shape[0]
    assert gate_weight.shape[1] == hidden and dense_out.shape[0] >= rows and dense_out.shape[1] == E
    assert y.is_contiguous() and gate_weight.is_contiguous() and dense_out.is_contiguous()
    L.check(L.load().pia_moe_router(_p(y), _p(gate_weight), rows, hidden, E, int(top_k), _p(dense_out), _s()))


def l2_prefetch(t, n_ranges=1, stride_bytes=0, range_bytes=None, gbytes_per_s=0.0, offset_bytes=0):
    """hint: pull (part of) an immutable weight tensor into L2 on the current stream (pia_l2_prefetch)"""
    if range_bytes is None:
        range_bytes = t.numel() * t.element_size() - offset_bytes
    L.check(L.load().pia_l2_prefetch(t.data_ptr() + offset_bytes, int(n_ranges), int(stride_bytes), int(range_bytes),
                                     float(gbytes_per_s), _s()))


def embed_gather(table, ids, n, out):
    rows, hidden = out.shape
    L.check(L.load().pia_embed_gather(_p(table), _p(ids), _p(n), rows, hidden, _p(out), _s()))


class AttnPlan(object):
    """pia_attn_plan_t: TMA descriptors over one model's KV cache(s) (KV splits merge on chip: no workspace).
    k_cache / v_cache: [n_layers, n_kv_heads, max_seq, head_dim], or [n_slots, ...] for the batched loop"""

    def __init__(self, k_cache, v_cache, n_q_heads, n_kv_heads, head_dim, max_nodes, kv_split_max=0):
        n_slots = k_cache.shape[0] if k_cache.dim() == 5 else 1
        n_layers, hkv, max_seq, hd = k_cache.shape[-4:]
        assert hkv == n_kv_heads and hd == head_dim and k_cache.is_contiguous() and v_cache.is_contiguous()
        self.cfg = L.AttnConfig(n_q_heads, n_kv_heads, head_dim, max_seq, max_nodes, n_layers, kv_split_max, n_slots)
        self.slot_stride = n_layers * hkv * max_seq * hd
        self.h = L.vp()
        self.lib = L.load()
        with torch.cuda.device(k_cache.device):
            L.check(self.lib.pia_attn_plan_create(C.byref(self.cfg), _p(k_cache), _p(v_cache), C.byref(self.h)))
        self._keep = (k_cache, v_cache)

    def forward(self, layer, q, mask, slots, out, scale_mul=1.0):
        assert q.shape[0] >= slots.rows and mask.shape[0] >= slots.rows and out.shape[0] >= slots.rows
        L.check(self.lib.pia_tree_attn_fwd(self.h, layer, _p(q), _p(mask), slots.ref(), float(scale_mul), _p(out), _s()))

    def forward_fused(self, layer, qkv, mask, slots, cos, sin, out, scale_mul=1.0):
        """RoPE + KV append + tree attention in one launch (pia_tree_attn_fused_fwd): qkv is the fused projection
        output; needs one cache per slot"""
        assert qkv.shape[0] >= slots.rows and mask.shape[0] >= slots.rows and out.shape[0] >= slots.rows
        L.check(self.lib.pia_tree_attn_fused_fwd(self.h, layer, _p(qkv), _p(cos), _p(sin), cos.shape[0], _p(mask),
                                                 slots.ref(), float(scale_mul), _p(out), _s()))

    def close(self):
        if self.h:
            self.lib.pia_attn_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Accept(object):
    """pia_accept + its config/workspace.  max_length is a device scalar (d_max_length) when given, so that one
    captured step serves every request length."""

    def __init__(self, vocab, max_nodes, repetition_penalty, eos_ids, max_length, device, bound_walk=False):
        eos = [int(e) for e in (eos_ids or []) if e is not None][:8]
        arr = (C.c_int32 * 8)(*(eos + [-1] * (8 - len(eos))))
        self.cfg = L.AcceptConfig(vocab, max_nodes, float(repetition_penalty), len(eos), arr, int(max_length),
                                  int(bool(bound_walk)))
        self.max_nodes = max_nodes
        self.lib = L.load()
        self.workspace = torch.empty((max(self.lib.pia_accept_workspace_bytes(C.byref(self.cfg)) // 4, 1),),
                                     dtype=torch.int32, device=device)

    def run(self, logits, ids, mask, n, seq, seq_len, acc_tokens, acc_count, acc_nodes, prefix_len, finished,
            batch=1, rows_per_slot=None, max_length=None, rng=None):
        """ids [batch * rows_per_slot], mask [batch * rows_per_slot, W], n / seq_len / prefix_len / finished /
        acc_count [batch], seq [batch, stride] (or 1-D for one slot), acc_tokens / acc_nodes [batch, max_nodes];
        max_length: optional int32 device scalar overriding the config's; rng: None (greedy) or an int32 device
        tensor {seed, counter} -> multinomial accept (do_sample)"""
        rps = int(rows_per_slot if rows_per_slot is not None else self.max_nodes // batch)
        stride = seq.shape[-1] if seq.dim() == 2 else seq.numel()
        L.check(self.lib.pia_accept(C.byref(self.cfg), _p(logits), _p(ids), _p(mask), mask.shape[-1], int(batch), rps,
                                    _p(n), _p(seq), _p(seq_len), int(stride), _p(max_length), _p(rng), _p(acc_tokens),
                                    _p(acc_count), _p(acc_nodes), _p(prefix_len), _p(finished), _p(self.workspace), _s()))


def kv_compact(k_cache, v_cache, acc_nodes, acc_count, prefix_len, batch=1):
    """k_cache / v_cache [n_layers, Hkv, S, D] (batch 1) or [batch_cap, n_layers, Hkv, S, D]"""
    n_layers, hkv, max_seq, hd = k_cache.shape[-4:]
    stride = n_layers * hkv * max_seq * hd if k_cache.dim() == 5 else 0
    nodes_stride = acc_nodes.shape[-1] if acc_nodes.dim() == 2 else acc_nodes.numel()
    L.check(L.load().pia_kv_compact(_p(k_cache), _p(v_cache), n_layers, hkv, max_seq, hd, int(batch), int(stride),
                                    _p(acc_nodes), int(nodes_stride), _p(acc_count), _p(prefix_len), _s()))


def launch_count():
    return int(L.load().pia_launch_count())
