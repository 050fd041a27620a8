# -*- coding: utf-8 -*-
"""FP8 weight-only projections on the B200 (csrc/gemm_ws.cu fp8 instantiations, LlamaForCausalLM.quantize_weights).

Kernel: against an fp32 evaluation of the dequantised product, and bit for bit against the bf16 k_gemm_ws plan.
Models: memory after quantisation, loop parity of the oracle loop and the fused device loop on the same fp8 model
(identical logits by construction, so tokens / dls / edls must match exactly), lossless lookahead against the fp8
model's own greedy output, and the verify logits against fp32 HF with the dequantised weights."""
import gc
import weakref

import pytest
import torch

from painlessinferenceacceleration_b200.common import ops
from tests.test_gpu_generate import OursBackend
from tests.tiny_models import prompts, tiny_hf_model
from tests.tiny_qwen2 import qwen2_hf_model

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _operands(N, K, rows, groups=1, seed=0, pow2=False):
    g = torch.Generator(device=DEV).manual_seed(seed)
    w = torch.randn((groups, N, K), generator=g, device=DEV) * 0.05
    w[:, 5] *= 1e-3            # rows whose values mostly land in e4m3's subnormal range
    w[:, 9] = 0                # all-zero row
    if pow2:                   # per-row power-of-two scales: bf16(Wq) * s is exact
        wq = (w * 448 / w.abs().amax(-1, keepdim=True).clamp_min(1e-30)).clamp(-448, 448).to(torch.float8_e4m3fn)
        s = torch.exp2(torch.randint(-12, -2, (groups, N), generator=g, device=DEV).float())
    else:
        wq, s = ops.quantize_fp8(w.to(torch.bfloat16))
    x = (torch.randn((rows, groups * K), generator=g, device=DEV)).to(torch.bfloat16)
    return wq, s.contiguous(), x


def _want(x, wq, s, bias=None):
    y = s[:, None].double() * (wq.double() @ x.double().t())          # [N, rows]
    if bias is not None:
        y = y + bias.double()[:, None]
    return y.t()


@pytest.mark.parametrize('rows,x_rows', [(64, 64), (37, 64), (128, 128), (100, 128), (256, 256), (200, 256)])
@pytest.mark.parametrize('split', [1, 4, -2, -4])
@pytest.mark.parametrize('with_bias', [False, True])
def test_fp8_gemm_against_fp32(rows, x_rows, split, with_bias):
    N, K = 384, 1024
    wq, s, x = _operands(N, K, x_rows, seed=rows + split)
    wq, s = wq[0], s[0]
    bias = (torch.randn(N, device=DEV) * 0.3).to(torch.bfloat16) if with_bias else None
    plan = ops.Gemm.fp8(ops.tile_weight_fp8(wq), s, x, bias=bias, split_k=split)
    assert plan.tok == (64 if x_rows <= 64 else 128 if x_rows <= 128 else 256)
    out = plan.run(rows)
    torch.cuda.synchronize()
    if plan.splits > 1:
        assert out.shape == (plan.splits, plan.tok, N)
        y = out[:, :rows].double().sum(0)                     # what rmsnorm_partials rounds once
    else:
        y = out[:rows].double()
    exact = _want(x[:rows], wq.float(), s, bias)
    # allowance: one bf16 ulp of the exact value (the single rounding) plus 2^-22 * (s * sum_k |x w| + |b|) for the
    # fp32 accumulation in the MMA's own order, the scale multiply and the bias add (fp32 unit roundoff 2^-24 times 4)
    mag = (s[:, None].double() * (wq.double().abs() @ x[:rows].double().abs().t())).t()
    if bias is not None:
        mag = mag + bias.double().abs()[None]
    err = (y - exact).abs()
    tol = mag * 2.0 ** -22 + (0 if plan.splits > 1 else 1) * torch.exp2(
        torch.floor(torch.log2(exact.abs().clamp_min(1e-30))) - 7)
    assert (err <= tol + 1e-30).all(), (err - tol).max().item()
    if plan.splits == 1:   # rows past `rows` are untouched
        assert out.shape[0] == x_rows


@pytest.mark.parametrize('E', [4, 8])
@pytest.mark.parametrize('x_rows', [64, 128, 256])
def test_fp8_grouped_gemm_against_fp32(E, x_rows):
    N, K = 256, 512
    wq, s, x = _operands(N, K, x_rows, groups=E, seed=E)
    plan = ops.Gemm.grouped_fp8(ops.tile_weight_fp8(wq), s, x)
    out = plan.run(x_rows)
    torch.cuda.synchronize()
    assert out.shape == (E, plan.tok, N)
    for e in range(E):
        exact = _want(x[:, e * K:(e + 1) * K], wq[e].float(), s[e])
        mag = (s[e][:, None].double() * (wq[e].double().abs() @ x[:, e * K:(e + 1) * K].double().abs().t())).t()
        ulp = torch.exp2(torch.floor(torch.log2(exact.abs().clamp_min(1e-30))) - 7)
        assert ((out[e, :x_rows].double() - exact).abs() <= mag * 2.0 ** -22 + ulp).all(), e


@pytest.mark.parametrize('split', [1, 4, -2, -4])
def test_fp8_plan_is_bit_identical_to_the_bf16_plan(split):
    """with power-of-two scales bf16(Wq) * s is exact in bf16 and s * sum(x * wq) == sum(x * (wq * s)) exactly, so the fp8
    plan at 64 token rows must reproduce the existing bf16 k_gemm_ws plan bit for bit: the same UMMA 128x64x16 sequence
    over the same K range per split (K = 1024: 8 fp8 chunks of 128 = 16 bf16 chunks of 64, so every split count used
    here cuts both at the same k).  The 128- and 256-row instantiations must then match the 64-row plan on every 64-row
    slice: the UMMA accumulates each output column independently of N, in the same k order."""
    N, K = 512, 1024
    wq, s, x = _operands(N, K, 256, seed=11, pow2=True)
    wq, s = wq[0], s[0]
    wb = (wq.float() * s[:, None]).to(torch.bfloat16)
    assert torch.equal(wb.float(), wq.float() * s[:, None])
    x64 = x[:64].contiguous()
    ref = ops.Gemm(wb.contiguous(), x64, split_k=split).run(64)
    got = ops.Gemm.fp8(ops.tile_weight_fp8(wq), s, x64, split_k=split).run(64)
    torch.cuda.synchronize()
    assert ref.dtype == got.dtype and ref.shape == got.shape
    assert torch.equal(ref.view(torch.int16) if ref.dtype == torch.bfloat16 else ref.view(torch.int32),
                       got.view(torch.int16) if got.dtype == torch.bfloat16 else got.view(torch.int32))
    for rows in (128, 256):
        xb = x[:rows].contiguous()
        big = ops.Gemm.fp8(ops.tile_weight_fp8(wq), s, xb, split_k=split).run(rows)
        for c in range(rows // 64):
            xs = x[64 * c:64 * (c + 1)].contiguous()
            small = ops.Gemm.fp8(ops.tile_weight_fp8(wq), s, xs, split_k=split).run(64)
            torch.cuda.synchronize()
            if big.dtype == torch.bfloat16:
                assert torch.equal(big[64 * c:64 * (c + 1)].view(torch.int16), small.view(torch.int16)), (rows, c)
            else:
                assert torch.equal(big[:, 64 * c:64 * (c + 1)].contiguous().view(torch.int32),
                                   small.view(torch.int32)), (rows, c)


def test_fp8_plan_rejects_bad_shapes():
    wq, s, x = _operands(256, 256, 64)
    with pytest.raises(AssertionError):
        ops.Gemm.fp8(ops.tile_weight_fp8(wq[0]), s[0], x[:, :128].contiguous())
    big = torch.zeros((300, 256), dtype=torch.bfloat16, device=DEV)
    with pytest.raises(AssertionError, match='1..256'):
        ops.Gemm.fp8(ops.tile_weight_fp8(wq[0]), s[0], big)
    plan = ops.Gemm.fp8(ops.tile_weight_fp8(wq[0]), s[0], x)
    with pytest.raises(AssertionError):
        plan.run(65)


# ---------------------------------------------------------------------------------------------------------------
# models
# ---------------------------------------------------------------------------------------------------------------
FAMILIES = ['llama', 'mistral', 'mixtral', 'qwen2_g7', 'qwen2_g6_tied']


def _hf(family, seed, dtype=torch.bfloat16):
    if family.startswith('qwen2'):
        return qwen2_hf_model(family[6:], seed=seed, dtype=dtype, device=DEV, vocab=200)
    return tiny_hf_model(family, seed=seed, dtype=dtype, device=DEV, vocab=200)


def _cls(family):
    from painlessinferenceacceleration_b200.models.llama.modeling_llama import LlamaForCausalLM
    from painlessinferenceacceleration_b200.models.mixtral.modeling_mixtral import MixtralForCausalLM
    from painlessinferenceacceleration_b200.models.qwen2.modeling_qwen2 import Qwen2ForCausalLM
    return {'mixtral': MixtralForCausalLM, 'qwen2_g7': Qwen2ForCausalLM, 'qwen2_g6_tied': Qwen2ForCausalLM}.get(
        family, LlamaForCausalLM)


def _ours(family, hf, cls=None):
    m = (cls or _cls(family))(hf.config, device=torch.device(DEV))
    missing = m.load_state_dict(hf.state_dict(), strict=False)
    assert not missing.missing_keys, missing
    if hf.config.tie_word_embeddings:
        with torch.no_grad():
            m.lm_head.weight.copy_(m.model.embed_tokens.weight)
    return m.quantize_weights()


def _forward_rt(m, ids, m01, P):
    """LookaheadPreTrainedModel.forward on the runtime as it is (forward() itself would rebuild a 128-node runtime
    for a draft of <= 64 nodes)"""
    import numpy as np
    rt = m._rt
    n = ids.shape[1]
    tree = m01[0, 0, :, P:].to('cpu').long().numpy()
    packed = np.packbits(np.pad(tree.astype(np.uint8), ((0, rt.max_nodes - n), (0, rt.max_nodes - n))), axis=1,
                         bitorder='little')
    rt.mask.copy_(torch.from_numpy(packed.view(np.int64).reshape(rt.max_nodes, rt.max_nodes // 64)).to(rt.device))
    rt.ids[:n] = ids[0].to(device=rt.device, dtype=torch.int32)
    rt.n.fill_(n)
    rt.prefix_len.fill_(P)
    rt.set_request(0, 0, 1 << 30)
    m._verify_layers(rt)
    return rt.logits[:n].clone()[None], P + n


class Backend(OursBackend):
    """OursBackend with the runtime's draft width fixed to the loop's (64 or 128 nodes)"""

    def __init__(self, ours, max_nodes, max_seq):
        super().__init__(ours, prefill_like_generate=True, max_seq=max_seq)
        self.max_nodes = max_nodes

    def forward(self, ids_in, m01, pos):
        n = ids_in.shape[1]
        if self.P == 0:
            rt = self.m._runtime(self.max_seq, self.max_nodes)
            rt.set_request(0, 0, 1 << 30)
            rt.seq[0, :n] = ids_in[0].to(device=rt.device, dtype=torch.int32)
            self.m._prefill_logits(rt, n)
            self.P = n
            return rt.logits[0:1].clone()[None]
        lg, self.P = _forward_rt(self.m, ids_in, m01, self.P)
        return lg


def _proj_shapes(m):
    c = m.config
    hd = m.geometry()['head_dim']
    kv = getattr(c, 'num_key_value_heads', None) or c.num_attention_heads
    H, nq, I = c.hidden_size, c.num_attention_heads * hd, c.intermediate_size
    shapes = {(nq + 2 * kv * hd, H), (nq, H), (kv * hd, H), (H, nq), (2 * I, H), (I, H), (H, I)}
    for (N, K) in list(shapes):   # bf16 HBM-tiled copies (ops.tile_weight)
        if N % 128 == 0 and K % 64 == 0:
            shapes.add((N // 128, K // 64, 128, 64))
    return shapes


def _reachable_tensors(m):
    """every tensor reachable from the model's modules (parameters, buffers, attributes) and its tiled-weight cache"""
    out = []
    for mod in m.modules():
        for v in list(mod._parameters.values()) + list(mod._buffers.values()) + list(vars(mod).values()):
            if isinstance(v, torch.Tensor):
                out.append(v)
    out += list(m.__dict__.get('_tiled_weights', {}).values())
    return out


@pytest.mark.parametrize('family', ['llama', 'qwen2_g7', 'mixtral'])
def test_quantize_weights_frees_the_bf16_projections(family):
    hf = _hf(family, seed=3)
    m = _cls(family)(hf.config, device=torch.device(DEV))
    m.load_state_dict(hf.state_dict(), strict=False)
    p = prompts(5, 1, 20, 200)[0].to(DEV)
    m.generate(input_ids=p, max_new_tokens=8, eos_token_id=2,
               decoding_kwargs={'use_lookahead': True, 'decoding_length': 64, 'branch_length': 8})
    m.fuse()
    watch = []
    for layer in m.model.layers:
        a = layer.self_attn
        watch += [a.qkv_weight, a.q_proj.weight, a.o_proj.weight]
        watch += [layer.mlp.experts.gate_up_proj] if family == 'mixtral' else [layer.mlp.gate_up_weight,
                                                                              layer.mlp.down_proj.weight]
    watch += list(m.__dict__.get('_tiled_weights', {}).values())
    refs = [weakref.ref(t) for t in watch]
    del watch
    m.quantize_weights()
    m.generate(input_ids=p, max_new_tokens=8, eos_token_id=2,
               decoding_kwargs={'use_lookahead': True, 'decoding_length': 64, 'branch_length': 8})
    gc.collect()
    assert all(r() is None for r in refs), 'a bf16 projection is still alive'
    shapes = _proj_shapes(m)
    for t in _reachable_tensors(m):
        assert not (t.dtype == torch.bfloat16 and tuple(t.shape) in shapes), tuple(t.shape)
    # parameter + buffer bytes = fp8 projections (1 B / weight) + fp32 scales + the bf16 remainder
    c = m.config
    hd = m.geometry()['head_dim']
    kv = getattr(c, 'num_key_value_heads', None) or c.num_attention_heads
    H, nq, I, V, L = c.hidden_size, c.num_attention_heads * hd, c.intermediate_size, c.vocab_size, c.num_hidden_layers
    E = getattr(c, 'num_local_experts', 1) if family == 'mixtral' else 1
    rows = [nq + 2 * kv * hd, H] + [2 * I * E, H * E]
    weights = (nq + 2 * kv * hd) * H + H * nq + E * (2 * I * H + H * I)
    # bf16: embedding + lm_head, the norms, Qwen2's qkv bias, Mixtral's router
    bf16 = 2 * (2 * V * H) + 2 * H * (2 * L + 1) + (2 * (nq + 2 * kv * hd) * L if family.startswith('qwen2') else 0)
    if family == 'mixtral':
        bf16 += 2 * E * H * L
    want = L * (weights + 4 * sum(rows)) + bf16
    have = sum(t.numel() * t.element_size() for t in m.parameters()) + sum(t.numel() * t.element_size() for t in m.buffers())
    assert have == want, (have, want)


@pytest.mark.parametrize('family,penalty,dl', [('llama', 1.0, 64), ('llama', 1.1, 128), ('mistral', 1.1, 64),
                                               ('mistral', 1.0, 128), ('mixtral', 1.0, 64), ('mixtral', 1.1, 128),
                                               ('qwen2_g7', 1.0, 64), ('qwen2_g7', 1.1, 128),
                                               ('qwen2_g6_tied', 1.1, 64), ('qwen2_g6_tied', 1.0, 128)])
def test_fp8_loop_is_exact_given_the_same_logits(family, penalty, dl):
    """the oracle loop (reference semantics, C oracle trie) drives one quantised copy through the backend interface,
    the fused device loop drives another; 90-token prompts (prefill at 256 rows), 64- or 128-node drafts (64- / 128-row
    decode plans).  Tokens, dls and edls must agree for every request, tries carried across requests."""
    from oracle.loop import lookahead_generate
    from oracle.trie import OracleLookaheadCache
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    hf = _hf(family, seed=6)
    a, b = _ours(family, hf), _ours(family, hf)
    del hf
    a.lookahead_cache = LookaheadCache(eos_ids=[2], device=DEV, vocab_capacity=1024, node_capacity=1 << 20)
    otrie = OracleLookaheadCache(eos_ids=[2])
    edl_all = []
    new = 56
    for rep in range(2):
        for p in prompts(55, 3, 90, 200):
            p = p.to(DEV)
            dk = {'use_lookahead': True, 'decoding_length': dl, 'branch_length': 12 if dl == 128 else 8}
            out = a.generate(input_ids=p, max_new_tokens=new, eos_token_id=2, repetition_penalty=penalty,
                             decoding_kwargs=dk, return_dict_in_generate=True)
            ref = lookahead_generate(None, otrie, p, max_new_tokens=new, eos_token_id=[2], repetition_penalty=penalty,
                                     decoding_length=dl, branch_length=dk['branch_length'],
                                     backend=Backend(b, 64 if dl <= 64 else 128, 90 + new + dl + 1))
            assert out.sequences[0].tolist() == ref['sequences'][0].tolist(), rep
            assert out.kwargs['edls'] == ref['edls'] and out.kwargs['dls'] == ref['dls'], rep
            edl_all += ref['edls'][1:]
    assert a._rt.max_nodes == (64 if dl <= 64 else 128)
    assert max(edl_all) > 2


def test_fp8_batched_loop_matches_the_per_request_loop():
    """batched loop (bs 3) on a quantised model: every request's tokens equal the per-request loop's output on the
    same fp8 model (greedy, lossless: neither loop changes what the model computes for the accepted tokens)"""
    from painlessinferenceacceleration_b200.models.llama.modeling_llama_batch import LlamaForCausalLM as Batch
    hf = _hf('llama', seed=9)
    batch, single = _ours('llama', hf, cls=Batch), _ours('llama', hf)
    ps = torch.cat([p for p in prompts(91, 3, 30, 200)], dim=0).to(DEV)
    out = batch.generate(input_ids=ps, max_new_tokens=32, eos_token_id=2,
                         decoding_kwargs={'use_lookahead': True, 'decoding_length': 64, 'branch_length': 8,
                                          'batch_share': 'rows'}, return_dict_in_generate=True)
    same = 0
    for i in range(3):
        g = single.generate(input_ids=ps[i:i + 1], max_new_tokens=32, eos_token_id=2,
                            decoding_kwargs={'use_lookahead': False})[0].tolist()
        L = out.kwargs['lengths'][i]
        same += int(out.sequences[i, :L].tolist() == g[:L])
    # greedy over different row sets: row-wise GEMMs and attention are identical per row, but a bf16 near-tie can flip
    assert same >= 2


def test_fp8_lookahead_equals_own_greedy():
    """lossless on our own kernels: lookahead output of the fp8 model = its use_lookahead=False greedy output"""
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    hf = _hf('llama', seed=4)
    ours = _ours('llama', hf)
    ours.lookahead_cache = LookaheadCache(eos_ids=[2], device=DEV, vocab_capacity=1024, node_capacity=1 << 20)
    same = 0
    ps = prompts(33, 6, 16, 200)
    for p in ps:
        p = p.to(DEV)
        g = ours.generate(input_ids=p, max_new_tokens=40, eos_token_id=2, decoding_kwargs={'use_lookahead': False})
        for _ in range(2):
            o = ours.generate(input_ids=p, max_new_tokens=40, eos_token_id=2,
                              decoding_kwargs={'use_lookahead': True, 'decoding_length': 64, 'branch_length': 8},
                              return_dict_in_generate=True)
        assert o.sequences.shape[1] <= 16 + 40
        assert sum(o.kwargs['edls']) == o.sequences.shape[1] - 16
        ok = o.sequences[0].tolist() == g[0].tolist()
        same += int(ok)
        if ok:
            assert max(o.kwargs['edls']) > 1
    assert same >= len(ps) - 2


def _dequantised_state(hf):
    """HF state dict with every quantised projection replaced by s * Wq (ops.quantize_fp8 is row-wise, so q/k/v and
    gate/up quantised apart equal the fused operands quantised at once)"""
    names = ('q_proj.weight', 'k_proj.weight', 'v_proj.weight', 'o_proj.weight', 'gate_proj.weight', 'up_proj.weight',
             'down_proj.weight', 'experts.gate_up_proj', 'experts.down_proj')
    out = {}
    for k, v in hf.state_dict().items():
        if k.endswith(names):
            wq, s = ops.quantize_fp8(v)
            v = wq.float() * s.unsqueeze(-1)
        out[k] = v.float()
    return out


@pytest.mark.parametrize('family', FAMILIES)
def test_fp8_verify_logits_within_tolerance(family):
    """the quantised model's verify logits vs HF eager fp32 with the dequantised weights s * Wq (the truth of the fp8
    model): max |error| <= 2 x the same dequantised model's eager bf16 error + 0.02"""
    hf = _hf(family, seed=8)
    ours = _ours(family, hf)
    deq = _dequantised_state(hf)
    hf32 = _hf(family, seed=0, dtype=torch.float32)
    hf32.load_state_dict(deq)
    hfb = _hf(family, seed=0, dtype=torch.bfloat16)
    hfb.load_state_dict({k: v.to(torch.bfloat16) for k, v in deq.items()})
    p = prompts(77, 1, 100, 200)[0].to(DEV)
    with torch.no_grad():
        truth = hf32(input_ids=p).logits[0].float()
        eager = hfb(input_ids=p).logits[0].float()
    m01 = torch.tril(torch.ones((1, 1, 100, 100), dtype=torch.long, device=DEV))
    got = OursBackend(ours).forward(p, m01, None)[0].float()
    e_ours, e_eager = (got - truth).abs().max().item(), (eager - truth).abs().max().item()
    assert e_ours <= 2 * e_eager + 0.02, (e_ours, e_eager)
    top = torch.topk(truth, 2, dim=-1).values
    sure = (top[:, 0] - top[:, 1]) > 2 * e_ours
    assert torch.equal(got.argmax(-1)[sure], truth.argmax(-1)[sure])


# ---------------------------------------------------------------------------------------------------------------
# model shapes
# ---------------------------------------------------------------------------------------------------------------
def _big_parity(cls, cfg, new=96):
    import bench
    from oracle.loop import lookahead_generate
    from oracle.trie import OracleLookaheadCache
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    a = bench.synth_fill(cls(cfg, device=torch.device(DEV)), cfg)
    b = cls(cfg, device=torch.device(DEV))
    b.load_state_dict(a.state_dict(), strict=True)
    a.quantize_weights()
    b.quantize_weights()
    a.lookahead_cache = LookaheadCache(eos_ids=[2], device=DEV, vocab_capacity=cfg.vocab_size)
    otrie = OracleLookaheadCache(eos_ids=[2])
    edl_all = []
    for rep in range(2):
        for p in bench.phrase_bank_prompts(2, cfg.vocab_size):
            p = torch.tensor([p], device=DEV)
            out = a.generate(input_ids=p, max_new_tokens=new, eos_token_id=2,
                             decoding_kwargs={'use_lookahead': True, 'decoding_length': 64, 'branch_length': 8},
                             return_dict_in_generate=True)
            ref = lookahead_generate(None, otrie, p, max_new_tokens=new, eos_token_id=[2],
                                     backend=Backend(b, 64, p.shape[1] + new + 65))
            assert out.sequences[0].tolist() == ref['sequences'][0].tolist(), rep
            assert out.kwargs['edls'] == ref['edls'] and out.kwargs['dls'] == ref['dls'], rep
            if rep == 1:
                edl_all += ref['edls'][1:]
    assert max(edl_all) > 2, 'the second pass never accepted a draft'


@pytest.mark.big
@pytest.mark.parametrize('shape', ['llama2-7b', 'qwen2-7b', 'mixtral-slice'])
def test_fp8_model_shape_loop_is_exact(shape):
    """loop parity of the quantised model at the Llama-2-7B, Qwen2-7B and 8-expert Mixtral-slice shapes
    (bench.synth_fill weights, 256-token phrase-bank prompts, 64-node / 8-branch drafts)"""
    from scripts.bench_fp8 import model_for
    cls, cfg = model_for(shape)
    _big_parity(cls, cfg)
