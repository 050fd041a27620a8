# -*- coding: utf-8 -*-
"""Qwen2 on the B200 path: the tree attention at odd GQA ratios (head pairs packed within a KV head), the biased
qkv projection, and the whole lookahead loop against the reference's semantics.

  * odd-G attention: (Hq, Hkv) in {(7, 1), (28, 4), (14, 2), (6, 2)}, plain and fused (RoPE + KV append inside the
    kernel) launches, single- and batched-slot forms, against the fp32 restatement of the reference's eager attention
    and against the one-head-per-CTA layout (PIA_ATTN_HEAD_PAIRS=0);
  * verify logits of tiny Qwen2 models (G = 7 untied, G = 6 tied) against an fp32 HF evaluation;
  * generate() against the oracle loop on the HF model, and the reference's own recorded loop (qwen2loop_*.npz)
    replayed through the fused device loop;
  * from_pretrained of save_pretrained checkpoints; the Qwen2-7B shape's loop parity (big)."""
import ctypes as C

import numpy as np
import pytest
import torch

from tests import loop_golden as G
from tests.test_gpu_generate import EPS, OursBackend
from tests.test_gpu_kernels import _mask_tensor, _random_tree, _ref_attention, _slots
from tests.tiny_models import prompts
from tests.tiny_qwen2 import golden_names, load_golden, qwen2_hf_model

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
HEADS = [(7, 1), (28, 4), (14, 2), (6, 2)]
# (P, n, pad): empty cache, ragged draft, root-only draft after a tile boundary, left padding, many tiles (KV splits)
CASES = [(0, 64, 0), (37, 33, 0), (129, 1, 0), (300, 64, 5), (2500, 47, 0)]


def _grid(plan):
    ns, ng = C.c_int(), C.c_int()
    assert plan.lib.pia_attn_plan_grid(plan.h, C.byref(ns), C.byref(ng)) == 0
    return ns.value, ng.value


def _plan(monkeypatch, pairs, *a):
    from painlessinferenceacceleration_b200.common import ops
    monkeypatch.setenv('PIA_ATTN_HEAD_PAIRS', pairs)
    return ops.AttnPlan(*a)


def _rope(max_pos, D=128, theta=1e6):
    inv = 1.0 / (theta ** (torch.arange(0, D, 2, device=DEV).float() / D))
    ang = torch.arange(max_pos, device=DEV).float()[:, None] * inv[None]
    return ang.cos().to(torch.bfloat16).contiguous(), ang.sin().to(torch.bfloat16).contiguous()


def test_head_group_counts(monkeypatch):
    """odd G: Hkv * ceil(G / 2) groups packed, Hq groups with PIA_ATTN_HEAD_PAIRS=0; even G and MHA as before"""
    D, R = 128, 64
    for Hq, Hkv, packed, single in [(7, 1, 4, 7), (28, 4, 16, 28), (14, 2, 8, 14), (6, 2, 4, 6), (32, 8, 16, 16),
                                    (32, 32, 32, 32)]:
        kc = torch.zeros((1, Hkv, 256, D), dtype=torch.bfloat16, device=DEV)
        assert _grid(_plan(monkeypatch, '1', kc, kc, Hq, Hkv, D, R))[1] == packed, (Hq, Hkv)
        assert _grid(_plan(monkeypatch, '0', kc, kc, Hq, Hkv, D, R))[1] == single, (Hq, Hkv)
    # 128-node drafts fill a tile with one head: one group per query head
    kc = torch.zeros((1, 4, 256, D), dtype=torch.bfloat16, device=DEV)
    assert _grid(_plan(monkeypatch, '1', kc, kc, 28, 4, D, 128))[1] == 28


@pytest.mark.parametrize('Hq,Hkv', HEADS)
@pytest.mark.parametrize('P,n,pad', CASES)
def test_odd_group_tree_attention(monkeypatch, Hq, Hkv, P, n, pad):
    """plain and fused launches, head pairs packed and not: each against the fp32 reference; the fused launch appends
    the same cache rows as RoPE/KV-append (bit for bit, in both layouts: the j == 0 group of every KV head writes);
    rows beyond the draft are never written"""
    from painlessinferenceacceleration_b200.common import ops
    rng = np.random.default_rng(P + n + Hq)
    torch.manual_seed(P * 7 + n + Hq)
    D, R, n_layers, layer = 128, 64, 2, 1
    max_seq = P + n + 70
    kc = (torch.randn((n_layers, Hkv, max_seq, D), device=DEV) * 0.7).to(torch.bfloat16)
    vc = (torch.randn((n_layers, Hkv, max_seq, D), device=DEV) * 0.7).to(torch.bfloat16)
    qkv = torch.randn((R, (Hq + 2 * Hkv) * D), device=DEV).to(torch.bfloat16)
    cos, sin = _rope(max_seq + 8)
    _, _, rows = _random_tree(rng, n)
    mask = _mask_tensor(rows, R)
    sl = _slots([n], [P], [pad], R)
    k0, v0 = kc.clone(), vc.clone()    # before the draft rows are appended
    q = torch.zeros((R, Hq, D), dtype=torch.bfloat16, device=DEV)
    ops.rope_kv_append(qkv, mask, sl, Hq, Hkv, D, cos, sin, q, kc[layer], vc[layer], max_seq)
    ref = _ref_attention(q, kc[layer], vc[layer], rows, n, P, pad, Hq // Hkv)
    outs = {}
    for pairs in ('1', '0'):
        plan = _plan(monkeypatch, pairs, kc, vc, Hq, Hkv, D, R)
        o = torch.full((R, Hq, D), 9.0, dtype=torch.bfloat16, device=DEV)
        plan.forward(layer, q, mask, sl, o)
        k2, v2 = k0.clone(), v0.clone()
        planf = _plan(monkeypatch, pairs, k2, v2, Hq, Hkv, D, R)
        of = torch.full((R, Hq, D), 9.0, dtype=torch.bfloat16, device=DEV)
        planf.forward_fused(layer, qkv, mask, sl, cos, sin, of)
        torch.cuda.synchronize()
        assert torch.equal(k2, kc) and torch.equal(v2, vc), pairs
        for name, t in (('plain', o), ('fused', of)):
            err = (t[:n].float() - ref).abs().max().item()
            assert torch.allclose(t[:n].float(), ref, atol=1.5e-2, rtol=2e-2), (pairs, name, err)
            assert float((t[n:].float() - 9.0).abs().sum()) == 0, (pairs, name)
            outs[(pairs, name)] = t
    # packed vs one head per CTA: the same math, another KV split count (fp32 summation order of the partials)
    for name in ('plain', 'fused'):
        assert torch.allclose(outs[('1', name)][:n].float(), outs[('0', name)][:n].float(), atol=4e-3, rtol=2e-2), name


@pytest.mark.parametrize('Hq,Hkv', [(7, 1), (28, 4)])
def test_odd_group_batched_slots(monkeypatch, Hq, Hkv):
    """the request-slot form (gridDim.z = slot): one launch over 6 slots with their own drafts, prefixes, padding and
    caches equals the fp32 reference per slot; the fused launch appends every slot's rows like RoPE/KV-append"""
    from painlessinferenceacceleration_b200.common import ops
    cases = [(8, 300, 0), (3, 0, 0), (0, 7, 0), (8, 310, 2), (1, 129, 0), (5, 900, 0)]
    rng = np.random.default_rng(Hq)
    torch.manual_seed(Hq)
    D, R, n_layers, B, rps, layer = 128, 64, 2, len(cases), 8, 1
    max_seq = max(P + n for n, P, _ in cases) + 70
    kc = (torch.randn((B, n_layers, Hkv, max_seq, D), device=DEV) * 0.7).to(torch.bfloat16)
    vc = (torch.randn((B, n_layers, Hkv, max_seq, D), device=DEV) * 0.7).to(torch.bfloat16)
    qkv = torch.randn((R, (Hq + 2 * Hkv) * D), device=DEV).to(torch.bfloat16)
    cos, sin = _rope(max_seq + 8)
    mask = torch.zeros((R, 1), dtype=torch.int64, device=DEV)
    trees = []
    for s_, (n, P, pad) in enumerate(cases):
        rows = _random_tree(rng, n)[2] if n else np.zeros((0,), dtype=np.uint64)
        trees.append(rows)
        if n:
            mask[s_ * rps:s_ * rps + n, 0] = torch.from_numpy(rows.view(np.int64)).to(DEV)
    ns, Ps, pads = [c[0] for c in cases], [c[1] for c in cases], [c[2] for c in cases]
    k0, v0 = kc.clone(), vc.clone()
    for pairs in ('1', '0'):
        kc.copy_(k0)
        vc.copy_(v0)
        plan = _plan(monkeypatch, pairs, kc, vc, Hq, Hkv, D, R)
        sl = _slots(ns, Ps, pads, rps, stride=plan.slot_stride)
        q = torch.zeros((R, Hq, D), dtype=torch.bfloat16, device=DEV)
        o = torch.full((R, Hq, D), 9.0, dtype=torch.bfloat16, device=DEV)
        ops.rope_kv_append(qkv, mask, sl, Hq, Hkv, D, cos, sin, q, kc[0, layer], vc[0, layer], max_seq)
        plan.forward(layer, q, mask, sl, o)
        k2, v2 = k0.clone(), v0.clone()
        planf = _plan(monkeypatch, pairs, k2, v2, Hq, Hkv, D, R)
        of = torch.full((R, Hq, D), 9.0, dtype=torch.bfloat16, device=DEV)
        planf.forward_fused(layer, qkv, mask, sl, cos, sin, of)
        torch.cuda.synchronize()
        assert torch.equal(k2, kc) and torch.equal(v2, vc), pairs
        for s_, (n, P, pad) in enumerate(cases):
            r0 = s_ * rps
            for name, t in (('plain', o), ('fused', of)):
                assert float((t[r0 + n:r0 + rps].float() - 9.0).abs().sum()) == 0, (pairs, name, s_)
                if n:
                    ref = _ref_attention(q[r0:], kc[s_, layer], vc[s_, layer], trees[s_], n, P, pad, Hq // Hkv)
                    assert torch.allclose(t[r0:r0 + n].float(), ref, atol=1.5e-2, rtol=2e-2), (pairs, name, s_)


# ---------------------------------------------------------------------------------------------------------------
# tiny Qwen2 models
# ---------------------------------------------------------------------------------------------------------------
def _pair(shape, seed):
    from painlessinferenceacceleration_b200.models.qwen2.modeling_qwen2 import Qwen2ForCausalLM
    hf = qwen2_hf_model(shape, seed=seed, dtype=torch.bfloat16, device=DEV, vocab=200)
    hf.fp32_twin = None
    ours = Qwen2ForCausalLM(hf.config, device=torch.device(DEV))
    missing = ours.load_state_dict(hf.state_dict(), strict=False)
    assert not missing.missing_keys, missing
    return hf, ours


def _fp32_twin(shape, hf):
    twin = qwen2_hf_model(shape, seed=0, dtype=torch.float32, device=DEV, vocab=200)
    twin.load_state_dict({k: v.float() for k, v in hf.state_dict().items()})
    return twin


@pytest.mark.parametrize('shape', ['g7', 'g6_tied'])
@pytest.mark.parametrize('gemm_set', [None, 'qkv,gate_up,down'])
def test_qwen2_verify_logits_within_tolerance(monkeypatch, shape, gemm_set):
    """our bf16 forward (biased qkv as one cuBLASLt GEMM with a bias epilogue) vs an fp32 evaluation of the same
    weights: max |logit error| <= 2 x the eager bf16 model's error + 0.02.  PIA_GEMM_SET=qkv must not move the biased
    projection onto k_gemm_ws (which has no bias)."""
    if gemm_set:
        monkeypatch.setenv('PIA_GEMM_SET', gemm_set)
    hf, ours = _pair(shape, seed=8)
    hf32 = _fp32_twin(shape, hf)
    p = prompts(77, 1, 100, 200)[0].to(DEV)
    with torch.no_grad():
        truth = hf32(input_ids=p).logits[0].float()
        eager = hf(input_ids=p).logits[0].float()
    m01 = torch.tril(torch.ones((1, 1, 100, 100), dtype=torch.long, device=DEV))
    got = OursBackend(ours).forward(p, m01, None)[0].float()
    e_ours, e_eager = (got - truth).abs().max().item(), (eager - truth).abs().max().item()
    assert e_ours <= 2 * e_eager + 0.02, (e_ours, e_eager)
    top = torch.topk(truth, 2, dim=-1).values
    sure = (top[:, 0] - top[:, 1]) > 2 * e_ours
    assert torch.equal(got.argmax(-1)[sure], truth.argmax(-1)[sure])
    plans = ours._rt.gemm_plans
    assert plans and all('qkv' not in lp for lp in plans['layers'])
    if gemm_set:
        assert all('gate_up' in lp for lp in plans['layers'])


def _legit_divergence(shape, hf, prefix, tok_a, tok_b, penalty):
    """as test_gpu_generate._legit_divergence: both candidates within the eager bf16 model's noise of the fp32 optimum"""
    if hf.fp32_twin is None:
        hf.fp32_twin = _fp32_twin(shape, hf)
    with torch.no_grad():
        truth = hf.fp32_twin(input_ids=prefix).logits[0, -1].float()
        noisy = hf(input_ids=prefix).logits[0, -1].float()
    noise = (noisy - truth).abs().max().item()
    if penalty != 1.0:
        from transformers import RepetitionPenaltyLogitsProcessor
        truth = RepetitionPenaltyLogitsProcessor(penalty)(prefix, truth[None])[0]
    gap = max((truth.max() - truth[tok_a]).item(), (truth.max() - truth[tok_b]).item())
    return gap <= 4 * noise + 0.05, gap, noise


@pytest.mark.parametrize('shape,penalty', [('g7', 1.0), ('g7', 1.1), ('g6_tied', 1.0)])
def test_qwen2_generate_matches_oracle(shape, penalty):
    """our generate() vs the oracle loop (reference semantics) driving the HF Qwen2 model: every divergence sits on
    an fp32 top-2 margin below EPS, and equal text implies equal drafts (dls) and accepted lengths (edls)"""
    from oracle.loop import lookahead_generate
    from oracle.trie import OracleLookaheadCache
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    hf, ours = _pair(shape, seed=2)
    ours.lookahead_cache = LookaheadCache(eos_ids=[2], device=DEV, vocab_capacity=1024, node_capacity=1 << 20)
    otrie = OracleLookaheadCache(eos_ids=[2])
    for rep in range(2):
        for p in prompts(21, 4, 24, 200):
            p = p.to(DEV)
            dk = {'use_lookahead': True, 'decoding_length': 64, 'branch_length': 8}
            out = ours.generate(input_ids=p, max_new_tokens=48, eos_token_id=2, repetition_penalty=penalty,
                                decoding_kwargs=dk, return_dict_in_generate=True)
            ref = lookahead_generate(hf, otrie, p, max_new_tokens=48, eos_token_id=[2], repetition_penalty=penalty)
            a, b = out.sequences[0].tolist(), ref['sequences'][0].tolist()
            if a == b:
                assert out.kwargs['edls'] == ref['edls'] and out.kwargs['dls'] == ref['dls']
            else:
                k = next(i for i in range(min(len(a), len(b))) if a[i] != b[i])
                ok, gap, noise = _legit_divergence(shape, hf, ref['sequences'][:, :k], a[k], b[k], penalty)
                assert ok, f'diverged at {k}: fp32 gap {gap:.3f} vs bf16 noise {noise:.3f}'
                assert gap < EPS, f'diverged at {k} although the fp32 top-2 margin is {gap:.3f} >= {EPS}'
                ours.lookahead_cache.fresh()
                otrie.fresh()


@pytest.mark.parametrize('name', golden_names())
def test_device_loop_reproduces_the_reference_loop_on_qwen2(name):
    """the reference's own loop on HF Qwen2 (qwen2loop_*.npz): its recorded logits fed to our fused device loop give
    the reference's drafts, tokens, dls and edls for every request (tries carried across requests)"""
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    from tests.test_gpu_loop_golden import _replay_model
    meta, z = load_golden(name)
    pen = meta['gen'].get('repetition_penalty', 1.0)
    dev = torch.device(DEV)
    model = _replay_model(meta['vocab'], dev)
    model.lookahead_cache = LookaheadCache(eos_ids=[2], device=dev, vocab_capacity=1024, node_capacity=1 << 20)
    multi = 0
    for ri, req in enumerate(meta['requests']):
        model.load(meta, z, req)
        dk = {'use_lookahead': True, 'decoding_length': meta['decoding_length'], 'branch_length': meta['branch_length']}
        out = model.generate(input_ids=torch.tensor([req['prompt']], device=dev), max_new_tokens=req['max_new_tokens'],
                             eos_token_id=2, repetition_penalty=pen, decoding_kwargs=dk, return_dict_in_generate=True)
        assert out.sequences[0].tolist() == req['sequences'], (name, ri)
        assert out.kwargs['dls'] == req['dls'] and out.kwargs['edls'] == req['edls'], (name, ri)
        ids_log, n_log, mask_log = model.ids_log.cpu(), model.n_log.cpu(), model.mask_log.cpu().numpy().view(np.uint64)
        for k, st in enumerate(req['steps'][1:]):
            n = len(st['decoding_ids'])
            assert int(n_log[k]) == n and ids_log[k, :n].tolist() == st['decoding_ids'], (name, ri, k)
            assert np.array_equal(mask_log[k, :n], G.step_mask(st)), (name, ri, k)
        multi += sum(e > 1 for e in req['edls'])
    assert multi >= 3


@pytest.mark.parametrize('shape', ['g7', 'g6_tied'])
def test_qwen2_from_pretrained(tmp_path, shape):
    """save_pretrained output (safetensors) loads with every parameter equal, the tied head from the embedding; a
    checkpoint without one of the q/k/v biases is refused"""
    from safetensors.torch import load_file, save_file
    from painlessinferenceacceleration_b200.models.qwen2.modeling_qwen2 import Qwen2ForCausalLM
    hf = qwen2_hf_model(shape, seed=5, dtype=torch.bfloat16, vocab=200)
    hf.save_pretrained(str(tmp_path))
    files = sorted(tmp_path.glob('*.safetensors'))
    assert files
    ours = Qwen2ForCausalLM.from_pretrained(str(tmp_path), device=torch.device(DEV))
    want = hf.state_dict()
    for k, v in ours.state_dict().items():
        assert torch.equal(v.cpu(), want[k]), k
    if hf.config.tie_word_embeddings:
        assert 'lm_head.weight' not in load_file(str(files[0]))
    sd = load_file(str(files[0]))
    del sd['model.layers.1.self_attn.k_proj.bias']
    save_file(sd, str(files[0]), metadata={'format': 'pt'})
    with pytest.raises(RuntimeError, match='missing'):
        Qwen2ForCausalLM.from_pretrained(str(tmp_path), device=torch.device(DEV))


@pytest.mark.big
def test_qwen2_7b_shape_loop_is_exact():
    """Qwen2-7B shape (28 layers, 3584 hidden, 18944 inter, 28 q / 4 KV heads: G = 7, V = 152064, rope_theta 1e6,
    q/k/v biases; bench.synth_fill weights): the oracle loop drives one copy through the backend interface, our fused
    device loop the other; 64-node / 8-branch drafts, 256-token phrase-bank prompts, two passes with the tries carried.
    Tokens, dls and edls must be identical for every request, and the second pass must accept drafts."""
    import bench
    from oracle.loop import lookahead_generate
    from oracle.trie import OracleLookaheadCache
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    from painlessinferenceacceleration_b200.models.qwen2.modeling_qwen2 import Qwen2ForCausalLM
    from scripts.bench_qwen2 import qwen2_7b_config
    cfg = qwen2_7b_config()
    a = bench.synth_fill(Qwen2ForCausalLM(cfg, device=torch.device(DEV)), cfg)
    b = Qwen2ForCausalLM(cfg, device=torch.device(DEV))
    b.load_state_dict(a.state_dict(), strict=True)
    a.lookahead_cache = LookaheadCache(eos_ids=[2], device=DEV, vocab_capacity=cfg.vocab_size)
    otrie = OracleLookaheadCache(eos_ids=[2])
    new = 96
    edl_all = []
    for rep in range(2):
        for p in bench.phrase_bank_prompts(3, cfg.vocab_size):
            p = torch.tensor([p], device=DEV)
            out = a.generate(input_ids=p, max_new_tokens=new, eos_token_id=2,
                             decoding_kwargs={'use_lookahead': True, 'decoding_length': 64, 'branch_length': 8},
                             return_dict_in_generate=True)
            ref = lookahead_generate(None, otrie, p, max_new_tokens=new, eos_token_id=[2],
                                     backend=OursBackend(b, prefill_like_generate=True, max_seq=256 + new + 65))
            assert out.sequences[0].tolist() == ref['sequences'][0].tolist(), rep
            assert out.kwargs['edls'] == ref['edls'] and out.kwargs['dls'] == ref['dls'], rep
            if rep == 1:
                edl_all += ref['edls'][1:]
    assert max(edl_all) > 2, 'the second pass never accepted a draft'
