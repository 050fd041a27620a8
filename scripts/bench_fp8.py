# -*- coding: utf-8 -*-
"""FP8 weight-only against bf16 on the lookahead path: bench.py's protocol (phrase-bank prompts, synth_fill weights,
warm-up requests, a first pass over unseen prompts, a second epoch from the trie the first pass left, 256 -> 256
tokens, 64-node / 8-branch drafts) on a bf16 model and its fp8 twin (the same weights through quantize_weights()),
built in one process and alternated pass by pass.  Also reported:
  * per-projection kernel time at 64 rows, fp8 plan against the bf16 path that runs today (k_gemm_ws or cuBLAS), each
    a CUDA graph over all layers (the layers' weights together exceed L2, so every launch reads HBM), with GB/s on
    the algorithmic weight bytes;
  * the whole verify forward (64 rows, one CUDA graph) for the split-K choices of the narrow fp8 projections;
  * prefill time per request (max_new_tokens = 1);
  * how far fp8 moves the model: verify logits of the fp8 twin against the bf16 model on the same prompts (max / mean
    |difference|, top-1 agreement) - diagnostics, not asserts.
Prints one JSON line.

    python scripts/bench_fp8.py --shape llama2-7b --steps 8 --warmup 3"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

SHAPES = ('llama2-7b', 'qwen2-7b', 'mixtral-slice')
MIXTRAL_SLICE_LAYERS = 4


def model_for(shape):
    """(model class, config) of a benchmark shape; the Mixtral slice is Mixtral-8x7B with its first layers only"""
    from painlessinferenceacceleration_b200.models.llama.modeling_llama import LlamaForCausalLM
    from painlessinferenceacceleration_b200.models.mixtral.modeling_mixtral import MixtralForCausalLM
    from painlessinferenceacceleration_b200.models.qwen2.modeling_qwen2 import Qwen2ForCausalLM
    if shape == 'qwen2-7b':
        from scripts.bench_qwen2 import qwen2_7b_config
        return Qwen2ForCausalLM, qwen2_7b_config()
    if shape == 'mixtral-slice':
        cfg, _ = bench.make_config('mixtral-8x7b')
        cfg.num_hidden_layers = MIXTRAL_SLICE_LAYERS
        return MixtralForCausalLM, cfg
    cfg, _ = bench.make_config(shape)
    return LlamaForCausalLM, cfg


def gpu_state():
    """card, power limit and SM clock, read in the same call as the measurement"""
    q = 'name,power.limit,clocks.sm,clocks.max.sm'
    try:
        out = subprocess.check_output(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader'], timeout=30).decode()
        return dict(zip(q.split(','), [v.strip() for v in out.splitlines()[0].split(',')]))
    except Exception as e:  # pragma: no cover
        return {'error': f'{type(e).__name__}: {e}'}


def weight_bytes(model):
    """decoder + lm_head weight bytes read per verify step (parameters and the fp8 buffers; embedding excluded)"""
    n = 0
    for name, t in list(model.named_parameters()) + list(model.named_buffers()):
        if 'embed_tokens' in name or 'qkv_bias' in name:
            continue
        n += t.numel() * t.element_size()
    return n


def _decode_state(model):
    rt = model._runtime(bench.PROMPT_LEN + bench.NEW_TOKENS + bench.DL + 1, 64)
    rt.n.fill_(bench.DL)
    rt.prefix_len.fill_(bench.PROMPT_LEN + bench.NEW_TOKENS // 2)
    rt.pad.zero_()
    rt.mask.copy_(rt.chain)
    return rt


def projection_times(bf, f8, reps=5):
    """us per launch (median of alternated repeats) for every projection at 64 rows: the fp8 plan vs the bf16 path"""
    import torch
    rb, rf = _decode_state(bf), _decode_state(f8)
    b = rb.decode_bufs
    lb = rb.gemm_plans['layers'] if rb.gemm_plans else [{} for _ in bf.model.layers]
    lf = rf.gemm_plans['layers']
    L = len(lf)
    jobs = {}
    for name in lf[0]:
        fp8 = (lambda name=name: [lp[name].run(64) for lp in lf])
        if name in lb[0]:
            bfj = (lambda name=name: [lp[name].run(64) for lp in lb])
            path = 'k_gemm_ws'
        elif name == 'qkv':
            def bfj():
                for layer in bf.model.layers:
                    a = layer.self_attn
                    if a.qkv_bias is not None:
                        torch.addmm(a.qkv_bias, b.y, a.qkv_weight.t(), out=b.qkv)
                    else:
                        torch.mm(b.y, a.qkv_weight.t(), out=b.qkv)
            path = 'cuBLAS'
        elif name == 'o':
            bfj = (lambda: [torch.mm(b.attn, layer.self_attn.o_proj.weight.t()) for layer in bf.model.layers])
            path = 'cuBLAS'
        else:
            continue
        w = lf[0][name].weight
        jobs[name] = (fp8, bfj, path, w.numel() * w.element_size())
    res = {}
    for name, (fp8, bfj, path, nbytes) in jobs.items():
        t8, tb = [], []
        for _ in range(reps):
            t8.append(bench._graph_time(fp8) / L)
            tb.append(bench._graph_time(bfj) / L)
        m8, mb = statistics.median(t8), statistics.median(tb)
        res[name] = {'fp8_us': m8, 'bf16_us': mb, 'bf16_path': path, 'fp8_weight_bytes': nbytes,
                     'fp8_gbs': nbytes / (m8 * 1e-6) / 1e9, 'bf16_gbs': 2 * nbytes / (mb * 1e-6) / 1e9,
                     'splits_fp8': lf[0][name].splits, 'fp8_all_us': t8, 'bf16_all_us': tb}
    return res


def forward_us(model, reps=5):
    import torch
    rt = _decode_state(model)
    ts = [bench._graph_time(lambda: model._verify_layers(rt), reps=10) for _ in range(reps)]
    torch.cuda.synchronize()
    return statistics.median(ts)


def split_sweep(model):
    """whole verify forward (64 rows) for the split-K of qkv / o / down, one choice changed at a time"""
    cls = type(model)
    base = dict(cls.FP8_SPLIT)
    variants = [dict(base)]
    for name, opts in (('qkv', (1, -4)), ('o', (1, 4, -2)), ('down', (1, 4, -2))):
        for v in opts:
            if v != base[name]:
                variants.append(dict(base, **{name: v}))
    out = []
    try:
        for v in variants:
            cls.FP8_SPLIT = v
            model._rt = None
            out.append({'split': v, 'forward_us': forward_us(model)})
    finally:
        cls.FP8_SPLIT = base
        model._rt = None
    return out


def prefill_ms(model, prompts, dev):
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ins = [torch.tensor([p], device=dev) for p in prompts]
    model.generate(input_ids=ins[0], max_new_tokens=1, eos_token_id=2, decoding_kwargs={'use_lookahead': False})
    torch.cuda.synchronize()
    e0.record()
    for x in ins:
        model.generate(input_ids=x, max_new_tokens=1, eos_token_id=2, decoding_kwargs={'use_lookahead': False})
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / len(ins)


def logit_drift(bf, f8, prompts, dev):
    import torch
    m01 = torch.tril(torch.ones((1, 1, 64, 64), dtype=torch.long, device=dev))
    mx, mean, agree, tot = 0.0, [], 0, 0
    for p in prompts:
        x = torch.tensor([p[:64]], device=dev)
        a = bf.forward(x, m01, past_key_values=None)[0][0].float()
        b = f8.forward(x, m01, past_key_values=None)[0][0].float()
        d = (a - b).abs()
        mx = max(mx, d.max().item())
        mean.append(d.mean().item())
        agree += int((a.argmax(-1) == b.argmax(-1)).sum())
        tot += a.shape[0]
    return {'rows': tot, 'max_abs_diff': mx, 'mean_abs_diff': sum(mean) / len(mean), 'top1_agreement': agree / tot,
            'note': 'fp8 twin vs bf16 model, verify logits of 64-token chains; diagnostics only'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--shape', choices=SHAPES, default='llama2-7b')
    ap.add_argument('--steps', type=int, default=8)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--no-sweep', action='store_true', help='skip the split-K sweep of the whole forward')
    args = ap.parse_args()
    import torch
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    cls, cfg = model_for(args.shape)
    bf = bench.synth_fill(cls(cfg, device=dev), cfg)
    f8 = cls(cfg, device=dev)
    f8.load_state_dict(bf.state_dict(), strict=True)
    f8.quantize_weights()
    models = {'bf16': bf, 'fp8': f8}
    for m in models.values():
        m.lookahead_cache = LookaheadCache(eos_ids=[2], device=dev, vocab_capacity=cfg.vocab_size)
    K, Wm = args.steps, args.warmup
    allp = bench.phrase_bank_prompts(64 + 8 * max(Wm, 1), cfg.vocab_size)
    timed = [allp[j] for j in bench.timed_requests(K)]
    warm = [allp[64 + i % (8 * max(Wm, 1))] for i in range(Wm)]
    gen = dict(max_new_tokens=bench.NEW_TOKENS, eos_token_id=2, return_dict_in_generate=True,
               decoding_kwargs={'use_lookahead': True, 'decoding_length': bench.DL, 'branch_length': bench.BL})
    for p in warm:
        for m in models.values():
            m.generate(input_ids=torch.tensor([p], device=dev), **gen)

    def timed_pass(model):
        ins = [torch.tensor([p], device=dev) for p in timed]
        toks, edls = 0, []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for x in ins:
            o = model.generate(input_ids=x, **gen)
            toks += o.sequences.shape[1] - bench.PROMPT_LEN
            edls += o.kwargs['edls'][1:]
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        return {'tok_s': toks / (ms / 1e3), 'ms': ms, 'tokens': toks,
                'mean_accepted_len_per_step': sum(edls) / max(len(edls), 1), 'verify_steps': len(edls),
                'ms_per_verify_step': ms / max(len(edls), 1)}

    state_before = gpu_state()
    sampler = bench.ClockSampler(0)
    sampler.start()
    res = {k: {} for k in models}
    for phase in ('first_pass', 'second_epoch'):     # alternated: both see the same neighbours on the shared host
        for k, m in models.items():
            res[k][phase] = timed_pass(m)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    for k, m in models.items():
        wb = weight_bytes(m)
        st = res[k]['first_pass']['ms_per_verify_step']
        res[k]['weight_bytes_per_step'] = wb
        res[k]['weight_gbs_per_step'] = wb / (st * 1e-3) / 1e9
    res['projections_64_rows'] = projection_times(bf, f8)
    res['verify_forward_us'] = {'bf16': forward_us(bf), 'fp8': forward_us(f8)}
    if not args.no_sweep:
        res['fp8_split_sweep'] = split_sweep(f8)
    pf = allp[:4]
    res['prefill_ms_per_request'] = {k: prefill_ms(m, pf, dev) for k, m in models.items()}
    res['logit_drift'] = logit_drift(bf, f8, allp[:4], dev)
    line = {
        'metric': f'fp8 vs bf16 weights @ {args.shape} {bench.DL}-draft/{bench.BL}-branch',
        'shape': args.shape, 'layers': cfg.num_hidden_layers, 'steps': K, 'warmup': Wm,
        'speedup_first_pass_tok_s': res['fp8']['first_pass']['tok_s'] / res['bf16']['first_pass']['tok_s'],
        **res,
        'gpu': gpu_state(), 'gpu_before': state_before, 'clocks': sampler.summary(),
        'data': f'synthetic (phrase-bank prompts, bench.synth_fill weights of the {args.shape} shape)',
    }
    print(json.dumps(line))


if __name__ == '__main__':
    main()
