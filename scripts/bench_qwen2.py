# -*- coding: utf-8 -*-
"""Qwen2-7B-shaped lookahead benchmark (28 layers, hidden 3584, inter 18944, 28 q / 4 KV heads, V = 152064,
rope_theta 1e6, q/k/v biases): bench.py's protocol (phrase-bank prompts, synth_fill weights, warm-up requests, a first
pass over unseen prompts, a second epoch from the trie the first pass left, 256 -> 256 tokens, 64-node / 8-branch
drafts), plus the two kernels the Qwen2 shape changes:
  * k_tree_attn per layer at G = 7 with head pairs packed (PIA_ATTN_HEAD_PAIRS=1, 16 head groups) and with one head
    per CTA (PIA_ATTN_HEAD_PAIRS=0, 28 head groups), alternated, each a CUDA graph over all 28 layers (the layers' KV
    planes together exceed L2, so every launch reads HBM);
  * k_row_argmax at V = 152064 (64 draft rows), from a torch.profiler trace of pia_accept.
Prints one JSON line.

    python scripts/bench_qwen2.py --steps 8 --warmup 3"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def qwen2_7b_config(layers=28):
    from transformers import Qwen2Config
    return Qwen2Config(vocab_size=152064, hidden_size=3584, intermediate_size=18944, num_hidden_layers=layers,
                       num_attention_heads=28, num_key_value_heads=4, max_position_embeddings=32768, rms_norm_eps=1e-6,
                       rope_theta=1e6, use_sliding_window=False, tie_word_embeddings=False, bos_token_id=1,
                       eos_token_id=2, pad_token_id=0)


def gpu_info(index):
    import torch
    out = {'name': torch.cuda.get_device_name(index)}
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        out['power_limit_w'] = nv.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
    except Exception as e:  # pragma: no cover
        out['power_limit_w'] = f'unavailable: {type(e).__name__}'
    return out


def attention_ab(model, reps=7):
    """us per k_tree_attn launch, head pairs on / off, on the runtime's own caches at the bench's mid-generation shape"""
    import torch
    from painlessinferenceacceleration_b200.common import ops
    rt, g = model._rt, model._rt.g
    P, n = bench.PROMPT_LEN + bench.NEW_TOKENS // 2, bench.DL
    rt.n.fill_(n)
    rt.prefix_len.fill_(P)
    rt.pad.zero_()
    rt.mask.copy_(rt.chain)
    plans, grids = {}, {}
    old = os.environ.get('PIA_ATTN_HEAD_PAIRS')
    for v in ('1', '0'):
        os.environ['PIA_ATTN_HEAD_PAIRS'] = v
        plans[v] = ops.AttnPlan(rt.k_cache, rt.v_cache, g['n_q_heads'], g['n_kv_heads'], g['head_dim'], rt.max_nodes)
        import ctypes as C
        ns, ng = C.c_int(), C.c_int()
        plans[v].lib.pia_attn_plan_grid(plans[v].h, C.byref(ns), C.byref(ng))
        grids[v] = {'n_split': ns.value, 'n_groups': ng.value}
    if old is None:
        del os.environ['PIA_ATTN_HEAD_PAIRS']
    else:
        os.environ['PIA_ATTN_HEAD_PAIRS'] = old
    outs = {v: torch.zeros_like(rt.attn) for v in plans}

    def sweep(v):
        return lambda: [plans[v].forward(li, rt.q, rt.mask, rt.decode_bufs.slots, outs[v]) for li in range(g['n_layers'])]

    times = {'1': [], '0': []}
    for _ in range(reps):     # alternated: both layouts see the same neighbours on the shared host
        for v in ('1', '0'):
            times[v].append(bench._graph_time(sweep(v)) / g['n_layers'])
    torch.cuda.synchronize()
    diff = (outs['1'][:n].float() - outs['0'][:n].float()).abs().max().item()
    L = P + n
    by = 2 * L * g['n_kv_heads'] * g['head_dim'] * 2 + 2 * n * g['n_q_heads'] * g['head_dim'] * 2
    res = {'shape': f'n={n} P={P} Hq={g["n_q_heads"]} Hkv={g["n_kv_heads"]} D={g["head_dim"]}',
           'algorithmic_bytes_per_launch': by, 'max_abs_diff_pairs_vs_single': diff}
    for v, name in (('1', 'head_pairs_1'), ('0', 'head_pairs_0')):
        res[name] = dict(grids[v], us_per_layer_median=statistics.median(times[v]), us_per_layer_all=times[v])
    return res


def row_argmax_us(vocab, dev, iters=50):
    """k_row_argmax (and the whole pia_accept) at this vocabulary: 64 draft rows of a chain, repetition penalty 1.1 so
    that the penalty bitmap is in play"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from painlessinferenceacceleration_b200.common import ops
    i32 = dict(dtype=torch.int32, device=dev)
    acc = ops.Accept(vocab, 64, 1.1, [2], 1 << 20, dev)
    logits = (torch.randn((64, vocab), device=dev)).to(torch.bfloat16)
    ids = torch.randint(3, vocab, (64,), **i32)
    mask = torch.tensor([(1 << (i + 1)) - 1 if i < 63 else -1 for i in range(64)], dtype=torch.int64, device=dev)[:, None]
    seq = torch.randint(3, vocab, (4096,), **i32)

    def run():
        seq_len, prefix = torch.tensor([512], **i32), torch.tensor([511], **i32)
        acc.run(logits, ids, mask, torch.tensor([64], **i32), seq, seq_len, torch.zeros((64,), **i32),
                torch.zeros((1,), **i32), torch.zeros((64,), **i32), prefix, torch.zeros((1,), **i32))
    for _ in range(5):
        run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            run()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        if 'k_row_argmax' in e.key or 'accept' in e.key.lower():
            per[e.key.split('(')[0]] = e.device_time_total / max(e.count, 1)
    return {'vocab': vocab, 'rows': 64, 'us_per_launch': per}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=8)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--penalty', type=float, default=1.0)
    args = ap.parse_args()
    import torch
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    from painlessinferenceacceleration_b200.models.qwen2.modeling_qwen2 import Qwen2ForCausalLM
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    cfg = qwen2_7b_config()
    model = Qwen2ForCausalLM(cfg, device=dev)
    bench.synth_fill(model, cfg)
    model.lookahead_cache = LookaheadCache(eos_ids=[2], device=dev, vocab_capacity=cfg.vocab_size)
    K, Wm = args.steps, args.warmup
    allp = bench.phrase_bank_prompts(64 + 8 * max(Wm, 1), cfg.vocab_size)
    timed = [allp[j] for j in bench.timed_requests(K)]
    warm = [allp[64 + i % (8 * max(Wm, 1))] for i in range(Wm)]
    gen = dict(max_new_tokens=bench.NEW_TOKENS, eos_token_id=2, return_dict_in_generate=True,
               repetition_penalty=args.penalty,
               decoding_kwargs={'use_lookahead': True, 'decoding_length': bench.DL, 'branch_length': bench.BL})
    for p in warm:
        model.generate(input_ids=torch.tensor([p], device=dev), **gen)

    def timed_pass():
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
        return {'value': toks / (ms / 1e3), 'unit': 'tokens/s', 'ms': ms, 'tokens': toks,
                'mean_accepted_len_per_step': sum(edls) / max(len(edls), 1), 'verify_steps': len(edls),
                'ms_per_verify_step': ms / max(len(edls), 1)}

    sampler = bench.ClockSampler(0)
    sampler.start()
    first = timed_pass()
    second = timed_pass()
    sampler.stop_flag = True
    sampler.join(timeout=2)
    hbm, _tf, src = bench.peaks()
    wbytes = bench.weight_bytes_per_step(model)
    step_ms = first['ms_per_verify_step']
    line = {
        'metric': f'accepted tokens/sec @ Qwen2-7B shape {bench.DL}-draft/{bench.BL}-branch; mean accepted len/step',
        'value': first['value'], 'unit': 'tokens/s', 'steps': K, 'warmup': Wm, 'repetition_penalty': args.penalty,
        'mean_accepted_len_per_step': first['mean_accepted_len_per_step'], 'ms_per_verify_step': step_ms,
        'first_pass': first, 'second_epoch': second,
        'roofline_step': {'bound': 'hbm', 'bytes_per_step': wbytes, 'ms_per_step': step_ms,
                          'achieved_gbs': wbytes / (step_ms * 1e-3) / 1e9, 'peak_gbs': hbm, 'peak_source': src,
                          'frac': wbytes / (step_ms * 1e-3) / 1e9 / hbm,
                          'note': 'decoder + lm_head weight bytes per verify step / measured time per verify step '
                                  '(host gaps, prefill and trie work included)'},
        'k_tree_attn': attention_ab(model),
        'k_row_argmax': row_argmax_us(cfg.vocab_size, dev),
        'gpu': gpu_info(0), 'clocks': sampler.summary(),
        'data': 'synthetic (phrase-bank prompts, bench.synth_fill weights of the Qwen2-7B shape)',
    }
    print(json.dumps(line))


if __name__ == '__main__':
    main()
