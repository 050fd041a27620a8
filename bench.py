# -*- coding: utf-8 -*-
"""bench.py -- accepted tokens/sec of the LOOKAHEAD draft-verify loop (BASELINE.json metric) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model llama2-7b|...]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" is one request through the hot path: a 256-token synthetic prompt -> greedy generation of 256 new tokens
with 64-token / 8-branch trie drafts (BASELINE config 2; SURVEY.md 8d).  No checkpoints exist offline, so the weights
are synthetic, of the named shape, and IDENTICAL in the GPU arm and the CPU arms (a counter-based hash of the element
index, synth_fill below): every decoder layer is plain random init (std 0.02); the embedding scale and the lm_head are
constructed so that greedy decoding is a noisy first-order chain over the vocabulary (next = succ(token) unless the
random layers' context-dependent contribution flips the arg-max).  Such text re-uses n-grams across requests like
real text does, so a trie warmed on OTHER prompts (the reference's warm-up, benchmarks/benchmark.py:159-169)
yields accepted lengths > 1 on prompts it has never seen - the headline is that first pass, not answer replay.
One JSON line is printed by rank 0; see README.md / DESIGN.md 5 for the keys.  N > 1 = independent data-parallel
replicas (the loop is per request, pretrained_model.py:1152): one NCCL broadcast of the weights, then no collective on
the data path; every replica runs the same K requests (identical work per rank, weak scaling).
"""
import argparse
import json
import os
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MODELS = {
    # name: (family, hidden, inter, layers, heads, kv_heads, vocab, repetition_penalty of its BASELINE config)
    'llama2-7b': ('llama', 4096, 11008, 32, 32, 32, 32000, 1.0),
    'mistral-7b': ('mistral', 4096, 14336, 32, 32, 8, 32000, 1.1),
    'mixtral-8x7b': ('mixtral', 4096, 14336, 32, 32, 8, 32000, 1.0),
    'tiny': ('llama', 512, 1024, 4, 4, 4, 32000, 1.0),
}
METRIC_NAMES = {'llama2-7b': 'Llama-2-7B', 'mistral-7b': 'Mistral-7B', 'mixtral-8x7b': 'Mixtral-8x7B', 'tiny': 'tiny'}
PROMPT_LEN, NEW_TOKENS, DL, BL = 256, 256, 64, 8
EMBED_STD = float(os.environ.get("PIA_BENCH_EMBED_STD", "5.5"))   # signal of the successor chain vs the layers' noise
LM_SCALE = 0.25
CPU_NEW_TOKENS = 16   # generated tokens per request of the bounded CPU samples (fixed, so the sample is reproducible)


def metric_name(model):
    return f'accepted tokens/sec @ {METRIC_NAMES[model]} {DL}-draft/{BL}-branch; mean accepted len/step'


def make_config(name):
    from transformers import LlamaConfig, MistralConfig, MixtralConfig
    fam, hid, inter, layers, heads, kv, vocab, _rp = MODELS[name]
    kw = dict(vocab_size=vocab, hidden_size=hid, intermediate_size=inter, num_hidden_layers=layers,
              num_attention_heads=heads, num_key_value_heads=kv, max_position_embeddings=4096, rms_norm_eps=1e-5,
              bos_token_id=1, eos_token_id=2, pad_token_id=0)
    if fam == 'mixtral':
        return MixtralConfig(sliding_window=None, num_local_experts=8, num_experts_per_tok=2, **kw), fam
    return (MistralConfig(sliding_window=None, **kw) if fam == 'mistral' else LlamaConfig(**kw)), fam


def phrase_bank_prompts(n, vocab, length=PROMPT_LEN, seed=1234):
    """SURVEY.md 8d: sequences drawn from 2000 phrases of 4-24 ids, ids Zipf(1.3) clipped to [3, V-1]"""
    rng = np.random.default_rng(seed)
    bank = [np.clip(rng.zipf(1.3, size=int(rng.integers(4, 25))), 3, vocab - 1) for _ in range(2000)]
    out = []
    for _ in range(n):
        toks = []
        while len(toks) < length:
            toks.extend(bank[int(rng.integers(0, len(bank)))].tolist())
        out.append(toks[:length])
    return out


# ----------------------------------------------------------------------------------------------- synthetic weights
def _hash32(i, seed):
    """murmur3 finaliser over int32 tensors (wrap-around arithmetic is identical on CPU and CUDA)"""
    import torch

    def lsr(x, k):  # logical shift right of an int32
        return (x >> k) & ((1 << (32 - k)) - 1)
    x = i ^ seed
    x = x ^ lsr(x, 16)
    x = x * torch.tensor(-2048144789, dtype=torch.int32, device=i.device)   # 0x85EBCA6B
    x = x ^ lsr(x, 13)
    x = x * torch.tensor(-1028477387, dtype=torch.int32, device=i.device)   # 0xC2B2AE35
    x = x ^ lsr(x, 16)
    return x


def hashed_normal_(t, seed, std):
    """fills tensor t (bf16) in place with zero-mean values of standard deviation std that are a pure function of
    (seed, element index) and identical on CPU and CUDA: a 24-bit uniform drawn from a two-round multiply/xorshift hash
    of the index (int32 wrap-around arithmetic), centred and scaled to the requested std"""
    import torch
    flat = t.view(-1)
    n = flat.numel()
    chunk = 1 << 24
    dev = t.device
    base = torch.arange(chunk, dtype=torch.int32, device=dev)
    c1 = torch.tensor(-1640531535, dtype=torch.int32, device=dev)   # 0x9E3779B1
    c2 = torch.tensor(-2048144789, dtype=torch.int32, device=dev)   # 0x85EBCA6B
    scale = std * (12.0 ** 0.5) / 16777216.0
    for k, s in enumerate(range(0, n, chunk)):
        e = min(n, s + chunk)
        salt = (int(seed) * 2654435761 + (k + 1) * 40503) & 0x7FFFFFFF
        x = (base[:e - s] ^ salt) * c1
        x = x ^ ((x >> 15) & 0x1FFFF)
        x = x * c2
        x = x ^ ((x >> 13) & 0x7FFFF)
        flat[s:e] = (((x & 0xFFFFFF).to(torch.float32) - 8388607.5) * scale).to(t.dtype)
    return t


def successor_map(vocab, seed=99):
    """succ(t): a fixed pseudo-random function [3, V) -> [3, V) (not injective: chains started from different tokens
    merge, which is what makes n-grams recur across requests)"""
    import torch
    t = torch.arange(vocab, dtype=torch.int32)
    h = _hash32(t, torch.tensor(seed, dtype=torch.int32)).to(torch.int64) & 0x7FFFFFFF
    return (3 + h % (vocab - 3)).to(torch.int64)


def synth_fill(model, cfg, seed=0, embed_std=None):
    """the benchmark's weights, identical on every device and in every arm (HF parameter names): norms = 1, decoder
    weights ~ U(std 0.02), embedding ~ U(std embed_std), lm_head row v = LM_SCALE * sum of the unit embeddings of the
    tokens t with succ(t) = v (hashed N(0, 0.02^2) for tokens without a predecessor)"""
    import torch
    embed_std = EMBED_STD if embed_std is None else embed_std
    emb = lm = None
    with torch.no_grad():
        for name, p in model.named_parameters():
            pseed = zlib.crc32(name.encode()) ^ (seed * 7919)
            if name.endswith('norm.weight') or name.endswith('layernorm.weight'):
                p.fill_(1.0)
            elif name.endswith('embed_tokens.weight'):
                hashed_normal_(p.data, pseed, embed_std)
                emb = p
            else:
                hashed_normal_(p.data, pseed, 0.02)
                if name.endswith('lm_head.weight'):
                    lm = p
        V = emb.shape[0]
        succ = successor_map(V).to(emb.device)
        unit = emb.data.double()
        unit = unit / unit.norm(dim=1, keepdim=True).clamp_min(1e-30)
        acc = torch.zeros_like(unit)
        acc.index_add_(0, succ[3:], unit[3:])          # float64: the order of the (few) addends cannot reach bf16
        has = torch.zeros((V,), dtype=torch.bool, device=emb.device)
        has[succ[3:]] = True
        lm.data[has] = (acc[has] * LM_SCALE).to(lm.dtype)
    return model


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region (B200_PROFILING.md clocks line), via NVML"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: 'hw_slowdown',
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: 'hw_thermal_slowdown',
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: 'sw_thermal_slowdown',
                     nv.nvmlClocksThrottleReasonSwPowerCap: 'sw_power_cap',
                     nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: 'hw_power_brake'}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.1)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f'nvml_unavailable:{type(e).__name__}')

    def summary(self):
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons)}


def peaks():
    """(HBM GB/s, dense bf16 TFLOP/s, source): the pool's measured numbers (MEASURED_PEAKS.json, driver-written) or the
    fallback B200_PROFILING.md states"""
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    try:
        d = json.load(open(p))
        return float(d['hbm_gbs']), float(d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1400.0))), 'measured'
    except (OSError, ValueError, KeyError, TypeError):
        return 6650.0, 1400.0, 'fallback'


def timed_requests(K, rank=0):
    """the K timed prompts: the same on every rank (identical work per replica: the aggregate scales with the hardware,
    not with which shard happens to accept longer drafts) and disjoint from the warm-up prompts"""
    return [i % 64 for i in range(K)]


# ----------------------------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from painlessinferenceacceleration_b200.common import ops
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    from painlessinferenceacceleration_b200.models.llama.modeling_llama import LlamaForCausalLM

    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)'
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    cfg, fam = make_config(args.model)
    penalty = MODELS[args.model][7]
    if fam == 'mixtral':
        from painlessinferenceacceleration_b200.models.mixtral.modeling_mixtral import MixtralForCausalLM as Cls
    else:
        Cls = LlamaForCausalLM
    model = Cls(cfg, device=dev)
    if rank == 0:
        synth_fill(model, cfg)
    if world > 1:  # the one collective of this path: weights from rank 0 over NVLink (SURVEY.md 8e)
        for p in model.parameters():
            dist.broadcast(p.data, src=0)
    model.lookahead_cache = LookaheadCache(eos_ids=[2], device=dev, vocab_capacity=cfg.vocab_size)
    K, Wm = args.steps, args.warmup
    allp = phrase_bank_prompts(64 + 8 * max(Wm, 1), cfg.vocab_size)
    timed = [allp[j] for j in timed_requests(K, rank)]
    warm = [allp[64 + i % (8 * max(Wm, 1))] for i in range(Wm)]
    dk = {'use_lookahead': True, 'decoding_length': DL, 'branch_length': BL}
    gen = dict(max_new_tokens=NEW_TOKENS, eos_token_id=2, decoding_kwargs=dk, return_dict_in_generate=True,
               repetition_penalty=penalty)
    for p in warm:  # untimed: CUDA graph capture, trie warm-up on a disjoint prompt set (benchmark.py:159-169)
        model.generate(input_ids=torch.tensor([p], device=dev), **gen)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_pass(host_io):
        ins = [torch.tensor([p]).pin_memory() if host_io else torch.tensor([p], device=dev) for p in timed]
        toks, edls, outs, last = 0, [], [], None
        l0 = ops.launch_count()
        r0 = model._rt.replays
        g0 = model._rt.graph_launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for x in ins:
            o = model.generate(input_ids=x.to(dev, non_blocking=True) if host_io else x, **gen)
            seq = o.sequences.cpu() if host_io else o.sequences
            outs.append(seq)
            last = o
            toks += seq.shape[1] - PROMPT_LEN
            edls += o.kwargs['edls'][1:]
        e1.record()
        barrier()
        ms_rank = e0.elapsed_time(e1)
        ms = ms_rank
        launches = (ops.launch_count() - l0) + (model._rt.replays - r0) * model._rt.kernels_per_graph + \
            (model._rt.graph_launches - g0)
        per_rank = [ms_rank]
        if world > 1:
            allms = [torch.zeros((1,), device=dev) for _ in range(world)]
            dist.all_gather(allms, torch.tensor([ms_rank], device=dev))
            per_rank = [float(t) for t in allms]
            ms = max(per_rank)
            agg = torch.tensor([float(toks), float(sum(edls)), float(len(edls)), float(launches)], device=dev)
            dist.all_reduce(agg)
            toks, s_e, n_e, launches = (float(v) for v in agg)
        else:
            s_e, n_e = float(sum(edls)), float(len(edls))
        return dict(ms=ms, tokens=toks, mean_edl=s_e / max(n_e, 1), steps=n_e, launches=int(launches), outs=outs,
                    per_rank_ms=per_rank, last=last)

    trie = model.lookahead_cache
    snap = trie.snapshot()              # the trie after the disjoint warm-up: both timed passes start from it
    sampler = ClockSampler(local)
    sampler.start()
    res = timed_pass(host_io=False)     # headline: first pass over prompts the trie has never seen
    trie.restore(snap)
    e2e = timed_pass(host_io=True)      # the same pass through host buffers, from the same trie state
    second = timed_pass(host_io=False)  # second pass: the trie has seen every answer once (the round-1 headline regime)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    my_clk = sampler.summary()          # every rank samples its own GPU; rank 0 prints them all
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res['last'])
    per_rank_clocks = [dict(my_clk, n_throttle_reasons=len(my_clk['reasons']))]
    if world > 1:
        t = torch.tensor([my_clk['sm_mhz'] or 0, my_clk['sm_max_mhz'] or 0, len(my_clk['reasons'])], device=dev)
        allc = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allc, t)
        per_rank_clocks = [{'sm_mhz': int(c[0]), 'sm_max_mhz': int(c[1]), 'n_throttle_reasons': int(c[2])} for c in allc]
    same_tokens = all(torch.equal(a.cpu(), b.cpu()) for a, b in zip(res['outs'], e2e['outs']))
    extra = {}
    if rank == 0:
        extra['roofline'] = gemm_roofline(model, dev)
        extra['roofline_attention'] = attention_roofline(model, dev)
        extra['roofline_attention_long_context'] = attention_roofline_long(dev)
        extra['roofline_trie_get'] = trie_roofline(dev)
        extra['trie_counters'] = trie_counters(dev)
        if world == 1 and fam != 'mixtral' and not args.no_batched:
            extra['batched'] = batched_line(args, cfg, model, dev, allp)
        if world == 1 and not args.no_cpu_baseline:
            extra['cpu_baseline'] = cpu_baseline(args, cfg, model, dev, allp)
    if rank == 0:
        hbm, _tf, src = peaks()
        step_ms = res['ms'] / max(res['steps'] / world, 1)
        wbytes = weight_bytes_per_step(model)
        line = {
            'metric': metric_name(args.model),
            'value': res['tokens'] / (res['ms'] / 1e3), 'unit': 'tokens/s', 'n_gpus': world, 'steps': K, 'warmup': Wm,
            'ms_per_step': res['ms'] / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'bf16', 'data': 'synthetic (phrase-bank prompts; hashed weights of the named shape whose greedy '
                                     'decoding is a noisy first-order chain, identical in the GPU and CPU arms)',
            'mean_accepted_len_per_step': res['mean_edl'], 'verify_steps': res['steps'],
            'ms_per_verify_step': step_ms,
            'second_epoch': {'value': second['tokens'] / (second['ms'] / 1e3), 'unit': 'tokens/s',
                             'mean_accepted_len_per_step': second['mean_edl'], 'verify_steps': second['steps'],
                             'ms_per_verify_step': second['ms'] / max(second['steps'] / world, 1)},
            'config': workload_config(args, world, src),
            'clocks': sampler.summary(),
            'per_rank_ms': res['per_rank_ms'],
            'per_rank_clocks': per_rank_clocks,
            'e2e': {'value': e2e['tokens'] / (e2e['ms'] / 1e3), 'unit': 'tokens/s',
                    'h2d_bytes_per_step': PROMPT_LEN * 8,
                    'd2h_bytes_per_step': int((PROMPT_LEN + NEW_TOKENS) * 8 + (e2e['steps'] / max(K * world, 1)) * 4 * (5 + DL)),
                    'mean_accepted_len_per_step': e2e['mean_edl'], 'verify_steps': e2e['steps'],
                    'ms_per_verify_step': e2e['ms'] / max(e2e['steps'] / world, 1),
                    'same_trie_state_as_value': True, 'same_tokens_as_value': bool(same_tokens)},
            'gpu_launches': res['launches'],
            'roofline_step': {'bound': 'hbm', 'bytes_per_step': wbytes, 'ms_per_step': step_ms,
                              'achieved': wbytes / (step_ms * 1e-3) / 1e9, 'peak': hbm, 'unit': 'GB/s',
                              'frac': wbytes / (step_ms * 1e-3) / 1e9 / hbm,
                              'note': 'decoder + lm_head weight bytes streamed by one verify step / measured time per '
                                      'verify step (host gaps, prefill and trie work included)'},
        }
        line.update(extra)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(d, o):
    """--dump-outputs: what generate() returned for the last request of the headline timed pass, as DIR/<name>.npy
    (float64, exact for these integers): the token ids (prompt + generated) and the per-step draft / accepted lengths.
    Prompts and weights are pure functions of the arguments, so two builds can be compared file by file."""
    os.makedirs(d, exist_ok=True)
    for name, v in (('sequences', o.sequences.cpu().numpy()), ('dls', o.kwargs['dls']), ('edls', o.kwargs['edls'])):
        np.save(os.path.join(d, f'{name}.npy'), np.asarray(v, dtype=np.float64))


def workload_config(args, world, peaks_src):
    penalty = MODELS[args.model][7]
    return {'workload': f'{args.model} bf16, greedy, {DL}-token/{BL}-branch trie draft, {PROMPT_LEN}-token prompt -> '
                        f'{NEW_TOKENS} new tokens, repetition_penalty {penalty}, 1 request per step per GPU',
            'l2': 'inputs larger than L2: every verify step streams the full weight set (>= 13 GB) and the KV cache of '
                  'all layers',
            'trie': 'warmed by the untimed warm-up requests on OTHER prompts only; value and e2e both start from that '
                    'trie state (snapshot / restore), second_epoch = a later pass that has seen each answer once',
            'weights': f'synth_fill: decoder N(0,0.02^2) hashed, embedding std {EMBED_STD}, successor lm_head x{LM_SCALE}',
            'parallelism': f'{world} independent replicas, identical requests on every replica' if world > 1 else 'single GPU',
            'peaks': peaks_src}


def weight_bytes_per_step(model):
    """algorithmic HBM bytes of one verify step: every decoder / lm_head weight once (the embedding is gathered)"""
    n = 0
    for name, p in model.named_parameters():
        if 'embed_tokens' in name:
            continue
        n += p.numel() * p.element_size()
    return n


def ncu_traffic(prefix, kernel):
    """DRAM bytes (read + written) per launch of `kernel` from the newest committed `ncu --set full` summary whose
    capture name starts with `prefix` (profiles/*_traffic.json, written by scripts/summarize_profiles.py); None when
    there is no such capture"""
    import glob
    for f in sorted(glob.glob(os.path.join(ROOT, 'profiles', '*_traffic.json')), reverse=True):
        try:
            for k, v in json.load(open(f)).items():
                name, _, kern = k.partition(':')
                if name.startswith(prefix) and kernel in kern:
                    return float(v)
        except (OSError, ValueError):
            continue
    return None


def _graph_time(fn, reps=20):
    """microseconds per replay of fn captured as a CUDA graph (so that the host launch path does not bound it)"""
    import torch
    fn()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fn()
    graph.replay()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps


def gemm_roofline(model, dev):
    """the step's dominant kernel by the committed launch list (profiles/*_launches.md): k_gemm_ws on the fused
    gate/up projection.  All layers' plans in turn (their weights together exceed L2, so every launch streams cold
    HBM), CUDA events around graph replays; algorithmic bytes = the weight once + the 64 activation rows + the output"""
    rt = model._rt
    plans = getattr(rt, 'gemm_plans', None)
    if not plans:
        return None
    key = 'gate_up_silu' if any('gate_up_silu' in p for p in plans['layers']) else 'gate_up'
    lp = [p for p in plans['layers'] if key in p]
    if not lp:
        return None
    b = rt.decode_bufs
    out = b.act if key == 'gate_up_silu' else b.gu   # the fused epilogue writes SiLU(gate) * up [64, N/2] directly

    def sweep():
        for p in lp:
            p[key].run(64, out=out)

    us = _graph_time(sweep) / len(lp)
    N, Kd = lp[0][key].N, b.y.shape[1]
    by = N * Kd * 2 + 64 * Kd * 2 + 64 * out.shape[1] * 2
    hbm, _tf, src = peaks()
    ach = by / (us * 1e-6) / 1e9
    return {'kernel': 'k_gemm_ws<4> (gate_up projection' + (' + SiLU*up epilogue' if key == 'gate_up_silu' else '') + ', one layer)', 'bound': 'hbm', 'achieved': ach, 'peak': hbm,
            'unit': 'GB/s', 'frac': ach / hbm, 'traffic': ncu_traffic('prof_gemm_ws', 'k_gemm_ws'),
            'bytes_per_launch': by, 'us_per_launch': us, 'shape': f'Y[64,{N}] = X[64,{Kd}] W[{N},{Kd}]^T',
            'peak_source': src}


def attention_roofline(model, dev):
    """k_tree_attn alone at the benchmark shape: 64 draft rows, prefix ~ mid-generation, all layers in turn (the
    layers' KV planes together exceed L2, so every launch reads cold HBM).  CUDA events on the launch stream."""
    rt = model._rt
    g = rt.g
    P, n = PROMPT_LEN + NEW_TOKENS // 2, DL
    rt.n.fill_(n)
    rt.prefix_len.fill_(P)
    rt.pad.zero_()
    rt.mask.copy_(rt.chain)
    L = P + n

    def sweep():
        for li in range(g['n_layers']):
            rt.plan.forward(li, rt.q, rt.mask, rt.decode_bufs.slots, rt.attn)

    us = _graph_time(sweep) / g['n_layers']
    # algorithmic bytes per launch (SURVEY.md 8d): K,V rows of every KV head + Q read + O write
    by = 2 * L * g['n_kv_heads'] * g['head_dim'] * 2 + 2 * n * g['n_q_heads'] * g['head_dim'] * 2
    fl = 4.0 * n * L * g['head_dim'] * g['n_q_heads']
    hbm, tf, src = peaks()
    ach = by / (us * 1e-6) / 1e9
    return {'kernel': 'k_tree_attn (one layer)', 'bound': 'hbm', 'achieved': ach, 'peak': hbm,
            'unit': 'GB/s', 'frac': ach / hbm, 'traffic': ncu_traffic('prof_attn_gqa_r' if g['n_kv_heads'] != g['n_q_heads'] else 'prof_attn_short', 'k_tree_attn'),
            'bytes_per_launch': by, 'us_per_launch': us, 'tensor_tflops': fl / (us * 1e-6) / 1e12,
            'tensor_frac': fl / (us * 1e-6) / 1e12 / tf,
            'shape': f'n={n} P={P} Hq={g["n_q_heads"]} Hkv={g["n_kv_heads"]} D={g["head_dim"]}', 'peak_source': src}


def attention_roofline_long(dev, P=3968, n=DL, hq=32, hkv=32, layers=4):
    """the same kernel where it is bandwidth- rather than latency-bound: a 4 k-token context (32 KV tiles per head, KV
    planes of the 4 layers = 270 MB > L2), stand-alone plan, CUDA-graph replay"""
    import torch
    from painlessinferenceacceleration_b200.common import ops
    D, R = 128, 64
    max_seq = P + n + 64
    kc = (torch.randn((layers, hkv, max_seq, D), device=dev) * 0.5).to(torch.bfloat16)
    vc = (torch.randn((layers, hkv, max_seq, D), device=dev) * 0.5).to(torch.bfloat16)
    q = (torch.randn((R, hq, D), device=dev) * 0.5).to(torch.bfloat16)
    out = torch.zeros_like(q)
    plan = ops.AttnPlan(kc, vc, hq, hkv, D, R)
    rows = np.array([(1 << (i + 1)) - 1 if i < 63 else 0xFFFFFFFFFFFFFFFF for i in range(R)], dtype=np.uint64)
    mask = torch.from_numpy(rows.view(np.int64)).to(dev).view(R, 1)
    slots = ops.Slots(torch.tensor([n], dtype=torch.int32, device=dev), torch.tensor([P], dtype=torch.int32, device=dev),
                      None, R)

    def sweep():
        for li in range(layers):
            plan.forward(li, q, mask, slots, out)

    us = _graph_time(sweep) / layers
    L = P + n
    by = 2 * L * hkv * D * 2 + 2 * n * hq * D * 2
    hbm, _tf, src = peaks()
    ach = by / (us * 1e-6) / 1e9
    return {'kernel': 'k_tree_attn (one layer, long context)', 'bound': 'hbm', 'achieved': ach, 'peak': hbm, 'unit': 'GB/s',
            'frac': ach / hbm, 'traffic': ncu_traffic('prof_attn_long', 'k_tree_attn') if P > 2000 else None,
            'bytes_per_launch': by, 'us_per_launch': us,
            'shape': f'n={n} P={P} Hq={hq} Hkv={hkv} D={D}', 'peak_source': src}


def _forest(dev, n_docs, full_walk=False):
    """full_walk: a handle whose queries visit the whole matched subtree like the reference (PIA_TRIE_PRUNE=0 is read
    when the handle is created) - used once to count the algorithmic bytes of the scan"""
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    old = os.environ.get('PIA_TRIE_PRUNE')
    if full_walk:
        os.environ['PIA_TRIE_PRUNE'] = '0'
    try:
        c = LookaheadCache(eos_ids=[2], device=dev, vocab_capacity=32000, node_capacity=1 << 23,
                           max_resident_queries=592)
    finally:
        if full_walk:
            if old is None:
                del os.environ['PIA_TRIE_PRUNE']
            else:
                os.environ['PIA_TRIE_PRUNE'] = old
    docs = phrase_bank_prompts(n_docs, 32000, length=256, seed=7)
    for d in docs:
        c.put(d, branch_length=9, mode='output', idx=-1)
    return c, docs


def trie_roofline(dev, n_docs=1500, n_queries=4096):
    """batched synthetic scan of SURVEY.md 8d: forest grown from phrase-bank documents, 4096 concurrent hier_get
    queries.  ALGORITHMIC bytes (SURVEY 8d: matched subtree x node record) = node records (32 B) + child entries
    (8 B) the reference's full walk of every matched subtree visits, counted by the kernel on a handle with the pruned
    walk switched off; `bytes_visited_per_launch` is what the timed (pruned) kernel really read."""
    import torch
    from painlessinferenceacceleration_b200 import _lib as L
    c, docs = _forest(dev, n_docs)
    rng = np.random.default_rng(8)
    qs = []
    for _ in range(n_queries):
        d = docs[int(rng.integers(0, len(docs)))]
        j = int(rng.integers(0, len(d) - 2))
        qs.append(d[j:j + 2])
    t = c._t
    dq = torch.tensor(qs, dtype=torch.int32, device=dev)
    dl = torch.full((n_queries,), 2, dtype=torch.int32, device=dev)
    o = t.out_buffers(n_queries, 64)

    def launch(t=t):
        L.check(t.lib.pia_trie_get(t.h, dq.data_ptr(), dl.data_ptr(), n_queries, 2, 2, None, 0, 64, 8, 0, 32,
                                   L.MODE['mix'], L.GET_HIER, 0, 0, None, o['ids'].data_ptr(), o['mask'].data_ptr(),
                                   o['n'].data_ptr(), o['sizes'].data_ptr(), o['nsizes'].data_ptr(),
                                   o['status'].data_ptr(), t.stream()))

    flush = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)
    launch()
    s0 = c.stats()
    times = []
    for _ in range(5):
        flush.fill_(1)  # L2 flush between timed launches (forest < L2)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        launch()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    s1 = c.stats()
    ms = float(np.median(times))
    out_bytes = n_queries * (64 * 4 + 64 * 8)
    visited = ((s1['nodes_visited'] - s0['nodes_visited']) * 32 + (s1['edges_visited'] - s0['edges_visited']) * 8) / 5.0
    visited += out_bytes
    mean_draft = float(o['n'].float().mean())
    ids_pruned = o['ids'].clone()
    n_pruned = o['n'].clone()
    del c
    cf, _ = _forest(dev, n_docs, full_walk=True)   # same forest, full walks: the algorithmic byte count (untimed)
    f0 = cf.stats()
    launch(cf._t)
    torch.cuda.synchronize()
    f1 = cf.stats()
    by = (f1['nodes_visited'] - f0['nodes_visited']) * 32 + (f1['edges_visited'] - f0['edges_visited']) * 8 + out_bytes
    same = bool(torch.equal(n_pruned, o['n']) and torch.equal(ids_pruned, o['ids']))
    hbm, _tf, src = peaks()
    ach = by / (ms * 1e-3) / 1e9
    return {'kernel': 'k_get<64,16> (4096 hier_get rows)', 'bound': 'hbm', 'achieved': ach, 'peak': hbm, 'unit': 'GB/s',
            'frac': ach / hbm, 'traffic': ncu_traffic('prof_trie_batch', 'k_get'), 'bytes_per_launch': by,
            'bytes_visited_per_launch': visited, 'achieved_on_visited_bytes': visited / (ms * 1e-3) / 1e9,
            'pruned_walk_equals_full_walk': same, 'ms_per_launch': ms, 'us_per_get': ms * 1e3 / n_queries,
            'forest_nodes': s1['nodes_used'], 'mean_draft': mean_draft, 'peak_source': src}


def trie_counters(dev, n_docs=200, n_ops=200):
    """perf_check_trie-style counters (benchmarks/benchmark.py:353-395): microseconds per get / stream_put / prompt put
    through the LookaheadCache API (host call, kernel, result back on the host), next to the same ops on the CPU trie
    restatement (oracle, 1 thread)"""
    import torch
    c, docs = _forest(dev, n_docs)
    rng = np.random.default_rng(9)
    qs = [docs[int(rng.integers(0, n_docs))][j:j + 2] for j in rng.integers(0, 250, size=n_ops).tolist()]
    out = {}

    def timeit(fn, n):
        torch.cuda.synchronize()
        t0 = time.time()
        for i in range(n):
            fn(i)
        torch.cuda.synchronize()
        return (time.time() - t0) / n * 1e6

    c.hier_get(qs[0], decoding_length=DL, branch_length=BL, min_output_size=DL // 2)
    out['gpu_us_per_hier_get'] = timeit(lambda i: c.hier_get(qs[i], decoding_length=DL, branch_length=BL,
                                                             min_output_size=DL // 2), n_ops)
    out['gpu_us_per_stream_put_4'] = timeit(lambda i: c.stream_put(docs[i % n_docs][8:12], branch_length=BL + 1), n_ops)
    out['gpu_us_per_prompt_put_256'] = timeit(lambda i: c.put(docs[i % n_docs], branch_length=BL + 1, mode='input', idx=0), 50)
    out['forest_nodes'] = c.stats()['nodes_used']
    try:
        from oracle.trie import OracleLookaheadCache
        o = OracleLookaheadCache(eos_ids=[2])
        for d in docs:
            o.put(d, branch_length=9, mode='output', idx=-1)

        def cput(fn, n):
            t0 = time.time()
            for i in range(n):
                fn(i)
            return (time.time() - t0) / n * 1e6

        out['cpu_port_us_per_hier_get'] = cput(lambda i: o.hier_get(qs[i], decoding_length=DL, branch_length=BL,
                                                                    min_output_size=DL // 2), n_ops)
        out['cpu_port_us_per_stream_put_4'] = cput(lambda i: o.stream_put(docs[i % n_docs][8:12], branch_length=BL + 1), n_ops)
        out['cpu_port_us_per_prompt_put_256'] = cput(lambda i: o.put(docs[i % n_docs], branch_length=BL + 1, mode='input', idx=0), 50)
        out['cpu_kind'] = 'port (oracle/trie_oracle.c, 1 thread); the Python reference measured 1.5-12 ms per get (BASELINE.md 2)'
    except Exception as e:  # pragma: no cover
        out['cpu_port_error'] = f'{type(e).__name__}: {e}'
    return out


def batched_line(args, cfg, model, dev, allp, bs=8):
    """BASELINE config 5's "batch=8/GPU" served as a true batch (common/pretrained_model_batch.py): 8 requests share
    the 64 draft rows of one verify step.  Two draft shares: 'reference' = decoding_length // active // active (what the
    reference's bat_get computes: 1 node per request at 8 requests, i.e. batched plain decoding) and 'rows' =
    decoding_length // active.  Same weights (the batch class shares the parameters), fresh trie warmed like the
    headline run."""
    import torch
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    from painlessinferenceacceleration_b200.models.llama.modeling_llama_batch import LlamaForCausalLM as BatchCls
    bm = BatchCls(cfg, device=dev)
    for (n1, p1), (n2, p2) in zip(bm.named_parameters(), model.named_parameters()):
        assert n1 == n2
        p1.data = p2.data
    bm._tiled_weights = getattr(model, '_tiled_weights', {})
    penalty = MODELS[args.model][7]
    out = {}
    for mode in ('rows', 'reference'):
        bm.lookahead_cache = LookaheadCache(eos_ids=[2], device=dev, vocab_capacity=cfg.vocab_size, n_input_slots=bs)
        dk = {'use_lookahead': True, 'decoding_length': DL, 'branch_length': BL, 'batch_share': mode}
        gen = dict(max_new_tokens=NEW_TOKENS, eos_token_id=2, decoding_kwargs=dk, return_dict_in_generate=True,
                   repetition_penalty=penalty)
        warm = torch.tensor(allp[64:64 + bs], device=dev)
        bm.generate(input_ids=warm, **gen)                     # untimed: graphs + trie warm-up on other prompts
        bm.generate(input_ids=warm, **dict(gen, max_new_tokens=2))   # untimed: the second pass of a runtime captures the prefill graphs
        ids = torch.tensor(allp[:bs], device=dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        o = bm.generate(input_ids=ids, **gen)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        toks = sum(o.kwargs['lengths']) - bs * PROMPT_LEN
        edls = o.kwargs['edls'][bs:]
        out[mode] = {'value': toks / (ms / 1e3), 'unit': 'tokens/s', 'batch': bs, 'tokens': toks, 'ms': ms,
                     'mean_accepted_len_per_request_step': float(np.mean(edls)) if edls else None}
    bm._rt = None
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------- CPU arms
def build_cpu_model(name):
    """HF eager model of the named shape on the host, bf16, the SAME synthetic weights as the GPU arm"""
    import torch
    from transformers import AutoModelForCausalLM
    cfg, _ = make_config(name)
    cfg._attn_implementation = 'eager'
    with torch.device('meta'):
        m = AutoModelForCausalLM.from_config(cfg, attn_implementation='eager', dtype=torch.bfloat16)
    m = m.to_empty(device='cpu')
    synth_fill(m, cfg)
    with torch.no_grad():
        for n_, b in m.named_buffers():
            if 'inv_freq' in n_:
                hd = cfg.hidden_size // cfg.num_attention_heads
                b.copy_(1.0 / (10000.0 ** (torch.arange(0, hd, 2).float() / hd)))
    return m.eval()


def cpu_threads():
    """host threads for the CPU arms: small-row GEMMs stop scaling (and then degrade) beyond a few dozen threads"""
    return max(1, min(os.cpu_count() or 1, 32))


def cpu_request(model, trie, prompt, penalty, new_tokens=CPU_NEW_TOKENS):
    """one request of the fixed CPU sample through the oracle loop (oracle/loop.py = the reference's CPU path restated):
    the full 256-token prompt, `new_tokens` generated tokens"""
    import torch
    from oracle.loop import lookahead_generate
    t0 = time.time()
    r = lookahead_generate(model, trie, torch.tensor([prompt]), max_new_tokens=new_tokens, eos_token_id=[2],
                           decoding_length=DL, branch_length=BL, repetition_penalty=penalty)
    return dict(tokens=r['sequences'][0, len(prompt):].tolist(), seconds=time.time() - t0, edls=r['edls'], dls=r['dls'],
                fts=r['fts'])


CPU_SAMPLE = ('{n} requests of the SAME workload cut to a fixed size: the full {p}-token prompt (prefill included) + '
              '{g} generated tokens each, 64/8 drafts, same synthetic weights and prompts as the GPU arm, trie warmed by '
              '{w} such requests on other prompts; oracle/loop.py + the C restatement of the trie over the installed HF '
              'eager bf16 model, {t} host threads')


def cpu_baseline(args, cfg, model, dev, allp, n_req=2):
    """rank 0, N=1: the CPU port on a bounded, fixed sample, and the cross-check BASELINE.md 3 promised: the same
    requests through the GPU path from the same (fresh) trie state must give the same tokens and the same accepted
    lengths (identical weights; bf16 near-ties are reported, not hidden)"""
    import torch
    from oracle.trie import OracleLookaheadCache
    from painlessinferenceacceleration_b200.common.lookahead_cache import LookaheadCache
    penalty = MODELS[args.model][7]
    threads = cpu_threads()
    torch.set_num_threads(threads)
    t0 = time.time()
    cpu_model = build_cpu_model(args.model)
    build_s = time.time() - t0
    ctrie = OracleLookaheadCache(eos_ids=[2])
    saved = model.lookahead_cache
    model.lookahead_cache = LookaheadCache(eos_ids=[2], device=dev, vocab_capacity=cfg.vocab_size)
    rows, secs, toks, edls = [], 0.0, 0, []
    try:
        for rep in range(2):   # the second pass drafts the first pass's answers: multi-token accepts on both sides
            for i in range(n_req):
                c = cpu_request(cpu_model, ctrie, allp[i], penalty)
                g = model.generate(input_ids=torch.tensor([allp[i]], device=dev), max_new_tokens=CPU_NEW_TOKENS,
                                   eos_token_id=2, repetition_penalty=penalty, return_dict_in_generate=True,
                                   decoding_kwargs={'use_lookahead': True, 'decoding_length': DL, 'branch_length': BL})
                gt = g.sequences[0, PROMPT_LEN:].tolist()
                same = gt == c['tokens']
                rows.append({'request': i, 'pass': rep, 'tokens_equal': same,
                             'edls_equal': bool(same and g.kwargs['edls'] == c['edls']),
                             'cpu_edl': float(np.mean(c['edls'][1:])) if len(c['edls']) > 1 else None,
                             'gpu_edl': float(np.mean(g.kwargs['edls'][1:])) if len(g.kwargs['edls']) > 1 else None})
                secs += c['seconds']
                toks += len(c['tokens'])
                edls += c['edls'][1:]
                if not same:  # a bf16 near-tie: the texts (and so the tries) part ways, resync both
                    ctrie.fresh()
                    model.lookahead_cache.fresh()
    finally:
        model.lookahead_cache = saved
    return {'value': toks / secs, 'unit': 'tokens/s', 'cores': threads, 'kind': 'port',
            'sample': CPU_SAMPLE.format(n=2 * n_req, p=PROMPT_LEN, g=CPU_NEW_TOKENS, w=0, t=threads)
            + f' (2 passes over {n_req} prompts from a fresh trie); {toks} tokens in {secs:.1f}s, model build {build_s:.0f}s untimed',
            'mean_accepted_len_per_step': float(np.mean(edls)) if edls else None,
            'cross_check_vs_gpu': {'requests': rows, 'all_tokens_equal': all(r['tokens_equal'] for r in rows),
                                   'edl_equal_where_tokens_equal': all(r['edls_equal'] for r in rows if r['tokens_equal'])}}


def run_reference(args):
    """--impl reference: the reference's own CPU path (restated: oracle/loop.py over the installed HF eager model +
    the C restatement of its trie) on the host cores; rank 0 only.  FIXED sample, independent of the host's speed:
    every step = one request with the full 256-token prompt and CPU_NEW_TOKENS generated tokens; warm-up = the same on
    the warm-up prompts.  Same metric / config / weights / prompts as the GPU arm."""
    import torch
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    from oracle.trie import OracleLookaheadCache
    threads = cpu_threads()
    torch.set_num_threads(threads)
    cfg, _ = make_config(args.model)
    penalty = MODELS[args.model][7]
    model = build_cpu_model(args.model)
    trie = OracleLookaheadCache(eos_ids=[2])
    K, Wm = args.steps, args.warmup
    allp = phrase_bank_prompts(64 + 8 * max(Wm, 1), cfg.vocab_size)
    for i in range(Wm):
        cpu_request(model, trie, allp[64 + i % (8 * max(Wm, 1))], penalty)
    samples = [cpu_request(model, trie, allp[j], penalty) for j in timed_requests(K)]
    toks = sum(len(s['tokens']) for s in samples)
    secs = sum(s['seconds'] for s in samples)
    edls = [e for s in samples for e in s['edls'][1:]]
    pre = float(np.mean([s['fts'][0] for s in samples]))
    ver = [t for s in samples for t in s['fts'][1:]]
    v = toks / secs
    sample = CPU_SAMPLE.format(n=K, p=PROMPT_LEN, g=CPU_NEW_TOKENS, w=Wm, t=threads) + f'; {toks} tokens in {secs:.0f}s'
    cpu = {'value': v, 'unit': 'tokens/s', 'cores': threads, 'kind': 'port', 'sample': sample,
           'prefill_s': pre, 'verify_step_s': float(np.mean(ver)) if ver else None,
           'full_request_tokens_per_s_extrapolated':
               (NEW_TOKENS / (pre + NEW_TOKENS / float(np.mean(edls)) * float(np.mean(ver)))) if ver and edls else None}
    print(json.dumps({
        'impl': 'reference', 'metric': metric_name(args.model),
        'value': v, 'unit': 'tokens/s', 'n_gpus': args.gpus, 'steps': K, 'warmup': Wm,
        'ms_per_step': secs / len(samples) * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'bf16', 'data': 'synthetic (phrase-bank prompts; hashed weights of the named shape whose greedy '
                                 'decoding is a noisy first-order chain, identical in the GPU and CPU arms)',
        'mean_accepted_len_per_step': float(np.mean(edls)) if edls else None,
        'config': workload_config(args, args.gpus, peaks()[2]),
        'cpu_baseline': cpu,
        'e2e': {'value': v, 'unit': 'tokens/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=8)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--model', default='llama2-7b', choices=sorted(MODELS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-batched', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the last timed request\'s outputs to DIR/<name>.npy')
    a = ap.parse_args()
    if a.dump_outputs and a.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl ours)')
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
