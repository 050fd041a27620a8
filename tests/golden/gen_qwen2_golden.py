# -*- coding: utf-8 -*-
"""Generates tests/golden/qwen2loop_*.npz by running the REFERENCE'S OWN loop code (tests/golden/ref_loop.py: the
unmodified loop functions of the reference's common/pretrained_model.py + the live reference trie) around the installed
Hugging Face Qwen2ForCausalLM (tests/tiny_qwen2.py: q/k/v biases, rope_theta 1e6, 7 or 6 query heads per KV head).
The reference's Qwen2 lookahead patch (models/qwen2/modeling_qwen2.py:997-1000) is Llama's, which is what ref_loop's
forward applies.  Needs the reference checkout, so it runs where that exists:

    python tests/golden/gen_qwen2_golden.py

Layout as gen_loop_golden.py's loop_*.npz (tests/loop_golden.step_logits / step_mask apply); the files are named
outside the loop_* glob so that the replay tests parametrised over loop_*.npz keep their case list."""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from tests.golden.gen_loop_golden import logits_bits, mask_rows  # noqa: E402
from tests.golden.ref_loop import import_reference, make_driver, run_reference_request  # noqa: E402
from tests.tiny_models import prompts  # noqa: E402
from tests.tiny_qwen2 import qwen2_hf_model  # noqa: E402


def scenario(name, shape, seed, vocab, requests, dl=64, bl=8, reps=2, **gen):
    _pm, _pmb, LookaheadCache = import_reference()
    torch.set_num_threads(4)
    hf = qwen2_hf_model(shape, seed=seed, dtype=torch.bfloat16, vocab=vocab)
    rec = []
    drv = make_driver(hf, LookaheadCache(), rec)
    reqs, arrays = [], {}
    for rep in range(reps):
        for q in requests:
            s0 = len(rec)
            r = run_reference_request(drv, q['prompt'], q['max_new_tokens'], decoding_length=dl, branch_length=bl, **gen)
            steps = []
            for si in range(s0, len(rec)):
                st = rec[si]
                key = f'logits_{si}'
                arrays[key] = logits_bits(st['logits'])
                steps.append(dict(context_len=len(st['context']), decoding_ids=[int(x) for x in st['decoding_ids']],
                                  mask=None if st['decoding_masks'] is None else [str(v) for v in mask_rows(st['decoding_masks'])],
                                  logits=key, tokens=[int(x) for x in st['tokens']], dl=int(st['dl']), edl=int(st['edl']),
                                  kv=st['kv']))
            reqs.append(dict(prompt=q['prompt'][0].tolist(), max_new_tokens=q['max_new_tokens'], attention_mask=None,
                             sequences=r['sequences'], dls=r['dls'], edls=r['edls'], steps=steps))
    meta = dict(name=name, family='qwen2', shape=shape, dtype='bfloat16', model_seed=seed, vocab=vocab,
                decoding_length=dl, branch_length=bl, gen=gen, requests=reqs)
    arrays['meta'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
    path = os.path.join(HERE, f'qwen2loop_{name}.npz')
    np.savez_compressed(path, **arrays)
    edl = [e for r in reqs for e in r['edls'][1:]]
    print(f'{name}: {len(reqs)} requests, {len(rec)} steps, mean edl {np.mean(edl):.2f}, max edl {max(edl)}, '
          f'edls of the last request {reqs[-1]["edls"]}, {os.path.getsize(path) // 1024} KB')


def main():
    V = 96
    scenario('g7_bf16', 'g7', 2, V, [dict(prompt=p, max_new_tokens=36) for p in prompts(41, 3, 24, V)])
    scenario('g7_bf16_rp11', 'g7', 3, V, [dict(prompt=p, max_new_tokens=32) for p in prompts(42, 3, 20, V)],
             repetition_penalty=1.1)
    scenario('g6_tied_bf16', 'g6_tied', 4, V, [dict(prompt=p, max_new_tokens=32) for p in prompts(43, 3, 20, V)])


if __name__ == '__main__':
    main()
