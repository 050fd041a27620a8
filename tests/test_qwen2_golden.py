# -*- coding: utf-8 -*-
"""oracle/loop.py against the reference's own loop run on HF Qwen2 models (tests/golden/qwen2loop_*.npz,
gen_qwen2_golden.py): the recorded logits are replayed step by step, and the drafts, accepted tokens, kv_idx, dls and
edls must be the reference's.  The G = 7 and tied G = 6 models, with and without repetition_penalty."""
import pytest
import torch

from oracle.loop import lookahead_generate
from oracle.trie import OracleLookaheadCache
from tests.test_loop_golden import ReplayBackend
from tests.tiny_qwen2 import golden_names, load_golden


def test_the_qwen2_goldens_exist():
    assert golden_names() == ['g6_tied_bf16', 'g7_bf16', 'g7_bf16_rp11']


@pytest.mark.parametrize('name', golden_names())
def test_oracle_loop_reproduces_the_reference_loop_on_qwen2(name):
    meta, z = load_golden(name)
    pen = meta['gen'].get('repetition_penalty', 1.0)
    trie = OracleLookaheadCache(eos_ids=[2])
    n_multi = 0
    for req in meta['requests']:
        be = ReplayBackend(meta, z, req)   # asserts the draft ids / tree mask / cursor of every forward
        out = lookahead_generate(None, trie, torch.tensor([req['prompt']]), max_new_tokens=req['max_new_tokens'],
                                 eos_token_id=[2], decoding_length=meta['decoding_length'],
                                 branch_length=meta['branch_length'], repetition_penalty=pen, backend=be, trace=True)
        assert out['sequences'][0].tolist() == req['sequences']
        assert out['dls'] == req['dls'] and out['edls'] == req['edls']
        assert be.i == len(req['steps'])
        ci = 0
        for st, tr in zip(req['steps'], out['steps']):
            assert tr['tokens'] == st['tokens']
            if st['kv'] is not None:
                assert be.compactions[ci] == st['kv']['kv_idx']
                ci += 1
            n_multi += len(st['tokens']) > 1
        assert ci == len(be.compactions)
    assert n_multi >= 3   # the second pass accepts drafts
