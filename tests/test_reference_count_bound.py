# -*- coding: utf-8 -*-
"""The premise of the pruned query walk (csrc/trie.cu tree_get), checked on the reference trie's forests: whatever
sequence of put / stream_put / reset_input_freqs / squeeze the reference executes, every node's counts bound its
children's (`_put` adds along root paths, lookahead_cache.py:40-56; `_squeeze` halves top-down and pops whole subtrees,
:302-310; `_reset_input_freq` zeroes top-down, :326-333).  Three seeded request streams were run through the live
reference and its whole forest hashed every 50 requests (tests/golden/gen_count_bound_golden.py); the CPU oracle
replays the streams, must reproduce each recorded forest node for node and count for count, and the bound is checked
on every node of those forests.  The CUDA trie asserts the same on its own forests in tests/test_gpu_trie.py."""
import hashlib
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'count_bound_streams.npz')
CASES = [(1, 12, False), (2, 3000, True), (3, 40, False)]
IDXS = 3                              # request slots: a node's counts are freqs[-1], freqs[0], freqs[1], freqs[2]
MAX_NODE, MAX_OUTPUT_NODE = 64, 24    # tiny limits: squeezes actually happen
PUT, STREAM_PUT, FINAL = 0, 1, 2      # op kinds of the recorded streams


def forest_digest(trees):
    """sha256 of a forest given as (tree token, node tokens, parent rows, counts) per tree, trees in token order"""
    h = hashlib.sha256()
    for token, tok, par, freq in sorted(trees, key=lambda t: t[0]):
        h.update(np.array([token, len(tok)], dtype=np.int64).tobytes())
        h.update(np.asarray(tok, dtype=np.int64).tobytes())
        h.update(np.asarray(par, dtype=np.int64).tobytes())
        h.update(np.asarray(freq, dtype=np.float64).tobytes())
    return h.hexdigest()


def _violations(par, freq):
    """(child, slot) pairs whose count exceeds the parent's; a tree's root carries no counts, its children are exempt"""
    kid = par >= 0
    return int((freq[kid] > freq[par[kid]]).sum())


@pytest.mark.parametrize('seed,vocab,zipf', CASES)
def test_reference_counts_bound_their_children(seed, vocab, zipf):
    from oracle.trie import OracleLookaheadCache
    z = np.load(GOLDEN)
    ops, toks, digests = z[f's{seed}_ops'], z[f's{seed}_toks'], z[f's{seed}_digest']
    c = OracleLookaheadCache(eos_ids=[2], max_node=MAX_NODE, max_output_node=MAX_OUTPUT_NODE)
    at, req, checks = 0, 0, 0
    for kind, n in ops.tolist():
        ids = toks[at:at + n].tolist()
        at += n
        idx = req % IDXS
        if kind == PUT:
            c.put(ids, branch_length=9, final=False, mode='input', idx=idx)
        else:
            c.stream_put(ids, branch_length=9, final=kind == FINAL, mode='output', idx=idx)
        if kind != FINAL:
            continue
        req += 1
        if req % 50 == 0:
            trees = []
            for t in range(vocab):
                tree = c.tree(t)
                if tree is not None:
                    trees.append((t, *tree.export(IDXS)))
            assert forest_digest(trees) == digests[req // 50 - 1], f'forest after request {req} differs from the reference'
            for _t, _tok, par, freq in trees:
                assert _violations(par, freq) == 0
                checks += 1
    assert at == len(toks) and req // 50 == len(digests)
    assert checks > 20
