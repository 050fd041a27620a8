# -*- coding: utf-8 -*-
"""tests/golden/count_bound_streams.npz: the data of tests/test_reference_count_bound.py, recorded from the LIVE
reference LookaheadCache (lookahead_cache.py:336) with tiny tree limits (max_node 64, max_output_node 24, so squeezes
happen).  Per case: a seeded request stream (prompt put in input mode, 1-9 stream_puts, a final stream_put that resets
the input counts and squeezes, :403-406) and, every 50 requests, a digest of the reference's whole forest
(tests/test_reference_count_bound.py forest_digest).  Run with the path of the reference's lookahead/ directory:

    python tests/golden/gen_count_bound_golden.py <reference>/lookahead
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from tests.test_reference_count_bound import (CASES, FINAL, IDXS, MAX_NODE, MAX_OUTPUT_NODE, PUT,  # noqa: E402
                                              STREAM_PUT, forest_digest)


def export(tree):
    """Tree.nodes in pre-order, children in insertion order (the layout of oracle/trie.py OracleTree.export)"""
    tok, par, freq = [], [], []

    def rec(nodes, parent):
        for t, node in nodes.items():
            r = len(tok)
            tok.append(t)
            par.append(parent)
            freq.append([node.freqs.get(k, 0.0) for k in range(-1, IDXS)])
            rec(node.children, r)
    rec(tree.nodes, -1)
    return tok, par, np.array(freq, dtype=np.float64).reshape(-1, IDXS + 1)


def main(ref):
    sys.path.insert(0, ref)
    from lookahead.common.lookahead_cache import LookaheadCache
    out = {}
    for seed, vocab, zipf in CASES:
        rng = np.random.default_rng(seed)

        def toks(k):
            if zipf:
                return np.clip(rng.zipf(1.3, size=k), 3, vocab - 1).tolist()
            return rng.integers(3, vocab, size=k).tolist()

        c = LookaheadCache(eos_ids=[2])
        c.max_node, c.max_output_node = MAX_NODE, MAX_OUTPUT_NODE
        ops, flat, digests, nodes = [], [], [], []
        for req in range(1500 if zipf else 300):
            idx = req % IDXS
            prompt = toks(int(rng.integers(4, 80)))
            c.put(prompt[1:], branch_length=9, final=False, mode='input', idx=idx)
            ops.append((PUT, len(prompt) - 1))
            flat += prompt[1:]
            for _ in range(int(rng.integers(1, 10))):
                t = toks(int(rng.integers(1, 9)))
                c.stream_put(t, branch_length=9, final=False, mode='output', idx=idx)
                ops.append((STREAM_PUT, len(t)))
                flat += t
            c.stream_put([], branch_length=9, final=True, mode='output', idx=idx)
            ops.append((FINAL, 0))
            if req % 50 == 49:
                trees = [(t, *export(tree)) for t, tree in c.mem.items()]
                digests.append(forest_digest(trees))
                nodes.append(sum(len(t[1]) for t in trees))
        out[f's{seed}_ops'] = np.array(ops, dtype=np.int32)
        out[f's{seed}_toks'] = np.array(flat, dtype=np.int16)
        out[f's{seed}_digest'] = np.array(digests)
        print(f'seed {seed}: {len(ops)} ops, {len(digests)} forests, {sum(nodes)} nodes checked')
    np.savez_compressed(os.path.join(HERE, 'count_bound_streams.npz'), **out)


if __name__ == '__main__':
    main(sys.argv[1])
