# -*- coding: utf-8 -*-
"""ctypes face of oracle/trie_oracle.c -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / ``--impl reference`` legs may import
this module; the product package (painlessinferenceacceleration_b200) never does.

The classes keep the method names of the reference so that parity tests read like the reference's own
(`/root/reference/lookahead/lookahead/common/lookahead_cache.py`: Tree :24, LookaheadCache :336).
`par_get` (:441-488) and `bat_get` (:519-561) are host-side list/numpy logic on top of hier_get/one_get
and are restated here in Python.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, '_ref', 'libtrie_oracle.so')
_MODES = {'input': 0, 'output': 1, 'mix': 2}


def build(force=False):
    src = os.path.join(_HERE, 'trie_oracle.c')
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(['make', '-C', _HERE, '-s'] + (['-B'] if force else []))
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        ip, u64p, vp = C.POINTER(C.c_int), C.POINTER(C.c_uint64), C.c_void_p
        L.orc_tree_new.restype = vp
        L.orc_tree_new.argtypes = [C.c_int, C.c_int, C.c_int]
        L.orc_tree_free.argtypes = [vp]
        L.orc_tree_put.argtypes = [vp, ip, C.c_int, C.c_int, C.c_int]
        L.orc_tree_get.restype = C.c_int
        L.orc_tree_get.argtypes = [vp, ip, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int,
                                   ip, u64p, ip]
        L.orc_tree_get_one_branch.restype = C.c_int
        L.orc_tree_get_one_branch.argtypes = [vp, ip, C.c_int, C.c_int, C.c_int, C.c_int, ip, ip]
        L.orc_tree_squeeze.argtypes = [vp]
        L.orc_tree_reset_input_freq.argtypes = [vp, C.c_int]
        L.orc_tree_n_node.restype = C.c_long
        L.orc_tree_n_node.argtypes = [vp]
        L.orc_tree_n_output_node.restype = C.c_long
        L.orc_tree_n_output_node.argtypes = [vp]
        L.orc_tree_export.restype = C.c_long
        L.orc_tree_export.argtypes = [vp, C.c_int, C.c_long, vp, vp, vp]
        L.orc_cache_new.restype = vp
        L.orc_cache_new.argtypes = [ip, C.c_int, C.c_int, C.c_int]
        L.orc_cache_free.argtypes = [vp]
        L.orc_cache_set_eos.argtypes = [vp, ip, C.c_int]
        L.orc_cache_set_stop_words.argtypes = [vp, ip, C.c_int]
        L.orc_cache_set_limits.argtypes = [vp, C.c_int, C.c_int]
        L.orc_cache_put.argtypes = [vp, ip, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_cache_stream_put.restype = C.c_int
        L.orc_cache_stream_put.argtypes = [vp, ip, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_cache_hier_get.restype = C.c_int
        L.orc_cache_hier_get.argtypes = [vp, ip, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip,
                                         u64p, ip, ip]
        L.orc_cache_one_get.restype = C.c_int
        L.orc_cache_one_get.argtypes = [vp, ip, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip, ip, ip]
        L.orc_cache_fresh.argtypes = [vp]
        L.orc_cache_reset_input_freqs.argtypes = [vp, C.c_int]
        L.orc_cache_squeeze_branch_counts.argtypes = [vp]
        L.orc_cache_tree.restype = vp
        L.orc_cache_tree.argtypes = [vp, C.c_int]
        L.orc_cache_n_update_trees.restype = C.c_int
        L.orc_cache_n_update_trees.argtypes = [vp]
        L.orc_cache_n_update_input_trees.restype = C.c_int
        L.orc_cache_n_update_input_trees.argtypes = [vp]
        L.orc_cache_total_nodes.restype = C.c_long
        L.orc_cache_total_nodes.argtypes = [vp]
        L.orc_cache_n_trees.restype = C.c_int
        L.orc_cache_n_trees.argtypes = [vp]
        _lib = L
    return _lib


def _iarr(xs):
    xs = list(xs)
    return (C.c_int * max(len(xs), 1))(*xs), len(xs)


def bits_to_mask(words, n, W):
    """rows of W uint64 words -> np.int64 [n, n] (bit j of row i == mask[i, j])"""
    m = np.zeros((n, n), dtype=np.int64)
    for i in range(n):
        for j in range(n):
            m[i, j] = (int(words[i * W + (j >> 6)]) >> (j & 63)) & 1
    return m


def _raise(rc):
    if rc == -2:
        raise IndexError('list index out of range')
    raise AssertionError(f'oracle error {rc}')


class OracleTree(object):
    """Tree (lookahead_cache.py:24)"""

    def __init__(self, token_id, max_node=65536, max_output_node=512, _handle=None):
        self.token_id = token_id
        self._own = _handle is None
        self._h = lib().orc_tree_new(token_id, max_node, max_output_node) if _handle is None else _handle

    def __del__(self):
        if getattr(self, '_own', False) and self._h:
            lib().orc_tree_free(self._h)
            self._h = None

    def put(self, token_ids, mode='output', idx=0, freq=1.0):
        assert mode in ('input', 'output') and freq == 1.0
        a, n = _iarr(token_ids)
        lib().orc_tree_put(self._h, a, n, _MODES[mode], idx)

    def get(self, token_ids, max_size=64, max_length=8, min_input_size=0, min_output_size=0, output_weight=1e-4,
            mode='mix', idx=0):
        assert mode in _MODES
        a, n = _iarr(token_ids)
        W = (max_size + 63) // 64
        ids = (C.c_int * max_size)()
        mask = (C.c_uint64 * (max_size * W))()
        sizes = (C.c_int * 2)()
        r = lib().orc_tree_get(self._h, a, n, max_size, max_length, min_input_size, min_output_size, output_weight,
                               _MODES[mode], idx, ids, mask, sizes)
        if r < 0:
            _raise(r)
        return list(ids[:r]), bits_to_mask(mask, r, W), [sizes[0], sizes[1]]

    def get_one_branch(self, token_ids, max_length=8, mode='mix', idx=0):
        a, n = _iarr(token_ids)
        ids = (C.c_int * (max_length + 2))()
        miss = C.c_int(0)
        r = lib().orc_tree_get_one_branch(self._h, a, n, max_length, _MODES[mode], idx, ids, C.byref(miss))
        if miss.value:
            return list(ids[:1]), np.ones((1, 1), dtype=np.int64), [0, 0]
        return list(ids[:r]), np.tril(np.ones((r, r), dtype=np.int64), 0), [r - 1]

    def squeeze(self):
        lib().orc_tree_squeeze(self._h)

    def reset_input_freq(self, idx):
        lib().orc_tree_reset_input_freq(self._h, idx)

    @property
    def n_node(self):
        return lib().orc_tree_n_node(self._h)

    @property
    def n_output_node(self):
        return lib().orc_tree_n_output_node(self._h)

    def export(self, n_idx):
        """Tree.nodes in pre-order, children in insertion order: (tokens int32 [n], parent rows int64 [n] with -1 for
        a child of the root, counts float64 [n, 1 + n_idx] = freqs[-1], freqs[0], ..., freqs[n_idx - 1])"""
        n = lib().orc_tree_export(self._h, n_idx, 0, None, None, None)
        tok, par = np.zeros(n, dtype=np.int32), np.zeros(n, dtype=np.int64)
        freq = np.zeros((n, 1 + n_idx), dtype=np.float64)
        lib().orc_tree_export(self._h, n_idx, n, tok.ctypes.data, par.ctypes.data, freq.ctypes.data)
        return tok, par, freq


class OracleLookaheadCache(object):
    """LookaheadCache (lookahead_cache.py:336)"""

    def __init__(self, debug=False, eos_ids=(2,), stop_words=None, max_node=65536, max_output_node=512):
        self.debug = debug
        self._eos_ids = list(eos_ids) if eos_ids is not None else [None]
        a, n = _iarr([e for e in self._eos_ids if e is not None])
        self._h = lib().orc_cache_new(a, n, max_node, max_output_node)
        self._max_node, self._max_output_node = max_node, max_output_node
        self._stop_words = {}
        self.stop_words = stop_words if stop_words is not None else {}
        self.default_mask = np.ones((1, 1), dtype=np.int64)

    def __del__(self):
        if getattr(self, '_h', None):
            lib().orc_cache_free(self._h)
            self._h = None

    # attributes the callers read/write (benchmark.py:270-273, pretrained_model.py:1088-1089)
    @property
    def eos_ids(self):
        return self._eos_ids

    @eos_ids.setter
    def eos_ids(self, v):
        self._eos_ids = list(v) if v is not None else [None]
        a, n = _iarr([e for e in self._eos_ids if e is not None])
        lib().orc_cache_set_eos(self._h, a, n)

    @property
    def stop_words(self):
        return self._stop_words

    @stop_words.setter
    def stop_words(self, v):
        self._stop_words = v if v is not None else {}
        a, n = _iarr(sorted(int(x) for x in self._stop_words))
        lib().orc_cache_set_stop_words(self._h, a, n)

    def put(self, token_ids, branch_length=8, final=False, mode='output', idx=0):
        a, n = _iarr(token_ids)
        lib().orc_cache_put(self._h, a, n, branch_length, int(final), _MODES[mode], idx)

    def stream_put(self, token_ids, branch_length=8, final=False, mode='output', idx=0):
        assert mode == 'output' and idx >= 0
        a, n = _iarr(token_ids)
        rc = lib().orc_cache_stream_put(self._h, a, n, branch_length, int(final), _MODES[mode], idx)
        if rc < 0:
            _raise(rc)

    def hier_get(self, token_ids, decoding_length=64, branch_length=8, min_input_size=0, min_output_size=0,
                 mode='mix', idx=0):
        assert mode in _MODES
        a, n = _iarr(token_ids)
        cap = max(decoding_length, 1)
        W = (cap + 63) // 64
        ids = (C.c_int * cap)()
        mask = (C.c_uint64 * (cap * W))()
        sizes = (C.c_int * 2)()
        ns = C.c_int(0)
        r = lib().orc_cache_hier_get(self._h, a, n, decoding_length, branch_length, min_input_size, min_output_size,
                                     _MODES[mode], idx, ids, mask, sizes, C.byref(ns))
        if r < 0:
            _raise(r)
        return list(ids[:r]), bits_to_mask(mask, r, W) if r else self.default_mask, list(sizes[:ns.value])

    def one_get(self, token_ids, decoding_length=64, branch_length=8, min_input_size=0, min_output_size=0,
                mode='mix', idx=0):
        assert mode in _MODES
        a, n = _iarr(token_ids)
        ids = (C.c_int * (branch_length + 2))()
        sizes = (C.c_int * 2)()
        ns = C.c_int(0)
        r = lib().orc_cache_one_get(self._h, a, n, decoding_length, branch_length, _MODES[mode], idx, ids, sizes,
                                    C.byref(ns))
        if r < 0:
            _raise(r)
        return list(ids[:r]), np.tril(np.ones((max(r, 1), max(r, 1)), dtype=np.int64), 0), list(sizes[:ns.value])

    def par_get(self, token_ids, decoding_length=16, branch_length=8, min_input_size=0, min_output_size=0,
                mode='mix', idx=0):
        """lookahead_cache.py:441-488 -- flatten hier_get's tree into parallel root-to-leaf branches."""
        out_ids, masks, _ = self.hier_get(token_ids, decoding_length=decoding_length, branch_length=branch_length,
                                          min_input_size=min_input_size, min_output_size=min_output_size, mode=mode,
                                          idx=idx)
        n_draft = len(out_ids) - 1
        kept = []  # ancestor sets of maximal paths, discovered from the last row upwards (:453-462)
        for i in range(n_draft, 0, -1):
            cols = set(np.nonzero(masks[i, 1:])[0].tolist())
            if all(len(cols - other) != 0 for other in kept):
                kept.append(cols)
        kept.reverse()
        total, branches = 0, []
        for cols in kept:
            take = sorted(cols)[:n_draft - total]
            total += len(take)
            branches.append([out_ids[i + 1] for i in take])
            if total >= n_draft:
                break
        ids = [out_ids[0]]
        par = np.tril(np.ones((total + 1, total + 1)), 0)
        pos = 1
        for br in branches:
            ids.extend(br)
            par[pos:pos + len(br), 1:pos] = 0
            pos += len(br)
        return ids, par, [pos - 1]

    def bat_get(self, token_id_list, decoding_length=64, branch_length=8, decoding_cursors=None, mode='output',
                indices=None, decoding_mode='hier'):
        """lookahead_cache.py:519-561"""
        assert mode in _MODES and decoding_mode in ('hier', 'one')
        bs = len(token_id_list)
        assert bs == len(decoding_cursors) and bs == len(indices)
        lo, hi = min(decoding_cursors), max(decoding_cursors)
        per_row = decoding_length // bs
        getter = getattr(self, decoding_mode + '_get')
        id_list, mask_list, size_list = [], [], []
        for b, q in enumerate(token_id_list):
            ids, m, s = getter(q, decoding_length=per_row, branch_length=branch_length, min_input_size=0,
                               min_output_size=max(per_row // 2, 1), mode=mode, idx=indices[b])
            id_list.append(ids)
            mask_list.append(m)
            size_list.append(s)
        width = max(len(x) for x in id_list)
        out = np.zeros((bs, width, hi - lo + width), dtype=np.int64)
        for b, ids in enumerate(id_list):
            k = len(ids)
            ids.extend([0] * (width - k))
            off = decoding_cursors[b] - lo
            out[b, :k, off:off + k] = mask_list[b]
            out[b, :, :off + 1] = 1
        return id_list, out, size_list

    def fresh(self):
        lib().orc_cache_fresh(self._h)

    def reset_input_freqs(self, idx):
        lib().orc_cache_reset_input_freqs(self._h, idx)

    def squeeze_branch_counts(self):
        lib().orc_cache_squeeze_branch_counts(self._h)

    # introspection used by tests / bench
    def tree(self, token_id):
        h = lib().orc_cache_tree(self._h, token_id)
        return OracleTree(token_id, _handle=h) if h else None

    def n_trees(self):
        return lib().orc_cache_n_trees(self._h)

    def total_nodes(self):
        return lib().orc_cache_total_nodes(self._h)

    def n_update_trees(self):
        return lib().orc_cache_n_update_trees(self._h)
