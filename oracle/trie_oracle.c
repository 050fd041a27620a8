/*
 * trie_oracle.c -- CPU restatement of PIA LOOKAHEAD's trie draft cache.
 *
 * TEST INFRASTRUCTURE ONLY.  This file is the parity oracle for the CUDA trie
 * (painlessinferenceacceleration_b200/csrc/trie.cu).  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs may load it; the product path never does.
 *
 * It restates, in plain C with insertion-ordered child vectors, the algorithm of
 *   /root/reference/lookahead/lookahead/common/lookahead_cache.py
 * (Node :13, Tree :24-333, LookaheadCache :336-587).  Every function cites the lines it follows.
 * The restatement is pinned by tests/test_oracle_trie.py against (i) the two golden vectors of
 * lookahead/tests/test_lookahead_cache.py:16-45 and (ii) recorded op streams produced by the live
 * reference module (tests/golden/gen_trie_golden.py -> tests/golden/trie_*.json).
 *
 * Frequencies are IEEE doubles exactly like the Python floats of the reference; `fm` is evaluated
 * as (1-w)*fi + w*fo with two roundings and no FMA contraction (compile with -ffp-contract=off).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_MODE_INPUT 0
#define ORC_MODE_OUTPUT 1
#define ORC_MODE_MIX 2
#define ORC_ERR_INDEX (-2) /* Python IndexError: k-th largest beyond the collected list */
#define ORC_ERR_ARG (-3)

typedef struct ONode {
  int token;
  double fo;      /* freqs[-1]  (output / global frequency) */
  double *fi;     /* freqs[idx] for idx >= 0 (per-request prompt frequency), default 0.0 */
  int nfi;
  struct ONode **kid; /* children in dict insertion order */
  int nkid, cap;
} ONode;

typedef struct OTree {
  int token_id;
  long n_node, n_output_node;
  int max_node, max_output_node;
  ONode root; /* root.kid == Tree.nodes */
  int in_update, in_update_input;
} OTree;

typedef struct OVec { int *v; int n, cap; } OVec;

typedef struct OCache {
  OTree **mem; int mem_cap;       /* mem: token -> Tree (lookahead_cache.py:342) */
  OVec *out_ids; int n_out;       /* _output_ids[idx] (:343) */
  OTree **upd; int n_upd, cap_upd;        /* _update_trees (:344) */
  OTree **updin; int n_updin, cap_updin;  /* _update_input_trees (:345) */
  int *eos; int n_eos;
  int *stop; int n_stop;
  int max_node, max_output_node;
} OCache;

/* ------------------------------------------------------------------ helpers */
static double node_fi(const ONode *p, int idx) { return (idx >= 0 && idx < p->nfi) ? p->fi[idx] : 0.0; }
static void node_add_fi(ONode *p, int idx, double f) {
  if (idx >= p->nfi) {
    p->fi = (double *)realloc(p->fi, sizeof(double) * (idx + 1));
    for (int i = p->nfi; i <= idx; ++i) p->fi[i] = 0.0;
    p->nfi = idx + 1;
  }
  p->fi[idx] += f;
}
static ONode *node_new(int token) {
  ONode *p = (ONode *)calloc(1, sizeof(ONode));
  p->token = token;
  return p;
}
static void node_push_kid(ONode *p, ONode *c) {
  if (p->nkid == p->cap) {
    p->cap = p->cap ? p->cap * 2 : 2;
    p->kid = (ONode **)realloc(p->kid, sizeof(ONode *) * p->cap);
  }
  p->kid[p->nkid++] = c;
}
static ONode *node_find(const ONode *p, int token) {
  for (int i = 0; i < p->nkid; ++i)
    if (p->kid[i]->token == token) return p->kid[i];
  return NULL;
}
static void node_free(ONode *p) {
  for (int i = 0; i < p->nkid; ++i) { node_free(p->kid[i]); free(p->kid[i]); }
  free(p->kid); free(p->fi);
  p->kid = NULL; p->fi = NULL; p->nkid = p->cap = 0; p->nfi = 0;
}
static void vec_push(OVec *v, int x) {
  if (v->n == v->cap) { v->cap = v->cap ? v->cap * 2 : 16; v->v = (int *)realloc(v->v, sizeof(int) * v->cap); }
  v->v[v->n++] = x;
}

/* ------------------------------------------------------------------ Tree */
/* Tree.__init__  lookahead_cache.py:25-31 */
OTree *orc_tree_new(int token_id, int max_node, int max_output_node) {
  OTree *t = (OTree *)calloc(1, sizeof(OTree));
  t->token_id = token_id; t->max_node = max_node; t->max_output_node = max_output_node;
  t->root.token = token_id;
  return t;
}
void orc_tree_free(OTree *t) { node_free(&t->root); free(t); }

/* Tree.put/_put/_pack  lookahead_cache.py:33-63.  mode output forces idx=-1 (:35-36). */
void orc_tree_put(OTree *t, const int *ids, int n, int mode, int idx) {
  ONode *cur = &t->root;
  const int out = (mode == ORC_MODE_OUTPUT);
  for (int i = 0; i < n; ++i) {
    ONode *c = node_find(cur, ids[i]);
    if (c == NULL) {
      /* _pack: chain of the remaining tokens, each with {idx: 1.0} (:57-63); counters (:48-50) */
      for (int j = i; j < n; ++j) {
        ONode *nn = node_new(ids[j]);
        if (out) nn->fo = 1.0; else node_add_fi(nn, idx, 1.0);
        node_push_kid(cur, nn);
        cur = nn;
      }
      t->n_node += n - i;
      if (out) t->n_output_node += n - i;
      return;
    }
    if (out) c->fo += 1.0; else node_add_fi(c, idx, 1.0); /* :53 */
    cur = c;
  }
}

/* Tree._match  lookahead_cache.py:224-246.
 * returns the node whose children are the candidate set ("nodes"), or NULL for the empty dict.
 * *mt receives the last query token looked at (match_token_id), *has_mt whether there was one. */
static const ONode *tree_match(const OTree *t, const int *q, int nq, int mode, int idx, int *mt, int *has_mt) {
  const ONode *cur = &t->root;
  *has_mt = 0; *mt = 0;
  if (nq == 0) return cur; /* :227-228 */
  for (int i = 0; i < nq; ++i) {
    *mt = q[i]; *has_mt = 1;
    const ONode *c = cur ? node_find(cur, q[i]) : NULL;
    if (c == NULL) { cur = NULL; break; }  /* :231-234 (nodes = {} then break) */
    int live;
    if (mode == ORC_MODE_INPUT) live = node_fi(c, idx) > 0;
    else if (mode == ORC_MODE_OUTPUT) live = c->fo > 0;
    else live = node_fi(c, idx) > 0 || c->fo > 0;
    cur = live ? c : NULL;   /* nodes = {} stays for the remaining tokens: next lookup fails -> break */
    if (cur == NULL) {
      /* the python loop continues with nodes={} : the next get() returns None and breaks, but
       * token_id has then advanced to the next query token (:230-234). */
      if (i + 1 < nq) { *mt = q[i + 1]; }
      break;
    }
  }
  return cur;
}

typedef struct { double fi, fo, fm; } OFreq;
typedef struct { OFreq *v; long n, cap; } OFreqVec;

/* Tree._dfs_get_freqs  lookahead_cache.py:146-154 */
static void dfs_get_freqs(const ONode *p, OFreqVec *out, int idx, double w) {
  for (int i = 0; i < p->nkid; ++i) {
    const ONode *c = p->kid[i];
    double fo = c->fo, fi = node_fi(c, idx);
    if (fo > 0 || fi > 0) {
      if (out->n == out->cap) { out->cap = out->cap ? out->cap * 2 : 256; out->v = (OFreq *)realloc(out->v, sizeof(OFreq) * out->cap); }
      OFreq r; r.fi = fi; r.fo = fo; r.fm = (1.0 - w) * fi + w * fo;
      out->v[out->n++] = r;
      if (c->nkid > 0) dfs_get_freqs(c, out, idx, w);
    }
  }
}

static int cmp_desc(const void *a, const void *b) {
  double x = *(const double *)a, y = *(const double *)b;
  return (x < y) - (x > y);
}
/* sorted(freqs, key=x[col], reverse=True)[k-1][col] with Python negative-index wrap (:85-86,:93-94,:102-108) */
static int kth_largest(const OFreqVec *f, int col, int k, double *out) {
  long n = f->n;
  long index = (long)k - 1;
  if (index < 0) index += n;
  if (index < 0 || index >= n) return ORC_ERR_INDEX;
  double *tmp = (double *)malloc(sizeof(double) * n);
  for (long i = 0; i < n; ++i) tmp[i] = col == 1 ? f->v[i].fi : f->v[i].fo;
  qsort(tmp, n, sizeof(double), cmp_desc);
  *out = tmp[index];
  free(tmp);
  return 0;
}

typedef struct {
  int *ids; uint64_t *mask; int W; int n; int max_size;
  double min_in, min_out, min_mix, w; int mode, idx; int sizes[2];
} ORavel;

typedef struct { const ONode *p; double fm; int ord; } OSort;
static int cmp_sort(const void *a, const void *b) {
  const OSort *x = (const OSort *)a, *y = (const OSort *)b;
  if (x->fm > y->fm) return -1;
  if (x->fm < y->fm) return 1;
  return x->ord - y->ord; /* stable: dict insertion order on ties (:254-258) */
}

/* Tree._ravel  lookahead_cache.py:248-293 */
static void ravel(const ONode *p, ORavel *r, int pid, int max_length) {
  if (r->n >= r->max_size || max_length <= 0) return;
  OSort *s = (OSort *)malloc(sizeof(OSort) * (p->nkid ? p->nkid : 1));
  for (int i = 0; i < p->nkid; ++i) {
    const ONode *c = p->kid[i];
    s[i].p = c; s[i].ord = i;
    s[i].fm = (1.0 - r->w) * node_fi(c, r->idx) + r->w * c->fo;
  }
  qsort(s, p->nkid, sizeof(OSort), cmp_sort);
  for (int i = 0; i < p->nkid; ++i) {
    if (r->n >= r->max_size) break;
    const ONode *c = s[i].p;
    double fi = node_fi(c, r->idx), fo = c->fo, fm = s[i].fm;
    if (r->mode == ORC_MODE_MIX) { if (fi < r->min_in && fo < r->min_out && fm < r->min_mix) continue; }
    else if (r->mode == ORC_MODE_INPUT) { if (fi < r->min_in) continue; }
    else { if (fo < r->min_out) continue; }
    if (fi > 0.0) r->sizes[0] += 1;
    if (fo > 0.0) r->sizes[1] += 1;
    int rid = r->n;
    r->ids[r->n++] = c->token;
    uint64_t *row = r->mask + (size_t)rid * r->W;
    if (pid > -1) memcpy(row, r->mask + (size_t)pid * r->W, sizeof(uint64_t) * r->W);
    row[rid >> 6] |= 1ull << (rid & 63);
    if (c->nkid > 0) ravel(c, r, rid, max_length - 1);
  }
  free(s);
}

/* Tree.get  lookahead_cache.py:65-144.
 * out_mask: max_size rows of W=ceil(max_size/64) uint64 words, bit j of row i == mask[i][j].
 * returns n (>=1) or a negative error. */
int orc_tree_get(const OTree *t, const int *q, int nq, int max_size, int max_length, int min_input_size,
                 int min_output_size, double output_weight, int mode, int idx, int *out_ids, uint64_t *out_mask,
                 int *out_sizes) {
  const int W = (max_size + 63) / 64;
  int mt, has_mt;
  const ONode *nodes = tree_match(t, q, nq, mode, idx, &mt, &has_mt);
  out_sizes[0] = out_sizes[1] = 0;
  if (nodes == NULL || nodes->nkid == 0) { /* :70-72 */
    out_ids[0] = nq > 0 ? q[nq - 1] : t->token_id;
    memset(out_mask, 0, sizeof(uint64_t) * W);
    out_mask[0] = 1;
    return 1;
  }
  OFreqVec fr = {0, 0, 0};
  dfs_get_freqs(nodes, &fr, idx, output_weight); /* :74-75 (weight as passed, before the mode override) */
  double min_mix = 1e9, min_in = 1e9, min_out = 1e9;
  int rc = 0;
  if (mode == ORC_MODE_INPUT) { /* :81-88 */
    output_weight = 0.0;
    long size = 0; for (long i = 0; i < fr.n; ++i) size += fr.v[i].fi > 0;
    if (size > max_size) rc = kth_largest(&fr, 1, min_input_size, &min_in); else min_in = 0.0;
  } else if (mode == ORC_MODE_OUTPUT) { /* :89-96 */
    output_weight = 1.0;
    long size = 0; for (long i = 0; i < fr.n; ++i) size += fr.v[i].fo > 0;
    if (size > max_size) rc = kth_largest(&fr, 2, min_output_size, &min_out); else min_out = 0.0;
  } else { /* :97-125 */
    long size = 0; for (long i = 0; i < fr.n; ++i) size += (fr.v[i].fi > 0 || fr.v[i].fo > 0);
    if (size > max_size) {
      if (min_input_size > 0) rc = kth_largest(&fr, 1, min_input_size, &min_in);
      if (rc == 0 && min_output_size > 0) rc = kth_largest(&fr, 2, min_output_size, &min_out);
      /* :111-123: every record carries None in slot 0, so `indices` is {None} (or empty) and the
       * refinement loop always hits `continue`; min_mix_freq keeps its 1e9 initial value. */
    } else {
      min_mix = 0.0;
    }
  }
  free(fr.v);
  if (rc) return rc;
  memset(out_mask, 0, sizeof(uint64_t) * (size_t)W * max_size);
  for (int i = 0; i < max_size; ++i) out_mask[(size_t)i * W] = 1; /* mask[:,0]=1 (:128) */
  ORavel r;
  r.ids = out_ids; r.mask = out_mask; r.W = W; r.n = 0; r.max_size = max_size;
  r.min_in = min_in; r.min_out = min_out; r.min_mix = min_mix; r.w = output_weight; r.mode = mode; r.idx = idx;
  r.sizes[0] = r.sizes[1] = 0;
  out_ids[r.n++] = (has_mt && mt != 0) ? mt : t->token_id; /* `match_token_id or self.token_id` (:129) */
  ravel(nodes, &r, -1, max_length);
  out_sizes[0] = r.sizes[0]; out_sizes[1] = r.sizes[1];
  return r.n;
}

/* Tree.get_one_branch  lookahead_cache.py:171-222 (note the swapped fo/fi names in mix mode :187-197).
 * returns number of ids (length+1); mask is lower-triangular and produced by the caller. */
int orc_tree_get_one_branch(const OTree *t, const int *q, int nq, int max_length, int mode, int idx, int *out_ids,
                            int *is_miss) {
  int mt, has_mt;
  const ONode *nodes = tree_match(t, q, nq, mode, idx, &mt, &has_mt);
  *is_miss = 0;
  if (nodes == NULL || nodes->nkid == 0) {
    out_ids[0] = nq > 0 ? q[nq - 1] : t->token_id;
    *is_miss = 1;
    return 1;
  }
  int n = 0, length = 0;
  out_ids[n++] = (has_mt && mt != 0) ? mt : t->token_id;
  while (nodes->nkid > 0 && length < max_length) {
    double max_freq = 0.0; const ONode *best = NULL;
    for (int i = 0; i < nodes->nkid; ++i) {
      const ONode *c = nodes->kid[i];
      double freq; int ok;
      if (mode == ORC_MODE_MIX) { double a = node_fi(c, idx), b = c->fo; ok = a > 0 || b > 0; freq = 10000 * b + a; }
      else if (mode == ORC_MODE_INPUT) { freq = node_fi(c, idx); ok = freq > 0; }
      else { freq = c->fo; ok = freq > 0; }
      if (ok && freq > max_freq) { max_freq = freq; best = c; }
    }
    if (!best) break;
    out_ids[n++] = best->token;
    nodes = best; length++;
  }
  return n;
}

/* Tree._squeeze/_count_node/squeeze  lookahead_cache.py:295-318 */
static void squeeze_rec(ONode *p) {
  int w = 0;
  for (int i = 0; i < p->nkid; ++i) {
    ONode *c = p->kid[i];
    if (c->fo > 1.0) {
      c->fo *= 0.5;
      if (c->nkid > 0) squeeze_rec(c);
      p->kid[w++] = c;
    } else {
      node_free(c); free(c);
    }
  }
  p->nkid = w;
}
static long count_nodes(const ONode *p) {
  long s = p->nkid;
  for (int i = 0; i < p->nkid; ++i) if (p->kid[i]->nkid > 0) s += count_nodes(p->kid[i]);
  return s;
}
void orc_tree_squeeze(OTree *t) {
  if (t->n_node > t->max_node || t->n_output_node > t->max_output_node) {
    squeeze_rec(&t->root);
    long c = count_nodes(&t->root);
    t->n_node = c; t->n_output_node = c;
  }
}
/* Tree.reset_input_freq  lookahead_cache.py:320-333 */
static void reset_rec(ONode *p, int idx) {
  for (int i = 0; i < p->nkid; ++i) {
    ONode *c = p->kid[i];
    if (node_fi(c, idx) == 0.0) continue;
    c->fi[idx] = 0.0;
    if (c->nkid > 0) reset_rec(c, idx);
  }
}
void orc_tree_reset_input_freq(OTree *t, int idx) { if (t->root.nkid) reset_rec(&t->root, idx); }
long orc_tree_n_node(const OTree *t) { return t->n_node; }
long orc_tree_n_output_node(const OTree *t) { return t->n_output_node; }

/* Tree.nodes in pre-order, children in insertion order: row r gets the node's token, its parent's row (-1 for a child
 * of the root) and freqs[-1], freqs[0], ..., freqs[n_idx - 1] (n_idx + 1 doubles).  Writes at most cap rows and
 * returns the number of nodes. */
static void export_rec(const ONode *p, long parent, int n_idx, long cap, long *row, int *tok, long *par, double *freq) {
  for (int i = 0; i < p->nkid; ++i) {
    const ONode *c = p->kid[i];
    const long r = (*row)++;
    if (r < cap) {
      tok[r] = c->token; par[r] = parent;
      freq[r * (n_idx + 1)] = c->fo;
      for (int k = 0; k < n_idx; ++k) freq[r * (n_idx + 1) + 1 + k] = node_fi(c, k);
    }
    export_rec(c, r, n_idx, cap, row, tok, par, freq);
  }
}
long orc_tree_export(const OTree *t, int n_idx, long cap, int *tok, long *par, double *freq) {
  long row = 0;
  export_rec(&t->root, -1, n_idx, cap, &row, tok, par, freq);
  return row;
}

/* ------------------------------------------------------------------ LookaheadCache */
/* LookaheadCache.__init__  lookahead_cache.py:337-347 */
OCache *orc_cache_new(const int *eos, int n_eos, int max_node, int max_output_node) {
  OCache *c = (OCache *)calloc(1, sizeof(OCache));
  c->n_eos = n_eos; c->eos = (int *)malloc(sizeof(int) * (n_eos ? n_eos : 1));
  memcpy(c->eos, eos, sizeof(int) * n_eos);
  c->max_node = max_node; c->max_output_node = max_output_node;
  return c;
}
void orc_cache_set_eos(OCache *c, const int *eos, int n) {
  free(c->eos); c->eos = (int *)malloc(sizeof(int) * (n ? n : 1)); memcpy(c->eos, eos, sizeof(int) * n); c->n_eos = n;
}
void orc_cache_set_stop_words(OCache *c, const int *w, int n) {
  free(c->stop); c->stop = (int *)malloc(sizeof(int) * (n ? n : 1)); memcpy(c->stop, w, sizeof(int) * n); c->n_stop = n;
}
void orc_cache_set_limits(OCache *c, int max_node, int max_output_node) { c->max_node = max_node; c->max_output_node = max_output_node; }
static int is_stop(const OCache *c, int t) { for (int i = 0; i < c->n_stop; ++i) if (c->stop[i] == t) return 1; return 0; }
static OTree *mem_get(const OCache *c, int token) { return (token >= 0 && token < c->mem_cap) ? c->mem[token] : NULL; }
static void mem_set(OCache *c, int token, OTree *t) {
  if (token >= c->mem_cap) {
    int nc = c->mem_cap ? c->mem_cap : 1024; while (nc <= token) nc *= 2;
    c->mem = (OTree **)realloc(c->mem, sizeof(OTree *) * nc);
    for (int i = c->mem_cap; i < nc; ++i) c->mem[i] = NULL;
    c->mem_cap = nc;
  }
  c->mem[token] = t;
}
static void set_add(OTree ***arr, int *n, int *cap, OTree *t) {
  if (*n == *cap) { *cap = *cap ? *cap * 2 : 64; *arr = (OTree **)realloc(*arr, sizeof(OTree *) * *cap); }
  (*arr)[(*n)++] = t;
}
static void add_update(OCache *c, OTree *t) { if (!t->in_update) { t->in_update = 1; set_add(&c->upd, &c->n_upd, &c->cap_upd, t); } }
static void add_update_input(OCache *c, OTree *t) { if (!t->in_update_input) { t->in_update_input = 1; set_add(&c->updin, &c->n_updin, &c->cap_updin, t); } }

/* eos truncation: for each eos in order, cut at its first occurrence (:350-352, :378-380) */
static int cut_eos(const OCache *c, const int *ids, int n) {
  for (int e = 0; e < c->n_eos; ++e)
    for (int i = 0; i < n; ++i) if (ids[i] == c->eos[e]) { n = i; break; }
  return n;
}

/* reset_input_freqs :566-570, squeeze_branch_counts :572-576 */
void orc_cache_reset_input_freqs(OCache *c, int idx) {
  for (int i = 0; i < c->n_updin; ++i) { orc_tree_reset_input_freq(c->updin[i], idx); c->updin[i]->in_update_input = 0; }
  c->n_updin = 0;
}
void orc_cache_squeeze_branch_counts(OCache *c) {
  if (c->n_upd >= 1024) {
    for (int i = 0; i < c->n_upd; ++i) { orc_tree_squeeze(c->upd[i]); c->upd[i]->in_update = 0; }
    c->n_upd = 0;
  }
}

/* LookaheadCache.put  lookahead_cache.py:349-373 */
void orc_cache_put(OCache *c, const int *ids, int n, int branch_length, int final, int mode, int idx) {
  n = cut_eos(c, ids, n);
  if (n >= 2) {
    for (int i = 0; i < n - 1; ++i) {
      int tok = ids[i];
      int len = n - (i + 1); if (len > branch_length) len = branch_length;
      OTree *t = mem_get(c, tok);
      if (t != NULL) {
        orc_tree_put(t, ids + i + 1, len, mode, idx);
        add_update(c, t);                      /* only pre-existing trees join _update_trees (:361-363) */
      } else {
        t = orc_tree_new(tok, c->max_node, c->max_output_node);
        orc_tree_put(t, ids + i + 1, len, mode, idx);
        mem_set(c, tok, t);
      }
      if (mode == ORC_MODE_INPUT) add_update_input(c, t);
    }
  }
  if (final) { orc_cache_reset_input_freqs(c, idx); orc_cache_squeeze_branch_counts(c); }
}

/* LookaheadCache.stream_put  lookahead_cache.py:375-406 */
int orc_cache_stream_put(OCache *c, const int *ids, int n, int branch_length, int final, int mode, int idx) {
  if (mode != ORC_MODE_OUTPUT || idx < 0) return ORC_ERR_ARG; /* assert (:377) */
  n = cut_eos(c, ids, n);
  if (idx >= c->n_out) {
    c->out_ids = (OVec *)realloc(c->out_ids, sizeof(OVec) * (idx + 1));
    for (int i = c->n_out; i <= idx; ++i) { c->out_ids[i].v = NULL; c->out_ids[i].n = c->out_ids[i].cap = 0; }
    c->n_out = idx + 1;
  }
  OVec *o = &c->out_ids[idx];
  for (int i = 0; i < n; ++i) vec_push(o, ids[i]);
  int ts = o->n;
  int min_bl = final ? 1 : branch_length;
  if (ts > min_bl) {
    for (int i = 0; i < ts - min_bl; ++i) {
      int tok = o->v[i];
      if (is_stop(c, tok)) continue;
      int len = ts - (i + 1); if (len > branch_length) len = branch_length;
      OTree *t = mem_get(c, tok);
      if (t == NULL) { t = orc_tree_new(tok, c->max_node, c->max_output_node); mem_set(c, tok, t); }
      orc_tree_put(t, o->v + i + 1, len, ORC_MODE_OUTPUT, idx);
      add_update(c, t);
    }
    if (!final) {
      int keep = branch_length; /* output_ids[ts - branch_length:] (:402) ; ts > branch_length here */
      memmove(o->v, o->v + ts - keep, sizeof(int) * keep);
      o->n = keep;
    }
  }
  if (final) { o->n = 0; orc_cache_reset_input_freqs(c, idx); orc_cache_squeeze_branch_counts(c); }
  return 0;
}

/* LookaheadCache.hier_get  lookahead_cache.py:408-439.
 * n_sizes: 0 when the early return (:413-414) fires (python returns sizes=[]), else 2. */
int orc_cache_hier_get(OCache *c, const int *q, int nq, int decoding_length, int branch_length, int min_input_size,
                       int min_output_size, int mode, int idx, int *out_ids, uint64_t *out_mask, int *out_sizes,
                       int *n_sizes) {
  const int W = (decoding_length > 0 ? decoding_length + 63 : 64) / 64;
  *n_sizes = 2; out_sizes[0] = out_sizes[1] = 0;
  if (decoding_length <= 1 || branch_length == 0) {
    *n_sizes = 0;
    if (nq == 0) return 0;
    out_ids[0] = q[nq - 1]; out_mask[0] = 1; return 1;
  }
  int n = -1;
  for (int i = 0; i < nq; ++i) {
    OTree *t = mem_get(c, q[i]);
    if (t == NULL) continue;
    int rest = nq - (i + 1);
    if (is_stop(c, q[i]) && rest == 0) continue; /* :422-423 */
    n = orc_tree_get(t, q + i + 1, rest, decoding_length, branch_length, min_input_size, min_output_size, 1e-4, mode, idx,
                     out_ids, out_mask, out_sizes);
    if (n < 0) return n;
    if (n >= branch_length) break; /* :433-434 */
  }
  if (n < 0) { /* decoding_ids is None (:436-437); mask stays default ones(1,1) */
    if (nq == 0) return 0;
    out_ids[0] = q[nq - 1]; memset(out_mask, 0, sizeof(uint64_t) * W); out_mask[0] = 1; return 1;
  }
  return n;
}

/* LookaheadCache.one_get  lookahead_cache.py:490-517; sizes=[length] on a hit, [0,0] on a tree miss. */
int orc_cache_one_get(OCache *c, const int *q, int nq, int decoding_length, int branch_length, int mode, int idx,
                      int *out_ids, int *out_sizes, int *n_sizes) {
  *n_sizes = 2; out_sizes[0] = out_sizes[1] = 0;
  if (decoding_length <= 1 || branch_length == 0) { *n_sizes = 0; if (nq == 0) return 0; out_ids[0] = q[nq - 1]; return 1; }
  int n = -1;
  for (int i = 0; i < nq; ++i) {
    OTree *t = mem_get(c, q[i]);
    if (t == NULL) continue;
    int rest = nq - (i + 1);
    if (is_stop(c, q[i]) && rest == 0) continue;
    int miss;
    n = orc_tree_get_one_branch(t, q + i + 1, rest, branch_length, mode, idx, out_ids, &miss);
    if (miss) { *n_sizes = 2; out_sizes[0] = out_sizes[1] = 0; } else { *n_sizes = 1; out_sizes[0] = n - 1; }
    if (n >= branch_length / 2) break; /* :512 */
  }
  if (n < 0) { if (nq == 0) return 0; out_ids[0] = q[nq - 1]; return 1; }
  return n;
}

/* LookaheadCache.fresh  lookahead_cache.py:563-564 (mem only; pending update sets keep the old trees) */
void orc_cache_fresh(OCache *c) { for (int i = 0; i < c->mem_cap; ++i) c->mem[i] = NULL; }

OTree *orc_cache_tree(OCache *c, int token) { return mem_get(c, token); }
int orc_cache_n_update_trees(const OCache *c) { return c->n_upd; }
int orc_cache_n_update_input_trees(const OCache *c) { return c->n_updin; }
long orc_cache_total_nodes(const OCache *c) {
  long s = 0;
  for (int i = 0; i < c->mem_cap; ++i) if (c->mem[i]) s += count_nodes(&c->mem[i]->root);
  return s;
}
int orc_cache_n_trees(const OCache *c) { int s = 0; for (int i = 0; i < c->mem_cap; ++i) s += c->mem[i] != NULL; return s; }
/* trees orphaned by fresh() are intentionally leaked (they may still sit in the update sets, as in python) */
void orc_cache_free(OCache *c) {
  for (int i = 0; i < c->mem_cap; ++i) if (c->mem[i]) orc_tree_free(c->mem[i]);
  for (int i = 0; i < c->n_out; ++i) free(c->out_ids[i].v);
  free(c->mem); free(c->out_ids); free(c->upd); free(c->updin); free(c->eos); free(c->stop); free(c);
}
