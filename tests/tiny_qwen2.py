# -*- coding: utf-8 -*-
"""seeded tiny random-init HF Qwen2 models (no checkpoints exist offline) and the loader of the qwen2loop_*.npz goldens.

`g7`: 7 query heads over 1 KV head (the odd group size of Qwen2-7B / Qwen2.5-7B, 28 / 4), head_dim 128, untied head.
`g6_tied`: 6 query heads over 1 KV head with tied input / output embeddings (the small Qwen2 checkpoints).
Both carry q/k/v biases, rope_theta 1e6 (the published checkpoints' value) and no sliding window."""
import glob
import json
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
SHAPES = {'g7': dict(num_attention_heads=7, tie_word_embeddings=False),
          'g6_tied': dict(num_attention_heads=6, tie_word_embeddings=True)}


def qwen2_config(shape, vocab=64, **over):
    from transformers import Qwen2Config
    s = SHAPES[shape]
    cfg = Qwen2Config(vocab_size=vocab, hidden_size=128 * s['num_attention_heads'], intermediate_size=256,
                      num_hidden_layers=2, num_attention_heads=s['num_attention_heads'], num_key_value_heads=1,
                      max_position_embeddings=1024, rms_norm_eps=1e-6, rope_theta=1e6, use_sliding_window=False,
                      tie_word_embeddings=s['tie_word_embeddings'], bos_token_id=1, eos_token_id=2, pad_token_id=0)
    for k, v in over.items():
        setattr(cfg, k, v)
    cfg._attn_implementation = 'eager'
    return cfg


def qwen2_hf_model(shape, seed=0, dtype=torch.float32, device='cpu', vocab=64, **over):
    from transformers import Qwen2ForCausalLM
    torch.manual_seed(seed)
    model = Qwen2ForCausalLM(qwen2_config(shape, vocab=vocab, **over))
    # std 0.08 like tests/tiny_models.py, biases included: a zero bias would leave the bias path untested
    with torch.no_grad():
        for n, p in model.named_parameters():
            if p.dim() >= 2 or n.endswith('.bias'):
                p.normal_(0.0, 0.08)
    return model.to(device=device, dtype=dtype).eval()


def golden_names():
    return sorted(os.path.basename(f)[len('qwen2loop_'):-4] for f in glob.glob(os.path.join(GOLD, 'qwen2loop_*.npz')))


def load_golden(name):
    """same layout as tests/golden/loop_*.npz: tests/loop_golden.step_logits / step_mask / mask01 apply"""
    z = np.load(os.path.join(GOLD, f'qwen2loop_{name}.npz'))
    return json.loads(bytes(z['meta']).decode()), z
