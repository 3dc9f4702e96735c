"""Deterministic synthetic workloads (BASELINE.json `configs`, SURVEY.md section 8(d)) and deterministic
parameter fill.  Everything is drawn from CPU `torch.Generator`s so that the reference (oracle side,
this container) and the B200 path (GPU box) see bit-identical inputs and weights without shipping
them.  No dependency on the reference or on `oracle/`.
"""
from __future__ import annotations

import zlib
import torch


def _gen(seed: int) -> torch.Generator:
    g = torch.Generator(device = 'cpu')
    g.manual_seed(int(seed))
    return g


def fill_parameters_(module: torch.nn.Module, seed: int = 0, scale: float = 1.0) -> None:
    """Overwrite every parameter / persistent buffer with values that depend only on (name, shape, seed).

    The reference zero-initialises most of the conditioning path (transfusion.py:659-669, 783), which
    would hide bugs (SURVEY.md section 7, hard part 6) - so parity fixtures randomise everything, with
    magnitudes chosen to keep activations O(1).
    """
    sd = module.state_dict()
    for name in sorted(sd.keys()):
        t = sd[name]
        if not t.is_floating_point():
            continue
        g = _gen(zlib.crc32(name.encode()) ^ (seed * 0x9E3779B1 & 0xFFFFFFFF))
        if name.endswith('rotary_emb.freqs'):
            continue                                      # keep the analytic RoPE frequencies
        shape = tuple(t.shape)
        r = torch.randn(shape, generator = g, dtype = torch.float32)
        if name.endswith('to_time_cond.0.weights'):
            v = r                                         # N(0,1) fourier frequencies, as the reference draws them
        elif t.ndim == 2:
            fan_in = shape[1]
            v = r * (scale / fan_in ** 0.5)
            if 'text_embed' in name:
                v = r * scale
        elif name.endswith('to_ada_ln_zero.bias'):
            v = r * 0.5 - 1.0
        elif name.endswith('pseudo_queries'):
            v = r * 0.5
        else:
            v = r * 0.2                                   # gammas, layerscales, biases: O(0.2) perturbation
        t.copy_(v.to(t.dtype))
    module.load_state_dict(sd)


def posemb_batch(seed: int = 77, dim_latent: int = 32, text_vocab: int = 64):
    """three ragged samples with 2-D latents of different (h, w) per instance: the axial positional embedding fixture (tests/golden/small_posemb.pt)"""
    g = _gen(seed)
    txt = lambda n: torch.randint(0, text_vocab, (n,), generator = g)
    lat = lambda h, w: torch.randn(h, w, dim_latent, generator = g)
    return [[txt(5), lat(2, 3), txt(4), lat(3, 2), txt(3)], [txt(7), lat(4, 2), txt(2)], [lat(1, 5), txt(6)]]


def config2_sample(seed: int, dim_latent: int = 384, text_vocab: int = 256,
                   text_lens = (200, 200, 99), span_len: int = 256):
    """One sample of the graded shape: [text200, latent 256xdl, text200, latent 256xdl, text99]
    -> 1025 positions after [sos]/[eos] and the 2x6 meta tokens -> n = 1024 after the shift."""
    g = _gen(1000003 * (seed + 1))
    out = []
    for i, tl in enumerate(text_lens):
        out.append(torch.randint(0, text_vocab, (tl,), generator = g))
        if i < len(text_lens) - 1:
            out.append(torch.randn(span_len, dim_latent, generator = g))
    return out


def config2_batch(batch: int, seed: int = 0, **kw):
    return [config2_sample(seed * 100003 + b, **kw) for b in range(batch)]


def config2_times(batch: int, seed: int = 0, num_modalities: int = 2) -> torch.Tensor:
    return torch.rand(batch, num_modalities, generator = _gen(77 + seed))


def small_sample(seed: int, dim_latent: int = 32, text_vocab: int = 64):
    """Small ragged sample: short text runs and spans of different lengths (parity-test sizes)."""
    g = _gen(424243 * (seed + 1))
    def ri(lo, hi):
        return int(torch.randint(lo, hi + 1, (1,), generator = g))
    out = [torch.randint(0, text_vocab, (ri(3, 20),), generator = g)]
    for _ in range(ri(1, 3)):
        out.append(torch.randn(ri(2, 40), dim_latent, generator = g))
        out.append(torch.randint(0, text_vocab, (ri(1, 25),), generator = g))
    return out


def small_batch(batch: int, seed: int = 0, **kw):
    return [small_sample(seed * 7919 + b, **kw) for b in range(batch)]


def config4_sample(seed: int, total_len: int = 1025, dims = (384, 192), text_vocab: int = 256):
    """Two modality types, many short alternating spans (span-mask stress), padded with text so that the
    packed length is exactly `total_len` after [sos]/[eos] and meta tokens."""
    g = _gen(9176 * (seed + 1))
    def pick(opts):
        return opts[int(torch.randint(0, len(opts), (1,), generator = g))]
    parts, used = [], 2                                    # sos + eos
    for i in range(8):
        tl = int(torch.randint(8, 41, (1,), generator = g))
        mtype = i % 2
        ml = pick((16, 32, 64, 96)) if mtype == 0 else pick((8, 24, 48))
        meta = 3 + len(str(ml))                            # [meta] digits [som] ... [eom]
        if used + tl + ml + meta + 8 > total_len:
            break
        parts.append(torch.randint(0, text_vocab, (tl,), generator = g))
        parts.append((mtype, torch.randn(ml, dims[mtype], generator = g)))
        used += tl + ml + meta
    parts.append(torch.randint(0, text_vocab, (total_len - used,), generator = g))
    return parts


def config4_batch(batch: int, seed: int = 0, **kw):
    return [config4_sample(seed * 65537 + b, **kw) for b in range(batch)]


def text_batch(batch: int, seq: int, vocab: int = 256, seed: int = 0) -> torch.Tensor:
    return torch.randint(0, vocab, (batch, seq), generator = _gen(31337 + seed))


def sampling_prompts(n_each: int, text_vocab: int, dim_latent: int, noise_len: int, seed: int):
    """(prompts, init_modality_noise) of the config-5 sampling fixtures: 4 x n_each mixed prompts (raw text / raw modality / None /
    text + modality) and the initial noise of the decoded modality"""
    g = _gen(seed)
    prompts = []
    for _ in range(n_each):
        prompts.append(torch.randint(0, text_vocab, (16,), generator = g))
        prompts.append((0, torch.randn(int(torch.randint(4, 33, (1,), generator = g)), dim_latent, generator = g)))
        prompts.append(None)
        prompts.append([torch.randint(0, text_vocab, (8,), generator = g), (0, torch.randn(int(torch.randint(6, 33, (1,), generator = g)), dim_latent, generator = g))])
    return prompts, torch.randn(noise_len, dim_latent, generator = g)
