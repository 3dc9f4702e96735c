"""Shared helpers of the parity tests: rebuild the exact inputs the golden fixtures were generated from."""
import os

import torch

from transfusion_pytorch_b200 import synth

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')

# constructors of the reference state_dict listing golden/state_dict_keys.json (configs 1, 2 and 4)
STATE_DICT_CTORS = dict(
    config1 = dict(num_text_tokens = 256, transformer = dict(dim = 128, depth = 2)),
    config2 = dict(num_text_tokens = 256, dim_latent = 384, modality_default_shape = (256,), transformer = dict(dim = 512, depth = 8)),
    config4 = dict(num_text_tokens = 256, dim_latent = (384, 192), modality_default_shape = ((4,), (2,)), transformer = dict(dim = 512, depth = 8)))


def load_golden(name):
    fx = torch.load(os.path.join(GOLDEN, f'{name}.pt'), weights_only = False)
    if 'prompt_args' in fx:                          # seeded sampling inputs are rebuilt rather than stored
        fx['prompts'], fx['noise'] = synth.sampling_prompts(**fx['prompt_args'])
    return fx


def hidden_rows(fx, n):
    """(slice of our token rows, number of fixture rows) for a sample of n tokens: fixtures may keep only every `hidden_stride`-th row"""
    step = fx.get('hidden_stride', 1)
    return slice(0, n, step), -(-n // step)


def golden_inputs(name):
    """(batch, times) exactly as oracle/make_golden.py built them."""
    if name in ('small_one_modality', 'small_laser_vres', 'small_velocity', 'small_clean'):
        return synth.small_batch(3, seed = 1, dim_latent = 32, text_vocab = 64)
    if name == 'small_posemb':
        return synth.posemb_batch()
    if name == 'small_two_modalities':
        return synth.config4_batch(2, seed = 2, total_len = 300, dims = (32, 16), text_vocab = 64)
    if name == 'config2_b2':
        return synth.config2_batch(2, seed = 4)
    if name == 'config4_d8':
        return synth.config4_batch(2, seed = 31)
    raise KeyError(name)


def golden_noise(fx, batch, dim_latents):
    """Per-type noise tensors in the order the reference's flat strategy drew them (one randn_like per type,
    types in order of first appearance)."""
    order = []
    for s in batch:
        for p in s:
            t = p[0] if isinstance(p, tuple) else (0 if (torch.is_tensor(p) and p.is_floating_point()) else None)
            if t is not None and t not in order:
                order.append(t)
    noise = [None] * len(dim_latents)
    for k, t in enumerate(order):
        rows, dl = fx['noise_shapes'][k]
        assert dl == dim_latents[t]
        noise[t] = torch.randn(rows, dl, generator = torch.Generator().manual_seed(9000 + k + 17 * fx['seed']))
    return noise


def grad_fingerprint(named_grads):
    out = {}
    for name, g in named_grads:
        g = g.detach().float().reshape(-1).cpu()
        proj = torch.randn(g.numel(), generator = torch.Generator().manual_seed(1234))
        out[name] = dict(stats = torch.stack([g.sum(), g.abs().sum(), (g * proj).sum(), g.norm()]).double(), head = g[:8].clone())
    return out


def unpack_rows(packed, rb, width = None):
    """packed [M, d] -> padded [B, n_max, d] like the reference's batch layout"""
    n_max = int(rb.seq_lens.max())
    d = packed.shape[1] if width is None else width
    out = packed.new_zeros((rb.B, n_max, d))
    for b in range(rb.B):
        out[b, :rb.seq_lens[b]] = packed[rb.cu[b]:rb.cu[b + 1], :d]
    return out


def flatten_sample(model, sample):
    """[('t', id) ...] / [('m', (type, latents))] items of one sample (list of text tensors and (type, latents) tuples)"""
    items = []
    for p in sample:
        if torch.is_tensor(p):
            items += [('t', int(v)) for v in p.reshape(-1).tolist()]
        else:
            items.append(('m', (p[0], p[1].detach().float().cpu())))
    return items


def compare_sampling(model, out, fx, bound, lat_tol):
    """Compare `sample_many` output with a reference fixture that carries the reference's top-2 logit margins per sampled token.

    Text must be IDENTICAL up to the first sampled token whose reference margin is below `bound` (the stated bf16 logit-noise bound): a
    mismatch at a larger margin fails; at a smaller one the sample has legitimately diverged (greedy decoding of two near-tied logits) and
    the comparison of that sample stops there.  Every modality decoded before that point must match within `lat_tol` of its max magnitude.
    Returns a per-sample report: dict(matched = sampled tokens that agree, total = sampled tokens in the fixture, diverged_at = index or None,
    margin = reference margin at the divergence, latent_err = [relative errors of the compared modalities])."""
    import copy
    report = []
    forced = fx['kw'].get('force_modality_at_start')
    for i, (ours, ref) in enumerate(zip(out, fx['samples'])):
        prep = model.prepare_prompt_sample(copy.deepcopy(fx['prompts'][i]), forced)[0]
        n_prompt = len(flatten_sample(model, prep))
        a, b = flatten_sample(model, ours), flatten_sample(model, ref)
        margins = fx['margins'][i]
        g, rep = 0, dict(matched = 0, total = len(margins), diverged_at = None, margin = None, latent_err = [])
        prev_mod = False
        for j, (x, y) in enumerate(zip(a, b)):
            sampled = j >= n_prompt and y[0] == 't' and not prev_mod            # the [eom] right after a decoded modality is appended, not sampled
            if x[0] != y[0]:
                assert sampled or (j >= n_prompt and x[0] == 't' and y[0] == 'm'), f'sample {i}: structure differs at item {j} inside the prompt'
            if y[0] == 'm' and x[0] == 'm':
                assert x[1][0] == y[1][0] and x[1][1].shape == y[1][1].shape, f'sample {i}: modality type / shape differs at item {j}'
                if j >= n_prompt:
                    err = ((x[1][1] - y[1][1]).abs().max() / y[1][1].abs().max().clamp(min = 1e-9)).item()
                    rep['latent_err'].append(err)
                    assert err < lat_tol, f'sample {i}: decoded modality at item {j} differs by {err:.3e} of its max magnitude'
                else:
                    assert torch.equal(x[1][1], y[1][1])
                prev_mod = True
                continue
            if x == y:
                if sampled:
                    g += 1; rep['matched'] += 1
                prev_mod = False
                continue
            # first difference
            assert j >= n_prompt, f'sample {i}: prompt token {j} differs'
            assert sampled, f'sample {i}: non-sampled token at item {j} differs: {x} vs {y}'
            assert margins[g] < bound, f'sample {i}: sampled token {g} differs ({x} vs {y}) although the reference margin {margins[g]:.4f} >= {bound}'
            rep['diverged_at'], rep['margin'] = g, margins[g]
            break
        else:
            assert len(a) == len(b), f'sample {i}: lengths differ without a token mismatch'
        report.append(rep)
    return report
