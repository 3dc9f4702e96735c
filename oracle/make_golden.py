"""TEST INFRASTRUCTURE ONLY - generates tests/golden/*.pt by running the UNMODIFIED reference
(/root/reference, imported through oracle/reference_loader.py with the shims) on the deterministic
synthetic inputs of transfusion_pytorch_b200/synth.py.  Runs in the build container only
(`python -m oracle.make_golden`); the fixtures it writes are committed and are what the GPU tests read.

The reference has no golden vectors of its own (SURVEY.md section 4): these fixtures ARE the pin of the
oracle - outputs of the reference itself on seeded inputs.
"""
from __future__ import annotations

import os
import sys
from unittest import mock

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from oracle.reference_loader import load_reference          # noqa: E402
from transfusion_pytorch_b200 import synth                   # noqa: E402
from helpers import STATE_DICT_CTORS                         # noqa: E402

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def compact(o):
    """clone every tensor of a fixture: torch.save writes the WHOLE storage of a view"""
    if torch.is_tensor(o): return o.detach().clone().contiguous()
    if isinstance(o, dict): return {k: compact(v) for k, v in o.items()}
    if isinstance(o, list): return [compact(v) for v in o]
    if isinstance(o, tuple): return tuple(compact(v) for v in o)
    return o


def grad_fingerprint(model):
    """Per-parameter gradient fingerprint: [sum, abs-sum, projection on a fixed pseudo-random vector, l2] + first 8 values."""
    out = {}
    for name, p in model.named_parameters():
        if p.grad is None:
            continue
        g = p.grad.detach().float().reshape(-1)
        gen = torch.Generator().manual_seed(1234)
        proj = torch.randn(g.numel(), generator = gen)
        out[name] = dict(stats = torch.stack([g.sum(), g.abs().sum(), (g * proj).sum(), g.norm()]).double(), head = g[:8].clone())
    return out


def count_modalities(batch):
    return max(sum(1 for p in s if isinstance(p, tuple) or (torch.is_tensor(p) and p.is_floating_point())) for s in batch)


def noise_for(rb_like_rows, dl, seed):
    return torch.randn(rb_like_rows, dl, generator = torch.Generator().manual_seed(seed))


def run_interleaved(ref, name, ctor, batch, times, seed, subsample_rows = None, keep_hiddens = True, hidden_stride = 1):
    """hidden_stride: keep every hidden_stride-th token row of the per-layer hiddens (keeps the fixture under 1 MB)"""
    torch.manual_seed(0)
    model = ref.Transfusion(**ctor, modality_processing = 'flat')
    synth.fill_parameters_(model, seed = seed)
    model.eval()                                   # no CFG dropout; nothing else depends on the mode
    n_types = model.num_modalities
    # deterministic noise: the flat strategy draws ONE randn_like per modality type, on the [S_t, dl] concatenation
    calls = []
    def fake_randn_like(t):
        e = noise_for(t.shape[0], t.shape[1], 9000 + len(calls) + 17 * seed)
        calls.append(tuple(t.shape))
        return e.to(t)
    with mock.patch('torch.randn_like', side_effect = fake_randn_like):
        loss, breakdown, hiddens = model(batch, times = times, return_breakdown = True, return_hiddens = True)
    loss.backward()
    # structural ground truth straight from the reference's pack/route
    from transfusion_pytorch.modality_processing import get_processing_strategy
    with torch.no_grad(), mock.patch('torch.randn_like', side_effect = lambda t: torch.zeros_like(t)):
        samples = [[torch.tensor([model.sos_id]), *s, torch.tensor([model.eos_id])] for s in batch]
        samples = [[(0, p) if (torch.is_tensor(p) and p.is_floating_point()) else p for p in s] for s in samples]
        proc = get_processing_strategy('flat')(samples, times, model, need_axial_pos_emb = False, return_loss = True, return_embed = False)
    fx = dict(
        name = name, ctor = ctor, seed = seed, times = times, noise_shapes = calls,
        loss = loss.detach().double(), text_loss = breakdown.text.detach().double(), flow_losses = [f.detach().double() for f in breakdown.flow],
        modality_positions = proc.modality_positions, total_tokens = proc.total_tokens, text = proc.text.clone(),
        grads = grad_fingerprint(model),
    )
    embed = hiddens[-1].detach()
    if subsample_rows is not None:
        fx['embed_rows'] = subsample_rows
        fx['embed'] = embed[:, subsample_rows].clone()
    else:
        fx['embed'] = embed.clone()
        if keep_hiddens:
            fx['hiddens'] = [h.detach()[:, ::hidden_stride].clone() for h in hiddens[:-1]]
            if hidden_stride > 1:
                fx['hidden_stride'] = hidden_stride
    torch.save(compact(fx), os.path.join(GOLDEN, f'{name}.pt'))
    print(f'{name}: loss {loss.item():.6f} text {breakdown.text.item():.6f} flow {[round(f.item(), 6) for f in breakdown.flow]} '
          f'positions[0] {proc.modality_positions[0]} total_tokens {proc.total_tokens}')


def run_text_only(ref, name, ctor, text, seed, prompt_len = 16, gen_len = 40):
    torch.manual_seed(0)
    model = ref.Transfusion(**ctor)
    synth.fill_parameters_(model, seed = seed)
    model.eval()
    loss = model(text)
    loss.backward()
    gen = model.generate_text_only(text[:, :prompt_len], gen_len, temperature = 0.)
    with torch.no_grad():
        logits = model.forward_text(text[:, :-1], return_loss = False)
        # top-2 logit margin of the reference at every generated position (teacher-forced on its own greedy continuation: a causal LM, so these
        # are the logits generation saw): lets the GPU test tell a bf16 near-tie from a real mismatch
        seq = torch.cat((text[:, :prompt_len], gen), dim = -1)
        lg = model.forward_text(seq[:, :-1], return_loss = False)[:, prompt_len - 1:]
        assert torch.equal(lg.argmax(dim = -1), gen)
        top2 = lg.topk(2, dim = -1).values
        margins = (top2[..., 0] - top2[..., 1]).clone()
    fx = dict(name = name, ctor = ctor, seed = seed, loss = loss.detach().double(), grads = grad_fingerprint(model), generated = gen.clone(),
              prompt_len = prompt_len, gen_len = gen_len, logits_last = logits[:, -1].detach().clone(), margins = margins)
    torch.save(compact(fx), os.path.join(GOLDEN, f'{name}.pt'))
    print(f'{name}: loss {loss.item():.6f} generated[0,:8] {gen[0, :8].tolist()}')


def run_sampling(ref, name, ctor, seed):
    """sample_many on mixed prompts, greedy text, fixed init noise, forced modality at start (SURVEY.md 8(d) config 5, shrunk)."""
    torch.manual_seed(0)
    model = ref.Transfusion(**ctor)
    synth.fill_parameters_(model, seed = seed)
    model.eval()
    g = torch.Generator().manual_seed(77)
    dl = ctor['dim_latent']
    prompts = [
        torch.randint(0, ctor['num_text_tokens'], (9,), generator = g),
        (0, torch.randn(5, dl, generator = g)),
        None,
        [torch.randint(0, ctor['num_text_tokens'], (4,), generator = g), (0, torch.randn(7, dl, generator = g))],
    ]
    noise = torch.randn(16, dl, generator = g)
    kw = dict(max_length = 14, text_temperature = 0., cfg_scale = 3., modality_steps = 4, init_modality_noise = noise, force_modality_at_start = (0, (6,)),
              return_unprocessed_modalities = True)
    import copy
    out = model.sample_many(copy.deepcopy(prompts), **kw)
    fx = dict(name = name, ctor = ctor, seed = seed, prompts = prompts, noise = noise, kw = {k: v for k, v in kw.items() if k != 'init_modality_noise'}, samples = out)
    torch.save(compact(fx), os.path.join(GOLDEN, f'{name}.pt'))
    for s in out:
        print('  sample:', [tuple(p.shape) if torch.is_tensor(p) else ('mod', p[0], tuple(p[1].shape)) for p in s])


def text_runs(model, sample, n_prompt_parts):
    """generated text of one output sample as a list of runs (one per text phase), prompt text excluded"""
    runs = []
    for j, part in enumerate(sample):
        if torch.is_tensor(part):
            runs.append(part.tolist())
    return runs


def run_sampling_sized(ref, name, ctor, seed, n_each, mod_len, steps, max_length, force = True):
    """config 5 of SURVEY.md 8(d) at a GPU-meaningful size: 4 x n_each mixed prompts (raw text / raw modality / None / text + modality), greedy text,
    seeded init noise, one forced modality of `mod_len` tokens at the start of every sample, `steps` midpoint steps, cfg 3.
    Besides the outputs, the fixture stores the reference's top-2 logit margin at EVERY sampled text token (`margins[i][k]`), recovered by
    replaying the reference's phase-grouped schedule over the recorded `sample_text_token` calls (every recorded token is checked against the
    output, so a wrong attribution cannot pass silently): the GPU test needs it to tell a bf16 near-tie from a real mismatch."""
    import copy
    torch.manual_seed(0)
    model = ref.Transfusion(**ctor)
    synth.fill_parameters_(model, seed = seed)
    model.eval()
    # the inputs are rebuilt from these arguments by tests/helpers.py:load_golden instead of being stored
    prompt_args = dict(n_each = n_each, text_vocab = ctor['num_text_tokens'], dim_latent = ctor['dim_latent'], noise_len = mod_len, seed = 1234 + seed)
    prompts, noise = synth.sampling_prompts(**prompt_args)
    kw = dict(max_length = max_length, text_temperature = 0., cfg_scale = 3., modality_steps = steps, init_modality_noise = noise, return_unprocessed_modalities = True)
    if force:
        kw['force_modality_at_start'] = (0, (mod_len,))
    calls = []
    tmod = sys.modules['transfusion_pytorch.transfusion']
    orig = tmod.sample_text_token
    def recording(logits, temperature = 1.0, min_p = 0.1):
        out = orig(logits, temperature, min_p)
        lg = logits.detach().float().reshape(-1, logits.shape[-1])
        top2 = lg.topk(2, dim = -1).values
        calls.append([(int(t), float(a - b)) for t, a, b in zip(out.reshape(-1).tolist(), top2[:, 0].tolist(), top2[:, 1].tolist())])
        return out
    with mock.patch.object(tmod, 'sample_text_token', recording):
        out = model.sample_many(copy.deepcopy(prompts), **kw)
    # ---- attribute the recorded rows to (sample, generated-token index) by replaying the schedule (T.py:2225-2250, 2563-2573)
    B = len(out)
    prep = [model.prepare_prompt_sample(copy.deepcopy(p), kw.get('force_modality_at_start'))[0] for p in prompts]
    n_prompt_text = []
    starts_in_modality = []
    runs = []
    for i in range(B):
        pp, oo = prep[i], out[i]
        last_prompt = pp[-1]
        assert torch.is_tensor(last_prompt)
        starts_in_modality.append(int(last_prompt[-1]) in model.som_ids)
        # generated text: the tail of the part that continues the last prompt text, then every later text part
        k0 = len(pp) - 1
        first = oo[k0][last_prompt.numel():].tolist()
        r = [first] if not starts_in_modality[-1] else []
        assert starts_in_modality[-1] is False or len(first) == 0
        r += [part.tolist() for part in oo[k0 + 1:] if torch.is_tensor(part)]
        # a text part right after a decoded modality starts with the [eom] the sampler appended itself (not a sampled token)
        fixed = []
        for j, run in enumerate(r):
            is_after_modality = not (j == 0 and not starts_in_modality[-1])
            fixed.append(run[1:] if is_after_modality else run)
        runs.append(fixed)
    margins = [[] for _ in range(B)]
    cur = [0] * B                       # run index per sample
    ci = 0
    # first tokens (1-D calls) for samples that start in the text phase
    for i in range(B):
        if not starts_in_modality[i]:
            (tok, mg), = calls[ci]; ci += 1
            assert tok == runs[i][0][0], (i, tok, runs[i][0][:3])
            margins[i].append(mg)
    pos = [1 if not starts_in_modality[i] else 0 for i in range(B)]      # next token inside the current run
    def in_text(i):
        return cur[i] < len(runs[i]) and pos[i] < len(runs[i][cur[i]])
    rnd = 0
    while ci < len(calls):
        active = [i for i in range(B) if (rnd > 0 or not starts_in_modality[i]) and cur[i] < len(runs[i]) and (pos[i] < len(runs[i][cur[i]]))]
        # a run that is already complete (e.g. its only token was the first-token sample) does not take part in this round
        while active:
            rows = calls[ci]; ci += 1
            assert len(rows) == len(active), (len(rows), active)
            for (tok, mg), i in zip(rows, active):
                assert tok == runs[i][cur[i]][pos[i]], (i, cur[i], pos[i], tok)
                margins[i].append(mg); pos[i] += 1
            active = [i for i in active if pos[i] < len(runs[i][cur[i]])]
        for i in range(B):               # next round: every sample that finished a run (or waited in the modality phase) moves to its next run
            if rnd > 0 or not starts_in_modality[i]:
                if cur[i] < len(runs[i]):
                    cur[i] += 1; pos[i] = 0
        rnd += 1
    assert all(len(margins[i]) == sum(len(r) for r in runs[i]) for i in range(B)), 'schedule replay did not consume every sampled token'
    fx = dict(name = name, ctor = ctor, seed = seed, prompt_args = prompt_args, kw = {k: v for k, v in kw.items() if k != 'init_modality_noise'}, samples = out,
              generated = [[t for r in runs[i] for t in r] for i in range(B)], margins = margins)
    torch.save(compact(fx), os.path.join(GOLDEN, f'{name}.pt'))
    for i, s in enumerate(out):
        print(f'  sample {i}:', [tuple(p.shape) if torch.is_tensor(p) else ('mod', p[0], tuple(p[1].shape)) for p in s], 'min margin %.4f' % min(margins[i], default = float('nan')))


def run_velocity(ref, name, ctor, batch, times, seed, delta = 1e-3):
    """velocity-consistency training step (T.py:2965-2971, 3084-3088, 3383-3418) with an EMA teacher whose parameters differ from the student's.
    randn_like calls: student draw(s) first, then the teacher's (one per modality type each) - both injected."""
    torch.manual_seed(0)
    model = ref.Transfusion(**ctor, modality_processing = 'flat')
    synth.fill_parameters_(model, seed = seed)
    model.eval()
    ema = model.create_ema(0.99)
    synth.fill_parameters_(ema.ema_model, seed = seed + 5)
    calls = []
    def fake_randn_like(t):
        e = noise_for(t.shape[0], t.shape[1], 9000 + len(calls) + 17 * seed)
        calls.append(tuple(t.shape))
        return e.to(t)
    with mock.patch('torch.randn_like', side_effect = fake_randn_like):
        loss, breakdown = model(batch, times = times, velocity_consistency_ema_model = ema, velocity_consistency_delta_time = delta, return_breakdown = True)
    loss.backward()
    fx = dict(name = name, ctor = ctor, seed = seed, times = times, delta = delta, noise_shapes = calls, loss = loss.detach().double(), text_loss = breakdown.text.detach().double(),
              flow_losses = [f.detach().double() for f in breakdown.flow], velocity_losses = [v.detach().double() for v in breakdown.velocity], grads = grad_fingerprint(model))
    torch.save(compact(fx), os.path.join(GOLDEN, f'{name}.pt'))
    print(f'{name}: loss {loss.item():.6f} flow {[round(f.item(), 6) for f in breakdown.flow]} velocity {[round(v.item(), 6) for v in breakdown.velocity]} draws {calls}')


def write_state_dict_keys(ref):
    """the reference's state_dict keys, shapes and dtypes for configs 1, 2 and 4 (the weight interchange contract of tests/test_host_cpu.py)"""
    import json
    listing = {name: {k: [list(v.shape), str(v.dtype)] for k, v in ref.Transfusion(**ctor).state_dict().items()} for name, ctor in STATE_DICT_CTORS.items()}
    with open(os.path.join(GOLDEN, 'state_dict_keys.json'), 'w') as f:
        json.dump(listing, f, indent = 0, sort_keys = True)


def main():
    os.makedirs(GOLDEN, exist_ok = True)
    ref = load_reference()
    only = os.environ.get('GOLDEN_ONLY', '')

    if only in ('', 'state_dict'):
        write_state_dict_keys(ref)
    if only in ('', 'config5'):
        ctor = dict(num_text_tokens = 256, dim_latent = 384, modality_default_shape = (64,), transformer = dict(dim = 512, depth = 8))
        run_sampling_sized(ref, 'config5_mid', ctor, seed = 21, n_each = 2, mod_len = 64, steps = 8, max_length = 96)
    if only in ('', 'config5free'):
        # no forced modality: samples start in the text phase, [som] tokens are SAMPLED (the never-cached-[som] path of T.py:2337-2349)
        ctor = dict(num_text_tokens = 16, dim_latent = 32, modality_default_shape = (6,), transformer = dict(dim = 128, depth = 2, heads = 2))
        run_sampling_sized(ref, 'sampling_free', ctor, seed = 5, n_each = 2, mod_len = 6, steps = 4, max_length = 40, force = False)
    if only in ('', 'config4'):
        # config 4 (two modalities, span-mask stress) at the graded width / depth, from the reference itself
        ctor = dict(num_text_tokens = 256, dim_latent = (384, 192), modality_default_shape = ((4,), (2,)), transformer = dict(dim = 512, depth = 8))
        batch = synth.config4_batch(2, seed = 31)
        times = torch.rand(2, count_modalities(batch), generator = torch.Generator().manual_seed(5))
        rows = torch.arange(0, 1024, 41)
        run_interleaved(ref, 'config4_d8', ctor, batch, times, seed = 13, subsample_rows = rows)
    if only in ('', 'config1'):
        ctor = dict(num_text_tokens = 256, transformer = dict(dim = 128, depth = 2))
        run_text_only(ref, 'config1_text_only', ctor, synth.text_batch(4, 257, seed = 3), seed = 3)
    if only in ('', 'velocity'):
        ctor = dict(num_text_tokens = 64, dim_latent = 32, modality_default_shape = (4,), transformer = dict(dim = 128, depth = 2, heads = 2))
        batch = synth.small_batch(3, seed = 1, dim_latent = 32, text_vocab = 64)
        times = torch.rand(3, count_modalities(batch), generator = torch.Generator().manual_seed(5))
        run_velocity(ref, 'small_velocity', ctor, batch, times, seed = 1)
    if only in ('', 'variants'):
        # optional attention variants of SURVEY 8(f) rank 4: LASER (T.py:981-983, 1021-1022; config 1's own script uses it, train_text_only.py:70) and
        # the learned value residual (T.py:956-960, 1234)
        ctor = dict(num_text_tokens = 256, transformer = dict(dim = 128, depth = 2, attn_laser = True))
        run_text_only(ref, 'config1_laser', ctor, synth.text_batch(4, 257, seed = 3), seed = 3)
        ctor = dict(num_text_tokens = 64, dim_latent = 32, modality_default_shape = (4,), transformer = dict(dim = 128, depth = 4, heads = 2, attn_laser = True, use_value_residual = True))
        batch = synth.small_batch(3, seed = 1, dim_latent = 32, text_vocab = 64)
        times = torch.rand(3, count_modalities(batch), generator = torch.Generator().manual_seed(5))
        run_interleaved(ref, 'small_laser_vres', ctor, batch, times, seed = 1, hidden_stride = 2)
        # model_output_clean (MP.py:100-126): the model predicts the clean modality in model space; times pushed towards 1 so that the eps clamp is exercised
        ctor = dict(num_text_tokens = 64, dim_latent = 32, modality_default_shape = (4,), model_output_clean = True, transformer = dict(dim = 128, depth = 2, heads = 2))
        times = (torch.rand(3, count_modalities(batch), generator = torch.Generator().manual_seed(7)) * 1.2).clamp(max = 0.999)
        run_interleaved(ref, 'small_clean', ctor, batch, times, seed = 1)
    if only in ('', 'posemb'):
        # axial positional embedding (T.py:1383-1403, 2792-2796; MP.py:1003-1046): 2-D latents of different (h, w) per instance, so that the factorised
        # per-axis tables are evaluated at the batch maximum and sliced per instance.  Upstream package unpinned: the shim's restatement is the oracle.
        ctor = dict(num_text_tokens = 64, dim_latent = 32, modality_default_shape = (2, 2), add_pos_emb = True, modality_num_dim = 2,
                    transformer = dict(dim = 128, depth = 2, heads = 2))
        batch = synth.posemb_batch()
        times = torch.rand(3, count_modalities(batch), generator = torch.Generator().manual_seed(5))
        run_interleaved(ref, 'small_posemb', ctor, batch, times, seed = 1)
    if only:
        return

    ctor = dict(num_text_tokens = 64, dim_latent = 32, modality_default_shape = (4,), transformer = dict(dim = 128, depth = 2, heads = 2))
    run_sampling(ref, 'sampling_small', ctor, seed = 8)
    if os.environ.get('GOLDEN_ONLY_SAMPLING'):
        return

    # (1) small single-modality, ragged, all hiddens kept
    ctor = dict(num_text_tokens = 64, dim_latent = 32, modality_default_shape = (4,), transformer = dict(dim = 128, depth = 2, heads = 2))
    batch = synth.small_batch(3, seed = 1, dim_latent = 32, text_vocab = 64)
    times = torch.rand(3, count_modalities(batch), generator = torch.Generator().manual_seed(5))
    run_interleaved(ref, 'small_one_modality', ctor, batch, times, seed = 1)

    # (2) small, depth 4 (two U-Net skips), two modality types, many short spans
    ctor = dict(num_text_tokens = 64, dim_latent = (32, 16), modality_default_shape = ((4,), (2,)), transformer = dict(dim = 128, depth = 4, heads = 4))
    batch = synth.config4_batch(2, seed = 2, total_len = 300, dims = (32, 16), text_vocab = 64)
    times = torch.rand(2, count_modalities(batch), generator = torch.Generator().manual_seed(6))
    run_interleaved(ref, 'small_two_modalities', ctor, batch, times, seed = 2, hidden_stride = 3)

    # (3) config 1: text-only pretrain shape (train_text_only.py), d=128 depth=2 heads=8
    ctor = dict(num_text_tokens = 256, transformer = dict(dim = 128, depth = 2))
    run_text_only(ref, 'config1_text_only', ctor, synth.text_batch(4, 257, seed = 3), seed = 3)

    # (4) config 2: the graded shape, b = 2 (CPU-feasible), embed subsampled
    ctor = dict(num_text_tokens = 256, dim_latent = 384, modality_default_shape = (256,), transformer = dict(dim = 512, depth = 8))
    batch = synth.config2_batch(2, seed = 4)
    times = synth.config2_times(2, seed = 4)
    rows = torch.tensor([0, 1, 5, 100, 205, 206, 207, 333, 461, 462, 500, 667, 668, 800, 923, 924, 1000, 1023])
    run_interleaved(ref, 'config2_b2', ctor, batch, times, seed = 4, subsample_rows = rows)


if __name__ == '__main__':
    main()
