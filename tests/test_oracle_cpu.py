"""CPU: the oracle restatement (oracle/torch_reference.py) is pinned against the golden fixtures, which are
outputs of the reference itself (oracle/make_golden.py).  Also exercises the product's host logic (pack/route,
API glue) end to end by injecting the oracle engine - the product itself never selects it."""
import pytest
import torch

from helpers import load_golden, golden_inputs, golden_noise, grad_fingerprint, hidden_rows
from transfusion_pytorch_b200 import Transfusion, synth
from oracle.torch_reference import OracleEngine

REL = 2e-5          # fp32 restatement vs fp32 reference


def build(fx):
    torch.manual_seed(0)
    model = Transfusion(**fx['ctor'])
    synth.fill_parameters_(model, seed = fx['seed'])
    model.eval()
    model._engine = OracleEngine(model)
    return model


def check_grads(model, fx, tol):
    fp = grad_fingerprint((n, p.grad) for n, p in model.named_parameters() if p.grad is not None)
    assert set(fx['grads']) <= set(fp), f'missing gradients: {sorted(set(fx["grads"]) - set(fp))[:5]}'
    for k, v in fx['grads'].items():
        ref_n = max(v['stats'][3].item(), 1e-12)
        assert abs(fp[k]['stats'][2].item() - v['stats'][2].item()) / ref_n < tol, k
        assert abs(fp[k]['stats'][3].item() - v['stats'][3].item()) / ref_n < tol, k


@pytest.mark.parametrize('name', ['small_one_modality', 'small_two_modalities'])
def test_oracle_matches_reference_small(name):
    fx = load_golden(name)
    model = build(fx)
    batch = golden_inputs(name)
    loss, bd = model(batch, times = fx['times'], return_breakdown = True, noise = golden_noise(fx, batch, model.dim_latents))
    rb = model._last_batch
    assert rb.modality_positions == fx['modality_positions']          # bit-exact span indices
    assert rb.total_tokens == fx['total_tokens']
    assert abs(loss.item() - fx['loss'].item()) / fx['loss'].item() < REL
    assert abs(bd.text.item() - fx['text_loss'].item()) / fx['text_loss'].item() < REL
    for a, b in zip(bd.flow, fx['flow_losses']):
        assert abs(a.item() - b.item()) / b.item() < REL
    st = model._engine.state
    for l, h in enumerate(fx['hiddens']):
        ours = st['hiddens'][l]
        for b in range(rb.B):
            rows, n = hidden_rows(fx, int(rb.seq_lens[b]))
            assert torch.allclose(ours[b, rows], h[b, :n], atol = 2e-4, rtol = 1e-4), f'hidden {l} sample {b}'
    loss.backward()
    check_grads(model, fx, 1e-3)


def test_oracle_matches_reference_text_only():
    fx = load_golden('config1_text_only')
    model = build(fx)
    text = synth.text_batch(4, 257, seed = 3)
    loss = model(text)
    assert abs(loss.item() - fx['loss'].item()) / fx['loss'].item() < REL
    loss.backward()
    check_grads(model, fx, 1e-3)
    logits = model.forward_text(text[:, :-1], return_loss = False)
    assert torch.allclose(logits[:, -1], fx['logits_last'], atol = 2e-4, rtol = 1e-4)
    gen = model.generate_text_only(text[:, :fx['prompt_len']], fx['gen_len'], temperature = 0.)
    assert torch.equal(gen.cpu(), fx['generated'])                    # greedy tokens bit-exact


def test_oracle_matches_reference_config2():
    fx = load_golden('config2_b2')
    model = build(fx)
    batch = golden_inputs('config2_b2')
    with torch.no_grad():
        rb_check = None
    loss, bd = model(batch, times = fx['times'], return_breakdown = True, noise = golden_noise(fx, batch, model.dim_latents))
    rb = model._last_batch
    assert rb.modality_positions == fx['modality_positions'] == [[(0, 206, 256), (0, 668, 256)]] * 2     # SURVEY.md 8(c) known answer
    assert rb.total_tokens == 2050 and rb.M == 2048
    assert abs(loss.item() - fx['loss'].item()) / fx['loss'].item() < REL
    emb = model._engine.state['embed']
    assert torch.allclose(emb[:, fx['embed_rows']], fx['embed'], atol = 2e-4, rtol = 1e-4)


def test_oracle_matches_reference_config4_depth8():
    """BASELINE.json configs[3] at the graded width / depth: two modality types, many short spans (fixture from the reference itself)"""
    fx = load_golden('config4_d8')
    model = build(fx)
    batch = golden_inputs('config4_d8')
    loss, bd = model(batch, times = fx['times'], return_breakdown = True, noise = golden_noise(fx, batch, model.dim_latents))
    rb = model._last_batch
    assert rb.modality_positions == fx['modality_positions'] and all(len(p) >= 8 for p in rb.modality_positions)
    assert rb.total_tokens == fx['total_tokens'] == 2050
    assert abs(loss.item() - fx['loss'].item()) / fx['loss'].item() < REL
    assert len(bd.flow) == 2 and all(abs(a.item() - b.item()) / b.item() < REL for a, b in zip(bd.flow, fx['flow_losses']))
    emb = model._engine.state['embed']
    assert torch.allclose(emb[:, fx['embed_rows']], fx['embed'], atol = 2e-4, rtol = 1e-4)
