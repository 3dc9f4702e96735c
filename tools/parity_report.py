#!/usr/bin/env python
"""Prints, per reference-generated fixture, the relative error of the loss / breakdown and the worst hidden-state and gradient-fingerprint errors of the
CUDA path (the numbers the parity tests bound).  Run once per engine option, e.g.  TFX_HIDDEN_BF16=1 python tools/parity_report.py"""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch
from helpers import load_golden, golden_inputs, golden_noise, grad_fingerprint, hidden_rows, unpack_rows
from transfusion_pytorch_b200 import Transfusion, synth

def rel(a, b): return abs(a - b) / max(abs(b), 1e-12)
print('options:', {k: v for k, v in os.environ.items() if k.startswith('TFX_')})
for name in ('small_one_modality', 'small_two_modalities', 'config2_b2', 'config4_d8', 'small_laser_vres', 'small_clean'):
    fx = load_golden(name)
    torch.manual_seed(0)
    model = Transfusion(**fx['ctor']).cuda(); synth.fill_parameters_(model, seed = fx['seed']); model.eval()
    batch = golden_inputs(name)
    loss, bd = model(batch, times = fx['times'], return_breakdown = True, noise = golden_noise(fx, batch, model.dim_latents))
    rb, st = model._last_batch, model.engine.state
    hid_err = 0.
    if 'hiddens' in fx:
        for l, h in enumerate(fx['hiddens']):
            ours = unpack_rows(st['hid'][l].float(), rb)
            for b in range(rb.B):
                rows, n = hidden_rows(fx, int(rb.seq_lens[b]))
                hid_err = max(hid_err, ((ours[b, rows].cpu() - h[b, :n]).abs().max() / h[b, :n].abs().max()).item())
    loss.backward()
    fp = grad_fingerprint((n, p.grad) for n, p in model.named_parameters() if p.grad is not None)
    gerr = max(max(abs(fp[k]['stats'][2].item() - v['stats'][2].item()), abs(fp[k]['stats'][3].item() - v['stats'][3].item())) / max(v['stats'][3].item(), 1e-12) for k, v in fx['grads'].items())
    print(f'{name:22s} loss {loss.item():.6f} ref {fx["loss"].item():.6f} rel {rel(loss.item(), fx["loss"].item()):.2e} | text rel {rel(bd.text.item(), fx["text_loss"].item()):.2e} | flow rel '
          f'{max(rel(a.item(), b.item()) for a, b in zip(bd.flow, fx["flow_losses"])):.2e} | hiddens {hid_err:.2e} | grad fingerprints {gerr:.2e}')
