"""Bring-up diagnostics on the GPU box: run the B200 path on a golden case and print, layer by layer, how far
each hidden state is from the reference's (tests/golden).  Not a test; prints only."""
import sys, os, traceback
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch
from helpers import load_golden, golden_inputs, golden_noise, grad_fingerprint, hidden_rows, unpack_rows
from transfusion_pytorch_b200 import Transfusion, synth


def rel(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).abs().max() / b.abs().max().clamp(min = 1e-9)).item(), ((a - b).norm() / b.norm().clamp(min = 1e-9)).item()


def run(name):
    fx = load_golden(name)
    torch.manual_seed(0)
    model = Transfusion(**fx['ctor']).cuda()
    synth.fill_parameters_(model, seed = fx['seed'])
    model.eval()
    batch = golden_inputs(name)
    noise = golden_noise(fx, batch, model.dim_latents)
    loss, bd = model(batch, times = fx['times'], return_breakdown = True, noise = noise)
    torch.cuda.synchronize()
    rb = model._last_batch
    print(f'== {name}: loss {loss.item():.6f} (ref {fx["loss"].item():.6f})  text {bd.text.item():.6f} (ref {fx["text_loss"].item():.6f})  '
          f'flow {[round(f.item(), 6) for f in bd.flow]} (ref {[round(f.item(), 6) for f in fx["flow_losses"]]})')
    print('   positions equal:', rb.modality_positions == fx['modality_positions'], ' total_tokens', rb.total_tokens, fx['total_tokens'])
    st = model.engine.state
    def tokens(ours, ref, fx_):
        """the rows of real tokens of every sample (the padding rows of the reference's batch layout are not ours to match), honouring hidden_stride"""
        pairs = [(ours[b, rows], ref[b, :n]) for b in range(rb.B) for rows, n in [hidden_rows(fx_, int(rb.seq_lens[b]))]]
        return torch.cat([o for o, _ in pairs]), torch.cat([r for _, r in pairs])
    if 'hiddens' in fx:
        for l, h in enumerate(fx['hiddens']):
            ours, ref = tokens(unpack_rows(st['hid'][l], rb), h, fx)
            print(f'   hidden[{l}] max-rel {rel(ours, ref)[0]:.3e}  l2-rel {rel(ours, ref)[1]:.3e}')
    emb = unpack_rows(st['out'], rb)
    if 'embed_rows' in fx:
        print('   embed rows rel', rel(emb[:, fx['embed_rows']], fx['embed']))
    else:
        print('   embed rel', rel(*tokens(emb, fx['embed'], {})))
    loss.backward()
    torch.cuda.synchronize()
    fp = grad_fingerprint((n, p.grad) for n, p in model.named_parameters() if p.grad is not None)
    worst = []
    for k, v in fx['grads'].items():
        if k not in fp:
            print('   MISSING grad', k); continue
        ref_n = v['stats'][3].item()
        d_proj = abs(fp[k]['stats'][2].item() - v['stats'][2].item())
        d_norm = abs(fp[k]['stats'][3].item() - ref_n)
        worst.append((max(d_proj, d_norm) / max(ref_n, 1e-12), k, fp[k]['stats'][3].item(), ref_n))
    worst.sort(reverse = True)
    for w in worst[:12]:
        print(f'   grad {w[1]:60s} err/|g| {w[0]:.3e}  |g| ours {w[2]:.4e} ref {w[3]:.4e}')
    print(f'   grads compared: {len(worst)}; median err {sorted(x[0] for x in worst)[len(worst) // 2]:.3e}')


if __name__ == '__main__':
    for name in (sys.argv[1:] or ['small_one_modality', 'small_two_modalities', 'config2_b2']):
        try:
            run(name)
        except Exception:
            traceback.print_exc()
