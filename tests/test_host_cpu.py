"""CPU: host logic - pack/route descriptor invariants against the reference's mask / position formulas,
special-token layout, state_dict parity, and that the C-ABI library loads and exports every symbol declared in
include/tfx_b200.h (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from transfusion_pytorch_b200 import Transfusion, synth, _lib
from transfusion_pytorch_b200.modality_processing import pack_batch, pack_text_only, get_processing_strategy

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def small_model(**kw):
    return Transfusion(num_text_tokens = 64, dim_latent = (32, 16), modality_default_shape = ((4,), (2,)), transformer = dict(dim = 128, depth = 2, heads = 2), **kw)


def test_special_token_layout_config2():
    m = Transfusion(num_text_tokens = 256, dim_latent = 384, modality_default_shape = (256,), transformer = dict(dim = 512, depth = 8))
    assert (m.sos_id, m.eos_id, m.null_text_id, m.som_ids, m.eom_ids, m.meta_id) == (256, 257, 258, [259], [260], 261)   # SURVEY.md 8(c)
    assert m.text_embed.weight.shape[0] == 390
    assert sum(p.numel() for p in m.parameters()) == 79_545_712
    assert m.char_tokenizer('256').tolist() == [312, 315, 316]
    assert m.decode_chars(m.char_tokenizer('12,7')) == '12,7'


def test_known_answer_positions_and_meta_tokens():
    m = Transfusion(num_text_tokens = 256, dim_latent = 384, modality_default_shape = (256,), transformer = dict(dim = 512, depth = 8))
    s = synth.config2_sample(0)
    rb = pack_batch([[torch.tensor([m.sos_id]), *s, torch.tensor([m.eos_id])]], torch.rand(1, 2), m, return_loss = True, return_embed = False)
    assert rb.modality_positions == [[(0, 206, 256), (0, 668, 256)]]
    assert rb.total_tokens == 1025 and rb.M == 1024
    ids = rb.text_id[201:206].tolist()
    assert ids == [261, 312, 315, 316, 259]                                 # [meta] '2' '5' '6' [som]
    assert rb.text_id[462] == 260                                           # [eom]
    assert rb.S == 512 and rb.n_cond == 2 and rb.n_type_tokens == [512]


def naive_mask(n, positions):
    """the reference's formula (transfusion.py:452-470): causal OR (i >= off AND j < off+len)"""
    i = np.arange(n)[:, None]; j = np.arange(n)[None, :]
    mask = i >= j
    for _, off, ln in positions:
        mask |= (i >= off) & (j < off + ln)
    return mask


def ref_rotary_positions(n, positions):
    """transfusion.py:398-415"""
    seq = np.arange(n)
    extra = np.zeros(n, dtype = bool)
    for _, off, ln in positions:
        extra |= (seq > off) & (seq < off + ln)
    return seq - np.cumsum(extra)


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_descriptor_equals_reference_mask_and_positions(seed):
    m = small_model()
    batch = synth.config4_batch(3, seed = seed, total_len = 200, dims = (32, 16), text_vocab = 64)
    samples = [[torch.tensor([m.sos_id]), *s, torch.tensor([m.eos_id])] for s in batch]
    n_mod = max(sum(isinstance(p, tuple) for p in s) for s in batch)
    rb = pack_batch(samples, torch.rand(3, n_mod), m, return_loss = True, return_embed = False)
    for b in range(rb.B):
        s0, n = int(rb.cu[b]), int(rb.seq_lens[b])
        lim = rb.kv_limit[s0:s0 + n] - s0
        ours = np.arange(n)[None, :] <= lim[:, None]
        assert (ours == naive_mask(n, rb.modality_positions[b])).all()
        assert (rb.rope_pos[s0:s0 + n] == ref_rotary_positions(n, rb.modality_positions[b])).all()
        is_mod = rb.cond_row[s0:s0 + n] >= 0
        ref_is_mod = np.zeros(n, dtype = bool)
        for _, off, ln in rb.modality_positions[b]:
            ref_is_mod[off:off + ln] = True
        assert (is_mod == ref_is_mod).all()
    # tiles cover every (query, visible key) pair and never straddle sequences
    seq_of = np.repeat(np.arange(rb.B), rb.seq_lens)
    for q0, qe, k0, ke in zip(rb.tile_q0, rb.tile_qend, rb.tile_kv0, rb.tile_kvend):
        assert seq_of[q0] == seq_of[qe - 1] and k0 == rb.cu[seq_of[q0]]
        assert rb.kv_limit[q0:qe].max() < ke
    for k0, ke, q0, qe in zip(rb.kt_kv0, rb.kt_kvend, rb.kt_q0, rb.kt_qend):
        b = seq_of[k0]
        rows = np.arange(rb.cu[b], rb.cu[b + 1])
        sees = rows[(rb.kv_limit[rows] >= k0)]
        sees = sees[(sees >= k0) | (rb.kv_limit[sees] >= k0)]
        first = rows[(rb.kv_limit[rows] >= k0) & ((rows >= k0) | True)].min()
        assert q0 <= first and qe == rb.cu[b + 1]
    # labels: next token, ignored at modality positions / null ids / last position
    assert rb.n_valid == int((rb.label >= 0).sum()) > 0


def test_empty_and_text_only_inputs():
    m = small_model()
    rb = pack_batch([[torch.tensor([m.sos_id]), torch.randint(0, 64, (5,)), torch.tensor([m.eos_id])], [torch.tensor([m.sos_id]), torch.tensor([m.eos_id])]],
                    None, m, return_loss = True, return_embed = False)
    assert rb.S == 0 and rb.n_cond == 0 and rb.modality_positions == [[], []] and rb.total_tokens == 9 and rb.M == 7
    rt = pack_text_only(torch.randint(0, 64, (2, 9)), return_loss = True)
    assert rt.M == 16 and (rt.kv_limit == np.arange(16)).all() and (rt.rope_pos[:8] == np.arange(8)).all()


def test_all_strategy_names_resolve_and_agree():
    m = small_model()
    batch = [[torch.tensor([m.sos_id]), *s, torch.tensor([m.eos_id])] for s in synth.config4_batch(2, seed = 5, total_len = 120, dims = (32, 16), text_vocab = 64)]
    times = torch.rand(2, 8)
    outs = [get_processing_strategy(n)(batch, times, m, need_axial_pos_emb = False, return_loss = True, return_embed = False) for n in ('naive', 'grouped', 'flat', 'hybrid', 'auto')]
    for o in outs[1:]:
        assert o.modality_positions == outs[0].modality_positions and (o.text_id == outs[0].text_id).all()
    with pytest.raises(AssertionError):
        get_processing_strategy('nope')


def test_validation_errors_match_reference_conventions():
    m = small_model()
    with pytest.raises(AssertionError):
        pack_batch([[(5, torch.randn(4, 32))]], torch.rand(1, 1), m, return_loss = False, return_embed = True)      # type out of range
    with pytest.raises(AssertionError):
        pack_batch([[(0, torch.randn(4, 31))]], torch.rand(1, 1), m, return_loss = False, return_embed = True)      # wrong latent dim
    with pytest.raises(NotImplementedError):
        Transfusion(num_text_tokens = 8, transformer = dict(dim = 128, depth = 1, dim_head = 32))


def test_state_dict_interchange_with_the_reference():
    """weight interchange contract (SURVEY.md 8(b)): identical state_dict keys, shapes and dtypes as the reference for configs 1, 2 and 4, checked
    against the reference's own listing (tests/golden/state_dict_keys.json, written by oracle/make_golden.py from the reference); a checkpoint with
    exactly the reference's keys, shapes and dtypes loads strictly into this model."""
    import json
    from helpers import STATE_DICT_CTORS
    listing = json.load(open(os.path.join(ROOT, 'tests', 'golden', 'state_dict_keys.json')))
    assert sorted(listing) == sorted(STATE_DICT_CTORS)
    for name, ctor in STATE_DICT_CTORS.items():
        ours = Transfusion(**ctor)
        sd = ours.state_dict()
        mine = {k: [list(v.shape), str(v.dtype)] for k, v in sd.items()}
        want = listing[name]
        assert mine == want, (sorted(set(mine) ^ set(want))[:6], name)
        theirs = {k: torch.full(shape, 0.5, dtype = getattr(torch, dtype.split('.')[1])) for k, (shape, dtype) in want.items()}
        ours.load_state_dict(theirs)                                          # reference-shaped checkpoint -> this model
        assert all(torch.equal(v, theirs[k]) for k, v in ours.state_dict().items())
    assert len(listing['config2']) == 206 and sum(int(np.prod(v[0])) for k, v in listing['config2'].items() if 'weights' not in k) >= 79_545_712


def test_cabi_library_exports_every_declared_symbol():
    assert _lib.library_present(), 'libtfx_b200.so not built (run __graft_entry__.build())'
    lib = ctypes.CDLL(_lib.LIB_PATH)
    header = open(os.path.join(ROOT, 'include', 'tfx_b200.h')).read()
    declared = set(re.findall(r'\b(tfx_[a-z0-9_]+)\s*\(', header))
    assert len(declared) >= 30
    for name in sorted(declared):
        assert hasattr(lib, name), f'{name} declared in include/tfx_b200.h but not exported'
    assert set(_lib.EXPORTED) == declared
    lib.tfx_version.restype = ctypes.c_int
    assert lib.tfx_version() == 200


def test_product_fails_loudly_without_cuda():
    m = small_model()
    if torch.cuda.is_available():
        pytest.skip('CUDA present')
    with pytest.raises(Exception) as ei:
        m(synth.config4_batch(1, seed = 0, total_len = 80, dims = (32, 16), text_vocab = 64))
    assert 'CUDA' in str(ei.value) or 'cuda' in str(ei.value)


def test_pack_is_the_host_half_of_forward_and_tile_tables_cover_the_mask():
    """`Transfusion.pack` (what DataParallelTrainer runs ahead of the device step) returns the descriptor `forward` would build;
    the 128-row tables of the tcgen05 attention kernels cover every visible (query, key) pair; the persistent-grid order is a
    permutation sorted by work."""
    m = small_model()
    batch = synth.small_batch(3, seed = 5, dim_latent = 32, text_vocab = 64)
    nm = max(sum(torch.is_tensor(p) and p.is_floating_point() for p in s) for s in batch)
    times = torch.rand(3, nm, generator = torch.Generator().manual_seed(0))
    m.eval()
    rb, t = m.pack(batch, times = times)
    assert t is times and rb.M == int(rb.seq_lens.sum()) and rb.has_labels
    seq_of = np.repeat(np.arange(rb.B), rb.seq_lens)
    for q0, qe, k0, ke in zip(rb.t2_q0, rb.t2_qend, rb.t2_kv0, rb.t2_kvend):
        assert qe - q0 <= 128 and seq_of[q0] == seq_of[qe - 1] and k0 == rb.cu[seq_of[q0]] and rb.kv_limit[q0:qe].max() < ke
    for k0, ke, q0, qe in zip(rb.k2_kv0, rb.k2_kvend, rb.k2_q0, rb.k2_qend):
        b = seq_of[k0]
        rows = np.arange(rb.cu[b], rb.cu[b + 1])
        first = rows[rb.kv_limit[rows] >= k0].min()                  # first query of the sequence that sees a key of this tile
        assert ke - k0 <= 128 and q0 <= first and (q0 - rb.cu[b]) % 128 == 0 and qe == rb.cu[b + 1]
    work = (rb.k2_qend - rb.k2_q0)[rb.k2_order]           # one L2-locality group here (< 8192 tokens): heaviest first
    assert sorted(rb.k2_order.tolist()) == list(range(len(rb.k2_kv0))) and (np.diff(work) <= 0).all()
    # forward work items of the persistent kernel: pairs of adjacent 128-row tiles of ONE sequence, every tile exactly once, heaviest pair first
    first, has_b = rb.p2 >> 1, rb.p2 & 1
    covered = sorted(first.tolist() + (first[has_b == 1] + 1).tolist())
    assert covered == list(range(len(rb.t2_q0)))
    for a, hb in zip(first, has_b):
        assert (rb.t2_q0[a] - rb.cu[seq_of[rb.t2_q0[a]]]) % 256 == 0
        if hb:
            assert seq_of[rb.t2_q0[a + 1]] == seq_of[rb.t2_q0[a]] and rb.t2_kv0[a + 1] == rb.t2_kv0[a] and rb.t2_q0[a + 1] == rb.t2_q0[a] + 128
        else:
            assert a + 1 == len(rb.t2_q0) or seq_of[rb.t2_q0[a + 1]] != seq_of[rb.t2_q0[a]]
    nkv = lambda t: (rb.t2_kvend[t] - rb.t2_kv0[t] + 127) // 128
    cost = np.array([nkv(a) + (nkv(a + 1) if hb else 0) for a, hb in zip(first, has_b)])
    assert (np.diff(cost) <= 0).all()


def test_step_graph_signature_ignores_data_but_not_shape():
    from transfusion_pytorch_b200.data_parallel import DataParallelTrainer
    from transfusion_pytorch_b200.engine import Engine
    m = small_model()
    a = synth.small_batch(2, seed = 1, dim_latent = 32, text_vocab = 64)
    b = [[p.clone() if torch.is_tensor(p) else p for p in s] for s in a]
    for s in b:
        for j, p in enumerate(s):
            if torch.is_tensor(p) and not p.is_floating_point():
                s[j] = (p + 1) % 64                                     # same shapes, different token ids
    nm = max(sum(torch.is_tensor(p) and p.is_floating_point() for p in s) for s in a)
    times = torch.rand(2, nm)
    ra, _ = m.pack(a, times = times)
    rb_, _ = m.pack(b, times = times)
    rc, _ = m.pack(a[:1], times = times[:1])
    sig = lambda r: DataParallelTrainer._signature(r, Engine)
    assert sig(ra) == sig(rb_) and sig(ra) != sig(rc)


def test_ctypes_signatures_match_the_header_prototypes():
    """every prototype of include/tfx_b200.h against the ctypes argtypes in _lib.SIGNATURES: same arity, same scalar classes
    (pointer / int / long long / float) in the same order - a mismatch would corrupt arguments silently."""
    import ctypes as C
    header = open(os.path.join(ROOT, 'include', 'tfx_b200.h')).read()
    header = re.sub(r'/\*.*?\*/', ' ', header, flags = re.S)
    protos = dict(re.findall(r'\bint\s+(tfx_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;', header, flags = re.S))
    def cls(arg):
        a = ' '.join(arg.split())
        if '*' in a: return C.c_void_p
        if a.startswith('unsigned long long'): return C.c_ulonglong
        if a.startswith('long long'): return C.c_longlong
        if a.startswith('float'): return C.c_float
        if a.startswith('int'): return C.c_int
        raise AssertionError(f'unrecognised parameter: {a!r}')
    checked = 0
    for name, argtypes in _lib.SIGNATURES.items():
        assert name in protos, f'{name} has ctypes argtypes but no prototype'
        params = [x for x in protos[name].split(',') if x.strip() and x.strip() != 'void']
        want = [cls(x) for x in params]
        assert len(want) == len(argtypes), f'{name}: header has {len(want)} parameters, _lib declares {len(argtypes)}'
        assert want == list(argtypes), f'{name}: parameter classes differ: {[w.__name__ for w in want]} vs {[a.__name__ for a in argtypes]}'
        checked += 1
    assert checked >= 35


def test_bench_clock_sampler_keeps_the_rows_of_the_timed_region(monkeypatch):
    """bench.py samples clocks from a separate process that starts long before the timed region: only rows stamped inside [start(), stop] are kept, and a
    region shorter than a polling period falls back to the nearest sample.  (The real poller talks to NVML; a fake one prints the same row format.)"""
    import importlib, sys, time
    sys.path.insert(0, ROOT)
    bench = importlib.import_module('bench')
    fake = ("import sys, time\nperiod = float(sys.argv[4])\nn = 0\nwhile True:\n"
            "    print(','.join([repr(time.time()), str(1500 + n), '1965', '700.0', 'Not Active', 'Not Active', 'Not Active', 'Active']), flush = True)\n"
            "    n += 1; time.sleep(period)\n")
    monkeypatch.setattr(bench.ClockSampler, 'POLLER', fake)
    s = bench.ClockSampler(0, period = 0.1)
    time.sleep(0.6)                      # "warm-up": rows before start() must not count
    s.start(); time.sleep(0.45); s.stop()
    out = s.summary()
    assert 3 <= out['samples'] <= 6 and out['sm_mhz'] >= 1504 and out['sm_max_mhz'] == 1965 and out['reasons'] == ['sw_power_cap']
    s = bench.ClockSampler(0, period = 0.2)
    time.sleep(0.5)
    s.start(); s.stop()                  # empty region: the nearest sample stands in
    assert s.summary()['samples'] == 1


def test_axial_pos_emb_tables_and_pack_coordinates_match_the_reference_module():
    """`add_pos_emb` (T.py:1383-1403, 2792-2796; MP.py:1003-1046): the engine's factorised tables + coordinate gather reproduce
    `ContinuousAxialPositionalEmbedding(axial_dims, flatten = True)` per instance (shim restatement of the un-vendored package: parity unpinned upstream),
    its parameter gradients match autograd, and pack_batch emits the row-major coordinates of every latent row."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, 'oracle', 'shims'))
    from axial_positional_embedding import ContinuousAxialPositionalEmbedding
    from transfusion_pytorch_b200.engine import posemb_tables, posemb_add, posemb_backward
    torch.manual_seed(0)
    D = 16
    ref = ContinuousAxialPositionalEmbedding(D, 2)
    params = [tuple(p.detach().clone() for p in (m[0].weight, m[0].bias, m[2].weight, m[2].bias)) for m in ref.mlps]
    shapes = [(2, 3), (3, 2), (4, 2), (1, 5)]
    lens = (8, 8)                                         # batch maximum (4, 5) rounded up to a multiple of 8
    coords = [torch.cat([torch.from_numpy(np.unravel_index(np.arange(h * w), (h, w))[a]) for h, w in shapes]).int() for a in range(2)]
    rows = torch.zeros(sum(h * w for h, w in shapes), D)
    tabs = posemb_tables(params, lens, 'cpu')
    posemb_add(rows, tabs, coords)
    want = torch.cat([ref(torch.tensor(sh), flatten = True) for sh in shapes])
    assert torch.allclose(rows, want.detach(), atol = 1e-5)
    d = torch.randn_like(rows)
    (want * d).sum().backward()
    grads = [tuple(torch.zeros_like(p) for p in ps) for ps in params]
    posemb_backward(d, tabs, coords, params, grads)
    for m, gs in zip(ref.mlps, grads):
        for p, g in zip((m[0].weight, m[0].bias, m[2].weight, m[2].bias), gs):
            assert torch.allclose(g, p.grad, atol = 1e-4, rtol = 1e-4)
    # pack: coordinates of the compact rows, table lengths
    model = Transfusion(num_text_tokens = 64, dim_latent = 32, modality_default_shape = (2, 2), add_pos_emb = True, modality_num_dim = 2,
                        transformer = dict(dim = 128, depth = 2, heads = 2))
    assert 'pos_emb_mlp.0.mlps.1.2.weight' in model.state_dict() and model.state_dict()['pos_emb_mlp.0.mlps.0.0.weight'].shape == (256, 1)
    batch = synth.posemb_batch()
    rb, _ = model.pack(batch, times = torch.rand(3, 2))
    assert rb.pos_max == ((8, 8),)
    off = 0
    for inst in rb.instances:                             # one type: compact rows are the instances in scan order
        c0, c1 = np.unravel_index(np.arange(inst.length), inst.axial_shape)
        assert (rb.pos_c0[off:off + inst.length] == c0).all() and (rb.pos_c1[off:off + inst.length] == c1).all()
        off += inst.length
    assert off == rb.S and (rb.pos_c2 == -1).all()
