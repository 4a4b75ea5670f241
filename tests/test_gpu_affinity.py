"""Affinity regressor on the B200: PropPredNet / PropPredNetEnc (libtdiff tdiff_prop_*) against the CPU restatement (oracle.prop) and
against the reference's pinned outputs (tests/golden/prop_pins.npz)."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import prop, restate, synth
from targetdiff_b200 import _lib
from targetdiff_b200.prop_model import PropPredNet, PropPredNetEnc

pytestmark = pytest.mark.gpu
PINS = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'prop_pins.npz'))
DEV = 'cuda:0'
PRED_TOL = dict(rtol=1e-4, atol=1e-3)
H_REL_TOL = 1e-4          # encoder h: max |error| over max |h|


def _model(config, seed, gain=1.0, ligand_dim=prop.LIGAND_FEATURE_DIM):
    if config['encoder']['name'] == 'egnn_enc':
        m = PropPredNetEnc(config, 27, ligand_dim, config['enc_ligand_dim'], config['enc_node_dim'], config['enc_graph_dim'], config['enc_feature_type'])
    else:
        m = PropPredNet(config, 27, ligand_dim)
    sd = prop.make_state_dict(config, seed, gain=gain, ligand_dim=ligand_dim)
    m.load_state_dict(sd, strict=True)
    return m.to(DEV), sd


def _run(model, config, x):
    d = {k: (v.to(DEV) if v is not None else None) for k, v in x.items()}
    args = (d['protein_pos'], d['protein_feat'], d['ligand_pos'], d['ligand_feat'], d['batch_protein'], d['batch_ligand'], d['output_kind'])
    if config['encoder']['name'] == 'egnn_enc':
        args += (d['enc_ligand'], d['enc_node'], d['enc_graph'])
    out, h = model(*args, return_h=True)
    return out.cpu(), h.cpu()


def _oracle(sd, config, x, trace=None):
    return prop.prop_forward(sd, config, x['protein_pos'], x['protein_feat'], x['ligand_pos'], x['ligand_feat'], x['batch_protein'], x['batch_ligand'],
                             x['output_kind'], x['enc_ligand'], x['enc_node'], x['enc_graph'], trace=trace)


def _h_close(got, want):
    err = (got - want).abs().max().item() / max(want.abs().max().item(), 1e-30)
    assert err <= H_REL_TOL, 'encoder h: max error %.3g of max |h|' % err


@pytest.mark.parametrize('name', sorted(prop.PIN_CASES))
def test_affinity_matches_oracle_and_reference(name):
    config, seed = prop.PIN_CASES[name][:2]
    x = prop.pin_inputs(name)
    model, sd = _model(config, seed)
    out, h = _run(model, config, x)
    tr = {}
    want = _oracle(sd, config, x, tr)
    torch.testing.assert_close(out, want, **PRED_TOL)
    _h_close(h, tr['h'])
    p = name + '__'
    torch.testing.assert_close(out, torch.from_numpy(PINS[p + 'pred']), **PRED_TOL)
    rows = torch.from_numpy(PINS[p + 'h_rows'])
    _h_close(h[rows], torch.from_numpy(PINS[p + 'h']))


@pytest.mark.parametrize('name', ['egnn_kinds', 'egnn_1h36'])
def test_edge_set_bit_exact(name):
    """The encoder's graph is the project's full-scan k-NN on the composed positions: same edge set as the reference's knn_graph."""
    config = prop.PIN_CASES[name][0]
    x = prop.pin_inputs(name)
    order = prop.compose_stable(x['batch_protein'], x['batch_ligand'])
    pos = torch.cat([x['protein_pos'], x['ligand_pos']])[order].contiguous().to(DEV)
    batch = torch.cat([x['batch_protein'], x['batch_ligand']])[order]
    counts = torch.bincount(batch).tolist()
    n, k = pos.shape[0], config['encoder']['knn']
    slots = torch.empty(n * k, dtype=torch.int32, device=DEV)
    ne = ctypes.c_int64()
    lib = _lib.load()
    _lib.check(lib.tdiff_knn_graph(ctypes.c_void_p(pos.data_ptr()), n, _lib.i32_array(counts), len(counts), k,
                                   ctypes.c_void_p(slots.data_ptr()), None, ctypes.byref(ne), None))
    s = slots.view(n, k).cpu().long()
    dst = torch.arange(n).unsqueeze(1).expand(n, k)
    keep = s >= 0
    key = (dst[keep] * n + s[keep]).sort().values
    assert torch.equal(key, torch.from_numpy(PINS[name + '__edges_sorted']))


def test_stressed_weights_gain3():
    config = prop.ENC_ALL_CONFIG
    x = prop.pin_inputs('enc_all')
    model, sd = _model(config, 7, gain=3.0)
    out, h = _run(model, config, x)
    tr = {}
    torch.testing.assert_close(out, _oracle(sd, config, x, tr), **PRED_TOL)
    _h_close(h, tr['h'])


def test_two_calls_bit_identical():
    x = prop.pin_inputs('egnn_kinds')
    model, _ = _model(prop.EGNN_CONFIG, 0)
    a, ha = _run(model, prop.EGNN_CONFIG, x)
    b, hb = _run(model, prop.EGNN_CONFIG, x)
    assert torch.equal(a, b) and torch.equal(ha, hb)


def test_alone_equals_inside_ragged_batch():
    """Per-destination padding of the edge tile: a complex's result does not depend on its neighbours in the batch (bit-identical),
    for every graph of a 66-graph ragged batch that includes an empty graph (pooled to 0) followed by a graph with an odd atom count."""
    config = prop.EGNN_CONFIG
    model, _ = _model(config, 0)
    rng = np.random.RandomState(5)
    psizes = [int(v) for v in rng.randint(20, 400, size=64)]
    lsizes = [int(v) for v in rng.randint(5, 40, size=64)]
    empty = 30
    psizes[empty:empty] = [0, 37]
    lsizes[empty:empty] = [0, 8]
    B = len(psizes)
    ppos, pfeat, lpos = [], [], []
    g = torch.Generator().manual_seed(11)
    for i, (npr, nl) in enumerate(zip(psizes, lsizes)):
        if npr == 0:
            ppos.append(torch.zeros(0, 3)), pfeat.append(torch.zeros(0, synth.PROTEIN_FEATURE_DIM)), lpos.append(torch.zeros(0, 3))
            continue
        p, f = synth.make_pocket(500 + i, npr)
        ppos.append(p), pfeat.append(f)
        lpos.append(p.mean(0, keepdim=True) + torch.randn(nl, 3, generator=g))
    lfeat = prop.make_ligand_features(9, sum(lsizes))
    bp = torch.repeat_interleave(torch.arange(B), torch.tensor(psizes))
    bl = torch.repeat_interleave(torch.arange(B), torch.tensor(lsizes))
    x = dict(protein_pos=torch.cat(ppos), protein_feat=torch.cat(pfeat), ligand_pos=torch.cat(lpos), ligand_feat=lfeat, batch_protein=bp,
             batch_ligand=bl, output_kind=None, enc_ligand=None, enc_node=None, enc_graph=None)
    full, hfull = _run(model, config, x)

    def sub(graphs):
        p0, l0 = sum(psizes[:graphs[0]]), sum(lsizes[:graphs[0]])
        ps, ls = [psizes[j] for j in graphs], [lsizes[j] for j in graphs]
        return dict(protein_pos=torch.cat([ppos[j] for j in graphs]), protein_feat=torch.cat([pfeat[j] for j in graphs]),
                    ligand_pos=torch.cat([lpos[j] for j in graphs]), ligand_feat=lfeat[l0:l0 + sum(ls)],
                    batch_protein=torch.repeat_interleave(torch.arange(len(graphs)), torch.tensor(ps)),
                    batch_ligand=torch.repeat_interleave(torch.arange(len(graphs)), torch.tensor(ls)), output_kind=None,
                    enc_ligand=None, enc_node=None, enc_graph=None), p0 + l0
    for j in range(B):
        if j == empty:          # a batch of one empty graph is rejected: score it together with its odd-sized neighbour
            one, n0 = sub([j, j + 1])
        elif j == empty + 1:
            continue
        else:
            one, n0 = sub([j])
        alone, halone = _run(model, config, one)
        assert torch.equal(alone, full[j:j + len(alone)]), j
        assert torch.equal(halone, hfull[n0:n0 + len(halone)]), j


def test_fetch_embedding_final_h_chain():
    """ScorePosNet3D.fetch_embedding(...)['final_h'] -> PropPredNetEnc(enc_node_feature=final_h), against the oracle chain."""
    from targetdiff_b200.config import default_model_config
    from targetdiff_b200.score_model import ScorePosNet3D
    sd_diff = synth.make_state_dict(0, schedules=restate.make_schedules())
    diff = ScorePosNet3D(default_model_config(), synth.PROTEIN_FEATURE_DIM, synth.LIGAND_NUM_CLASSES)
    diff.load_state_dict(sd_diff, strict=True)
    diff = diff.to(DEV)
    b = synth.make_batch(3, 2, n_protein=90, ligand_sizes=[14, 11])
    d = {k: v.to(DEV) for k, v in b.items()}
    emb = diff.fetch_embedding(d['protein_pos'], d['protein_v'], d['batch_protein'], d['init_ligand_pos'], d['init_ligand_v'], d['batch_ligand'])
    want_h = restate.forward(sd_diff, None, b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'], b['init_ligand_v'],
                             b['batch_ligand'], fix_x=True)['final_h']
    config = prop.EGNN_ENC_CONFIG
    model, sd = _model(config, 2)
    lfeat = prop.make_ligand_features(4, len(b['batch_ligand']))
    out = model(d['protein_pos'], d['protein_v'], d['init_ligand_pos'], lfeat.to(DEV), d['batch_protein'], d['batch_ligand'], None, None,
                emb['final_h'], None).cpu()
    want = prop.prop_forward(sd, config, b['protein_pos'], b['protein_v'], b['init_ligand_pos'], lfeat, b['batch_protein'], b['batch_ligand'],
                             enc_node=want_h)
    torch.testing.assert_close(out, want, **PRED_TOL)


def test_malformed_input_rejected():
    x = prop.pin_inputs('egnn_kinds')
    model, _ = _model(prop.EGNN_CONFIG, 0)
    d = {k: (v.to(DEV) if v is not None else None) for k, v in x.items()}
    base = [d['protein_pos'], d['protein_feat'], d['ligand_pos'], d['ligand_feat'], d['batch_protein'], d['batch_ligand'], d['output_kind']]
    bad_width = list(base)
    bad_width[3] = d['ligand_feat'][:, :-1]
    with pytest.raises(ValueError):
        model(*bad_width)
    bad_count = list(base)
    bad_count[2] = d['ligand_pos'][:-1]
    with pytest.raises(ValueError):
        model(*bad_count)
    for kind in ([0, 1, 2], [1, 4, 3]):
        bad_kind = list(base)
        bad_kind[6] = torch.tensor(kind, device=DEV)
        with pytest.raises(_lib.TdiffError, match='output_kind'):
            model(*bad_kind)
    out = model(*base)                       # the model stays usable after a rejected call
    assert out.shape == (3, 1) and bool(torch.isfinite(out).all())
