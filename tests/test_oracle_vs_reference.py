"""Pins oracle/restate.py against the UNMODIFIED reference (run under oracle/shims).  The reference's side of every comparison is
stored in tests/golden/reference_pins.npz (oracle/make_golden.py, `reference_pins`), so the pins hold on any machine: discrete
outputs (layouts, schedules, atom types, bond counts) bit for bit, floating-point outputs to a few ulp (see _assert_matches)."""
import os

import numpy as np
import pytest
import torch

from oracle import refload, restate, synth
from oracle.make_golden import (GOLDEN, PDB_1H36, PIN_CHAINS, PIN_DRIVER, PIN_FORWARD, PIN_LIKELIHOOD, PIN_OPTION_CONFIGS, PIN_OPTIONS,
                                layout_strings, stability_inputs)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def ref():
    """The reference's outputs (tests/golden/reference_pins.npz) as tensors, keyed '<pin>__<array>'."""
    with np.load(os.path.join(GOLDEN, 'reference_pins.npz')) as z:
        return {k: z[k] if z[k].dtype.kind == 'U' else torch.from_numpy(z[k]) for k in z.files}


@pytest.fixture
def knn_shim(monkeypatch):
    """`torch_geometric.nn.knn_graph` as the reference imports it: the pure-torch stand-in under oracle/shims."""
    monkeypatch.syspath_prepend(refload.SHIMS)
    from torch_geometric.nn import knn_graph
    return knn_graph


def _assert_matches(want, got, name):
    """Integer outputs (atom types) bit for bit; floating-point outputs to a few ulp (rtol 1e-5, atol 1e-6, as for the other stored
    reference vectors in tests/test_oracle_golden.py).  torch's CPU kernels round the last bits differently per vector ISA and thread
    count, so vectors stored on one host do not reproduce bit for bit on another."""
    want, got = torch.as_tensor(want), torch.as_tensor(got)
    if want.dtype.is_floating_point:
        torch.testing.assert_close(got, want, rtol=1e-5, atol=1e-6, msg=lambda m: name + ': ' + m)
    else:
        assert torch.equal(got, want), name


def _assert_chain_equal(ref, prefix, got):
    _assert_matches(ref[prefix + '__pos'], got['pos'], 'pos')
    _assert_matches(ref[prefix + '__v'], got['v'], 'v')
    for k in ('pos_traj', 'v_traj', 'v0_traj', 'vt_traj'):
        assert len(ref[prefix + '__' + k]) == len(got[k]), k
        _assert_matches(ref[prefix + '__' + k], torch.stack(got[k]), k)


def test_state_dict_layout_matches_reference(ref):
    spec = synth.state_dict_spec()
    assert ref['layout'].tolist() == ['%s:%s' % (k, 'x'.join(str(s) for s in shape)) for k, shape, _ in spec]
    assert len(spec) == 384


def test_schedules_bit_exact(ref):
    sched = restate.make_schedules()
    for k in synth.SCHEDULE_KEYS:
        assert torch.equal(ref['schedule__' + k], sched[k]), k


def test_knn_shim_equals_canonical_restatement(knn_shim):
    b = synth.make_batch(11, 3, n_protein=70, ligand_sizes=[5, 9, 1])
    x = torch.cat([b['protein_pos'], b['init_ligand_pos']])
    batch = torch.cat([b['batch_protein'], b['batch_ligand']])
    order = torch.sort(batch, stable=True).indices
    x, batch = x[order], batch[order]
    for k in (8, 32, 48):
        assert torch.equal(knn_shim(x, k=k, batch=batch, flow='source_to_target'), restate.knn_graph_canonical(x, k, batch))


def test_knn_small_graph_and_ties(knn_shim):
    # graph 0 has 5 nodes (< k+1) incl. exact duplicate points and equidistant neighbours; graph 1 has 40 on a lattice
    g0 = torch.tensor([[0., 0, 0], [1, 0, 0], [-1, 0, 0], [0, 0, 0], [0, 1, 0]])
    g1 = torch.stack(torch.meshgrid(torch.arange(5.), torch.arange(4.), torch.arange(2.), indexing='ij'), -1).reshape(-1, 3)
    x = torch.cat([g0, g1])
    batch = torch.cat([torch.zeros(5, dtype=torch.long), torch.ones(40, dtype=torch.long)])
    a = knn_shim(x, k=32, batch=batch)
    b = restate.knn_graph_canonical(x, 32, batch)
    assert torch.equal(a, b)
    assert (a[1] < 5).sum() == 5 * 4              # fewer than k edges per node in the small graph
    assert ((a[1] >= 5).sum()) == 40 * 32


def test_forward_bit_exact(ref):
    sd = synth.make_state_dict(PIN_FORWARD['weight_seed'], schedules=restate.make_schedules())
    b = synth.make_batch(**PIN_FORWARD['batch'])
    pp2, lp2, _ = restate.center_pos(b['protein_pos'], b['init_ligand_pos'], b['batch_protein'], b['batch_ligand'])
    _assert_matches(ref['forward__protein_pos'], pp2, 'protein_pos')
    _assert_matches(ref['forward__ligand_pos'], lp2, 'ligand_pos')
    got = restate.forward(sd, None, pp2, b['protein_v'], b['batch_protein'], lp2, b['init_ligand_v'], b['batch_ligand'])
    for k in ('pred_ligand_pos', 'pred_ligand_v', 'final_h', 'final_ligand_h'):
        _assert_matches(ref['forward__' + k], got[k], k)


def _pinned_chain(name):
    c = PIN_CHAINS[name]
    sd = synth.make_state_dict(c['weight_seed'], schedules=restate.make_schedules())
    b = synth.make_batch(**c['batch'])
    S = c['tape'][1]
    pn, vu = synth.make_tape(c['tape'][0], S, len(b['batch_ligand']))
    args = (b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'], b['init_ligand_v'], b['batch_ligand'])
    return restate.sample_diffusion(sd, c['cfg'] or None, *args, pn, vu, num_steps=S)


def test_sampling_chain_bit_exact(ref):
    _assert_chain_equal(ref, 'chain', _pinned_chain('chain'))


@pytest.mark.parametrize('steps', PIN_LIKELIHOOD['steps'])
def test_likelihood_estimation_matches_reference(ref, steps):
    """SURVEY 8(f) n3: the second consumer of `forward` (reference models/molopt_score_model.py:565-617), incl. the decoder
    branch (t = 0) and the prior branch (time_step == T)."""
    c = PIN_LIKELIHOOD
    i = c['steps'].index(steps)
    sd = synth.make_state_dict(c['weight_seed'], schedules=restate.make_schedules())
    b = synth.make_batch(**c['batch'])
    Nl = len(b['batch_ligand'])
    pn, vu = synth.make_tape(c['tape_seed'], 1, Nl)
    t = torch.tensor(steps) if steps is not None else torch.full((2,), 1000)
    args = (b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'], b['init_ligand_v'], b['batch_ligand'])
    got = restate.likelihood_estimation(sd, None, *args, t, pn[0], vu[0])
    for w, g in zip((ref['likelihood%d__kl_pos' % i], ref['likelihood%d__kl_v' % i]), got):
        assert w.shape == g.shape == (2,)
        torch.testing.assert_close(g, w, rtol=1e-6, atol=1e-7)


def test_sampling_chain_noise_mean_type_bit_exact(ref):
    """SURVEY 8(f) n2: model_mean_type='noise' (reference models/molopt_score_model.py:663-666, :419-422)."""
    _assert_chain_equal(ref, 'chain_noise', _pinned_chain('chain_noise'))


@pytest.mark.parametrize('cfgd', PIN_OPTION_CONFIGS, ids=lambda c: ','.join('%s=%s' % kv for kv in c.items()))
def test_backbone_options_restatement_bit_exact(ref, cfgd):
    """SURVEY 8(f) n2: num_blocks > 1, ew_net_type r / m / none, x2h_out_fc, time_emb_mode 'simple', cutoff_mode 'hybrid' -- state_dict layout (key order and
    shapes) and a 3-step sampling chain of the restatement against the unmodified reference, bit for bit."""
    prefix = 'option%d' % PIN_OPTION_CONFIGS.index(cfgd)
    c = PIN_OPTIONS
    sd = synth.make_state_dict(c['weight_seed'], cfgd, schedules=restate.make_schedules(cfgd))
    assert ref[prefix + '__layout'].tolist() == layout_strings(sd).tolist()
    b = synth.make_batch(**c['batch'])
    S = c['tape'][1]
    pn, vu = synth.make_tape(c['tape'][0], S, len(b['batch_ligand']))
    args = (b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'], b['init_ligand_v'], b['batch_ligand'])
    _assert_chain_equal(ref, prefix, restate.sample_diffusion(sd, cfgd, *args, pn, vu, num_steps=S))


def test_sampling_driver_restatement_bit_exact(ref):
    """a1: oracle.restate.sample_diffusion_ligand against the UNMODIFIED reference driver (scripts/sample_diffusion.py:31-116, imported with
    placeholders for rdkit / openbabel / lmdb) on the 1h36 pocket: same seeds -> the same prior sizes, positions, types and trajectories."""
    import json
    from targetdiff_b200.pocket import pdb_to_pocket_data
    from targetdiff_b200.sampling import seed_all
    # the product's PDB ingest gives the reference's tensors
    data = pdb_to_pocket_data(PDB_1H36)
    assert torch.equal(data.protein_pos, ref['driver__protein_pos'])
    assert torch.equal(data.protein_atom_feature, ref['driver__protein_atom_feature'])
    c = PIN_DRIVER
    sd = synth.make_state_dict(0, schedules=restate.make_schedules())
    prior = json.load(open(os.path.join(ROOT, 'targetdiff_b200', 'data', 'atom_num_prior.json')))
    seed_all(c['seed'])
    out = restate.sample_diffusion_ligand(sd, None, data.protein_pos, data.protein_atom_feature, c['num_samples'], prior,
                                          batch_size=c['batch_size'], num_steps=c['num_steps'])
    for name, got in zip(('pos', 'v', 'pos_traj', 'v_traj', 'v0_traj', 'vt_traj'), out[:6]):
        assert len(got) == c['num_samples'], name
        for i, y in enumerate(got):
            _assert_matches(ref['driver__%s%d' % (name, i)], torch.from_numpy(np.asarray(y)), '%s[%d]' % (name, i))


def test_check_stability_restatement_equals_reference(ref):
    """n4: the bond-count stability screen (utils/evaluation/analyze.py:106-143) on random molecule-like point sets."""
    for n, hs, pos, z in stability_inputs():
        got = restate.check_stability(pos, z, hs=hs)
        assert ref['stability%d_%d__counts' % (n, hs)].tolist() == [int(bool(got[0])), got[1], got[2]]
        assert np.array_equal(ref['stability%d_%d__nr_bonds' % (n, hs)].numpy(), got[3])
