"""Affinity regressor, host side: the CPU restatement (oracle.prop) against the reference's pinned outputs, the Python mirror's
state_dict layout, and the configurations it rejects."""
import os

import numpy as np
import pytest
import torch

from oracle import prop
from targetdiff_b200.prop_model import PropPredNet, PropPredNetEnc, get_model

PINS = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'prop_pins.npz'))


def _mirror(config, ligand_dim=prop.LIGAND_FEATURE_DIM):
    if config['encoder']['name'] == 'egnn_enc':
        return PropPredNetEnc(config, 27, ligand_dim, config['enc_ligand_dim'], config['enc_node_dim'], config['enc_graph_dim'],
                              config['enc_feature_type'])
    return PropPredNet(config, 27, ligand_dim)


@pytest.mark.parametrize('name', sorted(prop.PIN_CASES))
def test_state_dict_layout_matches_reference(name):
    config, seed = prop.PIN_CASES[name][:2]
    want = list(PINS[name + '__layout'])
    spec = ['%s:%s' % (k, 'x'.join(map(str, s))) for k, s, _ in prop.state_dict_spec(config)]
    model = _mirror(config)
    got = ['%s:%s' % (k, 'x'.join(map(str, v.shape))) for k, v in model.state_dict().items()]
    assert spec == want and got == want
    model.load_state_dict(prop.make_state_dict(config, seed), strict=True)


def test_published_configs_entry_counts():
    assert len(_mirror(prop.EGNN_CONFIG).state_dict()) == 75
    assert len(_mirror(prop.EGNN_ENC_CONFIG).state_dict()) == 79


@pytest.mark.parametrize('name', sorted(prop.PIN_CASES))
def test_restatement_matches_reference(name):
    config, seed = prop.PIN_CASES[name][:2]
    x = prop.pin_inputs(name)
    p = name + '__'
    for k in ('protein_pos', 'protein_feat', 'ligand_pos', 'ligand_feat', 'enc_node'):
        if x[k] is not None:
            assert torch.equal(x[k], torch.from_numpy(PINS[p + k])), k
    tr = {}
    out = prop.prop_forward(prop.make_state_dict(config, seed), config, x['protein_pos'], x['protein_feat'], x['ligand_pos'], x['ligand_feat'],
                            x['batch_protein'], x['batch_ligand'], x['output_kind'], x['enc_ligand'], x['enc_node'], x['enc_graph'], trace=tr)
    n = len(x['batch_protein']) + len(x['batch_ligand'])
    ei = tr['edge_index']
    assert torch.equal((ei[1] * n + ei[0]).sort().values, torch.from_numpy(PINS[p + 'edges_sorted']))      # edge set, bit-exact
    # the reference sums messages / pools with torch_scatter, the restatement with index_add_: last-bit differences only
    torch.testing.assert_close(out, torch.from_numpy(PINS[p + 'pred']), rtol=1e-5, atol=1e-5)
    torch.testing.assert_close(tr['h'][torch.from_numpy(PINS[p + 'h_rows'])], torch.from_numpy(PINS[p + 'h']), rtol=1e-5, atol=1e-5)


def _with(config, **enc):
    c = dict(config, encoder=dict(config['encoder'], **{k: v for k, v in enc.items() if k != 'hidden_channels'}))
    if 'hidden_channels' in enc:
        c['hidden_channels'] = enc['hidden_channels']
    return c


@pytest.mark.parametrize('change', [dict(name='egnn_x'), dict(hidden_dim=128), dict(hidden_channels=128), dict(num_r_gaussian=65),
                                    dict(act_fn='silu'), dict(norm=True), dict(edge_dim=4), dict(knn=0), dict(knn=65)])
def test_unsupported_configs_rejected(change):
    with pytest.raises(NotImplementedError):
        PropPredNet(_with(prop.EGNN_CONFIG, **change), 27, 30)


def test_get_model_and_host_errors():
    m = get_model({'model': prop.EGNN_ENC_CONFIG}, 27, 30)
    assert isinstance(m, PropPredNetEnc) and m.output_dim == 1
    m = get_model({'model': prop.EGNN_CONFIG}, 27, 30)
    assert isinstance(m, PropPredNet) and m.output_dim == 3
    with pytest.raises(NotImplementedError):
        m.get_loss(None, 0.1)
    x = prop.pin_inputs('egnn_none')
    with pytest.raises(RuntimeError, match='no CPU path'):
        m(x['protein_pos'], x['protein_feat'], x['ligand_pos'], x['ligand_feat'], x['batch_protein'], x['batch_ligand'], None)
