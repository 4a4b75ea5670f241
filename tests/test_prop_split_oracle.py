"""The bf16-split emulating oracle (oracle.prop.split_linear / emulate_split), host side: its error bound, its exactness on
bf16-representable operands, the float64 forward against the fp32 one, and the explanation of the stressed-weight deviations that
DESIGN.md section 9 gives (the split's own error, reproduced by emulation)."""
import pytest
import torch
import torch.nn.functional as F

from oracle import prop
from targetdiff_b200.prop_model import PropPredNet, PropPredNetEnc


def _rel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


def _h(sd, config, x, linear=prop.plain_linear):
    tr = {}
    out = prop.forward_float64(sd, config, x, linear=linear, trace=tr)
    return out, tr['h']


def _mixed(g, rows, cols):
    """fp32 values spread over six decades, random signs."""
    return (torch.randn(rows, cols, generator=g) * 10.0 ** (6 * torch.rand(rows, cols, generator=g) - 3)).float()


@pytest.mark.parametrize('gain', [1.0, 3.0])
@pytest.mark.parametrize('name', sorted(prop.PIN_CASES))
def test_float64_forward_matches_fp32(name, gain):
    """The fp32 oracle is not the source of the GPU's error: it is within 2e-5 of max |h| of the float64 forward (measured maximum
    1.0e-5, enc_final_h at gain 3, with torch 2.11 on x86-64; the last bits depend on the CPU kernels)."""
    config, seed = prop.PIN_CASES[name][:2]
    x = prop.pin_inputs(name)
    sd = prop.make_state_dict(config, seed, gain=gain)
    tr = {}
    out32 = prop.prop_forward(sd, config, x['protein_pos'], x['protein_feat'], x['ligand_pos'], x['ligand_feat'], x['batch_protein'],
                              x['batch_ligand'], x['output_kind'], x['enc_ligand'], x['enc_node'], x['enc_graph'], trace=tr)
    out64, h64 = _h(sd, config, x)
    assert out64.dtype == torch.float64 and h64.dtype == torch.float64
    assert _rel(tr['h'].double(), h64) <= 2e-5
    torch.testing.assert_close(out32.double(), out64, rtol=5e-5, atol=1e-6)


def test_split_linear_error_bound():
    """|split - exact| <= 3.1 * 2^-16 * (|x|.|w|^T) elementwise: |x - x1 - x2| <= 2^-16 |x|, and the dropped terms are x2.w2 and the
    two residuals.  The bound is also nearly reached, so a product that forgot to split would fail the second assertion."""
    g = torch.Generator().manual_seed(0)
    x, w, b = _mixed(g, 96, 300), _mixed(g, 80, 300), _mixed(g, 1, 80)[0]
    exact = x.double() @ w.double().T
    y = prop.split_linear(x, w)
    bound = 3.1 * 2.0 ** -16 * (x.double().abs() @ w.double().abs().T)
    assert bool(((y - exact).abs() <= bound).all())
    assert ((y - exact).abs() / bound).max().item() > 0.05
    torch.testing.assert_close(prop.split_linear(x, w, b), y + b.double(), rtol=0, atol=0)      # the bias comes after, unsplit


def test_split_linear_exact_on_bf16_operands():
    g = torch.Generator().manual_seed(1)
    x = _mixed(g, 64, 200).to(torch.bfloat16).float()
    w = _mixed(g, 48, 200).to(torch.bfloat16).float()
    torch.testing.assert_close(prop.split_linear(x, w), F.linear(x.double(), w.double()), rtol=1e-13, atol=0)


def test_tensor_core_linears_are_the_split_ones():
    """Embeddings, both edge-MLP Linears, both node-MLP Linears and enc_node_layer are split; the gate and out_block are plain."""
    g = torch.Generator().manual_seed(2)
    x, w = _mixed(g, 8, 64).double(), _mixed(g, 4, 64).double()
    b = torch.zeros(4, dtype=torch.float64)
    config = dict(prop.ENC_ALL_CONFIG, encoder=dict(prop.ENC_ALL_CONFIG['encoder'], num_layers=2))
    split = {k[:-len('.weight')] for k, _, kind in prop.state_dict_spec(config) if kind == 'lin_w'
             and not torch.equal(prop.tensor_core_linear(k, x, w, b), F.linear(x, w, b))}
    want = {'protein_atom_emb', 'ligand_atom_emb', 'enc_node_layer.0', 'enc_node_layer.2'}
    want |= {'encoder.net.%d.%s' % (l, n) for l in range(2) for n in ('edge_mlp.net.0', 'edge_mlp.net.2', 'node_mlp.net.0', 'node_mlp.net.2')}
    assert split == want


# max |h_emulated - h_float64| / max |h_float64| with every Linear x3, per pinned case (DESIGN.md section 9)
GAIN3_SPLIT_ERROR = {'egnn_none': 1.50e-2, 'enc_final_h': 1.61e-2, 'egnn_kinds': 3.1e-5, 'egnn_1h36': 2.7e-5, 'enc_all': 1.76e-2}
# the edge gate (layer index, src, dst) whose logit the split moves across 0 in those cases
GAIN3_GATE_FLIPS = {'egnn_none': (5, 98, 91), 'enc_final_h': (4, 1, 11), 'enc_all': (5, 120, 110)}


@pytest.mark.parametrize('name', sorted(prop.PIN_CASES))
def test_split_error_with_stressed_weights(name):
    """The emulated split reproduces the gain-3 deviations the B200 shows against the fp32 oracle, and each large one is a single edge
    gate: its logit, on a scale of 1e6 to 1e8, lies within the split's error of 0, so the sigmoid switches a whole message on or off.  With
    that gate put back on the float64 side the emulation is within 4e-4 of the float64 forward.  At gain 1 nothing flips and the split
    stays within 1.5e-5 of max |h|."""
    config, seed = prop.PIN_CASES[name][:2]
    x = prop.pin_inputs(name)
    sd1 = prop.make_state_dict(config, seed, gain=1.0)
    assert _rel(_h(sd1, config, x, prop.tensor_core_linear)[1], _h(sd1, config, x)[1]) <= 1.5e-5
    assert not prop.gate_flips(sd1, config, x)[0]
    sd = prop.make_state_dict(config, seed, gain=3.0)
    _, h64 = _h(sd, config, x)
    _, hemu = _h(sd, config, x, prop.tensor_core_linear)
    assert _rel(hemu, h64) == pytest.approx(GAIN3_SPLIT_ERROR[name], rel=0.1)
    flips, z64, ei = prop.gate_flips(sd, config, x)
    got = [(l, ei[0, i].item(), ei[1, i].item()) for l, idx in flips.items() for i in idx]
    assert got == ([GAIN3_GATE_FLIPS[name]] if name in GAIN3_GATE_FLIPS else [])
    if flips:
        assert max(z64[l].abs().max().item() for l in flips) > 1e6
        ov = {l: (i, z64[l][i]) for l, i in flips.items()}
        _, hov, _, _ = prop.forward_with_gates(sd, config, x, linear=prop.tensor_core_linear, gate_override=ov)
        assert _rel(hov, h64) <= 4e-4


@pytest.mark.parametrize('output_dim', [1, 5, 32])
def test_output_dim_layout(output_dim):
    for config in (prop.EGNN_CONFIG, prop.ENC_ALL_CONFIG):
        if config['encoder']['name'] == 'egnn_enc':
            m = PropPredNetEnc(config, 27, 30, 13, 128, 20, 'full', output_dim=output_dim)
        else:
            m = PropPredNet(config, 27, 30, output_dim=output_dim)
        spec = [(k, s) for k, s, _ in prop.state_dict_spec(config, output_dim=output_dim)]
        assert spec == [(k, tuple(v.shape)) for k, v in m.state_dict().items()]
        m.load_state_dict(prop.make_state_dict(config, 1, output_dim=output_dim), strict=True)
