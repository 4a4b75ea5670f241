"""CPU restatement of targetdiff's binding-affinity regressor (TEST INFRASTRUCTURE, see oracle/__init__.py).

PropPredNet / PropPredNetEnc with the EnEquiEncoder (reference models/property_pred/prop_model.py,
models/property_pred/prop_egnn.py; paths relative to the reference tree), op by op in torch-CPU fp32 on a
reference-layout state_dict, plus seeded weights / ligand features and the generator of the reference pins
(tests/golden/prop_pins.npz):

    python -m oracle.prop          # build container only: runs the UNMODIFIED reference under oracle/shims

Node order: per graph, protein atoms (input order) then ligand atoms (input order) -- a STABLE sort of the batch
vector, which is also the order of ScorePosNet3D.fetch_embedding()['final_h'].  The reference's compose_context_prop
uses the unstable `argsort()` (models/common.py:142); the pins record the permutation it produced.
"""
import math
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

from .restate import gaussian_smearing, knn_graph_canonical
from .synth import PROTEIN_FEATURE_DIM

# configs/prop/pdbbind_general_egnn.yml and configs/prop/pdbbind_general_egnn_enc_final_h.yml (model sections, values only)
EGNN_CONFIG = dict(hidden_channels=256, encoder=dict(name='egnn', num_layers=6, hidden_dim=256, edge_dim=0, num_r_gaussian=64,
                                                     act_fn='relu', norm=False, cutoff=10.0, knn=48))
EGNN_ENC_CONFIG = dict(hidden_channels=256, enc_ligand_dim=0, enc_node_dim=128, enc_graph_dim=0, enc_feature_type='final_h',
                       encoder=dict(EGNN_CONFIG['encoder'], name='egnn_enc'))
# ligand_atom_feature_full width of the synthetic data.  The real width comes from the checkpoint (ligand_atom_emb.weight): it depends
# on the rdkit version that featurised PDBbind (utils/transforms_prop.py:31-68), so nothing here may assume a constant.
LIGAND_FEATURE_DIM = 30
OUTPUT_KINDS = {1: 'Ki', 2: 'Kd', 3: 'IC50'}        # utils/misc_prop.py KMAP


def _lin(key, out_dim, in_dim):
    return [(key + '.weight', (out_dim, in_dim), 'lin_w'), (key + '.bias', (out_dim,), 'lin_b:%d' % in_dim)]


def state_dict_spec(config, protein_dim=PROTEIN_FEATURE_DIM, ligand_dim=LIGAND_FEATURE_DIM, output_dim=None):
    """Ordered (key, shape, kind) list == the reference module's state_dict() (prop_model.py:29-45,99-128, prop_egnn.py:8-26,49-72).
    output_dim None: the reference's get_model choice (3 for PropPredNet, 1 for PropPredNetEnc)."""
    enc = config['encoder']
    H, G, L = config['hidden_channels'], enc['num_r_gaussian'], enc['num_layers']
    is_enc = enc['name'] == 'egnn_enc'
    spec = _lin('protein_atom_emb', H, protein_dim)
    spec += _lin('ligand_atom_emb', H, ligand_dim + (config.get('enc_ligand_dim', 0) if is_enc else 0))
    spec += [('encoder.distance_expansion.offset', (G,), 'offset:%r' % float(enc['cutoff']))]
    for l in range(L):
        p = 'encoder.net.%d' % l
        if G > 1:
            spec += [(p + '.r_expansion.offset', (G,), 'offset:100.0')]         # r_max = 10**2 (prop_egnn.py:12-13,21); never read
        spec += _lin(p + '.edge_mlp.net.0', H, 2 * H + enc['edge_dim'] + G) + _lin(p + '.edge_mlp.net.2', H, H)
        spec += _lin(p + '.edge_inf.0', 1, H)
        spec += _lin(p + '.node_mlp.net.0', H, 2 * H) + _lin(p + '.node_mlp.net.2', H, H)
    if is_enc and config.get('enc_node_dim', 0) > 0:
        spec += _lin('enc_node_layer.0', H, H + config['enc_node_dim']) + _lin('enc_node_layer.2', H, H)
    gdim = config.get('enc_graph_dim', 0) if is_enc else 0
    if output_dim is None:
        output_dim = 1 if is_enc else 3
    spec += _lin('out_block.0', H, H + gdim) + _lin('out_block.2', output_dim, H)
    return spec


def make_state_dict(config, seed=0, gain=1.0, protein_dim=PROTEIN_FEATURE_DIM, ligand_dim=LIGAND_FEATURE_DIM, output_dim=None):
    """Deterministic weights, Linear: U(-1/sqrt(in), 1/sqrt(in)) * gain (nn.Linear's default bound), like oracle.synth."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for key, shape, kind in state_dict_spec(config, protein_dim, ligand_dim, output_dim):
        if kind.startswith('offset'):
            sd[key] = torch.linspace(0.0, float(kind.split(':')[1]), shape[0])              # GaussianSmearing(fixed_offset=False)
        elif kind == 'lin_w':
            sd[key] = (torch.rand(shape, generator=g) * 2 - 1) * (gain / math.sqrt(shape[1]))
        else:
            sd[key] = (torch.rand(shape, generator=g) * 2 - 1) * (gain / math.sqrt(int(kind.split(':')[1])))
    return sd


def make_ligand_features(seed, n_atoms, dim=LIGAND_FEATURE_DIM):
    """Seeded stand-in for ligand_atom_feature_full: a one-hot element block (first 8 columns) and sparse binary flags."""
    g = torch.Generator().manual_seed(seed)
    f = (torch.rand(n_atoms, dim, generator=g) < 0.25).float()
    f[:, :8] = 0.0
    f[torch.arange(n_atoms), torch.randint(0, 8, (n_atoms,), generator=g)] = 1.0
    return f


def compose_stable(batch_protein, batch_ligand):
    """Permutation of cat([protein, ligand]) into the stable per-graph protein-then-ligand order."""
    return torch.sort(torch.cat([batch_protein, batch_ligand]), stable=True).indices


def plain_linear(key, x, w, b):
    """The default `linear` hook: F.linear.  `key` is the state_dict key of the weight (which Linear this is)."""
    return F.linear(x, w, b)


def _apply(linear, sd, prefix, x):
    return linear(prefix + '.weight', x, sd[prefix + '.weight'], sd[prefix + '.bias'])


def _linear_relu_linear(sd, prefix, x, act=F.relu, i0=0, i1=2, linear=plain_linear):
    y = act(_apply(linear, sd, '%s.%d' % (prefix, i0), x))
    return _apply(linear, sd, '%s.%d' % (prefix, i1), y)


def shifted_softplus(x):
    return F.softplus(x) - torch.log(torch.tensor(2.0)).item()                               # models/common.py:156-162


def encoder_forward(sd, enc, h, pos, batch, trace=None, linear=plain_linear):
    """EnEquiEncoder.forward (prop_egnn.py:74-83), update_x=False, norm=False, act_fn='relu'.  The edge set comes from the fp32
    positions (knn_graph_canonical casts); the edge lengths from `pos` as given, so a float64 run widens the fp32 values."""
    ei = knn_graph_canonical(pos, enc['knn'], batch)          # rows (src, dst) == knn_graph(flow='target_to_source') unpacked dst, src
    src, dst = ei[0], ei[1]
    edge_length = torch.norm(pos[dst] - pos[src], dim=1)                                      # :79
    edge_attr = gaussian_smearing(edge_length, sd['encoder.distance_expansion.offset'])      # :80, common.py:7-26
    for l in range(enc['num_layers']):                                                        # :82-83
        p = 'encoder.net.%d' % l
        m = F.relu(_linear_relu_linear(sd, p + '.edge_mlp.net', torch.cat([edge_attr, h[dst], h[src]], -1), linear=linear))   # :34-35
        e = torch.sigmoid(_apply(linear, sd, p + '.edge_inf.0', m))                                                    # :36
        mi = torch.zeros_like(h).index_add_(0, dst, m * e)                                                     # :37 scatter_sum
        h = h + _linear_relu_linear(sd, p + '.node_mlp.net', torch.cat([mi, h], -1), linear=linear)          # :41, :83
    if trace is not None:
        trace['edge_index'] = ei
    return h


def prop_forward(sd, config, protein_pos, protein_feat, ligand_pos, ligand_feat, batch_protein, batch_ligand, output_kind=None,
                 enc_ligand=None, enc_node=None, enc_graph=None, trace=None, linear=plain_linear):
    """PropPredNet.forward (prop_model.py:48-74) / PropPredNetEnc.forward (:130-165).  `enc_node` is in the stable composed order.
    `linear(key, x, w, b)` computes every Linear (key: the state_dict key of its weight); see tensor_core_linear."""
    enc = config['encoder']
    if enc_ligand is not None:
        ligand_feat = torch.cat([ligand_feat, enc_ligand], -1)                                 # :133-134
    h_p = _apply(linear, sd, 'protein_atom_emb', protein_feat)
    h_l = _apply(linear, sd, 'ligand_atom_emb', ligand_feat)
    order = compose_stable(batch_protein, batch_ligand)                                       # common.py:140-153
    h = torch.cat([h_p, h_l])[order]
    pos = torch.cat([protein_pos, ligand_pos])[order]
    batch = torch.cat([batch_protein, batch_ligand])[order]
    h = encoder_forward(sd, enc, h, pos, batch, trace, linear)
    if trace is not None:
        trace['h'] = h
    if enc_node is not None:                                                                  # :146-148
        h = _linear_relu_linear(sd, 'enc_node_layer', torch.cat([h, enc_node], -1), linear=linear)
    n_graphs = int(max(batch_protein.max().item() if len(batch_protein) else -1, batch_ligand.max().item() if len(batch_ligand) else -1)) + 1
    pre = torch.zeros(n_graphs, h.shape[1], dtype=h.dtype).index_add_(0, batch, h)                            # :151 scatter sum
    if enc_graph is not None:
        pre = torch.cat([pre, enc_graph], -1)                                                 # :152-153
    out = _linear_relu_linear(sd, 'out_block', pre, act=shifted_softplus, linear=linear)      # :155
    if output_kind is not None:                                                               # :156-158
        out = torch.sum(out * F.one_hot(output_kind - 1, out.shape[1]), dim=-1, keepdim=True)
    return out


# ----------------------------------------------------------------------------------------------------- bf16-split emulation
# csrc/prop.cu runs every Linear below on tcgen05 in the two-piece bf16 split; edge_inf.0 (gate) and out_block run as fp32 FMA on
# CUDA cores.  edge_mlp.net.0 is one product over all G + 512 input columns: the kernels' gaussian / h_dst / h_src blocks sum to it.
TENSOR_CORE_LINEARS = ('protein_atom_emb', 'ligand_atom_emb', 'edge_mlp.net.0', 'edge_mlp.net.2', 'node_mlp.net.0', 'node_mlp.net.2',
                       'enc_node_layer.0', 'enc_node_layer.2')


def bf16_split(t):
    """fp32 t -> (t1, t2) in float64: t1 = bf16_rn(t), t2 = bf16_rn(t - t1) (t - t1 is exact in fp32)."""
    t = t.to(torch.float32)
    t1 = t.to(torch.bfloat16).to(torch.float32)
    t2 = (t - t1).to(torch.bfloat16).to(torch.float32)
    return t1.double(), t2.double()


def split_linear(x, w, b=None):
    """prop_gemm_kernel / prop_edge_kernel arithmetic: both operands rounded to fp32 and split, y = x1.w1^T + x1.w2^T + x2.w1^T
    accumulated in float64 (the kernels accumulate in fp32), then the fp32 bias.  |y - x.w^T| <= ~3 * 2^-16 * |x|.|w|^T."""
    x1, x2 = bf16_split(x)
    w1, w2 = bf16_split(w)
    y = x1 @ w1.T + x1 @ w2.T + x2 @ w1.T
    return y if b is None else y + b.to(torch.float32).double()


def tensor_core_linear(key, x, w, b):
    """`linear` hook of prop_forward that emulates the split on the Linears that run on tensor cores, plain F.linear elsewhere."""
    name = key[:-len('.weight')]
    if any(name == t or name.endswith('.' + t) for t in TENSOR_CORE_LINEARS):
        return split_linear(x, w, b)
    return F.linear(x, w, b)


def to_float64(sd_or_inputs):
    """float tensors of a state_dict / an input dict widened to float64 (integer tensors and None unchanged)."""
    return {k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in sd_or_inputs.items()}


def forward_float64(sd, config, x, linear=plain_linear, trace=None):
    """prop_forward on the float64 widening of `sd` and the input dict `x` (pin_inputs keys)."""
    sd, x = to_float64(sd), to_float64(x)
    return prop_forward(sd, config, x['protein_pos'], x['protein_feat'], x['ligand_pos'], x['ligand_feat'], x['batch_protein'],
                        x['batch_ligand'], x['output_kind'], x['enc_ligand'], x['enc_node'], x['enc_graph'], trace=trace, linear=linear)


def emulate_split(sd, config, x, trace=None):
    """What the B200 kernels compute, up to their fp32 accumulation: float64 everywhere, bf16 split on the tensor-core Linears."""
    return forward_float64(sd, config, x, linear=tensor_core_linear, trace=trace)


def forward_with_gates(sd, config, x, linear=plain_linear, gate_override=None):
    """forward_float64 that also returns every layer's edge-gate logits (edge_inf.0 outputs, edge order of trace['edge_index']).
    gate_override {layer: (edge indices, logits)} replaces those logits before the sigmoid.  Returns (pred, h, [logits per layer])."""
    gates, tr = [], {}

    def hooked(key, xx, w, b):
        y = linear(key, xx, w, b)
        if key.endswith('.edge_inf.0.weight'):
            if gate_override and len(gates) in gate_override:
                idx, z = gate_override[len(gates)]
                y = y.clone()
                y[idx, 0] = z.to(y.dtype)
            gates.append(y[:, 0])
        return y
    out = forward_float64(sd, config, x, linear=hooked, trace=tr)
    return out, tr['h'], gates, tr['edge_index']


def gate_flips(sd, config, x):
    """Edges whose gate the split's own error switches: sigmoid(logit) differs by more than 1/2 between the float64 forward and
    emulate_split.  With large weights the logits reach ~1e8 and the sigmoid is a step, so a logit within the split's error of 0 decides
    whether a whole message enters its destination's sum: a knife edge, not a kernel defect.  Returns {layer: edge indices} and the
    float64 logits, so forward_with_gates(..., gate_override=...) can put the emulation on the float64 side of every flipped gate."""
    _, _, z64, ei = forward_with_gates(sd, config, x)
    _, _, zemu, _ = forward_with_gates(sd, config, x, linear=tensor_core_linear)
    flips = {}
    for l, (a, b) in enumerate(zip(z64, zemu)):
        idx = torch.nonzero((torch.sigmoid(a) - torch.sigmoid(b)).abs() > 0.5).flatten()
        if len(idx):
            flips[l] = idx
    return flips, z64, ei


# ----------------------------------------------------------------------------------------------------- reference pins
GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')
PIN_PATH = os.path.join(GOLDEN, 'prop_pins.npz')
ENC_ALL_CONFIG = dict(EGNN_ENC_CONFIG, enc_ligand_dim=13, enc_node_dim=128, enc_graph_dim=20, enc_feature_type='full')
# name -> (config, weight seed, protein sizes per graph (None: the 1h36 pocket), ligand sizes, output_kind, enc inputs)
PIN_CASES = {
    'egnn_kinds': (EGNN_CONFIG, 0, [60, 30, 80], [12, 10, 20], [1, 2, 3], ()),      # graph 1 has 40 < k + 1 atoms
    'egnn_none': (EGNN_CONFIG, 1, [50, 36], [15, 9], None, ()),
    'enc_final_h': (EGNN_ENC_CONFIG, 2, [60, 30], [12, 10], None, ('node',)),    # output_dim 1: only kind 1 (or None) is valid
    'enc_all': (ENC_ALL_CONFIG, 3, [45, 70], [14, 11], [1, 1], ('ligand', 'node', 'graph')),
    'egnn_1h36': (EGNN_CONFIG, 4, None, [25], [1], ()),
}
PIN_H_ROWS = 48          # encoder rows stored per case (a seeded sample): the predictions are pinned in full


def pin_inputs(name):
    """The inputs of one pin case (seeded; the 1h36 pocket comes from tests/golden/1h36_pocket10.pdb)."""
    from . import synth
    config, seed, psizes, lsizes, kinds, encs = PIN_CASES[name]
    ppos, pfeat = [], []
    if psizes is None:
        sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
        from targetdiff_b200.pocket import pdb_to_pocket_data
        d = pdb_to_pocket_data(os.path.join(GOLDEN, '1h36_pocket10.pdb'))
        ppos, pfeat = [d.protein_pos.float()], [d.protein_atom_feature.float()]
        psizes = [len(d.protein_pos)]
    else:
        for i, n in enumerate(psizes):
            p, f = synth.make_pocket(100 * seed + i, n)
            ppos.append(p), pfeat.append(f)
    g = torch.Generator().manual_seed(1000 + seed)
    lpos = [ppos[i].mean(0, keepdim=True) + 1.5 * torch.randn(n, 3, generator=g) for i, n in enumerate(lsizes)]
    out = dict(protein_pos=torch.cat(ppos), protein_feat=torch.cat(pfeat), ligand_pos=torch.cat(lpos),
               ligand_feat=make_ligand_features(2000 + seed, sum(lsizes)),
               batch_protein=torch.repeat_interleave(torch.arange(len(psizes)), torch.tensor(psizes)),
               batch_ligand=torch.repeat_interleave(torch.arange(len(lsizes)), torch.tensor(lsizes)))
    out['output_kind'] = torch.tensor(kinds) if kinds is not None else None
    n_nodes, B = sum(psizes) + sum(lsizes), len(lsizes)
    out['enc_ligand'] = torch.randn(sum(lsizes), config['enc_ligand_dim'], generator=g) if 'ligand' in encs else None
    out['enc_node'] = torch.randn(n_nodes, config['enc_node_dim'], generator=g) if 'node' in encs else None
    out['enc_graph'] = torch.randn(B, config['enc_graph_dim'], generator=g) if 'graph' in encs else None
    return out


def _reference_model(config, sd):
    from . import refload
    refload.import_reference()
    from easydict import EasyDict
    from models.property_pred.prop_model import PropPredNet, PropPredNetEnc
    cfg = EasyDict(config)
    L = sd['ligand_atom_emb.weight'].shape[1]
    if config['encoder']['name'] == 'egnn_enc':
        model = PropPredNetEnc(cfg, PROTEIN_FEATURE_DIM, L - cfg.enc_ligand_dim, cfg.enc_ligand_dim, cfg.enc_node_dim, cfg.enc_graph_dim,
                               cfg.enc_feature_type, output_dim=1)
    else:
        model = PropPredNet(cfg, PROTEIN_FEATURE_DIM, L, output_dim=3)
    model.load_state_dict(sd, strict=True)
    return model.eval()


def run_reference_pins():
    """The reference's outputs for every PIN_CASES entry, mapped to the stable node order."""
    out = {}
    for name, (config, seed, _, _, _, _) in PIN_CASES.items():
        sd = make_state_dict(config, seed)
        x = pin_inputs(name)
        model = _reference_model(config, sd)
        ref_order = torch.cat([x['batch_protein'], x['batch_ligand']]).argsort()           # what compose_context_prop does
        stable = compose_stable(x['batch_protein'], x['batch_ligand'])
        inv_stable = torch.empty_like(stable)
        inv_stable[stable] = torch.arange(len(stable))
        to_stable = inv_stable[ref_order]            # reference node i == stable node to_stable[i]
        captured = {}
        enc_mod = model.encoder
        h_hook = enc_mod.register_forward_hook(lambda m, a, o: captured.__setitem__('h', o.detach().clone()))
        import models.property_pred.prop_egnn as pe
        orig_knn = pe.knn_graph

        def knn_spy(*a, **k):
            ei = orig_knn(*a, **k)
            captured['edge_index'] = ei.clone()
            return ei
        pe.knn_graph = knn_spy
        try:
            with torch.no_grad():
                kw = dict(output_kind=x['output_kind'])
                if config['encoder']['name'] == 'egnn_enc':
                    kw.update(enc_ligand_feature=x['enc_ligand'], enc_graph_feature=x['enc_graph'],
                              enc_node_feature=x['enc_node'][to_stable] if x['enc_node'] is not None else None)
                pred = model(x['protein_pos'], x['protein_feat'], x['ligand_pos'], x['ligand_feat'], x['batch_protein'], x['batch_ligand'], **kw)
        finally:
            pe.knn_graph = orig_knn
            h_hook.remove()
        h_stable = torch.empty_like(captured['h'])
        h_stable[to_stable] = captured['h']
        dst, src = captured['edge_index']                                                    # flow='target_to_source' (prop_egnn.py:77-78)
        ei = torch.stack([to_stable[src], to_stable[dst]])                                   # rows (src, dst) in the stable order
        key = ei[1] * len(stable) + ei[0]
        n = len(stable)
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:PIN_H_ROWS].sort().values
        p = name + '__'
        for k, v in x.items():
            if v is not None:
                out[p + k] = v
        out[p + 'pred'] = pred
        out[p + 'h_rows'] = rows
        out[p + 'h'] = h_stable[rows]
        out[p + 'edges_sorted'] = (key.sort().values).to(torch.int64)                        # dst * N + src, canonical set
        out[p + 'ref_order'] = ref_order
        out[p + 'layout'] = np.array(['%s:%s' % (k, 'x'.join(map(str, v.shape))) for k, v in model.state_dict().items()])
    return {k: v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v) for k, v in out.items()}


def main():
    arrs = run_reference_pins()
    np.savez_compressed(PIN_PATH, **arrs)
    print(PIN_PATH, os.path.getsize(PIN_PATH), 'bytes')


if __name__ == '__main__':
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    main()
