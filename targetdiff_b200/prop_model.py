"""PropPredNet / PropPredNetEnc -- drop-in for the reference's binding-affinity regressor (inference).

Mirrors the reference's Python surface (models/property_pred/prop_model.py:27-165, utils/misc_prop.py:45-64): constructor
signatures, `state_dict` layout (including the unused per-layer `r_expansion.offset` buffers, so `load_state_dict(ckpt['model'])`
is strict-compatible), `forward` signatures and `get_model`.

The modules below only *hold parameters*: every computation goes through libtdiff.so (tdiff_prop_*, hand-written sm_100a kernels,
include/tdiff.h).  There is no PyTorch/CPU execution path; calling forward on CPU tensors raises.
"""
import ctypes

import torch
import torch.nn as nn

from . import _lib
from .config import Config

HIDDEN = 256      # the only hidden width the kernels are built for


def _cfg(config):
    return config if isinstance(config, Config) else Config(dict(config))


def check_supported(config):
    """Raise NotImplementedError, with the reason, for a model config the B200 kernels do not implement."""
    enc = config.encoder
    if enc.name not in ('egnn', 'egnn_enc'):
        raise NotImplementedError("encoder.name=%r: only 'egnn' / 'egnn_enc' (EnEquiEncoder) exist in the reference" % enc.name)
    if config.hidden_channels != HIDDEN or enc.hidden_dim != HIDDEN:
        raise NotImplementedError('hidden_channels=%s, encoder.hidden_dim=%s: the kernels are built for 256' % (config.hidden_channels, enc.hidden_dim))
    if not 2 <= enc.num_r_gaussian <= 64:
        raise NotImplementedError('num_r_gaussian=%s: the gaussian block is one 64-wide MMA K-block (and the reference needs >= 2)' % enc.num_r_gaussian)
    if enc.act_fn != 'relu':
        raise NotImplementedError("act_fn=%r: only 'relu' is implemented" % enc.act_fn)
    if enc.norm:
        raise NotImplementedError('norm=True (LayerNorm inside the edge / node MLPs) is not implemented')
    if enc.edge_dim > 0:
        raise NotImplementedError('edge_dim=%s: the encoder has no edge features in any published config' % enc.edge_dim)
    if not 1 <= enc.knn <= 64:
        raise NotImplementedError('knn=%s outside 1..64 (neighbour slots per destination)' % enc.knn)


class _Offsets(nn.Module):
    def __init__(self, stop, n):
        super().__init__()
        self.register_buffer('offset', torch.linspace(0.0, stop, n))     # GaussianSmearing(fixed_offset=False), models/common.py:7-19


class _Net(nn.Module):
    def __init__(self, *layers):
        super().__init__()
        self.net = nn.Sequential(*layers)


class _EnBaseLayer(nn.Module):
    """parameter holder of EnBaseLayer (prop_egnn.py:8-26; same module order = same state_dict order)"""

    def __init__(self, H, G):
        super().__init__()
        self.r_expansion = _Offsets(10.0 ** 2, G)        # never read by the reference's forward either
        self.edge_mlp = _Net(nn.Linear(2 * H + G, H), nn.ReLU(), nn.Linear(H, H), nn.ReLU())
        self.edge_inf = nn.Sequential(nn.Linear(H, 1), nn.Sigmoid())
        self.node_mlp = _Net(nn.Linear(2 * H, H), nn.ReLU(), nn.Linear(H, H))


class _Encoder(nn.Module):
    def __init__(self, enc):
        super().__init__()
        self.distance_expansion = _Offsets(float(enc.cutoff), enc.num_r_gaussian)
        self.net = nn.ModuleList([_EnBaseLayer(enc.hidden_dim, enc.num_r_gaussian) for _ in range(enc.num_layers)])


class _ShiftedSoftplus(nn.Module):
    pass


def _counts(batch, name, B):
    if batch.numel() > 1 and bool((batch[1:] < batch[:-1]).any()):
        raise ValueError('%s must be sorted ascending (PyG Batch order)' % name)
    return torch.bincount(batch, minlength=B).cpu().tolist()


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


class _PropBase(nn.Module):
    def _init_common(self, config, protein_atom_feature_dim, ligand_in_dim, output_dim, enc_graph_dim):
        config = _cfg(config)
        check_supported(config)
        self.config = config
        self.hidden_dim = config.hidden_channels
        self.output_dim = output_dim
        self.protein_atom_feature_dim = protein_atom_feature_dim
        self.protein_atom_emb = nn.Linear(protein_atom_feature_dim, self.hidden_dim)
        self.ligand_atom_emb = nn.Linear(ligand_in_dim, self.hidden_dim)
        self.encoder = _Encoder(config.encoder)
        self._out_in = self.hidden_dim + enc_graph_dim
        self.__dict__['_engine'] = None
        self.__dict__['_engine_device'] = None

    def _add_out_block(self):
        self.out_block = nn.Sequential(nn.Linear(self._out_in, self.hidden_dim), _ShiftedSoftplus(), nn.Linear(self.hidden_dim, self.output_dim))
        self.requires_grad_(False)          # inference engine: the CUDA path has no backward

    # ------------------------------------------------------------------ engine management
    def _apply(self, fn, *a, **k):
        self._drop_engine()
        return super()._apply(fn, *a, **k)

    def load_state_dict(self, *a, **k):
        self._drop_engine()
        return super().load_state_dict(*a, **k)

    def _drop_engine(self):
        eng = self.__dict__.get('_engine')
        if eng is not None:
            _lib.load().tdiff_prop_destroy(eng)
        self.__dict__['_engine'] = None

    def __del__(self):
        try:
            self._drop_engine()
        except Exception:
            pass

    def engine(self, device):
        """The libtdiff model for `device` (created on first use from the current state_dict)."""
        device = torch.device(device)
        if device.type != 'cuda':
            raise RuntimeError('%s (targetdiff_b200) only runs on CUDA devices; got %s. There is no CPU path.' % (type(self).__name__, device))
        index = device.index if device.index is not None else torch.cuda.current_device()
        if self._engine is not None and self._engine_device == index:
            return self._engine
        self._drop_engine()
        lib = _lib.load()
        sd = {k: v.detach().to('cpu', torch.float32).contiguous() for k, v in self.state_dict().items()}
        entries = (_lib.tdiff_tensor * len(sd))()
        keep = []
        for i, (k, v) in enumerate(sd.items()):
            name = k.encode()
            keep.append((name, v))
            entries[i].name, entries[i].data, entries[i].numel = name, v.data_ptr(), v.numel()
        enc = self.config.encoder
        cfg = _lib.tdiff_prop_config(self.hidden_dim, enc.num_layers, enc.knn, enc.num_r_gaussian, enc.edge_dim, int(bool(enc.norm)),
                                     self.protein_atom_feature_dim, self.ligand_atom_feature_dim, self._enc_dims[0], self._enc_dims[1],
                                     self._enc_dims[2], self.output_dim)
        out = ctypes.c_void_p()
        _lib.check(lib.tdiff_prop_create(ctypes.byref(cfg), entries, len(sd), index, ctypes.byref(out)))
        self.__dict__['_engine'], self.__dict__['_engine_device'] = out, index
        return out

    @torch.no_grad()
    def _run(self, protein_pos, protein_atom_feature, ligand_pos, ligand_atom_feature, batch_protein, batch_ligand, output_kind,
             enc_ligand_feature=None, enc_node_feature=None, enc_graph_feature=None, return_h=False):
        dev = protein_pos.device
        eng = self.engine(dev)
        lib = _lib.load()
        B = int(max(batch_protein.max().item() if batch_protein.numel() else -1, batch_ligand.max().item() if batch_ligand.numel() else -1)) + 1
        if B < 1:
            raise ValueError('empty batch')
        pc, lc = _counts(batch_protein, 'batch_protein', B), _counts(batch_ligand, 'batch_ligand', B)
        Np, Nl = sum(pc), sum(lc)
        N = Np + Nl

        def f32(t, rows, cols, name):
            if t is None:
                return None
            if t.device != dev:
                raise ValueError('%s is on %s, expected %s' % (name, t.device, dev))
            t = t.detach().to(torch.float32).contiguous()
            if t.dim() != 2 or t.shape[0] != rows or t.shape[1] != cols:
                raise ValueError('%s must be [%d, %d], got %s' % (name, rows, cols, list(t.shape)))
            return t
        ppos = f32(protein_pos, Np, 3, 'protein_pos')
        pfeat = f32(protein_atom_feature, Np, self.protein_atom_feature_dim, 'protein_atom_feature')
        lpos = f32(ligand_pos, Nl, 3, 'ligand_pos')
        lfeat = f32(ligand_atom_feature, Nl, self.ligand_atom_feature_dim, 'ligand_atom_feature')
        el = f32(enc_ligand_feature, Nl, self._enc_dims[0], 'enc_ligand_feature')
        en = f32(enc_node_feature, N, self._enc_dims[1], 'enc_node_feature')
        eg = f32(enc_graph_feature, B, self._enc_dims[2], 'enc_graph_feature')
        kind = None
        if output_kind is not None:
            kind = output_kind.detach().to(dev, torch.int64).reshape(-1).contiguous()
            if kind.numel() != B:
                raise ValueError('output_kind must have one entry per graph (%d), got %d' % (B, kind.numel()))
        out = torch.empty(B, 1 if kind is not None else self.output_dim, device=dev)
        h = torch.empty(N, self.hidden_dim, device=dev) if return_h else None
        st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(lib.tdiff_prop_forward(eng, B, _lib.i32_array(pc), _lib.i32_array(lc), _ptr(ppos), _ptr(pfeat), _ptr(lpos), _ptr(lfeat),
                                          _ptr(el), _ptr(en), _ptr(eg), _ptr(kind), _ptr(out), _ptr(h), st))
        return (out, h) if return_h else out

    def get_loss(self, *a, **k):
        raise NotImplementedError('training is out of scope of the B200 engine: the affinity kernels have no backward')


class PropPredNet(_PropBase):
    """reference models/property_pred/prop_model.py:27-95 (output_dim 3: Ki / Kd / IC50 columns)."""

    def __init__(self, config, protein_atom_feature_dim, ligand_atom_feature_dim, output_dim=3):
        super().__init__()
        self.ligand_atom_feature_dim = ligand_atom_feature_dim
        self._enc_dims = (0, 0, 0)
        self._init_common(config, protein_atom_feature_dim, ligand_atom_feature_dim, output_dim, 0)
        self._add_out_block()

    def forward(self, protein_pos, protein_atom_feature, ligand_pos, ligand_atom_feature, batch_protein, batch_ligand, output_kind,
                return_h=False):
        """Prediction [B,1] (the `output_kind` column of each graph) or [B,output_dim] with output_kind None.  return_h=True also
        returns the encoder output [N,256] in composed node order (per graph: protein atoms, then ligand atoms)."""
        return self._run(protein_pos, protein_atom_feature, ligand_pos, ligand_atom_feature, batch_protein, batch_ligand, output_kind,
                         return_h=return_h)


class PropPredNetEnc(_PropBase):
    """reference models/property_pred/prop_model.py:98-165: TargetDiff-derived features in three places (ligand atoms, every node,
    the pooled graph vector).  enc_node_feature rows are in composed node order, e.g. ScorePosNet3D.fetch_embedding(...)['final_h']."""

    def __init__(self, config, protein_atom_feature_dim, ligand_atom_feature_dim, enc_ligand_dim, enc_node_dim, enc_graph_dim,
                 enc_feature_type=None, output_dim=1):
        super().__init__()
        self.ligand_atom_feature_dim = ligand_atom_feature_dim
        self.enc_ligand_dim, self.enc_node_dim, self.enc_graph_dim = enc_ligand_dim, enc_node_dim, enc_graph_dim
        self.enc_feature_type = enc_feature_type
        self._enc_dims = (enc_ligand_dim, enc_node_dim, enc_graph_dim)
        self._init_common(config, protein_atom_feature_dim, ligand_atom_feature_dim + enc_ligand_dim, output_dim, enc_graph_dim)
        if enc_node_dim > 0:
            self.enc_node_layer = nn.Sequential(nn.Linear(self.hidden_dim + enc_node_dim, self.hidden_dim), nn.ReLU(),
                                                nn.Linear(self.hidden_dim, self.hidden_dim))
        self._add_out_block()

    def forward(self, protein_pos, protein_atom_feature, ligand_pos, ligand_atom_feature, batch_protein, batch_ligand, output_kind,
                enc_ligand_feature, enc_node_feature, enc_graph_feature, return_h=False):
        if enc_node_feature is not None and self.enc_node_dim == 0:
            raise ValueError('enc_node_feature given but the model has enc_node_dim 0 (no enc_node_layer)')
        return self._run(protein_pos, protein_atom_feature, ligand_pos, ligand_atom_feature, batch_protein, batch_ligand, output_kind,
                         enc_ligand_feature, enc_node_feature, enc_graph_feature, return_h=return_h)


def get_model(config, protein_atom_feat_dim, ligand_atom_feat_dim):
    """reference utils/misc_prop.py:45-64 (`config` is the whole training config; its `model` section builds the network)."""
    config = _cfg(config)
    if config.model.encoder.name == 'egnn_enc':
        return PropPredNetEnc(config.model, protein_atom_feature_dim=protein_atom_feat_dim, ligand_atom_feature_dim=ligand_atom_feat_dim,
                              enc_ligand_dim=config.model.enc_ligand_dim, enc_node_dim=config.model.enc_node_dim,
                              enc_graph_dim=config.model.enc_graph_dim, enc_feature_type=config.model.enc_feature_type, output_dim=1)
    return PropPredNet(config.model, protein_atom_feature_dim=protein_atom_feat_dim, ligand_atom_feature_dim=ligand_atom_feat_dim, output_dim=3)
