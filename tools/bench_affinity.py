"""Throughput of the affinity regressor (PropPredNet, published `egnn` config) on one GPU, with its precision against the CPU oracle.

    python tools/bench_affinity.py --complexes 4096 --batch 1024 --out result.json

Workload: `--complexes` protein-ligand complexes of realistic size (pockets of 300-600 atoms, ligands of 20-30 atoms), every complex a
distinct rigid placement + jitter of one of 32 synthetic pockets, resident on the device.  The working set (node states, projections,
neighbour lists: about 12 KB per atom) is far larger than the 126 MB L2.  Timed with CUDA events after a warm-up pass; the in-situ
edge-kernel time comes from a separate profiling pass (events around every edge-kernel launch).  A sample of the timed outputs is
checked against oracle.prop in the same run, the pinned reference cases (tests/golden/prop_pins.npz) give the maximum errors, and a
CPU baseline runs the oracle on the host cores.  Prints one JSON object and writes it to --out.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import prop, synth  # noqa: E402
from targetdiff_b200 import _lib  # noqa: E402
from targetdiff_b200.prop_model import PropPredNet, PropPredNetEnc  # noqa: E402

DATASHEET_BF16_TFLOPS = 2250.0      # HGX B200 data sheet, dense BF16, one GPU at 1000 W


def make_workload(n, seed=0):
    rng = np.random.RandomState(seed)
    bases = [synth.make_pocket(7000 + i, int(rng.randint(300, 601))) for i in range(32)]
    g = torch.Generator().manual_seed(seed)
    ppos, pfeat, lpos, ps, ls = [], [], [], [], []
    for i in range(n):
        p, f = bases[i % 32]
        p = p + torch.from_numpy(rng.uniform(-50, 50, size=(1, 3)).astype(np.float32)) + 0.05 * torch.randn(p.shape, generator=g)
        nl = int(rng.randint(20, 31))
        ppos.append(p), pfeat.append(f), ps.append(len(p)), ls.append(nl)
        lpos.append(p.mean(0, keepdim=True) + 1.5 * torch.randn(nl, 3, generator=g))
    return dict(protein_pos=torch.cat(ppos), protein_feat=torch.cat(pfeat), ligand_pos=torch.cat(lpos),
                ligand_feat=prop.make_ligand_features(seed + 1, sum(ls)), psizes=ps, lsizes=ls)


def batches(w, batch):
    """Split the workload into forward calls of `batch` complexes: list of dicts of device tensors + the graph range."""
    out, p0, l0 = [], 0, 0
    for g0 in range(0, len(w['psizes']), batch):
        ps, ls = w['psizes'][g0:g0 + batch], w['lsizes'][g0:g0 + batch]
        np_, nl = sum(ps), sum(ls)
        out.append(dict(g0=g0, p0=p0, l0=l0, protein_pos=w['protein_pos'][p0:p0 + np_], protein_feat=w['protein_feat'][p0:p0 + np_],
                        ligand_pos=w['ligand_pos'][l0:l0 + nl], ligand_feat=w['ligand_feat'][l0:l0 + nl],
                        batch_protein=torch.repeat_interleave(torch.arange(len(ps)), torch.tensor(ps)),
                        batch_ligand=torch.repeat_interleave(torch.arange(len(ls)), torch.tensor(ls))))
        p0, l0 = p0 + np_, l0 + nl
    return out


def gpu_info():
    try:
        r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True,
                           timeout=30)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 else 'nvidia-smi failed: ' + r.stderr.strip()
    except Exception as e:          # noqa: BLE001
        return 'nvidia-smi unavailable: %s' % e


def precision_on_pins(dev):
    pins = np.load(os.path.join(ROOT, 'tests', 'golden', 'prop_pins.npz'))
    res = {}
    for name, (config, seed, *_rest) in prop.PIN_CASES.items():
        x = prop.pin_inputs(name)
        for gain in (1.0, 3.0):
            sd = prop.make_state_dict(config, seed, gain=gain)
            if config['encoder']['name'] == 'egnn_enc':
                m = PropPredNetEnc(config, 27, prop.LIGAND_FEATURE_DIM, config['enc_ligand_dim'], config['enc_node_dim'], config['enc_graph_dim'])
            else:
                m = PropPredNet(config, 27, prop.LIGAND_FEATURE_DIM)
            m.load_state_dict(sd, strict=True)
            m = m.to(dev)
            d = {k: (v.to(dev) if v is not None else None) for k, v in x.items()}
            args = [d['protein_pos'], d['protein_feat'], d['ligand_pos'], d['ligand_feat'], d['batch_protein'], d['batch_ligand'], d['output_kind']]
            if config['encoder']['name'] == 'egnn_enc':
                args += [d['enc_ligand'], d['enc_node'], d['enc_graph']]
            out, h = m(*args, return_h=True)
            out, h = out.cpu(), h.cpu()
            tr = {}
            want = prop.prop_forward(sd, config, x['protein_pos'], x['protein_feat'], x['ligand_pos'], x['ligand_feat'], x['batch_protein'],
                                     x['batch_ligand'], x['output_kind'], x['enc_ligand'], x['enc_node'], x['enc_graph'], trace=tr)
            r = dict(pred_max_abs_err_vs_oracle=(out - want).abs().max().item(),
                     pred_max_rel_err_vs_oracle=((out - want).abs() / want.abs().clamp_min(1e-30)).max().item(),
                     h_max_err_over_max_abs_h_vs_oracle=(h - tr['h']).abs().max().item() / tr['h'].abs().max().item())
            # against the float64 emulation of the kernels' bf16 split; where the split's error switches an edge gate (a logit
            # within that error of 0), also against the emulation with those gates on the float64 side
            flips, z64, ei = prop.gate_flips(sd, config, x)
            sides = {'split_emulation': None}
            if flips:
                sides['split_emulation_fp64_gates'] = {l: (i, z64[l][i]) for l, i in flips.items()}
            for label, ov in sides.items():
                eo, eh, _, _ = prop.forward_with_gates(sd, config, x, linear=prop.tensor_core_linear, gate_override=ov)
                r['h_max_err_over_max_abs_h_vs_' + label] = (h.double() - eh).abs().max().item() / eh.abs().max().item()
                r['pred_max_err_over_max_abs_pred_vs_' + label] = (out.double() - eo).abs().max().item() / max(eo.abs().max().item(), 1.0)
            r['gate_flips_layer_src_dst'] = [(l, ei[0, i].item(), ei[1, i].item()) for l, idx in flips.items() for i in idx]
            if gain == 1.0:
                ref = torch.from_numpy(pins[name + '__pred'])
                hr = torch.from_numpy(pins[name + '__h'])
                r.update(pred_max_abs_err_vs_reference=(out - ref).abs().max().item(),
                         h_max_err_over_max_abs_h_vs_reference=(h[torch.from_numpy(pins[name + '__h_rows'])] - hr).abs().max().item() / hr.abs().max().item())
            res['%s_gain%g' % (name, gain)] = r
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--complexes', type=int, default=4096)
    ap.add_argument('--batch', type=int, default=1024)
    ap.add_argument('--iters', type=int, default=5)
    ap.add_argument('--check', type=int, default=4, help='complexes of the timed pass checked against the CPU oracle')
    ap.add_argument('--cpu-complexes', type=int, default=4)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_affinity needs a CUDA device (there is no CPU path to time)')
    dev = torch.device('cuda:0')
    config = prop.EGNN_CONFIG
    sd = prop.make_state_dict(config, 0)
    model = PropPredNet(config, 27, prop.LIGAND_FEATURE_DIM)
    model.load_state_dict(sd, strict=True)
    model = model.to(dev)
    w = make_workload(a.complexes)
    host_batches = batches(w, a.batch)
    dev_batches = [{k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in b.items()} for b in host_batches]
    outs = [torch.empty(0)] * len(dev_batches)

    def one_pass():
        for i, b in enumerate(dev_batches):
            outs[i] = model(b['protein_pos'], b['protein_feat'], b['ligand_pos'], b['ligand_feat'], b['batch_protein'], b['batch_ligand'], None)

    one_pass()                                        # warm-up: module load, smem opt-in, buffer growth
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.iters):
        one_pass()
    e1.record()
    torch.cuda.synchronize()
    ms_pass = e0.elapsed_time(e1) / a.iters
    n_atoms = sum(w['psizes']) + sum(w['lsizes'])
    # in-situ edge-kernel time (separate pass: profiling synchronises after each edge launch)
    lib = _lib.load()
    eng = model.engine(dev)
    _lib.check(lib.tdiff_prop_profile(eng, 1))
    one_pass()
    torch.cuda.synchronize()
    ms_edge, n_launch, n_rows = ctypes.c_double(), ctypes.c_int64(), ctypes.c_int64()
    _lib.check(lib.tdiff_prop_profile_read(eng, ctypes.byref(ms_edge), ctypes.byref(n_launch), ctypes.byref(n_rows)))
    _lib.check(lib.tdiff_prop_profile(eng, 0))
    G, H = config['encoder']['num_r_gaussian'], 256
    mac_per_row = 64 * H + H * H                       # gaussian block (K padded to 64) + second Linear
    executed_flop = 2.0 * mac_per_row * n_rows.value * 3          # three bf16 passes per product (a1b1 + a1b2 + a2b1)
    n_edges_useful = n_atoms * config['encoder']['knn']            # every graph here has > k atoms
    useful_flop = 2.0 * (G * H + H * H) * n_edges_useful * (n_launch.value // len(dev_batches))
    peak, peak_src = DATASHEET_BF16_TFLOPS, 'data sheet (HGX B200 dense BF16, 1000 W); MEASURED_PEAKS.json not present'
    pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(pk):
        peak, peak_src = float(json.load(open(pk))['bf16_tflops_sustained']), 'MEASURED_PEAKS.json bf16_tflops_sustained'
    edge_tflops = executed_flop / (ms_edge.value * 1e-3) / 1e12
    # outputs of the timed pass against the oracle (first graphs of the first batch)
    b0 = host_batches[0]
    nchk = min(a.check, len(w['psizes']))
    pn, ln = sum(w['psizes'][:nchk]), sum(w['lsizes'][:nchk])
    want = prop.prop_forward(sd, config, b0['protein_pos'][:pn], b0['protein_feat'][:pn], b0['ligand_pos'][:ln], b0['ligand_feat'][:ln],
                             b0['batch_protein'][:pn], b0['batch_ligand'][:ln])
    got = outs[0][:nchk].cpu()
    check_err = (got - want).abs().max().item()
    check_ok = bool(torch.allclose(got, want, rtol=1e-4, atol=1e-3))
    # CPU baseline: the oracle on the host cores
    cb = batches(w, a.cpu_complexes)[0]
    t0 = time.perf_counter()
    prop.prop_forward(sd, config, cb['protein_pos'], cb['protein_feat'], cb['ligand_pos'], cb['ligand_feat'], cb['batch_protein'], cb['batch_ligand'])
    cpu_s = time.perf_counter() - t0
    res = dict(
        workload=dict(config='pdbbind_general_egnn (hidden 256, knn 48, 6 layers, 64 gaussians)', complexes=a.complexes, batch=a.batch,
                      atoms=n_atoms, mean_atoms_per_complex=n_atoms / a.complexes, pocket_atoms='300-600', ligand_atoms='20-30', iters=a.iters),
        gpu=gpu_info(),
        complexes_per_s=a.complexes / (ms_pass * 1e-3), ms_per_pass=ms_pass,
        edge_kernel=dict(ms_total_per_pass=ms_edge.value, launches=n_launch.value, tile_rows=n_rows.value,
                         executed_tensor_tflops=edge_tflops, useful_fp32_equiv_tflops=useful_flop / (ms_edge.value * 1e-3) / 1e12,
                         share_of_bf16_peak=edge_tflops / peak, peak_tflops=peak, peak_source=peak_src,
                         share_of_pass=ms_edge.value / ms_pass,
                         note='executed = 3 bf16 MMA passes x (64x256 + 256x256) MAC x 128 rows per tile (2 destinations x 64 padded slots)'),
        check_vs_oracle=dict(complexes=nchk, max_abs_err=check_err, within_tolerance=check_ok, tolerance="rtol 1e-4, atol 1e-3"),
        cpu_baseline=dict(complexes=a.cpu_complexes, seconds=cpu_s, complexes_per_s=a.cpu_complexes / cpu_s, threads=torch.get_num_threads(),
                          what='oracle.prop.prop_forward, torch CPU fp32'),
        precision=precision_on_pins(dev),
    )
    s = json.dumps(res, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(s + '\n')
    if not check_ok:
        raise SystemExit('outputs of the timed pass disagree with the oracle')


if __name__ == '__main__':
    main()
