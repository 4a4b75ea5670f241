"""Regenerate tests/golden/*.npz by running the UNMODIFIED reference (under oracle/shims) -- build container only.

    python -m oracle.make_golden

Inputs/weights/noise come from oracle.synth seeds (rebuildable anywhere); only the reference's OUTPUTS are
stored.  Cases:
  forward_small   ScorePosNet3D.forward, 2 graphs (60 protein + 9 / 7 ligand atoms), default config
  chain_trunc     sample_diffusion, T=1000, num_steps=5 (t = 999..995: truncated chain, never reaches t==0)
  chain_full_T20  sample_diffusion, num_diffusion_timesteps=20, num_steps=None (reaches the t==0 no-noise branch)
  likelihood      likelihood_estimation at mixed time steps + the prior branch
Long cases (minutes of CPU each; `python -m oracle.make_golden <name>`):
  chain_1000_cfg1   BASELINE configs[0] shape (1 graph, 300 + 20 atoms), the FULL chain t = 999..0 on one noise tape
  chain_cfg5        BASELINE configs[4] shape (1 graph, 1200 + 40 atoms, knn = 48), 20 steps
  pocket_1h36_s50   the reference DRIVER (scripts/sample_diffusion.py:31-116 via scripts/sample_for_pocket.py:18-31) on
                    tests/golden/1h36_pocket10.pdb (= reference examples/1h36_A_rec_1h36_r88_lig_tt_docked_0_pocket10.pdb),
                    seed 2021, 3 samples in batches of 2, prior sizes, 50 steps -- all draws from the global CPU generators
  pocket_1h36_full  same, 2 samples, the full 1000 steps (BASELINE configs[1] at a CPU-feasible sample count)
Reference pins (`python -m oracle.make_golden reference_pins`, about a minute):
  reference_pins    the reference's side of every comparison in tests/test_oracle_vs_reference.py (state_dict layouts,
                    schedules, forward, 3-step chains, likelihood_estimation, backbone options, the sampling driver on
                    the 1h36 pocket, check_stability), so that those bit-exact pins hold without the reference tree
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import refload, restate, synth  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(HERE), 'tests', 'golden')

CASES = {
    'forward_small': dict(cfg={}, weight_seed=0, batch=dict(seed=1, n_graphs=2, n_protein=60, ligand_sizes=[9, 7])),
    'chain_trunc': dict(cfg={}, weight_seed=3, batch=dict(seed=2, n_graphs=2, n_protein=48, ligand_sizes=[8, 6]),
                        tape_seed=7, num_steps=5),
    'chain_full_T20': dict(cfg={'num_diffusion_timesteps': 20}, weight_seed=4,
                           batch=dict(seed=5, n_graphs=1, n_protein=50, ligand_sizes=[10]), tape_seed=9, num_steps=None),
    # SURVEY 8(f) n3: likelihood_estimation at mixed time steps (incl. the decoder branch t = 0) and the prior branch (t = T)
    'likelihood': dict(cfg={}, weight_seed=5, batch=dict(seed=4, n_graphs=3, n_protein=64, ligand_sizes=[7, 10, 4]), tape_seed=9,
                       time_steps=[0, 999, 417]),
}


LONG_CASES = {
    'chain_1000_cfg1': dict(cfg={}, weight_seed=0, batch=dict(seed=100, n_graphs=1, n_protein=300, ligand_sizes=[20]), tape_seed=7,
                            num_steps=None, stride=25),
    # stressed weights: every Linear scaled x3 (attention logits ~ x9, value / coordinate messages ~ x3) -- sharper, less benign dynamics than
    # the default initialisation; stand-in for a trained checkpoint in the precision audit (tools/precision_audit.py)
    'chain_1000_cfg1_gain3': dict(cfg={}, weight_seed=0, gain=3.0, batch=dict(seed=100, n_graphs=1, n_protein=300, ligand_sizes=[20]), tape_seed=7,
                                  num_steps=None, stride=25),
    'chain_cfg5': dict(cfg={'knn': 48}, weight_seed=6, batch=dict(seed=55, n_graphs=1, n_protein=1200, ligand_sizes=[40]), tape_seed=8,
                       num_steps=20, stride=1),
    'pocket_1h36_s50': dict(cfg={}, weight_seed=0, seed=2021, num_samples=3, batch_size=2, num_steps=50, stride=1),
    'pocket_1h36_full': dict(cfg={}, weight_seed=0, seed=2021, num_samples=2, batch_size=2, num_steps=1000, stride=25),
}
PDB_1H36 = os.path.join(GOLDEN, '1h36_pocket10.pdb')


def run_long_case(name):
    """Outputs of the unmodified reference for the long cases.  Trajectories of log-probabilities are kept every `stride` steps
    (positions and types at every step)."""
    import time
    case = LONG_CASES[name]
    ref, model, sd = build_reference_model(case)
    t0 = time.time()
    with torch.no_grad():
        if 'batch' in case:
            b = synth.make_batch(**case['batch'])
            T = sd['betas'].shape[0]
            S = case['num_steps'] or T
            pn, vu = synth.make_tape(case['tape_seed'], S, len(b['batch_ligand']))
            with refload.noise_tape(pn, vu):
                r = model.sample_diffusion(b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'],
                                           b['init_ligand_v'], b['batch_ligand'], num_steps=case['num_steps'], center_pos_mode='protein')
            st = case['stride']
            out = dict(pos=r['pos'], v=r['v'], pos_traj=torch.stack(r['pos_traj']), v_traj=torch.stack(r['v_traj']).to(torch.int8),
                       v0_traj=torch.stack(r['v0_traj'])[::st], vt_traj=torch.stack(r['vt_traj'])[::st])
        else:
            sd_mod, sfp = refload.import_reference_scripts()
            import utils.misc as misc
            import utils.transforms as trans
            data = trans.FeaturizeProteinAtom()(sfp.pdb_to_pocket_data(PDB_1H36))
            misc.seed_all(case['seed'])
            res = sd_mod.sample_diffusion_ligand(model, data, case['num_samples'], batch_size=case['batch_size'], device='cpu',
                                                 num_steps=case['num_steps'], pos_only=False, center_pos_mode='protein',
                                                 sample_num_atoms='prior')
            pos, v, pos_traj, v_traj, v0_traj, vt_traj, _ = res
            st = case['stride']
            out = dict(sizes=torch.tensor([len(p) for p in pos]), pos=torch.from_numpy(np.concatenate(pos)), v=torch.from_numpy(np.concatenate(v)),
                       pos_traj=torch.from_numpy(np.concatenate(pos_traj, axis=1)).float(),
                       v_traj=torch.from_numpy(np.concatenate(v_traj, axis=1)).to(torch.int8),
                       v0_traj=torch.from_numpy(np.concatenate(v0_traj, axis=1))[::st],
                       vt_traj=torch.from_numpy(np.concatenate(vt_traj, axis=1))[::st])
    out['cpu_seconds'] = torch.tensor(time.time() - t0)
    return {k: v.detach().cpu().numpy() for k, v in out.items()}


def build_reference_model(case):
    ref = refload.import_reference()
    cfg = refload.default_model_config()
    cfg.update(case['cfg'])
    model = ref.ScorePosNet3D(cfg, synth.PROTEIN_FEATURE_DIM, synth.LIGAND_NUM_CLASSES)
    sd = synth.make_state_dict(case['weight_seed'], case['cfg'], schedules=restate.make_schedules(case['cfg']), gain=case.get('gain', 1.0))
    for k in synth.SCHEDULE_KEYS:       # our fp64->fp32 tables must equal the reference's own
        assert torch.equal(model.state_dict()[k], sd[k]), k
    model.load_state_dict(sd, strict=True)
    return ref, model.eval(), sd


def run_case(name):
    case = CASES[name]
    ref, model, sd = build_reference_model(case)
    b = synth.make_batch(**case['batch'])
    out = {}
    with torch.no_grad():
        if 'time_steps' in case:
            pn, vu = synth.make_tape(case['tape_seed'], 1, len(b['batch_ligand']))
            args = (b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'], b['init_ligand_v'], b['batch_ligand'])
            with refload.noise_tape(pn, vu):
                kp, kv = model.likelihood_estimation(*args, time_step=torch.tensor(case['time_steps']))
            T = sd['betas'].shape[0]
            kp_T, kv_T = model.likelihood_estimation(*args, time_step=torch.full((len(case['time_steps']),), T))
            out = dict(kl_pos=kp, kl_v=kv, kl_pos_prior=kp_T, kl_v_prior=kv_T)
        elif 'num_steps' not in case:
            pp, lp, _ = ref.center_pos(b['protein_pos'], b['init_ligand_pos'], b['batch_protein'], b['batch_ligand'])
            # capture the backbone's intermediate state through its own return_all / a forward hook
            grabbed = {}
            net = model.refine_net
            orig = net._connect_edge
            net._connect_edge = lambda x, m, bt: grabbed.setdefault('edge_index', orig(x, m, bt))
            layer_out = []
            hooks = [l.register_forward_hook(lambda mod, inp, o: layer_out.append((o[0].clone(), o[1].clone())))
                     for l in net.base_block]
            ew = []
            hooks.append(net.edge_pred_layer.register_forward_hook(lambda mod, inp, o: ew.append(torch.sigmoid(o))))
            preds = model(pp, b['protein_v'], b['batch_protein'], lp, b['init_ligand_v'], b['batch_ligand'])
            for h in hooks:
                h.remove()
            net._connect_edge = orig
            out = dict(pred_ligand_pos=preds['pred_ligand_pos'], pred_ligand_v=preds['pred_ligand_v'],
                       final_h=preds['final_h'], edge_index=grabbed['edge_index'], e_w=ew[0].view(-1),
                       layer_x=torch.stack([x for _, x in layer_out]), layer0_h=layer_out[0][0],
                       layer4_h=layer_out[4][0])
        else:
            T = sd['betas'].shape[0]
            S = case['num_steps'] or T
            pn, vu = synth.make_tape(case['tape_seed'], S, len(b['batch_ligand']))
            with refload.noise_tape(pn, vu):
                r = model.sample_diffusion(b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'],
                                           b['init_ligand_v'], b['batch_ligand'], num_steps=case['num_steps'],
                                           center_pos_mode='protein')
            out = dict(pos=r['pos'], v=r['v'], pos_traj=torch.stack(r['pos_traj']), v_traj=torch.stack(r['v_traj']),
                       v0_traj=torch.stack(r['v0_traj']), vt_traj=torch.stack(r['vt_traj']))
    return {k: v.detach().cpu().numpy() for k, v in out.items()}


# ---- reference pins: inputs of tests/test_oracle_vs_reference.py; the reference's outputs go to reference_pins.npz
PIN_FORWARD = dict(weight_seed=0, batch=dict(seed=1, n_graphs=2, n_protein=60, ligand_sizes=[9, 7]))
PIN_CHAINS = {     # name -> model config, weight seed, batch, noise tape (seed, steps)
    'chain': dict(cfg={}, weight_seed=3, batch=dict(seed=2, n_graphs=2, n_protein=48, ligand_sizes=[8, 6]), tape=(7, 3)),
    'chain_noise': dict(cfg={'model_mean_type': 'noise'}, weight_seed=6, batch=dict(seed=8, n_graphs=2, n_protein=48, ligand_sizes=[8, 6]),
                        tape=(7, 3)),
}
PIN_LIKELIHOOD = dict(weight_seed=5, batch=dict(seed=4, n_graphs=2, n_protein=52, ligand_sizes=[7, 10]), tape_seed=9,
                      steps=[[0, 999], [417, 3], None])          # None: the prior branch, time_step == T
PIN_OPTION_CONFIGS = [{'num_blocks': 2}, {'ew_net_type': 'r'}, {'ew_net_type': 'm'}, {'ew_net_type': 'none'}, {'x2h_out_fc': True},
                      {'time_emb_dim': 1, 'time_emb_mode': 'simple'}, {'num_blocks': 2, 'ew_net_type': 'r', 'x2h_out_fc': True, 'time_emb_dim': 1},
                      {'cutoff_mode': 'hybrid'}, {'cutoff_mode': 'hybrid', 'knn': 8, 'num_blocks': 2}]
PIN_OPTIONS = dict(weight_seed=0, batch=dict(seed=3, n_graphs=2, n_protein=60, ligand_sizes=[9, 7]), tape=(5, 3))
PIN_DRIVER = dict(seed=2021, num_samples=3, batch_size=2, num_steps=2)
PIN_STABILITY = dict(seed=0, sizes=(1, 2, 9, 25, 40))


def stability_inputs():
    """Random molecule-like point sets of the check_stability pin: (n, hs, pos, z) in draw order."""
    rng = np.random.RandomState(PIN_STABILITY['seed'])
    for n in PIN_STABILITY['sizes']:
        for hs in (False, True):
            pos = np.cumsum(rng.normal(scale=0.85, size=(n, 3)), axis=0)          # chain-like: neighbours at bonding distance
            z = rng.choice([1, 6, 7, 8, 9, 15, 16, 17], size=n, p=[0.1, 0.5, 0.12, 0.15, 0.03, 0.02, 0.05, 0.03])
            yield n, hs, pos, z


def layout_strings(sd):
    """state_dict layout as 'key:shape' strings, in key order."""
    return np.array(['%s:%s' % (k, 'x'.join(str(s) for s in v.shape)) for k, v in sd.items()])


def run_reference_pins():
    """The reference's outputs for every comparison of tests/test_oracle_vs_reference.py (keys '<pin>__<array>')."""
    ref = refload.import_reference()
    out = {}

    def ref_model(cfgd=None):
        cfg = refload.default_model_config()
        cfg.update(cfgd or {})
        return ref.ScorePosNet3D(cfg, synth.PROTEIN_FEATURE_DIM, synth.LIGAND_NUM_CLASSES).eval()

    def chain(model, b, tape_seed, S, n_lig, prefix):
        pn, vu = synth.make_tape(tape_seed, S, n_lig)
        args = (b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'], b['init_ligand_v'], b['batch_ligand'])
        with torch.no_grad(), refload.noise_tape(pn, vu):
            r = model.sample_diffusion(*args, num_steps=S, center_pos_mode='protein')
        out.update({prefix + '__pos': r['pos'], prefix + '__v': r['v']})
        for k in ('pos_traj', 'v_traj', 'v0_traj', 'vt_traj'):
            out[prefix + '__' + k] = torch.stack(r[k])

    model = ref_model()
    out['layout'] = layout_strings(model.state_dict())
    for k in synth.SCHEDULE_KEYS:
        out['schedule__' + k] = model.state_dict()[k]

    model.load_state_dict(synth.make_state_dict(PIN_FORWARD['weight_seed'], schedules=restate.make_schedules()), strict=True)
    b = synth.make_batch(**PIN_FORWARD['batch'])
    with torch.no_grad():
        pp, lp, _ = ref.center_pos(b['protein_pos'], b['init_ligand_pos'], b['batch_protein'], b['batch_ligand'])
        want = model(pp, b['protein_v'], b['batch_protein'], lp, b['init_ligand_v'], b['batch_ligand'])
    out.update({'forward__protein_pos': pp, 'forward__ligand_pos': lp})
    for k in ('pred_ligand_pos', 'pred_ligand_v', 'final_h', 'final_ligand_h'):
        out['forward__' + k] = want[k]

    for name, c in PIN_CHAINS.items():
        model = ref_model(c['cfg'])
        model.load_state_dict(synth.make_state_dict(c['weight_seed'], schedules=restate.make_schedules()), strict=True)
        b = synth.make_batch(**c['batch'])
        chain(model, b, c['tape'][0], c['tape'][1], len(b['batch_ligand']), name)

    c = PIN_LIKELIHOOD
    model = ref_model()
    model.load_state_dict(synth.make_state_dict(c['weight_seed'], schedules=restate.make_schedules()), strict=True)
    b = synth.make_batch(**c['batch'])
    args = (b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'], b['init_ligand_v'], b['batch_ligand'])
    for i, steps in enumerate(c['steps']):
        pn, vu = synth.make_tape(c['tape_seed'], 1, len(b['batch_ligand']))
        t = torch.tensor(steps) if steps is not None else torch.full((2,), 1000)
        with torch.no_grad(), refload.noise_tape(pn, vu):
            kp, kv = model.likelihood_estimation(*args, time_step=t)
        out.update({'likelihood%d__kl_pos' % i: kp, 'likelihood%d__kl_v' % i: kv})

    c = PIN_OPTIONS
    for i, cfgd in enumerate(PIN_OPTION_CONFIGS):
        model = ref_model(cfgd)
        out['option%d__layout' % i] = layout_strings(model.state_dict())
        model.load_state_dict(synth.make_state_dict(c['weight_seed'], cfgd, schedules=restate.make_schedules(cfgd)), strict=True)
        b = synth.make_batch(**c['batch'])
        chain(model, b, c['tape'][0], c['tape'][1], len(b['batch_ligand']), 'option%d' % i)

    sd_mod, sfp = refload.import_reference_scripts()
    import utils.misc as misc
    import utils.transforms as trans
    data = trans.FeaturizeProteinAtom()(sfp.pdb_to_pocket_data(PDB_1H36))
    model = ref_model()
    model.load_state_dict(synth.make_state_dict(0, schedules=restate.make_schedules()), strict=True)
    c = PIN_DRIVER
    misc.seed_all(c['seed'])
    res = sd_mod.sample_diffusion_ligand(model, data, c['num_samples'], batch_size=c['batch_size'], device='cpu', num_steps=c['num_steps'],
                                         center_pos_mode='protein', sample_num_atoms='prior')
    for j, name in enumerate(('pos', 'v', 'pos_traj', 'v_traj', 'v0_traj', 'vt_traj')):
        for i, arr in enumerate(res[j]):
            out['driver__%s%d' % (name, i)] = arr
    out.update({'driver__protein_pos': data.protein_pos, 'driver__protein_atom_feature': data.protein_atom_feature})

    import importlib
    analyze = importlib.import_module('utils.evaluation.analyze')
    for n, hs, pos, z in stability_inputs():
        w = analyze.check_stability(pos, z, hs=hs, return_nr_bonds=True)
        out['stability%d_%d__counts' % (n, hs)] = np.array([bool(w[0]), w[1], w[2]], dtype=np.int64)
        out['stability%d_%d__nr_bonds' % (n, hs)] = np.asarray(w[3])
    return {k: v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v) for k, v in out.items()}


def main():
    import sys
    os.makedirs(GOLDEN, exist_ok=True)
    for name in (sys.argv[1:] or CASES):
        arrs = run_reference_pins() if name == 'reference_pins' else run_long_case(name) if name in LONG_CASES else run_case(name)
        path = os.path.join(GOLDEN, name + '.npz')
        np.savez_compressed(path, **arrs)
        print(name, {k: v.shape for k, v in arrs.items()}, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main()
