#!/usr/bin/env python
"""bench.py -- molecules/sec of the 1000-step denoising sampler (BASELINE.json metric) on N B200s, one process per GPU.

    python bench.py --gpus 1 --steps K --warmup W            (driver contract; N>1 is launched through torchrun)
    python bench.py --impl reference ...                      (the reference's algorithm on the host cores: CPU oracle port)

What a "step" is: one pass of the hot path -- one denoising step (k-NN graph + 9 attention layers + type head +
posterior update) over the whole in-flight batch.  Every step of the 1000-step chain costs the same (N and E = k*N do
not change along the chain), so   molecules/sec = graphs_in_flight / (1000 * seconds_per_step).
The timed K steps are consecutive steps of a real chain (Philox noise on the device), inputs resident in HBM.
Workload (default --workload cfg3 = BASELINE.json configs[2], "synthetic CrossDocked-shape batch"): 64 distinct synthetic pockets x
10 samples = 640 graphs of 300 protein + 20 ligand atoms per GPU, k=32, 9 layers.  Scaling is weak: every rank runs its own batch
(pocket-sharded, no data-path collective; NCCL only broadcasts the weights once).  Other presets: cfg1 (1 graph, 300+20), cfg2 (the
1h36 pocket of tests/golden x 100 samples with prior-sampled ligand sizes), cfg5 (64 graphs of 1200+40 atoms, k=48).
The timed region writes all four trajectories (positions, types, v0 / vt log-probabilities) like the reference's loop does;
--full-chain times one REAL 1000-step chain (t = 999 ... 0) instead of K steps x 1000.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CHAIN_STEPS = 1000
# BASELINE.json `configs` as workload presets (per GPU)
WORKLOADS = {
    'cfg1': dict(pockets=1, samples=1, n_protein=300, n_ligand=20, knn=32),
    'cfg2': dict(pockets=1, samples=100, n_protein=572, n_ligand=25, knn=32),
    'cfg3': dict(pockets=64, samples=10, n_protein=300, n_ligand=20, knn=32),
    'cfg5': dict(pockets=64, samples=1, n_protein=1200, n_ligand=40, knn=48),
}
DTYPE = 'f32 (storage, LayerNorm, softmax, accumulation); GEMM operands as 2-piece bf16 splits on tcgen05 (3 products, ~16-bit operand mantissa)'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg3', choices=sorted(WORKLOADS), help='BASELINE.json configuration preset')
    ap.add_argument('--pockets', type=int)
    ap.add_argument('--samples', type=int)
    ap.add_argument('--n-protein', type=int)
    ap.add_argument('--n-ligand', type=int)
    ap.add_argument('--knn', type=int)
    ap.add_argument('--full-chain', action='store_true', help='time one real 1000-step chain (overrides --steps)')
    ap.add_argument('--e2e-steps', type=int, default=100, help='denoising steps per end-to-end public-API call')
    ap.add_argument('--profile-steps', type=int, default=3, help='eager steps timed per kernel with CUDA events for the roofline')
    ap.add_argument('--cpu-graphs', type=str, default='1,16', help='batch sizes of the CPU arm (BASELINE.md section 3: 1 and 16)')
    ap.add_argument('--cpu-steps', type=int, default=3)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed for rank 0 as DIR/<name>.npy: pos (lab-frame ligand '
                         'positions, f32), v (atom types, f64), log_v0 / log_vt (the last v0_traj / vt_traj entry, f32); at most '
                         '64 MB in all, beyond that a fixed seeded sample of ligand atoms, their indices in rows.npy')
    a = ap.parse_args()
    for k, v in WORKLOADS[a.workload].items():
        if getattr(a, k) is None:
            setattr(a, k, v)
    if a.full_chain:
        a.steps = CHAIN_STEPS
    if not 1 <= a.steps <= CHAIN_STEPS:
        ap.error('--steps must be in 1..%d: the timed steps are consecutive steps of one chain' % CHAIN_STEPS)
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of the GPU path (--impl ours)')
    return a


def workload_name(a):
    what = 'the 1h36 pocket (tests/golden/1h36_pocket10.pdb, 572 atoms) x %d samples, prior-sampled ligand sizes' % a.samples \
        if a.workload == 'cfg2' else '%d synthetic pockets x %d samples = %d graphs x (%d protein + %d ligand atoms)' % (
            a.pockets, a.samples, a.pockets * a.samples, a.n_protein, a.n_ligand)
    return '%s: %s, k=%d, 9 layers' % (a.workload, what, a.knn)


def make_workload(a, rank):
    """Host batch of this rank in the reference's calling convention + (graphs, nodes, ligand atoms)."""
    import numpy as np
    import torch
    from oracle import synth
    G = a.pockets * a.samples
    if a.workload == 'cfg2':
        from targetdiff_b200 import atom_num
        from targetdiff_b200.pocket import pdb_to_pocket_data
        data = pdb_to_pocket_data(os.path.join(ROOT, 'tests', 'golden', '1h36_pocket10.pdb'))
        np.random.seed(2021 + rank)
        size = atom_num.get_space_size(data.protein_pos.numpy())
        sizes = [int(atom_num.sample_atom_num(size)) for _ in range(G)]
        n_p = data.protein_pos.shape[0]
        g = torch.Generator().manual_seed(2021 + rank)
        bl = torch.repeat_interleave(torch.arange(G), torch.tensor(sizes))
        b = dict(protein_pos=data.protein_pos.repeat(G, 1), protein_v=data.protein_atom_feature.float().repeat(G, 1),
                 batch_protein=torch.repeat_interleave(torch.arange(G), n_p),
                 init_ligand_pos=data.protein_pos.mean(0, keepdim=True) + torch.randn(len(bl), 3, generator=g),
                 init_ligand_v=torch.randint(0, synth.LIGAND_NUM_CLASSES, (len(bl),), generator=g), batch_ligand=bl)
        a.n_protein, a.n_ligand = n_p, round(sum(sizes) / G, 2)
    else:
        b = synth.make_batch(100 + rank, G, n_protein=a.n_protein, n_ligand=a.n_ligand, distinct_pockets=a.pockets)
    return b, G, int(b['protein_pos'].shape[0] + b['init_ligand_pos'].shape[0]), int(b['init_ligand_pos'].shape[0])


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write `arrays` (name -> host tensor with one row per ligand atom) as out_dir/<name>.npy in f32 / f64.  Above DUMP_LIMIT bytes
    in all, the same seeded sample of rows goes into every file and the sampled row indices into rows.npy."""
    import numpy as np
    import torch
    arrays = {k: v if v.is_floating_point() else v.double() for k, v in arrays.items()}      # class indices: exact in f64
    n = len(next(iter(arrays.values())))
    row_bytes = sum(v[0].numel() * v.element_size() for v in arrays.values())
    if n * row_bytes > DUMP_LIMIT:
        keep = (DUMP_LIMIT - 4096) // (row_bytes + 8)                                      # 8 bytes per index, npy headers
        rows = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        arrays = dict({k: v[rows] for k, v in arrays.items()}, rows=rows.double())
    os.makedirs(out_dir, exist_ok=True)
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), v.numpy())


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(',')])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace('.', '').isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        reasons = set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons),
                'samples': len(self.rows)}


# ------------------------------------------------------------------------------------------------- CPU arm
def _best_thread_count(sd, a, b):
    """torch-CPU throughput on these small per-edge ops collapses when oversubscribed (128 threads are ~100x slower than 16 on
    the GPU box), so the CPU arm uses the fastest of a few thread counts (one forward each) -- reported as `cores`."""
    import torch
    from oracle import restate
    ncpu = os.cpu_count() or 1
    best, best_t = 1, float('inf')
    pp, lp, _ = restate.center_pos(b['protein_pos'], b['init_ligand_pos'], b['batch_protein'], b['batch_ligand'])
    for n in sorted({min(ncpu, c) for c in (8, 16, 32, 64)}):
        torch.set_num_threads(n)
        dts = []
        for rep in range(3):          # first call after a thread-count change is a warm-up
            t0 = time.perf_counter()
            restate.forward(sd, {'knn': a.knn}, pp, b['protein_v'], b['batch_protein'], lp, b['init_ligand_v'], b['batch_ligand'])
            dts.append(time.perf_counter() - t0)
        dt = min(dts[1:])
        if dt < best_t:
            best, best_t = n, dt
        if dt > 3 * best_t:
            break
    return best


def cpu_oracle_rate(a, graphs, steps, warmup=3, cores=None):
    """The reference's algorithm on the host cores (oracle/restate.py, torch CPU) on a bounded sample of the same workload:
    `graphs` graphs of the same shape x `steps` denoising steps.  Returns (molecules/s, s/step, info)."""
    import torch
    from oracle import restate, synth
    sd = synth.make_state_dict(0, {'knn': a.knn}, schedules=restate.make_schedules())
    b = synth.make_batch(1, graphs, n_protein=a.n_protein, n_ligand=int(round(a.n_ligand)), distinct_pockets=graphs)
    if cores is None:
        cores = _best_thread_count(sd, a, b)
    torch.set_num_threads(cores)
    S = warmup + steps
    pn, vu = synth.make_tape(7, S, len(b['batch_ligand']))
    marks = []
    restate.sample_diffusion(sd, {'knn': a.knn}, b['protein_pos'], b['protein_v'], b['batch_protein'], b['init_ligand_pos'],
                             b['init_ligand_v'], b['batch_ligand'], pn, vu, num_steps=S,
                             step_callback=lambda s, i, *r: marks.append(time.perf_counter()))
    per_step = (marks[-1] - marks[warmup - 1]) / steps if warmup >= 1 else (marks[-1] - marks[0]) / max(1, steps - 1)
    rate = graphs / (CHAIN_STEPS * per_step)
    info = {'value': rate, 'unit': 'molecules/s', 'cores': cores, 'host_cpus': os.cpu_count(), 'kind': 'port',
            'sample': '%d graphs (%d+%d atoms) x %d denoising steps after %d warm-up, %.3f s/step, extrapolated x%d steps; '
                      'torch threads = fastest of {8,16,32,64}' % (graphs, a.n_protein, a.n_ligand, steps, warmup, per_step, CHAIN_STEPS)}
    return rate, per_step, info


def cpu_arm(a, steps, warmup=3):
    """CPU arm at every batch size of --cpu-graphs (BASELINE.md section 3: 1 and 16); the best rate is the reported value."""
    best = None
    runs = []
    cores = None                       # thread count chosen once, on the first (smallest) batch size
    for g in [max(1, int(x)) for x in str(a.cpu_graphs).split(',') if x.strip()]:
        # larger batches cost seconds per step on the CPU: bounded sample (the per-step cost does not depend on the step index)
        rate, per_step, info = cpu_oracle_rate(a, g, steps if g == 1 else min(steps, 5), warmup if g == 1 else 3, cores)
        cores = info['cores']
        runs.append({'graphs': g, 'molecules_per_s': rate, 's_per_step': per_step, 'cores': info['cores']})
        if best is None or rate > best[0]:
            best = (rate, per_step, info)
    rate, per_step, info = best
    info['runs'] = runs
    info['sample'] = 'best of batch sizes %s; ' % [r['graphs'] for r in runs] + info['sample']
    return rate, per_step, info


def run_reference_arm(a, rank, world):
    if rank != 0:
        return
    steps = max(1, min(a.steps, 20))
    rate, per_step, info = cpu_arm(a, steps, warmup=max(3, min(a.warmup, 5)))
    line = {'impl': 'reference', 'metric': 'molecules/sec (1000-step sampling, CrossDocked pocket shape)', 'value': rate, 'unit': 'molecules/s',
            'n_gpus': a.gpus, 'steps': a.steps, 'warmup': a.warmup, 'ms_per_step': per_step * 1e3, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': workload_name(a), 'chain_steps': CHAIN_STEPS,
                       'note': 'reference algorithm (oracle port of the PyG path, torch CPU) on the host cores; bounded sample'},
            'cpu_baseline': info, 'e2e': {'value': rate, 'unit': 'molecules/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------- GPU arm
def main():
    a = parse_args()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if a.impl == 'reference':
        run_reference_arm(a, rank, world)
        return

    import ctypes
    import torch
    import torch.distributed as dist
    from targetdiff_b200 import _lib
    from targetdiff_b200.config import default_model_config
    from targetdiff_b200.score_model import ScorePosNet3D
    from oracle import synth            # synthetic inputs only (seeded pockets / weights); not on the measured path

    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _lib.load()

    # ---- model: rank 0 builds the seeded weights, NCCL broadcast over NVLink to the other ranks (the only collective)
    cfg = default_model_config()
    cfg.knn = a.knn
    model = ScorePosNet3D(cfg, synth.PROTEIN_FEATURE_DIM, synth.LIGAND_NUM_CLASSES)
    if rank == 0:
        sd = synth.make_state_dict(0, {'knn': a.knn}, schedules={k: getattr(model, k).data for k in synth.SCHEDULE_KEYS})
        model.load_state_dict(sd, strict=True)
    model = model.to(dev)
    if world > 1:
        flat = torch.cat([p.data.view(-1) for p in model.state_dict().values()])
        dist.broadcast(flat, 0)
        off = 0
        for p in model.state_dict().values():
            p.data.copy_(flat[off:off + p.numel()].view_as(p))
            off += p.numel()
        model._drop_engine()

    # ---- synthetic batch of this rank (different pockets per rank), staged in pinned host memory
    b, G, N, Nl = make_workload(a, rank)
    host = {k: v.pin_memory() for k, v in b.items()}
    E = N * a.knn
    K = synth.LIGAND_NUM_CLASSES

    def to_dev():
        return {k: v.to(dev, non_blocking=True) for k, v in host.items()}

    d = to_dev()
    args = (d['protein_pos'], d['protein_v'], d['batch_protein'], d['init_ligand_pos'], d['init_ligand_v'], d['batch_ligand'])
    eng = model.engine(dev)
    st = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    model._bind(eng, d['protein_pos'], d['protein_v'], d['batch_protein'], d['batch_ligand'], 1)
    _lib.check(lib.tdiff_set_ligand(eng, ctypes.c_void_p(d['init_ligand_pos'].data_ptr()), ctypes.c_void_p(d['init_ligand_v'].data_ptr()), 1, st))

    # all four trajectories are written inside the timed region, like the reference's loop (models/molopt_score_model.py:687-693)
    S_traj = max(a.steps, a.warmup, a.profile_steps, 3)
    traj = (torch.empty(S_traj, Nl, 3, device=dev), torch.empty(S_traj, Nl, dtype=torch.int64, device=dev),
            torch.empty(S_traj, Nl, K, device=dev), torch.empty(S_traj, Nl, K, device=dev))
    PT = lambda t: ctypes.c_void_p(t.data_ptr())

    def chain(steps, seed):
        _lib.check(lib.tdiff_sample(eng, steps, None, None, ctypes.c_uint64(seed), PT(traj[0]), PT(traj[1]), PT(traj[2]), PT(traj[3]), 0, st))

    def reset_state():
        _lib.check(lib.tdiff_set_ligand(eng, ctypes.c_void_p(d['init_ligand_pos'].data_ptr()), ctypes.c_void_p(d['init_ligand_v'].data_ptr()), 1, st))

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- warm-up, then EXACTLY K timed denoising steps (device events, max over ranks)
    chain(max(3, a.warmup), 1)
    if a.full_chain:
        reset_state()                 # the real chain starts from the initial state at t = T - 1
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = lib.tdiff_launch_count(eng)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(torch.cuda.current_stream(dev))
    chain(a.steps, 2)
    ev1.record(torch.cuda.current_stream(dev))
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = lib.tdiff_launch_count(eng) - l0
    clocks = sampler.stop()
    if a.dump_outputs and rank == 0:    # before the profiling chain below overwrites the trajectories
        last = a.steps - 1
        dump_outputs(a.dump_outputs, {'pos': traj[0][last].cpu(), 'v': traj[1][last].cpu(), 'log_v0': traj[2][last].cpu(),
                                      'log_vt': traj[3][last].cpu()})
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    ms_per_step = ms / a.steps
    value = world * G / (CHAIN_STEPS * ms_per_step * 1e-3)

    # ---- per-kernel timing (eager launches bracketed by CUDA events on the launch stream) for the roofline
    roofline, extra = None, {}
    if rank == 0 and a.profile_steps > 0:
        _lib.check(lib.tdiff_profile(eng, 1))
        chain(a.profile_steps, 3)
        vals = [ctypes.c_double() for _ in range(4)]
        cnts = [ctypes.c_int64() for _ in range(3)]
        _lib.check(lib.tdiff_profile_read(eng, ctypes.byref(vals[0]), ctypes.byref(cnts[0]), ctypes.byref(vals[1]), ctypes.byref(cnts[1]),
                                          ctypes.byref(vals[2]), ctypes.byref(cnts[2]), ctypes.byref(vals[3])))
        _lib.check(lib.tdiff_profile(eng, 0))
        peak, peak_src = measured_peaks()
        ms_h, n_h = vals[0].value, cnts[0].value
        ms_x, n_x = vals[1].value, cnts[1].value
        ms_mlp, n_mlp = vals[2].value, cnts[2].value
        tot = vals[3].value
        mode = lib.tdiff_edge_mlp_mode(eng)
        fused = mode == 5
        if n_h:
            t_h = ms_h / n_h * 1e-3
            if fused:   # keys never reach HBM: per edge 16 logits (64 B) + v 512 + e_w 4; per node h in + out
                bytes_h, kname = E * 580 + N * 1024, 'aggregate_h_logits_kernel (scatter_softmax->scatter_sum on fused logits, x2h)'
            else:       # SURVEY.md 8(d): k 512 + v 512 + e_w 4 per edge; q, h, out per node
                bytes_h, kname = E * 1028 + N * 1536, 'aggregate_h_kernel (fused scatter_softmax->scatter_sum, x2h)'
            ach = bytes_h / t_h / 1e9
            traffic = None
            try:        # dram__bytes_read+write of one launch from the committed ncu --set full capture (profiles/, same workload)
                tj = json.load(open(os.path.join(ROOT, 'profiles', 'aggregate_traffic.json')))
                if tj.get('kernel', '').startswith(kname.split()[0]) and tj.get('graphs') == G:
                    traffic = tj['dram_bytes_per_launch']
            except Exception:
                pass
            roofline = {'kernel': kname, 'bound': 'hbm', 'achieved': ach,
                        'peak': peak, 'unit': 'GB/s', 'frac': ach / peak, 'traffic': traffic, 'peak_source': peak_src,
                        'algorithmic_bytes_per_launch': bytes_h, 'avg_launch_ms': t_h * 1e3, 'launches_timed': n_h,
                        'share_of_step': ms_h / tot if tot else None}
        if n_x:
            El = Nl * a.knn
            bytes_x = El * (148 if fused else 596) + Nl * (25 if fused else 537)
            t_x = ms_x / n_x * 1e-3
            extra['roofline_aggregate_x'] = {'kernel': 'aggregate_x_kernel (h2x, ligand destinations only)', 'bound': 'hbm',
                                             'achieved': bytes_x / t_x / 1e9, 'peak': peak, 'unit': 'GB/s', 'frac': bytes_x / t_x / 1e9 / peak,
                                             'avg_launch_ms': t_x * 1e3, 'share_of_step': ms_x / tot if tot else None}
        if n_mlp:
            # tensor-core work actually executed by the edge MLPs of one layer (x2h: hk + hv on all E rows; h2x: xk + xv on ligand
            # destinations): per row 3 bf16 products x (128 x NOUT second Linear + 32 x 128 gaussian block) MAC on tcgen05
            El = Nl * a.knn
            # (v4: the gaussian/type block of both edge types of a destination class is one K = 64 MMA: 2 x 21 useful slots of 64)
            kpre = 64 if fused else 0
            mac_row = lambda nout: 3 * (128 * nout + kpre * 128)
            flops = 2.0 * (E * 2 * mac_row(128) + El * (mac_row(128) + mac_row(16)))
            useful = 2.0 * (E * 2 * 3 * (128 * 128 + 21 * 128) + El * 3 * (128 * 128 + 21 * 128 + 128 * 16 + 21 * 128))
            t_m = ms_mlp / (n_mlp / 2) * 1e-3                       # per layer (x2h pair + h2x pair, incl. the slow-row pre-passes)
            tpeak = None
            try:
                tpeak = float(json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['bf16_tflops_sustained'])
                tsrc = 'measured (MEASURED_PEAKS.json bf16_tflops_sustained: kernel timed inside a long step)'
            except Exception:
                tpeak, tsrc = 1400.0, 'fallback (B200_PROFILING.md sustained 1.4 PFLOP/s)'
            ach = flops / t_m / 1e12
            # DRAM bytes of one value-MLP (+ aggregation) launch: not measurable inside this run (needs ncu); taken from this round's
            # committed `ncu --set full` capture of the same workload when there is one, else null
            mlp_traffic, traffic_src = None, None
            try:
                tj = json.load(open(os.path.join(ROOT, 'profiles', 'r02_edge_mlp_traffic.json')))
                if tj.get('graphs') == G and tj.get('workload') == a.workload:
                    mlp_traffic, traffic_src = tj['dram_bytes_per_launch'], 'profiles/r02_edge_mlp_traffic.json (ncu --set full, value launch)'
            except Exception:
                pass
            extra['edge_mlp'] = {'kernel': 'edge_mlp_v4_kernel x4 per layer (engine mode %d)' % mode, 'bound': 'tensor', 'achieved': ach, 'peak': tpeak,
                                 'unit': 'TFLOP/s', 'frac': ach / tpeak, 'traffic': mlp_traffic, 'traffic_source': traffic_src, 'peak_source': tsrc,
                                 'executed_flops_per_layer': flops, 'useful_flops_per_layer': useful, 'frac_useful': useful / t_m / 1e12 / tpeak,
                                 'ms_per_layer': t_m * 1e3, 'share_of_step': ms_mlp / tot if tot else None,
                                 'note': 'executed flops = every issued tcgen05 MMA (3 bf16 products per fp32-class product, K = 64 gaussian block '
                                         'incl. its zero padding); useful = the same without padding slots; the kernel is bound by its '
                                         'CUDA-core LayerNorm/split stage, see DESIGN.md section 6'}
            if roofline is None:            # aggregation fused into the value-MLP epilogue: the dominant kernel is the edge MLP itself
                roofline = dict(extra['edge_mlp'])
        extra['profile_ms_per_step_eager'] = tot / a.profile_steps if tot else None
        # canonical (unfused) attention aggregation on the same problem size through the stand-alone C-ABI operator: keys AND values
        # in HBM, algorithmic bytes E*1028 + N*1536 (SURVEY.md 8(d)); timed with CUDA events on the launch stream
        try:
            kk = a.knn
            gk = torch.randn(E, 128, device=dev)
            gv = torch.randn(E, 128, device=dev)
            gw = torch.rand(E, device=dev)
            gs = torch.randint(0, N, (N, kk), device=dev, dtype=torch.int32)
            gq = torch.randn(N, 128, device=dev)
            gh = torch.randn(N, 128, device=dev)
            go = torch.empty_like(gh)
            P_ = lambda t: ctypes.c_void_p(t.data_ptr())
            def agg():
                _lib.check(lib.tdiff_attn_aggregate_h(P_(gk), P_(gv), P_(gw), P_(gs), P_(gq), P_(gh), P_(go), N, kk, st))
            for _ in range(3):
                agg()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record(torch.cuda.current_stream(dev))
            reps = 10
            for _ in range(reps):
                agg()
            e1.record(torch.cuda.current_stream(dev))
            torch.cuda.synchronize(dev)
            t_u = e0.elapsed_time(e1) / reps * 1e-3
            bytes_u = E * 1028 + N * 1536
            traffic_u = None             # DRAM bytes of one launch from this round's committed ncu capture of the same problem size
            try:
                tj = json.load(open(os.path.join(ROOT, 'profiles', 'r02_aggregate_h_traffic.json')))
                if tj.get('nodes') == N and tj.get('k') == kk:
                    traffic_u = tj['dram_bytes_per_launch']
            except Exception:
                pass
            extra['roofline_unfused_aggregate'] = {'kernel': 'aggregate_h_kernel (tdiff_attn_aggregate_h: keys + values from HBM)', 'bound': 'hbm',
                                                   'achieved': bytes_u / t_u / 1e9, 'peak': peak, 'unit': 'GB/s', 'frac': bytes_u / t_u / 1e9 / peak,
                                                   'traffic': traffic_u,
                                                   'algorithmic_bytes_per_launch': bytes_u, 'avg_launch_ms': t_u * 1e3,
                                                   'note': 'stand-alone operator on random data of the bench problem size; the engine itself fuses the '
                                                           'logits into the key-MLP epilogue (roofline above)'}
            del gk, gv, gw, gs, gq, gh, go
        except Exception as ex:      # never fail the bench line because of the auxiliary measurement
            extra['roofline_unfused_aggregate'] = {'error': str(ex)[:200]}

    # ---- end to end through the public API with HOST buffers (H2D of the inputs, the chain, D2H of results + trajectories)
    e2e = None
    if not a.no_e2e:
        S = CHAIN_STEPS if a.full_chain else max(3, a.e2e_steps)
        h2d = sum(v.numel() * v.element_size() for v in host.values())
        d2h = Nl * 12 + Nl * 8 + S * Nl * (12 + 8 + 2 * K * 4)
        reps = 1 if a.full_chain else 2

        def one_call(seed):
            dd = to_dev()
            r = model.sample_diffusion(dd['protein_pos'], dd['protein_v'], dd['batch_protein'], dd['init_ligand_pos'], dd['init_ligand_v'],
                                       dd['batch_ligand'], num_steps=S, center_pos_mode='protein', seed=seed, stack_traj=True)
            return r['pos'].cpu(), r['v'].cpu()

        if not a.full_chain:
            one_call(11)
        barrier()
        t0 = time.perf_counter()
        for i in range(reps):
            one_call(12 + i)
        torch.cuda.synchronize(dev)
        t_call = (time.perf_counter() - t0) / reps
        if world > 1:
            t = torch.tensor([t_call], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            t_call = float(t.item())
        e2e = {'value': world * G / (CHAIN_STEPS * (t_call / S)), 'unit': 'molecules/s', 'h2d_bytes_per_step': h2d / S,
               'd2h_bytes_per_step': d2h / S,
               'note': 'ScorePosNet3D.sample_diffusion(num_steps=%d) per call from pinned host tensors incl. batch binding, H2D, chain, '
                       'D2H of final state and all four trajectories; per-step cost x1000 (a real 1000-step call amortises the copies '
                       '%dx better)' % (S, CHAIN_STEPS // S)}

    # ---- CPU baseline (rank 0, N=1 only; bounded sample)
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        _, _, cpu = cpu_arm(a, a.cpu_steps)

    if rank == 0:
        line = {'metric': 'molecules/sec (1000-step sampling, CrossDocked pocket shape)', 'value': value, 'unit': 'molecules/s', 'n_gpus': world,
                'steps': a.steps, 'warmup': max(3, a.warmup), 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': DTYPE, 'data': 'synthetic',
                'config': {'workload': workload_name(a), 'graphs_per_gpu': G, 'nodes': N, 'edges': E, 'chain_steps': CHAIN_STEPS,
                           'step': ('one REAL 1000-step chain (t = 999 ... 0) timed in full' if a.full_chain else
                                    'one denoising step of the whole in-flight batch; value = graphs / (1000 * s_per_step)') +
                                   '; all four trajectories written inside the timed region',
                           'parallelism': 'pocket-sharded x%d (no data-path collective)' % world,
                           'l2': 'per-step working set (k,v edge tensors %.1f GB) >> 126 MB L2; no explicit flush' % (2 * E * 512 / 1e9),
                           'noise': 'device Philox4x32-10'},
                'clocks': clocks, 'gpu_launches': int(launches), 'e2e': e2e, 'roofline': roofline, 'cpu_baseline': cpu}
        line.update(extra)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
