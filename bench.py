#!/usr/bin/env python
"""Benchmark of the diffusion-sampling hot path (BASELINE.json metric: ligands/sec sampled,
1000-step denoise, batch 64 pockets of ~300 protein + 24 ligand atoms per GPU).

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA path)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port)
    torchrun --nproc-per-node N ... bench.py --gpus N ...    # N > 1: one rank per GPU, weak scaling

A "step" is ONE denoise step of the whole batch: ligand embedding -> device kNN -> edge gate ->
9 x (node GEMMs, fused X2H, fused H2X) -> classifier -> reverse diffusion step (+ the two torch
RNG draws).  value = ligands/s = (64 x N) / (T x seconds per step), T = 1000.
Timing: W >= 3 warm-up steps, then K steps each bracketed by CUDA events on the launching
stream with an L2 flush (256 MiB write) between timed steps, barrier + synchronize around the
region, max over ranks.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

T_STEPS = 1000
WORKLOADS = {
    # name: (graphs per GPU, protein atoms, ligand atoms, gen_mode, encoder overrides, description)
    'c2': (64, 300, 24, 'denovo', {}, 'de novo denoise, batch 64 pockets x (300 protein + 24 ligand atoms), 1000 steps, fp32'),
    'c3': (128, 300, 24, 'partial', {'cutoff_mode': 'radius', 'r_max': 10.0},
           'linker task, batch 128, radius graph r=10 A (cap 32), 1000 steps'),
    'c1': (1, 200, 24, 'denovo', {}, 'de novo, 1 pocket 200+24 atoms (plumbing case)'),
    # ragged pockets 100..800 protein atoms (mean 450), 24 ligand atoms, context fixed: 32 pockets per GPU (256 over 8)
    'c5': (32, None, 24, 'partial', {}, 'scaffold task, ragged pockets 100-800 atoms, 32 pockets per GPU (256 over 8 GPUs)'),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference', 'reference-gpu'])
    ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS))
    ap.add_argument('--e2e-steps', type=int, default=T_STEPS, help='denoise steps of the end-to-end sample() call')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--profile-steps', type=int, default=3)
    ap.add_argument('--scaling', default=None, choices=['weak', 'strong'],
                    help="weak: every rank gets the workload's pockets (default for c2/c3/c1); strong: ONE global batch is "
                         'partitioned over the ranks by atom count (default for c5: 256 ragged pockets over the box)')
    ap.add_argument('--global-graphs', type=int, default=None, help='pockets of the global batch for --scaling strong')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the ligand state the last timed step computed (coordinates x_lig '
                         '[n_lig, 3] and atom-type one-hots c_lig [n_lig, K], float32) as DIR/<name>.npy; the inputs are '
                         'seeded, so two builds run with the same arguments can be compared output for output')
    return ap.parse_args()


def dump_outputs(out_dir, arrays, rank, world):
    """Write each device tensor as out_dir/<name>.npy (float32); with several ranks every rank writes <name>.rank<r>.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    suffix = '' if world == 1 else f'.rank{rank}'
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f'{name}{suffix}.npy'), t.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU every 100 ms (NVML) while running."""
    REASONS = {0x4: 'sw_power_cap', 0x8: 'hw_slowdown', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown',
               0x80: 'hw_power_brake_slowdown', 0x2: 'applications_clocks_setting', 0x10: 'sync_boost'}

    def __init__(self, torch_index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self.nv = pynvml
            try:
                uuid = str(torch.cuda.get_device_properties(torch_index).uuid)
                self.h = pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + uuid).encode() if not uuid.startswith('GPU-') else uuid.encode())
            except Exception:
                vis = os.environ.get('CUDA_VISIBLE_DEVICES')
                idx = int(vis.split(',')[torch_index]) if vis and vis.split(',')[torch_index].isdigit() else torch_index
                self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:   # NVML missing: report nulls rather than fail the bench
            self.nv, self.err = None, repr(e)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                fn = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                mask = int(fn(self.h))
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._loop, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr is not None:
            self._thr.join()

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons), 'samples': 0}
        return {'sm_mhz': statistics.median(self.samples), 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons), 'samples': len(self.samples)}


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), 'measured'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0}, 'fallback'


def workload_batch(name, rank, n_graphs=None):
    from cbgbench_b200 import synthetic
    import numpy as np
    B, n_prot, n_lig, gen_mode, enc, _ = WORKLOADS[name]
    B = n_graphs or B
    if n_prot is None:
        sizes = [int(v) for v in np.random.RandomState(77 + rank).randint(100, 801, size=B)]
    else:
        sizes = [n_prot] * B
    return synthetic.make_batch(sizes, [n_lig] * B, seed=2024 + rank, gen_mode=gen_mode), enc


# ---------------------------------------------------------------------------------------------
# Reference legs.  What is timed is the UNMODIFIED reference: TargetDiff.sample(batch) (repo/models/diffusion/
# targetdiff.py:127-184) imported from baseline/_ref (staged copy of /root/reference, see baseline/ref_runner.py) with the
# bench's seeded weights, on the FULL batch of the workload.  One sample() call with T = n steps is n denoise steps.
def reference_enc(workload):
    """Encoder overrides the reference can run: its radius branch is dead code (unitransformer.py:76-77), so the c3
    workload falls back to the kNN graph there (said in the line)."""
    enc = dict(WORKLOADS[workload][4])
    note = None
    if enc.get('cutoff_mode') == 'radius':
        enc, note = {}, "reference cannot build a radius graph (dead code upstream): timed with its kNN graph"
    return enc, note


def cpu_thread_candidates():
    ncpu = os.cpu_count() or 1
    cands = []
    for c in (min(64, ncpu), 32, 16, ncpu):
        if c <= ncpu and c not in cands:
            cands.append(c)
    return cands


def reference_cpu_probe(workload, max_probe_s=240.0):
    """Pick the torch thread count on the REAL batch: one 2-step sample() call per candidate (these calls are the
    warm-up of the reference arm).  Returns (threads, {threads: s/step}, steps_run)."""
    from baseline import ref_runner
    batch, _ = workload_batch(workload, 0)
    enc, _ = reference_enc(workload)
    tried, t0, steps_run = {}, time.perf_counter(), 0
    for c in cpu_thread_candidates():
        if tried and time.perf_counter() - t0 > max_probe_s:
            break
        sec, _ = ref_runner.time_sample(batch, enc, 2, 'cpu', threads=c)
        tried[c] = sec / 2
        steps_run += 2
    return min(tried, key=tried.get), {k: round(v, 3) for k, v in tried.items()}, steps_run


def run_reference(args):
    """--impl reference / reference-gpu: the reference's own implementation of the path on this box (host cores, or
    eager PyTorch on one GPU), same metric and config, rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    from baseline import ref_runner
    if ref_runner.ref_root() is None:
        print(json.dumps({'impl': args.impl, 'unavailable': 'baseline/_ref missing and /root/reference absent'}), flush=True)
        return
    B, n_prot, n_lig, _, _, desc = WORKLOADS[args.workload]
    enc, note = reference_enc(args.workload)
    batch, _ = workload_batch(args.workload, 0)
    gpu = args.impl == 'reference-gpu'
    if gpu:
        dev = 'cuda:%d' % int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(dev)
        warm_steps = max(2, args.warmup)
        ref_runner.time_sample(batch, enc, warm_steps, dev)                      # warm-up call (allocator, kernels)
        sec, _ = ref_runner.time_sample(batch, enc, max(2, args.steps), dev)
        threads, tried = torch.get_num_threads(), None
        kind = 'reference eager PyTorch on one GPU (unmodified TargetDiff.sample, torch-op shims for pyg/scatter)'
    else:
        threads, tried, warm_steps = reference_cpu_probe(args.workload)
        while warm_steps < args.warmup:                                         # top up to the requested warm-up
            ref_runner.time_sample(batch, enc, 2, 'cpu', threads=threads)
            warm_steps += 2
        sec, _ = ref_runner.time_sample(batch, enc, max(2, args.steps), 'cpu', threads=threads)
        kind = 'reference CPU path (unmodified TargetDiff.sample, torch CPU fp32)'
    n_timed = max(2, args.steps)
    sec_step = sec / n_timed
    value = B / (T_STEPS * sec_step)
    sample = (f'all {B} pockets ({n_prot}+{n_lig} atoms each): one TargetDiff.sample() call of {n_timed} denoise steps after '
              f'{warm_steps} warm-up steps; ligands/s = pockets / (1000 x s/step)')
    if not gpu:
        sample += f'; {threads} torch threads of {os.cpu_count()} host cores (s/step on the full batch per thread count: {tried})'
    line = {
        'impl': args.impl, 'metric': 'ligands/sec sampled (1000-step denoise, batch 64)', 'value': value,
        'unit': 'ligands/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': sec_step * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': {'workload': f'{args.workload}: {desc}', 'graphs_per_gpu': B, 'graphs_timed': B, 'kind': kind,
                   'denoise_steps_per_ligand': T_STEPS, 'step': 'one denoise step of the whole batch', 'note': note},
        'cpu_baseline': {'value': value, 'unit': 'ligands/s', 'cores': threads, 'kind': 'reference', 'sample': sample},
        'e2e': {'value': value, 'unit': 'ligands/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    if gpu:
        line['cpu_baseline'] = None
        line['config']['device'] = torch.cuda.get_device_name()
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    from cbgbench_b200 import _lib, synthetic
    from cbgbench_b200.targetdiff import TargetDiffB200

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torchrun)'
    if args.warmup < 3:
        raise SystemExit('--warmup must be >= 3')
    if args.steps < 1:
        raise SystemExit('--steps must be >= 1')
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    torch.set_grad_enabled(False)
    L = _lib.lib()

    B, n_prot, n_lig, gen_mode, enc, desc = WORKLOADS[args.workload]
    scaling = args.scaling or ('strong' if args.workload == 'c5' else 'weak')
    shard = None
    if scaling == 'strong':
        # ONE global batch, identical on every rank (same seed), partitioned by atom count (LPT, cbgbench_b200/sharding.py);
        # every rank samples its share with no communication, the final states meet in one all-gather
        from cbgbench_b200 import sharding
        total = args.global_graphs or (256 if args.workload == 'c5' else B)
        full, _ = workload_batch(args.workload, 0, total)
        sizes = sharding.graph_sizes(full).tolist()
        parts = sharding.assign_graphs(sizes, world)
        batch = sharding.take_graphs(full, parts[rank])
        lig_per_graph = torch.bincount(full['ligand_element_batch'], minlength=total)
        shard = {'parts': parts, 'counts': [int(lig_per_graph[torch.as_tensor(p_, dtype=torch.long)].sum()) for p_ in parts],
                 'atoms': [int(sum(sizes[g] for g in p_)) for p_ in parts], 'total_graphs': total}
        B_total, B = total, len(parts[rank])
    else:
        batch, _ = workload_batch(args.workload, rank)
        B_total = B * world
    model = TargetDiffB200(synthetic.targetdiff_config(num_steps=T_STEPS, **enc))
    model.load_state_dict(synthetic.seeded_state_dict(model, seed=0), strict=True)
    model = model.to(dev).eval()
    torch.manual_seed(2024 + rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident steps (inputs already in HBM) ------------------------------------------
    state = model.prepare(batch)
    n_lig_tot, K = state['n_lig'], model.num_classes
    N = state['n_nodes']
    need = args.warmup + args.steps + args.profile_steps
    assert need < T_STEPS
    X = torch.empty((T_STEPS + 1, n_lig_tot, 3), device=dev)
    Cc = torch.empty((T_STEPS + 1, n_lig_tot, K), device=dev)
    X[T_STEPS].copy_(state['x_lig'])
    Cc[T_STEPS].copy_(state['c_lig'])
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2
    t_seq = list(reversed(range(T_STEPS)))
    model.run_steps(state, t_seq[:args.warmup], X, Cc)
    barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    launches0 = L.cbg_launch_count()
    with ClockSampler(local_rank) as clocks:
        for i in range(args.steps):
            flush.zero_()                                  # L2 flush between timed steps (outside the events)
            starts[i].record()
            model.run_steps(state, [t_seq[args.warmup + i]], X, Cc)
            ends[i].record()
        barrier()
    gpu_launches = L.cbg_launch_count() - launches0
    if args.dump_outputs:
        t_out = t_seq[args.warmup + args.steps - 1]        # slot t of X / Cc holds the result of step t
        dump_outputs(args.dump_outputs, {'x_lig': X[t_out], 'c_lig': Cc[t_out]}, rank, world)
    step_ms = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    ms_per_step = sum(step_ms) / len(step_ms)
    t = torch.tensor([ms_per_step], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_per_step = float(t.item())
    ms_rank = sum(step_ms) / len(step_ms)
    value = B_total / (T_STEPS * ms_per_step * 1e-3)

    # ---- per-kernel CUDA-event profile of a few more steps (roofline of the dominant kernel) ------
    prof = None
    if args.profile_steps > 0:
        L.cbg_profile_enable(1)
        p0 = args.warmup + args.steps
        model.run_steps(state, t_seq[p0:p0 + args.profile_steps], X, Cc)
        prof = _lib.profile_collect()
        L.cbg_profile_enable(0)
    peaks, peak_kind = measured_peaks()
    roofline, kernels = None, None
    if prof:
        kernels = {k: {'ms_per_step': v[0] / args.profile_steps, 'launches_per_step': v[1] / args.profile_steps}
                   for k, v in prof.items() if v[1]}
        dom = max(('x2h_k', 'x2h_v'), key=lambda k: prof[k][0])
        dom_ms = prof[dom][0] / prof[dom][1]
        # rows one launch processes: with receptive-field pruning layer l only updates the nodes that can still reach a
        # sampled atom, so the per-launch average over the layers is what the measured launch time corresponds to
        n_layers = state['plan'].num_layers
        rows = float(N)
        if model.use_prune:
            import ctypes
            cnt = (ctypes.c_int32 * (n_layers + 1))()
            _lib.check(L.cbg_sample_prune_counts_host(ctypes.byref(state['plan']), cnt, _lib.stream_ptr(dev)))
            rows = sum(cnt[l + 1] for l in range(n_layers)) / n_layers
            rows_src = sum(cnt[l] for l in range(n_layers)) / n_layers          # rows whose Pj plane a launch may gather
        else:
            rows_src = rows
        traffic, ncu_info = None, None
        tpath = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')      # dram bytes/launch from the last ncu --set full capture
        if os.path.exists(tpath):
            with open(tpath) as f:
                rec = json.load(f).get(dom + '_tc') or {}
            traffic = rec.get('dram_bytes_per_launch')
            ncu_info = rec.get('ncu')
        # The fused X2H kernels (csrc/x2h_tc.cu) are TENSOR-bound, not HBM-bound (DESIGN.md section 5): per 128-edge tile
        # they issue 17 + 48 tcgen05 MMAs, nothing of size [E, 128] crosses HBM.
        #   executed tensor FLOPs per tile = 17 x (128 x 128 x 16 x 2) + 48 x (128 x 64 x 16 x 2); the (hi, lo) f16 split
        #   runs three f16 products per fp32 product and pads K = 84 to 96
        #   algorithmic (fp32-equivalent) FLOPs per edge and kernel = (84 + 128) x 128 x 2   (first-Linear RBF part + second Linear)
        #   algorithmic HBM bytes per launch: node planes read once + per-row neighbour / gate / coordinate rows + w / h
        tiles = rows / 4.0
        exec_flops = tiles * (17 * 128 * 128 * 16 * 2 + 48 * 128 * 64 * 16 * 2)
        alg_flops = rows * 32 * (84 + 128) * 128 * 2
        per_row = {'x2h_k': 512 + 512 + 128 + 128 + 16 + 2048, 'x2h_v': 512 + 128 + 16 + 2048 + 1024}[dom]
        alg_bytes = per_row * rows + 512 * rows_src
        tf_peak = peaks.get('bf16_tflops_sustained') or peaks.get('bf16_tflops')
        ach_exec = exec_flops / (dom_ms * 1e-3) / 1e12
        ach_alg = alg_flops / (dom_ms * 1e-3) / 1e12
        hbm = alg_bytes / (dom_ms * 1e-3) / 1e9
        roofline = {'kernel': dom + ' (x2h_tc_kernel)', 'bound': 'tensor', 'achieved': ach_alg, 'peak': tf_peak / 3.0, 'unit': 'TFLOP/s',
                    'frac': ach_alg / (tf_peak / 3.0), 'traffic': traffic,
                    'peak_source': f'{peak_kind} bf16 cuBLAS TFLOP/s sustained (MEASURED_PEAKS.json: {tf_peak}) / 3: the fp32-accurate '
                                   '(hi, lo) f16 split needs three tensor-core products per algorithmic product',
                    'algorithmic_flops_per_launch': alg_flops, 'launch_ms': dom_ms, 'rows_per_launch': rows,
                    'executed': {'tflops': ach_exec, 'peak_tflops': tf_peak, 'frac': ach_exec / tf_peak,
                                 'note': 'tcgen05 FLOPs actually issued (3 products, K padded 84 -> 96)'},
                    'hbm': {'algorithmic_bytes_per_launch': alg_bytes, 'achieved_gbs': hbm, 'peak_gbs': peaks['hbm_gbs'],
                            'frac': hbm / peaks['hbm_gbs'],
                            'note': "the north-star's 60 % HBM target assumed per-edge k/v tensors crossing HBM (9.9 GB/step); they are "
                                    'never materialised, the kernel moves ~4 KB per node and is bounded on the compute side'},
                    # what shares the SM with the tensor pipe (DESIGN.md section 5.2): LSU wavefronts of the last ncu capture of
                    # this kernel (unpruned launch, 5184 tiles) and the B-operand bytes the 41 MMAs of a tile read from shared memory
                    'shared_memory': {'ncu_capture': ncu_info, 'mma_b_operand_bytes_per_tile': 41 * 128 * 16 * 2,
                                      'note': 'static evidence from profiles/ncu_traffic.json (ncu --set full), not measured in this run'}}

    # ---- end to end through the public API: host batch -> model.sample() -> host trajectory -------
    e2e = None
    if not args.no_e2e:
        host_batch = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in batch.items()}
        h2d = sum(v.numel() * v.element_size() for v in host_batch.values() if torch.is_tensor(v))
        steps_e2e = min(args.e2e_steps, T_STEPS)
        # warm-up of the public-API path (allocations, R-cache buffers, NCCL channels of the final gather)
        model.sample(host_batch, num_steps=2, traj_mode='final')
        if world > 1:
            from cbgbench_b200 import sharding
            gid_map = (torch.as_tensor(shard['parts'][rank], dtype=torch.long) if shard else torch.arange(B) + rank * B).to(dev)
            counts = shard['counts'] if shard else [n_lig_tot] * world
            gid0 = gid_map[batch['ligand_element_batch'].to(dev)]
            sharding.gather_final(torch.zeros(n_lig_tot, 3, device=dev), torch.zeros(n_lig_tot, dtype=torch.int64, device=dev),
                                  gid0, counts=counts)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        traj = model.sample(host_batch, num_steps=steps_e2e)          # H2D + steps + D2H of the trajectory
        t_last = T_STEPS - steps_e2e
        if world > 1:                                                  # the single gather of final coordinates, device to device:
            xd, cd, _ = traj[t_last - 1]                               # the state after the last step is still on the GPU (traj[-1] at full T)
            sharding.gather_final(xd, cd.argmax(-1), gid0, counts=counts)
        ev1.record()
        barrier()
        e2e_ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
        d2h = sum(traj[t][0].numel() * 4 + traj[t][1].numel() * 4 for t in traj if t >= 0)
        e2e_value = B_total / (float(e2e_ms.item()) * 1e-3) * (steps_e2e / T_STEPS)
        e2e = {'value': e2e_value, 'unit': 'ligands/s', 'h2d_bytes_per_step': h2d / steps_e2e,
               'd2h_bytes_per_step': d2h / steps_e2e, 'seconds': float(e2e_ms.item()) * 1e-3, 'denoise_steps': steps_e2e,
               'api': 'TargetDiffB200.sample(host batch) -> traj (CPU), H2D/D2H and final gather inside the timed region'}

    # ---- the reference beside it (rank 0, N = 1): its CPU path on the host cores (bounded sample: one 2-step
    # sample() call on the full batch) and its eager-PyTorch path on this GPU (the same-box GPU comparator)
    cpu, ref_gpu = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from baseline import ref_runner
        if ref_runner.ref_root() is not None:
            enc_r, note_r = reference_enc(args.workload)
            threads = min(64, os.cpu_count() or 1)
            sec, _ = ref_runner.time_sample(batch, enc_r, 2, 'cpu', threads=threads)
            cpu = {'value': B / (T_STEPS * sec / 2), 'unit': 'ligands/s', 'cores': threads, 'kind': 'reference',
                   'sample': f'all {B} pockets, one unmodified TargetDiff.sample() call of 2 denoise steps (no warm-up), torch CPU '
                             f'fp32, {threads} threads of {os.cpu_count()} host cores; extrapolated: pockets / (1000 x s/step); '
                             f'the --impl reference arm times more steps and picks the thread count on the full batch'}
            try:
                ref_runner.time_sample(batch, enc_r, 2, str(dev))
                n_ref = 5
                sec_g, _ = ref_runner.time_sample(batch, enc_r, n_ref, str(dev))
                ref_gpu = {'ms_per_step': sec_g / n_ref * 1e3, 'value': B / (T_STEPS * sec_g / n_ref), 'unit': 'ligands/s',
                           'kind': 'reference eager PyTorch on this GPU (unmodified TargetDiff.sample, torch-op shims for '
                                   'pyg/scatter), one call of %d steps after a 2-step warm-up call' % n_ref, 'note': note_r}
            except Exception as e:     # the comparator must never take the bench line down
                ref_gpu = {'unavailable': repr(e)[:200]}
            torch.set_grad_enabled(False)

    ranks = None
    if world > 1:
        mine = {'rank': rank, 'graphs': B, 'nodes': int(N), 'ms_per_step': ms_rank}
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        ranks = allr
        slow = max(allr, key=lambda r_: r_['ms_per_step'])
        ranks_summary = {'per_rank': allr, 'limiting_rank': slow['rank'],
                         'imbalance': slow['ms_per_step'] / (sum(r_['ms_per_step'] for r_ in allr) / world)}
    if rank == 0:
        line = {
            'metric': 'ligands/sec sampled (1000-step denoise, batch 64)', 'value': value, 'unit': 'ligands/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step,
            'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': f'{args.workload}: {desc}', 'graphs_per_gpu': B, 'graphs_total': B_total, 'nodes_per_gpu': N,
                       'denoise_steps_per_ligand': T_STEPS, 'step': 'one denoise step of the whole batch',
                       'l2': 'flushed (256 MiB write) between timed steps', 'parallelism': f'dp{world} (pockets sharded, no data-path collective)'},
            'clocks': clocks.summary(), 'gpu_launches': int(gpu_launches), 'e2e': e2e, 'roofline': roofline,
            'cpu_baseline': cpu, 'reference_gpu': ref_gpu, 'kernels': kernels,
        }
        if ranks is not None:
            line['ranks'] = ranks_summary
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl in ('reference', 'reference-gpu'):
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
