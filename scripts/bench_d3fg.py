#!/usr/bin/env python
"""Measurement of the D3FG sampler (DESIGN.md section 13): one JSON line.

Workload: the shipped width (hidden 256, 9 IPA layers, 28 FG types, T = 1000 schedule) at 64 pockets x (100 residues +
8 functional groups), synthetic data and seeded weights.  The pocket shape is an assumption, not taken from data.
Method as scripts/bench_f2.py: warm-up steps, then K timed reverse steps each bracketed by CUDA events with a 256 MiB L2
flush in between, the launch counter, and a per-kernel-family breakdown over a few extra steps.  The eager-torch oracle
(oracle/diffusion_fg.py) is timed the same way on the same GPU and batch, and one step of both from the same state and
draws is compared.  The card's name and power limit come from a read-only nvidia-smi query in the same run.
Building the T = 1000 histograms takes about a minute of CPU time before anything is timed.

    python scripts/bench_d3fg.py [--steps 20] [--warmup 3] [--oracle-steps 3]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

T, B, N_RES, N_FG, K = 1000, 64, 100, 8, 28


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        name, power = [s.strip() for s in out.split(',')[:2]]
        return {'gpu': name, 'power_limit': power}
    except Exception as e:          # the measurement stands without it; say so
        return {'gpu': 'not measured', 'power_limit': 'not measured', 'query_error': str(e)}


def timed(fn, steps, flush):
    import torch
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    for i in range(steps):
        flush.zero_()
        starts[i].record()
        fn(i)
        ends[i].record()
    torch.cuda.synchronize()
    return sum(s.elapsed_time(e) for s, e in zip(starts, ends)) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--oracle-steps', type=int, default=3)
    args = ap.parse_args()
    import torch
    from cbgbench_b200 import _lib, synthetic as S
    from cbgbench_b200.difffg import D3FGB200
    from oracle import diffusion_fg as OF
    from oracle.diffusion import type_reverse_step
    from oracle.diffusion_bp import pos_reverse_step_score
    torch.set_grad_enabled(False)
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    L = _lib.lib()
    model = D3FGB200(S.d3fg_config(num_steps=T))
    sd = S.seeded_state_dict(model, seed=0, skip_prefixes=S.D3FG_SKIP)
    model.load_state_dict(sd, strict=True)
    model = model.to(dev).eval()
    batch = S.make_fg_batch([N_RES] * B, [N_FG] * B, seed=2024)
    n = B * N_FG
    state = model.prepare(batch)
    buf = torch.empty((T + 1, n * (6 + K)), device=dev)
    split = lambda r: (r[:3 * n].view(n, 3), r[6 * n:].view(n, K), r[3 * n:6 * n].view(n, 3))
    x0, c0, o0 = split(buf[T])
    x0.copy_(state['x_lig'])
    c0.copy_(state['c_lig'])
    o0.copy_(state['o_lig'])
    slots = lambda t: split(buf[t])
    t_seq = list(reversed(range(T)))
    torch.manual_seed(2024)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    model.run_steps(state, t_seq[:args.warmup], slots)
    torch.cuda.synchronize()
    l0 = L.cbg_launch_count()
    ms = timed(lambda i: model.run_steps(state, [t_seq[args.warmup + i]], slots), args.steps, flush)
    launches = (L.cbg_launch_count() - l0) / args.steps
    L.cbg_profile_enable(1)
    nprof = 3
    done = args.warmup + args.steps
    model.run_steps(state, t_seq[done:done + nprof], slots)
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    L.cbg_profile_enable(0)
    kern = {k: round(v[0] / nprof, 4) for k, v in prof.items() if v[0] > 0}

    # eager-torch oracle on the same GPU and batch, and one step of both from the same state and draws.  The oracle's
    # kNN (oracle/graph_ops.py) builds its neighbour table on the CPU; its edge list is moved to the GPU here.
    from oracle import graph_ops as G
    to_edges = G.table_to_edge_index
    G.table_to_edge_index = lambda nbr: to_edges(nbr).to(dev)
    sd_d = {k: v.to(dev) for k, v in model.state_dict().items()}
    bd = {k: v.to(dev) for k, v in batch.items()}
    cdf = state['keep']['cdf']
    t = t_seq[done + nprof]
    x_t, c_t, o_t = (a.clone() for a in slots(t + 1))
    pn, rn, tu = S.make_d3fg_noise(1, n, K, seed=3)
    pn, tu = pn.to(dev), tu.to(dev)
    rn = {k: v.to(dev) for k, v in rn.items()}
    gen = bd['ligand_lig_flag']

    def oracle_step(_):
        eps, o_pred, logits = OF.denoise(sd_d, bd, x_t, c_t, o_t, K)
        x_n = pos_reverse_step_score(sd_d, eps, x_t, t, gen, pn[0])
        o_n, _ = OF.rot_reverse_step(sd_d, o_pred, o_t, t, gen, rn['dir'][0], rn['bin_u'][0], rn['in_u'][0],
                                     rn['gauss'][0], cdf=cdf)
        c_n, _ = type_reverse_step(sd_d, logits, c_t, t, gen, tu[0], K)
        return x_n, c_n, o_n, o_pred

    oracle_step(0)
    torch.cuda.synchronize()
    ms_oracle = timed(oracle_step, args.oracle_steps, flush)
    want = oracle_step(0)
    # the CUDA step at the same t with the same draws: slot 1 -> slot 0 of a scratch trajectory
    scratch = torch.empty((2, n * (6 + K)), device=dev)
    for dst, src in zip(split(scratch[1]), (x_t, c_t, o_t)):
        dst.copy_(src)
    at_t = lambda a: {t: a[0]}
    model.run_steps(state, [t], lambda s: split(scratch[s - t]), pos_noise=at_t(pn),
                    rot_noise={k: at_t(v) for k, v in rn.items()}, type_uniform=at_t(tu))
    torch.cuda.synchronize()
    got = split(scratch[0])
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))
    from oracle.ipa import so3vec_to_rotation
    # rotations of the FGs whose input o and both log maps of the step (encoder o_pred, step o) are well conditioned
    # (angle < pi - 0.05): the fp32 log map amplifies rounding by 1 / sin(theta) near pi (DESIGN.md section 13)
    well = lambda o: o.double().norm(dim=-1) < torch.pi - 0.05
    ok = well(want[2]) & well(got[2]) & well(want[3]) & well(o_t)
    d_rot = (so3vec_to_rotation(got[2][ok].double()) - so3vec_to_rotation(want[2][ok].double())).abs().max()
    diff = {'x': rel(got[0], want[0]), 'exp_o_abs': float(d_rot), 'o_rows_compared': int(ok.sum()), 'o_rows': n,
            'fg_types_equal': bool(torch.equal(got[1].argmax(-1), want[1].argmax(-1)))}
    out = {'model': 'difffg', 'workload': f'{B} pockets x ({N_RES} residues + {N_FG} FGs), hidden 256, 9 layers, K={K}, '
                                          f'T={T} (assumed shape, not from data)',
           'n_gpus': 1, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(ms, 4),
           'samples_per_s': round(B / (T * ms * 1e-3), 4), 'launches_per_step': launches, 'kernel_ms_per_step': kern,
           'oracle_eager_torch_ms_per_step': round(ms_oracle, 3), 'oracle_steps': args.oracle_steps,
           'speedup_vs_oracle': round(ms_oracle / ms, 2), 'max_rel_diff_vs_oracle_step': diff,
           'dtype': 'f32', 'data': 'synthetic', 'l2_flush_between_steps': True, **card()}
    print(json.dumps(out), flush=True)


if __name__ == '__main__':
    main()
