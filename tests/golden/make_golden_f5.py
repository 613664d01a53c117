"""Golden fixtures of the D3FG sampler from the UNMODIFIED reference ``D3FG`` (/root/reference
repo/models/diffusion/difffg.py), imported through tests/golden/ref_shims.py.

    python tests/golden/make_golden_f5.py          (needs /root/reference; the fixtures are committed)

The reference's ``sample()`` runs on the CPU with its random draws queued from cbgbench_b200.synthetic.make_d3fg_noise,
in the order the reference consumes them; ``torch.multinomial`` is replaced by the project's inverse-CDF definition
(oracle/diffusion_fg.py: multinomial_bin).  Inputs and weights are regenerated bit-identically by the tests (numpy
RandomState seeds), so only OUTPUTS are stored:
  d3fg_trajectory.npz   per case: x / o [T+1, n, 3] and FG types [T+1, n] for keys T-1 ... -1
  d3fg_tables_T1000.npz the 12 VP tables of the pos / rot / fg schedulers, the 4 TypeVP log tables, the forward and inverse
                        angular stddev / approx_flag vectors and their Y rows at t in ROWS, at the shipped T = 1000
  d3fg_state_keys.json  state-dict keys and shapes of the shipped configuration (hidden 256, 9 layers, 28 classes, T 1000)
The oracle restatement is asserted equal to the reference (1e-5) at every state of every case.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ref_shims  # noqa: E402
from cbgbench_b200 import synthetic as S  # noqa: E402

ROWS = [0, 1, 2, 10, 500, 999]
VP_NAMES = ['betas', 'alphas', 'alphas_cumprod', 'alphas_cumprod_prev', 'sqrt_alphas_cumprod',
            'sqrt_one_minus_alphas_cumprod', 'sqrt_recip_alphas_cumprod', 'sqrt_recipm1_alphas_cumprod',
            'posterior_mean_c0_coef', 'posterior_mean_ct_coef', 'posterior_var', 'posterior_logvar']
TYPE_NAMES = ['log_alphas_v', 'log_one_minus_alphas_v', 'log_alphas_cumprod_v', 'log_one_minus_alphas_cumprod_v']


def ref_cfg(num_steps):
    c = S.d3fg_config(num_steps=num_steps)
    return ref_shims.EasyDict(json.loads(json.dumps(c)))


class DrawQueue:
    """Replaces torch's random functions while the reference samples: each call pops the next queued draw."""

    def __init__(self):
        self.q = []

    def push(self, kind, value):
        self.q.append((kind, value))

    def pop(self, kind, shape):
        k, v = self.q.pop(0)
        assert k == kind and tuple(v.shape) == tuple(shape), (k, kind, tuple(v.shape), tuple(shape))
        return v.clone()

    def install(self):
        from oracle.diffusion_fg import multinomial_bin
        self.saved = {n: getattr(torch, n) for n in ('randn', 'randn_like', 'rand_like', 'multinomial')}
        torch.randn = lambda *size, device=None, **kw: self.pop('randn', size[0] if len(size) == 1 else size)
        torch.randn_like = lambda t, **kw: self.pop('randn_like', t.shape)
        torch.rand_like = lambda t, **kw: self.pop('rand_like', t.shape)

        def multinomial(prob, num_samples):
            u = self.pop('multinomial', prob.shape[:1])
            return multinomial_bin(torch.cumsum(prob.double(), dim=1), u)[:, None]
        torch.multinomial = multinomial

    def uninstall(self):
        for n, f in self.saved.items():
            setattr(torch, n, f)
        assert not self.q, f'{len(self.q)} draws left over'


def main():
    ref_shims.install()
    torch.set_grad_enabled(False)
    from repo.models.diffusion.difffg import D3FG
    from cbgbench_b200.difffg import D3FGB200
    from oracle import diffusion_fg as OF
    T = S.D3FG_STEPS
    ref = D3FG(ref_cfg(T)).eval()
    ours = D3FGB200(S.d3fg_config(num_steps=T))
    rsd, osd = ref.state_dict(), ours.state_dict()
    assert list(rsd.keys()) == list(osd.keys())
    assert all(tuple(a.shape) == tuple(b.shape) for a, b in zip(rsd.values(), osd.values()))
    for k in rsd:                                  # schedule tables are bit-equal at the test size
        if k.startswith(S.D3FG_SKIP):
            assert torch.equal(rsd[k], osd[k]), k
    sd = S.seeded_state_dict(ours, seed=S.D3FG_WEIGHT_SEED, skip_prefixes=S.D3FG_SKIP)
    ref.load_state_dict(sd, strict=True)
    out = {}
    for name, n_res, n_fg, seed, mode in S.D3FG_CASES:
        batch = S.make_fg_batch(n_res, n_fg, seed, mode)
        n = sum(n_fg)
        pn, rn, tu = S.make_d3fg_noise(T, n, 28, seed=S.D3FG_NOISE_SEED)
        dq = DrawQueue()
        for t in reversed(range(T)):
            for kind, v in (('randn_like', pn[t]), ('randn', rn['dir'][t]), ('multinomial', rn['bin_u'][t]),
                            ('rand_like', rn['in_u'][t]), ('randn_like', rn['gauss'][t]), ('rand_like', tu[t])):
                dq.push(kind, v)
        dq.install()
        try:
            traj = ref.sample(batch)
        finally:
            dq.uninstall()
        want = OF.sample(sd, batch, T, pn, rn, tu)
        keys = list(range(T - 1, -2, -1))
        for t in keys:
            for i, nm in enumerate(('x', 'c', 'o')):
                a, w = traj[t][i].float(), want[t][i]
                err = float((a - w).abs().max() / (w.abs().max() + 1e-12))
                assert err < 1e-5, (name, t, nm, err)
        out[f'{name}/x'] = np.stack([traj[t][0].numpy() for t in keys])
        out[f'{name}/o'] = np.stack([traj[t][2].numpy() for t in keys])
        out[f'{name}/v'] = np.stack([traj[t][1].argmax(-1).numpy() for t in keys]).astype(np.int8)
        print(name, 'ok', n, 'FGs')
    np.savez_compressed(os.path.join(HERE, 'd3fg_trajectory.npz'), **out)

    big = D3FG(ref_cfg(1000)).eval()                  # the shipped configuration (about a minute of histograms)
    with open(os.path.join(HERE, 'd3fg_state_keys.json'), 'w') as f:
        json.dump({k: list(v.shape) for k, v in big.state_dict().items()}, f, indent=0)
    tab = {}
    for sched in ('pos_scheduler', 'rot_scheduler', 'type_scheduler'):
        for nm in VP_NAMES:
            tab[f'{sched}/{nm}'] = getattr(big, sched).__getattr__(nm).detach().numpy()
    for nm in TYPE_NAMES:
        tab[f'type_scheduler/{nm}'] = getattr(big.type_scheduler, nm).detach().numpy()
    for which in ('fwd', 'inv'):
        d = getattr(big.rot_scheduler, f'angular_distrib_{which}')
        tab[f'{which}/stddevs'] = d.stddevs.numpy()
        tab[f'{which}/approx_flag'] = d.approx_flag.numpy()
        tab[f'{which}/Y_rows'] = d.Y[ROWS].numpy()
    tab['rows'] = np.asarray(ROWS)
    np.savez_compressed(os.path.join(HERE, 'd3fg_tables_T1000.npz'), **tab)
    for fn in ('d3fg_trajectory.npz', 'd3fg_tables_T1000.npz', 'd3fg_state_keys.json'):
        print(fn, os.path.getsize(os.path.join(HERE, fn)), 'bytes')


if __name__ == '__main__':
    main()
