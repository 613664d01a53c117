"""Golden for tests/test_reference_plugin.py: what the UNMODIFIED reference computes on the plugin test's inputs, so that
the test needs no copy of the reference (needs the reference checkout, imported through ref_shims.py):

    python tests/golden/make_golden_plugin.py      ->  tests/golden/plugin_seam.npz

The reference's ``TargetDiff.sample`` runs with its own denoiser on two pockets (120 + 14 and 70 + 9 atoms), T = 6 steps,
with injected noise.  Stored: ligand coordinates and atom types of every state, and the keyword arguments and outputs of
the loop's first denoiser call (``self.denoiser(batch_idx=batch_idx, **context_composed)``, targetdiff.py:166), i.e. the
calling convention a drop-in denoiser has to accept.  Inputs and weights are regenerated bit-identically by the test
(cbgbench_b200/synthetic.py).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import ref_shims  # noqa: E402
from cbgbench_b200 import synthetic  # noqa: E402
from cbgbench_b200.targetdiff import TargetDiffB200  # noqa: E402

# must match tests/test_reference_plugin.py
T = 6
N_PROT, N_LIG = [120, 70], [14, 9]
DATA_SEED, NOISE_SEED = 61, 17


def main():
    torch.set_grad_enabled(False)
    ref = ref_shims.load_targetdiff(ref_shims.targetdiff_cfg(num_steps=T))
    mine = TargetDiffB200(synthetic.targetdiff_config(num_steps=T))
    ref.load_state_dict(synthetic.seeded_state_dict(mine, seed=0), strict=True)
    batch = synthetic.make_batch(N_PROT, N_LIG, seed=DATA_SEED)
    pn, tu = synthetic.make_noise(T, sum(N_LIG), 13, seed=NOISE_SEED)
    calls = {'randn': 0, 'rand': 0}
    seen = []

    def record(module, args, kwargs, output):
        if not seen:
            seen.append((args, dict(kwargs), output))

    def fake_randn_like(a, *aa, **kk):      # once per step, t = T-1 ... 0 (diffusion_scheduler.py:163)
        t = T - 1 - calls['randn']
        calls['randn'] += 1
        return pn[t]

    def fake_rand_like(a, *aa, **kk):       # categorical.py:27
        t = T - 1 - calls['rand']
        calls['rand'] += 1
        return tu[t]

    hook = ref.denoiser.register_forward_hook(record, with_kwargs=True)
    orig_randn, orig_rand = torch.randn_like, torch.rand_like
    torch.randn_like, torch.rand_like = fake_randn_like, fake_rand_like
    try:
        traj = ref.sample(batch)
    finally:
        torch.randn_like, torch.rand_like = orig_randn, orig_rand
        hook.remove()
    assert calls == {'randn': T, 'rand': T}, calls
    args, kwargs, (x_out, h_out, v_out) = seen[0]
    assert not args and sorted(kwargs) == ['batch_idx', 'gen_flag', 'h', 'lig_flag', 'x'], (args, sorted(kwargs))
    out = {f'call/in/{k}': v.cpu().numpy() for k, v in kwargs.items()}
    out.update({'call/out/x': x_out.cpu().numpy(), 'call/out/h': h_out.cpu().numpy(), 'call/out/v': v_out.cpu().numpy()})
    for t in range(-1, T):
        out[f'x{t}'] = traj[t][0].cpu().numpy()
        out[f'v{t}'] = traj[t][1].cpu().argmax(-1).numpy().astype(np.int16)
    np.savez_compressed(os.path.join(HERE, 'plugin_seam.npz'), **out)
    print('plugin seam T=6: call nodes', kwargs['x'].shape[0], 'final types', out['v-1'])


if __name__ == '__main__':
    main()
