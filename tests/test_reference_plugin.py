"""The drop-in seams of INTEGRATION.md section 2, against what the UNMODIFIED reference computes on the same inputs
(tests/golden/plugin_seam.npz, written by tests/golden/make_golden_plugin.py from the reference's own
``TargetDiff.sample`` with its own denoiser and injected noise):

* seam 1: ``UniTransformerB200`` (what the patched ``get_e3_gnn`` returns) is called exactly the way the reference's
  sample loop calls its denoiser - ``denoiser(batch_idx=..., x=..., h=..., gen_flag=..., lig_flag=...)`` -> ``(x, h, v)``,
  with the arguments recorded from the loop's first step - and returns the reference denoiser's outputs;
* seam 2: ``get_model(cfg)`` returns ``TargetDiffB200`` for the reference's EasyDict config, loads the same state dict and
  samples the reference's trajectory.

Atom types bit-exact, coordinates within 1e-4 of the reference and of the oracle."""
import numpy as np
import pytest
import torch

from cbgbench_b200 import synthetic
from helpers import assert_close, golden, make_model, rel_err

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
TOL = 1e-4
# must match tests/golden/make_golden_plugin.py
T = 6
N_PROT, N_LIG = [120, 70], [14, 9]
DATA_SEED, NOISE_SEED = 61, 17


def test_reference_sample_loop_with_b200_denoiser_and_get_model_seam():
    from baseline import ref_runner
    from cbgbench_b200 import TargetDiffB200, UniTransformerB200, get_model
    from oracle import diffusion as OD
    g = golden('plugin_seam.npz')
    dev = torch.device('cuda:0')
    _, sd = make_model(T)
    batch = synthetic.make_batch(N_PROT, N_LIG, seed=DATA_SEED)
    pn, tu = synthetic.make_noise(T, sum(N_LIG), 13, seed=NOISE_SEED)
    want = OD.sample(sd, batch, T, pn, tu)

    # ---- seam 2: get_model(cfg) -> TargetDiffB200 built from the reference's EasyDict config
    mine = get_model(ref_runner.targetdiff_cfg(T))
    assert isinstance(mine, TargetDiffB200) and isinstance(mine.denoiser, UniTransformerB200)
    mine.load_state_dict(sd, strict=True)                      # identical keys / shapes
    mine = mine.to(dev).eval()

    # ---- seam 1: the denoiser call of the reference's sample loop, keyword for keyword
    call = {k[len('call/in/'):]: torch.from_numpy(g[k]).to(dev) for k in g.files if k.startswith('call/in/')}
    assert sorted(call) == ['batch_idx', 'gen_flag', 'h', 'lig_flag', 'x']
    x, h, v = mine.denoiser(**call)
    for got, k in ((x, 'x'), (h, 'h'), (v, 'v')):
        assert rel_err(got.cpu(), g[f'call/out/{k}']) < TOL, (k, rel_err(got.cpu(), g[f'call/out/{k}']))
    assert_close(x.cpu(), g['call/out/x'], rtol=1e-4, atol=1e-4, what='seam 1 denoiser x')

    dbatch = {k: (v_.to(dev) if torch.is_tensor(v_) else v_) for k, v_ in batch.items()}
    traj = mine.sample(dbatch, pos_noise=pn, type_uniform=tu)
    for t in range(-1, T - 1):
        xg, vg = traj[t][0].cpu(), traj[t][1].cpu().argmax(-1)
        assert np.array_equal(vg.numpy(), g[f'v{t}'].astype(np.int64)), t
        assert torch.equal(vg, want[t][1].argmax(-1)), t
        assert rel_err(xg, g[f'x{t}']) < TOL, (t, rel_err(xg, g[f'x{t}']))
        assert_close(xg, g[f'x{t}'], rtol=1e-4, atol=1e-5, what=f'seam 2 x t={t}')
        assert rel_err(xg, want[t][0]) < TOL, (t, rel_err(xg, want[t][0]))
