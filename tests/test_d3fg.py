"""D3FG sampler: context embedder, SO(3) reverse step and the ``difffg`` model (DESIGN.md section 13).

CPU: the oracle restatement (oracle/diffusion_fg.py) against the live-reference fixtures (tests/golden/make_golden_f5.py),
the state-dict and schedule-table contracts, the factory, the unsupported-configuration errors, the 28-class IPA packer.
GPU: csrc/d3fg.cu and csrc/ipa.cu through the C-ABI against the oracle and the fixtures.

Bars (tests/helpers.py): x and logits within 1e-4 relative (max norm and element-wise), FG types bit-exact.  Rotations are
compared as exp(o) (3x3 entries) and o element-wise.  The fp32 log map amplifies rounding by about 1 / sin(theta) near
the angle pi (where o and -o are the same rotation): measured against float64, the oracle's own error reaches 8e-5 at
pi - 0.07.  So one step is compared within 1e-4 where the angle is below pi - 0.2; a 20-step trajectory, which carries
each step's difference into the next, within 5e-4 on the FGs whose log maps all stayed below pi - 0.05, and their
positions (which see o only through exp(o)) at the position bars; every FG's positions within 1e-2 (no gross error)."""
import ctypes as C
import json
import os
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from cbgbench_b200 import _lib, get_model, synthetic as S
from cbgbench_b200.difffg import D3FGB200
from cbgbench_b200.ipatransformer import IPATransformerB200, pack_ipa_blob
from cbgbench_b200.schedulers import TypeVPTables, VPTables, angular_histogram, rot_stddevs
from helpers import GOLDEN, assert_close, rel_err

torch.set_grad_enabled(False)
T = S.D3FG_STEPS


def _gold(name):
    return np.load(os.path.join(GOLDEN, name))


_MODEL = {}


def _model():
    """T = 20 model at the shipped width with the fixtures' seeded weights (built once: the histograms take seconds)."""
    if not _MODEL:
        m = D3FGB200(S.d3fg_config(num_steps=T))
        sd = S.seeded_state_dict(m, seed=S.D3FG_WEIGHT_SEED, skip_prefixes=S.D3FG_SKIP)
        m.load_state_dict(sd, strict=True)
        _MODEL['m'], _MODEL['sd'] = m.eval(), sd
    return _MODEL['m'], _MODEL['sd']


def _case(case):
    name, n_res, n_fg, seed, mode = case
    batch = S.make_fg_batch(n_res, n_fg, seed, mode)
    return batch, S.make_d3fg_noise(T, sum(n_fg), 28, seed=S.D3FG_NOISE_SEED)


def so3_exp(o):
    from oracle.ipa import so3vec_to_rotation
    return so3vec_to_rotation(o.double())


def angle(o):
    return o.double().cpu().norm(dim=-1)


WELL = np.pi - 0.05       # trajectory: FGs whose log maps stayed below this angle
WELL_STEP = np.pi - 0.2   # one step: the fp32 log map's own error stays below 3e-5 here


def assert_rot_close(got, want, what, rows=None, tol=1e-4, well=WELL_STEP):
    """exp(o) entries within ``tol`` and o element-wise (1e-4 relative, ``tol`` rad absolute) on ``rows`` (default: all)
    whose angle is below ``well`` on both sides."""
    got, want = got.double().cpu(), want.double().cpu()
    ok = (angle(want) < well) & (angle(got) < well)
    if rows is not None:
        ok &= rows
    d = (so3_exp(got[ok]) - so3_exp(want[ok])).abs().max() if bool(ok.any()) else torch.zeros(())
    assert float(d) < tol, f'{what}: exp(o) differs by {float(d):.3e} ({int(ok.sum())} rows compared)'
    assert_close(got[ok], want[ok], atol=tol, what=what)


# ---- CPU ------------------------------------------------------------------------------------------------------------------
def test_state_dict_keys_and_shapes_match_reference():
    with open(os.path.join(GOLDEN, 'd3fg_state_keys.json')) as f:
        want = json.load(f)                                     # shipped config at T = 1000
    m, _ = _model()
    got = {k: list(v.shape) for k, v in m.state_dict().items()}
    assert list(got) == list(want)
    for k, shape in want.items():
        if k.startswith(S.D3FG_SKIP[:3]) and shape and shape[0] == 1000:
            shape = [T] + shape[1:]                             # schedule tables: leading dim = T
        assert got[k] == shape, k


def test_schedule_tables_match_reference_T1000():
    g = _gold('d3fg_tables_T1000.npz')
    pos = VPTables(1000, beta_start=1e-7, beta_end=2e-3, type='sigmoid')
    typ = TypeVPTables(1000, num_classes=28, type='cosine', cosine_s=0.01)
    rot = VPTables(1000, type='cosine', cosine_s=0.01)           # RotVPTables' VP part (its histograms: below)
    for sched, tab in (('pos_scheduler', pos), ('type_scheduler', typ), ('rot_scheduler', rot)):
        for nm in ('betas', 'alphas', 'alphas_cumprod', 'alphas_cumprod_prev', 'sqrt_alphas_cumprod',
                   'sqrt_one_minus_alphas_cumprod', 'sqrt_recip_alphas_cumprod', 'sqrt_recipm1_alphas_cumprod',
                   'posterior_mean_c0_coef', 'posterior_mean_ct_coef', 'posterior_var', 'posterior_logvar'):
            assert torch.equal(getattr(tab, nm).detach(), torch.from_numpy(g[f'{sched}/{nm}'])), (sched, nm)
    for nm in ('log_alphas_v', 'log_one_minus_alphas_v', 'log_alphas_cumprod_v', 'log_one_minus_alphas_cumprod_v'):
        assert torch.equal(getattr(typ, nm).detach(), torch.from_numpy(g[f'type_scheduler/{nm}'])), nm
    fwd, inv = rot_stddevs(rot.alphas_cumprod.detach(), rot.betas.detach())
    for which, sd in (('fwd', fwd), ('inv', inv)):
        sd = torch.tensor(sd, dtype=torch.float32)
        assert torch.equal(sd, torch.from_numpy(g[f'{which}/stddevs'])), which
        assert torch.equal(sd <= 0.1, torch.from_numpy(g[f'{which}/approx_flag'])), which
        want = torch.from_numpy(g[f'{which}/Y_rows'])
        for i, t in enumerate(g['rows']):
            x, y = angular_histogram(sd[t].item())
            assert torch.equal(x, torch.linspace(0, np.pi, 8192))
            # bit-equal on the fixture machine; the fp32 sum over 1024 terms may round differently with another SIMD width
            assert_close(y, want[i], rtol=1e-6, atol=1e-6 * float(want[i].abs().max()), what=f'{which} Y[{t}]')


@pytest.mark.parametrize('case', S.D3FG_CASES, ids=[c[0] for c in S.D3FG_CASES])
def test_oracle_matches_reference_trajectory(case):
    from oracle import diffusion_fg as OF
    _, sd = _model()
    batch, (pn, rn, tu) = _case(case)
    want = OF.sample(sd, batch, T, pn, rn, tu)
    g = _gold('d3fg_trajectory.npz')
    for i, t in enumerate(range(T - 1, -2, -1)):
        x, c, o = want[t]
        assert rel_err(x, torch.from_numpy(g[f'{case[0]}/x'][i])) < 1e-5, t
        assert rel_err(o, torch.from_numpy(g[f'{case[0]}/o'][i])) < 1e-5, t
        assert torch.equal(c.argmax(-1), torch.from_numpy(g[f'{case[0]}/v'][i]).long()), t


def test_get_model_and_unsupported_configs():
    for name in ('difffg', 'difffg_v2'):
        cfg = S.d3fg_config(num_steps=4, hidden=128, num_layers=1)
        cfg['type'] = name
        assert type(get_model(cfg)) is D3FGB200
    bad = [lambda c: c.embedder.__setitem__('time', dict(type='sin')),
           lambda c: c.embedder.__setitem__('vec', dict(type='x', vec_emb_dim=4)),
           lambda c: c.embedder.residue.__setitem__('type', 'linear'),
           lambda c: c.embedder.__setitem__('emb_dim', 128),
           lambda c: c.__setitem__('num_fgtype', 33)]
    for edit in bad:
        cfg = S.d3fg_config(num_steps=4)
        edit(cfg)
        with pytest.raises(NotImplementedError):
            D3FGB200(cfg)


def test_cpu_model_raises():
    m = D3FGB200(S.d3fg_config(num_steps=4, hidden=128, num_layers=1))
    with pytest.raises(RuntimeError):
        m.sample(S.make_fg_batch([12], [3], 1))
    with pytest.raises(NotImplementedError):
        m(S.make_fg_batch([12], [3], 1))


def test_ipa_packer_places_28_class_classifier():
    H = 256
    model = IPATransformerB200(S.ipa_config(H, 1, 28))
    sd = S.seeded_state_dict(model, seed=1, skip_prefixes=())
    L = _lib.lib()
    blob = pack_ipa_blob(sd, H, 1, 1, 28)
    g0 = _lib.blob_layout()['global_floats']
    head = {L.cbg_ipa_head_field_name(f).decode(): (L.cbg_ipa_head_field_offset(H, f), L.cbg_ipa_head_field_size(H, f))
            for f in range(L.cbg_ipa_head_fields())}
    o, n = head['CLS_W1']
    assert n == 32 * H
    w = blob[g0 + o: g0 + o + n].view(32, H)
    assert torch.equal(w[:28], sd['classifier.2.weight']) and not bool(w[28:].any())
    o, n = head['CLS_B1']
    assert torch.equal(blob[g0 + o: g0 + o + 28], sd['classifier.2.bias'])
    with pytest.raises(NotImplementedError):
        IPATransformerB200(S.ipa_config(H, 1, 33))


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('num_classes', [28, 32])
def test_cuda_ipa_forward_many_classes(num_classes):
    from oracle import ipa as OI
    dev = torch.device('cuda:0')
    model = IPATransformerB200(S.ipa_config(256, 2, num_classes))
    sd = S.seeded_state_dict(model, seed=9, skip_prefixes=())
    model.load_state_dict(sd, strict=True)
    model = model.to(dev)
    inp = S.make_ipa_inputs(256, [60, 25], [8, 5], 77, 'partial')
    got = [t.cpu() for t in model(*[t.to(dev) for t in inp])]
    want = OI.ipatransformer_forward(sd, *inp)
    for a, w, nm in zip(got, want, ('eps_pos', 'h', 'o_next', 'R_next', 'c')):
        assert rel_err(a, w) < 1e-4, (nm, rel_err(a, w))
        if nm == 'o_next':
            assert_rot_close(a, w, nm)
        else:
            assert_close(a, w, what=nm)


def _reverse_inputs(n, K, seed):
    rs = np.random.RandomState(seed)
    f = lambda *s: torch.from_numpy(rs.normal(size=s).astype(np.float32))
    v = torch.from_numpy(rs.randint(0, K, size=n))
    gen = torch.from_numpy(rs.random_sample(n) < 0.75)
    return dict(eps=f(n, 3), logits=2 * f(n, K), o_pred=f(n, 3), x_t=f(n, 3), c_t=F.one_hot(v, K).float(),
                o_t=f(n, 3), gen=gen)


@pytest.mark.gpu
def test_cuda_reverse_step_matches_oracle():
    """cbg_d3fg_reverse_f32 alone at the shipped T = 1000 schedule: only the histogram rows the steps use are built."""
    from oracle import diffusion_fg as OF
    from oracle.diffusion import type_reverse_step
    from oracle.diffusion_bp import pos_reverse_step_score
    dev = torch.device('cuda:0')
    Tb, K, n, steps = 1000, 28, 96, [0, 1, 2, 500, 999]
    pos = VPTables(Tb, beta_start=1e-7, beta_end=2e-3, type='sigmoid')
    typ = TypeVPTables(Tb, num_classes=K, type='cosine', cosine_s=0.01)
    rot = VPTables(Tb, type='cosine', cosine_s=0.01)
    _, inv = rot_stddevs(rot.alphas_cumprod.detach(), rot.betas.detach())
    stddevs = torch.tensor(inv, dtype=torch.float32)
    X = torch.zeros(Tb, 8192)
    Y = torch.zeros(Tb, 8192)
    for t in steps:
        X[t], Y[t] = angular_histogram(inv[t])
    pre = 'rot_scheduler.angular_distrib_inv.'
    sd = {pre + 'X': X, pre + 'Y': Y, pre + 'stddevs': stddevs, pre + 'approx_flag': stddevs <= 0.1}
    sd.update({'pos_scheduler.' + k: v.detach() for k, v in pos.state_dict().items()})
    sd.update({'type_scheduler.' + k: v.detach() for k, v in typ.state_dict().items()})
    cdf = OF.inverse_cdf(sd)
    cdf_d, X_d = cdf.to(dev), X.to(dev)
    host = types.SimpleNamespace(pos_scheduler=pos, type_scheduler=typ)
    L = _lib.lib()
    for t in steps:
        inp = _reverse_inputs(n, K, 100 + t)
        pn, rn, tu = S.make_d3fg_noise(1, n, K, seed=200 + t)
        rnd = dict(pos_noise=pn[0], rot_dir=rn['dir'][0], rot_bin_u=rn['bin_u'][0], rot_in_u=rn['in_u'][0],
                   rot_gauss=rn['gauss'][0], type_u=tu[0])
        d = {k: v.to(dev).contiguous() for k, v in {**inp, **rnd}.items()}
        gen8 = d['gen'].to(torch.uint8)
        x_n, c_n, o_n = torch.empty(n, 3, device=dev), torch.empty(n, K, device=dev), torch.empty(n, 3, device=dev)
        v_n = torch.empty(n, dtype=torch.int64, device=dev)
        bins = torch.empty(n, dtype=torch.int32, device=dev)
        coef = D3FGB200.step_coef(host, t, inv, (stddevs <= 0.1).tolist())
        _lib.check(L.cbg_d3fg_reverse_f32(
            C.byref(coef), cdf_d.data_ptr(), X_d.data_ptr(), 8191, *[d[k].data_ptr() for k in (
                'eps', 'logits', 'o_pred', 'x_t', 'c_t', 'o_t')], gen8.data_ptr(), *[d[k].data_ptr() for k in (
                    'pos_noise', 'rot_dir', 'rot_bin_u', 'rot_in_u', 'rot_gauss', 'type_u')], n, K,
            x_n.data_ptr(), c_n.data_ptr(), o_n.data_ptr(), v_n.data_ptr(), bins.data_ptr(), _lib.stream_ptr(dev)))
        torch.cuda.synchronize()
        gen = inp['gen']
        x_w = pos_reverse_step_score(sd, inp['eps'], inp['x_t'], t, gen, rnd['pos_noise'])
        o_w, b_w = OF.rot_reverse_step(sd, inp['o_pred'], inp['o_t'], t, gen, rnd['rot_dir'], rnd['rot_bin_u'],
                                       rnd['rot_in_u'], rnd['rot_gauss'], cdf=cdf)
        c_w, v_w = type_reverse_step(sd, inp['logits'], inp['c_t'], t, gen, rnd['type_u'], K)
        assert torch.equal(bins.cpu().long(), b_w), t
        assert rel_err(x_n.cpu(), x_w) < 1e-4 and torch.equal(v_n.cpu(), v_w) and torch.equal(c_n.cpu(), c_w), t
        assert_close(x_n.cpu(), x_w, what=f'x t={t}')
        assert_rot_close(o_n.cpu(), o_w, f'o t={t}')
        assert torch.equal(o_n.cpu()[~gen], inp['o_t'][~gen]) and torch.equal(x_n.cpu()[~gen], inp['x_t'][~gen])


def _gpu_model():
    m, sd = _model()
    return m.to('cuda:0'), sd


@pytest.mark.gpu
@pytest.mark.parametrize('case', S.D3FG_CASES, ids=[c[0] for c in S.D3FG_CASES])
def test_cuda_trajectory_matches_reference(case):
    model, sd = _gpu_model()
    batch, (pn, rn, tu) = _case(case)
    outs = {}
    traj = model.sample(batch, pos_noise=pn, rot_noise=rn, type_uniform=tu, outs=outs)
    g = _gold('d3fg_trajectory.npz')
    assert sorted(traj) == list(range(-1, T))
    assert traj[-1][0].is_cuda and not traj[0][0].is_cuda and len(traj[0]) == 4
    # rotations are compared on FGs whose every log map so far (the encoder's o_pred and the step's o) was well
    # conditioned: one at the pi end perturbs the axis, and the difference is then carried along the trajectory
    clean = angle(batch['ligand_o_fg']) < WELL
    for i, t in enumerate(range(T - 1, -2, -1)):
        x, c, o, bl = (a.cpu() for a in traj[t])
        xw, ow = torch.from_numpy(g[f'{case[0]}/x'][i]), torch.from_numpy(g[f'{case[0]}/o'][i])
        if t < T - 1:
            clean &= (angle(outs[t + 1][2]) < WELL) & (angle(o) < WELL) & (angle(ow) < WELL)
        assert rel_err(x[clean], xw[clean]) < 1e-4, (t, rel_err(x[clean], xw[clean]))
        assert_close(x[clean], xw[clean], what=f'x t={t}')
        assert rel_err(x, xw) < 1e-2, (t, rel_err(x, xw))            # every FG: no gross error
        assert_rot_close(o, ow, f'o t={t}', rows=clean, tol=5e-4, well=WELL)
        assert torch.equal(c.argmax(-1), torch.from_numpy(g[f'{case[0]}/v'][i]).long()), t
        assert torch.equal(c.sum(-1), torch.ones(c.shape[0]))
        assert torch.equal(bl, batch['ligand_type_fg_batch'])
    assert float(clean.float().mean()) >= 0.25, f'only {int(clean.sum())} of {clean.numel()} FGs compared'
    # encoder outputs of the first step vs the oracle (logits bar)
    from oracle import diffusion_fg as OF
    x0 = batch['ligand_pos_heavyatom'][:, 1]
    eps_w, o_w, lg_w = OF.denoise(sd, batch, x0, F.one_hot(batch['ligand_type_fg'], 28).float(), batch['ligand_o_fg'], 28)
    eps, lg, o_pred = (a.cpu() for a in outs[T - 1])
    assert rel_err(lg, lg_w) < 1e-4 and rel_err(eps, eps_w) < 1e-4
    assert_close(lg, lg_w, what='logits')
    assert_rot_close(o_pred, o_w, 'o_pred')
    if 'ligand_gen_flag' in batch:                               # rows without gen_flag keep their input, bit for bit
        fixed = ~batch['ligand_gen_flag']
        for t in range(-1, T):
            x, c, o = (a.cpu() for a in traj[t][:3])
            assert torch.equal(x[fixed], x0[fixed]) and torch.equal(o[fixed], batch['ligand_o_fg'][fixed])
            assert torch.equal(c.argmax(-1)[fixed], batch['ligand_type_fg'][fixed])


@pytest.mark.gpu
def test_cuda_graph_alone_equals_graph_in_batch_and_repeats():
    model, _ = _gpu_model()
    batch, (pn, rn, tu) = _case(S.D3FG_CASES[0])
    steps = 6
    full = model.sample(batch, pos_noise=pn, rot_noise=rn, type_uniform=tu, num_steps=steps)
    again = model.sample(batch, pos_noise=pn, rot_noise=rn, type_uniform=tu, num_steps=steps)
    for t in full:
        for a, b in zip(full[t], again[t]):
            assert torch.equal(a.cpu(), b.cpu()), t
    g = 2                                          # last graph: its chain ids do not touch the previous graph's
    bl, br = batch['ligand_type_fg_batch'], batch['protein_type_fg_batch']
    ml, mr = bl == g, br == g
    sub = {}
    for k, v in batch.items():
        if k == 'protein_num_chains':
            sub[k] = v[g:g + 1]
        elif k.startswith('ligand'):
            sub[k] = v[ml]
        else:
            sub[k] = v[mr]
    sub['ligand_type_fg_batch'] = torch.zeros(int(ml.sum()), dtype=torch.long)
    sub['protein_type_fg_batch'] = torch.zeros(int(mr.sum()), dtype=torch.long)
    alone = model.sample(sub, pos_noise=pn[:, ml], rot_noise={k: v[:, ml] for k, v in rn.items()},
                         type_uniform=tu[:, ml], num_steps=steps)
    for t in alone:
        for a, b in zip(alone[t][:3], full[t][:3]):
            assert torch.equal(a.cpu(), b.cpu()[ml]), t
