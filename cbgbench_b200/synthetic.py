"""Synthetic pockets + seeded weights (no dataset or checkpoint is reachable offline).

Input distributions follow SURVEY.md section 8(d): protein_pos ~ N(0, 8^2) centred
(``center_pos``, repo/datasets/transforms/translation.py:5-25), ligand_pos ~ N(0, I)
(``assign_molpos`` gaussian, init_lig.py:415-432), ligand types ~ U{0..K-1}
(``assign_atomtype`` uniform, init_lig.py:377-412), protein feature = one-hot(6) | backbone bit
(protein_featurizer.py:21-26), residue ~ U{0..19}.

Everything is drawn from ``numpy.random.RandomState`` (bit-stable across numpy/torch
versions and machines) so golden fixtures only need to store OUTPUTS.
"""
import numpy as np
import torch

from .modules import cfg_get


class Cfg(dict):
    """Minimal attr-dict with the ``cfg.get(name, default)`` protocol the reference's
    EasyDict configs offer (repo/utils/misc.py:141-146)."""

    def __init__(self, d=None, **kw):
        super().__init__()
        for k, v in dict(d or {}, **kw).items():
            self[k] = v

    def __setitem__(self, k, v):
        if isinstance(v, dict) and not isinstance(v, Cfg):
            v = Cfg(v)
        super().__setitem__(k, v)

    __setattr__ = __setitem__

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e


def targetdiff_config(num_steps=1000, num_layers=9, num_atomtype=13, k=None, cutoff_mode=None, r_max=None):
    """configs/denovo/train/targetdiff.yml:1-23 (+ num_atomtype, configuration.py:13-38)."""
    enc = dict(type='unitransformer', node_feat_dim=128, n_heads=16, num_layers=num_layers)
    if k is not None:
        enc['k'] = k
    if cutoff_mode is not None:
        enc['cutoff_mode'] = cutoff_mode
    if r_max is not None:
        enc['r_max'] = r_max
    return Cfg(dict(
        type='targetdiff', num_atomtype=num_atomtype, encoder=enc,
        generator=dict(pos_schedule=dict(type='sigmoid', beta_start=1.e-7, beta_end=2.e-3),
                       atom_schedule=dict(type='cosine', cosine_s=0.01),
                       num_diffusion_timesteps=num_steps, time_sampler='symmetric'),
        embedder=dict(emb_dim=128, atom=dict(type='linear'), residue=dict(type='linear'))))


def diffsbdd_config(num_steps=1000, num_layers=9, num_atomtype=13, k=None):
    """configs/denovo/train/diffsbdd.yml:1-22 (+ num_atomtype)."""
    enc = dict(type='unitransformer', node_feat_dim=128, n_heads=16, num_layers=num_layers)
    if k is not None:
        enc['k'] = k
    return Cfg(dict(
        type='diffsbdd', num_atomtype=num_atomtype, encoder=enc,
        generator=dict(pos_schedule=dict(type='polynomial_2'), atom_schedule=dict(type='polynomial_2'),
                       num_diffusion_timesteps=num_steps, time_sampler='random'),
        embedder=dict(emb_dim=128, atom=dict(type='linear'), residue=dict(type='linear'))))


def diffbp_config(num_steps=1000, num_layers=9, num_atomtype=13, k=None, num_layers_com=None):
    """configs/denovo/train/diffbp.yml:1-26 (+ num_atomtype)."""
    enc = dict(type='unitransformer', node_feat_dim=128, n_heads=16, num_layers=num_layers)
    if k is not None:
        enc['k'] = k
    if num_layers_com is not None:
        enc['num_layers_com'] = num_layers_com
    return Cfg(dict(
        type='diffbp', num_atomtype=num_atomtype, encoder=enc,
        generator=dict(pos_schedule=dict(type='sigmoid', beta_start=1.e-7, beta_end=2.e-3),
                       atom_schedule=dict(type='uniform'), num_diffusion_timesteps=num_steps, time_sampler='symmetric',
                       com_schedule=dict(type='log', sigma_min=1.e-7, sigma_max=5.0)),
        embedder=dict(emb_dim=128, atom=dict(type='linear'), residue=dict(type='linear'))))


def make_bp_noise(num_steps, n_lig, seed=7):
    """Injected draws of one DiffBP.sample call: positions N(0,1) [T,n_lig,3], type change mask U[0,1) [T,n_lig]."""
    rs = np.random.RandomState(seed)
    pn = torch.from_numpy(rs.normal(size=(num_steps, n_lig, 3)).astype(np.float32))
    tu = torch.from_numpy(rs.random_sample(size=(num_steps, n_lig)).astype(np.float32))
    return pn, tu


def make_sbdd_noise(num_steps, n_lig, num_classes=13, seed=7):
    """Injected normal draws of one DiffSBDD.sample call (order of the reference: x then c)."""
    rs = np.random.RandomState(seed)
    f = lambda *shape: torch.from_numpy(rs.normal(size=shape).astype(np.float32))
    return {'init_x': f(n_lig, 3), 'init_c': f(n_lig, num_classes),
            'step_x': f(num_steps, n_lig, 3), 'step_c': f(num_steps, n_lig, num_classes),
            'final_x': f(n_lig, 3), 'final_c': f(n_lig, num_classes)}


def make_batch(n_prot, n_lig, seed=2024, num_classes=13, gen_mode='denovo', protein_sigma=8.0):
    """Flat ragged batch with the reference's keys (SURVEY.md section 8b).

    n_prot / n_lig: per-graph atom counts (sequences of equal length).
    gen_mode: 'denovo' (all ligand atoms generated) or 'partial' (linker/scaffold-like:
    the first two thirds of every ligand are fixed context, the rest is generated)."""
    rs = np.random.RandomState(seed)
    n_prot, n_lig = list(n_prot), list(n_lig)
    assert len(n_prot) == len(n_lig)
    pp, lp, lt, pf, pa, lb, pb, gen = [], [], [], [], [], [], [], []
    for g, (np_, nl) in enumerate(zip(n_prot, n_lig)):
        p = rs.normal(0.0, protein_sigma, size=(np_, 3))
        if np_:
            p = p - p.mean(0, keepdims=True)
        pp.append(p)
        lp.append(rs.normal(0.0, 1.0, size=(nl, 3)))
        lt.append(rs.randint(0, num_classes, size=nl))
        f = np.zeros((np_, 7))
        f[np.arange(np_), rs.randint(0, 6, size=np_)] = 1.0
        f[:, 6] = rs.randint(0, 2, size=np_)
        pf.append(f)
        pa.append(rs.randint(0, 20, size=np_))
        lb.append(np.full(nl, g))
        pb.append(np.full(np_, g))
        gflag = np.ones(nl, dtype=bool)
        if gen_mode == 'partial':
            gflag[: (2 * nl) // 3] = False
        gen.append(gflag)
    cat = lambda xs, dt: torch.from_numpy(np.concatenate(xs, 0).astype(dt))
    n_l, n_p = int(sum(n_lig)), int(sum(n_prot))
    batch = {
        'ligand_pos': cat(lp, np.float32), 'ligand_atom_type': cat(lt, np.int64),
        'protein_pos': cat(pp, np.float32), 'protein_atom_feature': cat(pf, np.float32),
        'protein_aa_type': cat(pa, np.int64),
        'ligand_lig_flag': torch.ones(n_l, dtype=torch.bool),
        'protein_lig_flag': torch.zeros(n_p, dtype=torch.bool),
        'ligand_element_batch': cat(lb, np.int64), 'protein_element_batch': cat(pb, np.int64),
        'protein_translation': torch.zeros(n_p, 3),     # one row per protein atom, like center_pos (translation.py:11-24)
    }
    if gen_mode == 'partial':
        batch['ligand_gen_flag'] = cat(gen, np.bool_)
    return batch


def make_noise(num_steps, n_lig, num_classes, seed=7):
    """Pre-generated per-step noise for parity runs: pos_noise [T,n_lig,3] ~ N(0,1),
    type_uniform [T,n_lig,K] ~ U[0,1)."""
    rs = np.random.RandomState(seed)
    pn = torch.from_numpy(rs.normal(size=(num_steps, n_lig, 3)).astype(np.float32))
    tu = torch.from_numpy(rs.random_sample(size=(num_steps, n_lig, num_classes)).astype(np.float32))
    return pn, tu


def seeded_state_dict(model, seed=0, skip_prefixes=('pos_scheduler.', 'type_scheduler.')):
    """Deterministic weights for every learnable tensor of ``model`` (state-dict order):
    matrices ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in)) (nn.Linear default scale), LayerNorm gains
    ~ N(1, 0.2^2), biases / LayerNorm shifts ~ N(0, 0.2^2) so that no affine term is trivial.
    The H2X value heads (xv_func.net.3) are scaled by 0.1 so random-weight coordinate updates stay
    of trained-model magnitude.  Buffers (``offset``) and schedule tables are left alone."""
    rs = np.random.RandomState(seed)
    sd = model.state_dict()
    out = {}
    for name, t in sd.items():
        if name.startswith(tuple(skip_prefixes)) or name.endswith('.offset'):
            out[name] = t.clone()
            continue
        shape = tuple(t.shape)
        if t.dim() == 2:
            bound = 1.0 / np.sqrt(shape[1])
            v = rs.uniform(-bound, bound, size=shape)
            if 'xv_func.net.3' in name:
                v = v * 0.1
        elif name.endswith('net.1.weight'):
            v = rs.normal(1.0, 0.2, size=shape)
        else:
            v = rs.normal(0.0, 0.2, size=shape)
            if 'xv_func.net.3' in name:
                v = v * 0.1
        out[name] = torch.from_numpy(np.asarray(v, dtype=np.float32)).reshape(shape)
    return out


__all__ = ['Cfg', 'targetdiff_config', 'diffsbdd_config', 'make_sbdd_noise', 'diffbp_config', 'make_bp_noise', 'make_batch', 'make_noise', 'seeded_state_dict', 'cfg_get']


# ---- SURVEY.md section 8 row f4: IPATransformer (D3FG encoder) -----------------------------------------------------------
# (name, hidden, num_layers, num_classes, nodes per graph, functional-group ("ligand") nodes per graph, data seed, gen mode)
IPA_CASES = [
    ('h256_two_graphs', 256, 3, 8, [70, 45], [6, 4], 31, 'denovo'),        # shipped width (d3fg_fg.yml:5), one graph > k + 1
    ('h256_ragged', 256, 2, 12, [120, 20, 9], [8, 3, 2], 32, 'partial'),   # graphs below k + 1 nodes, partial generation
    ('h128_single', 128, 2, 8, [90], [7], 33, 'denovo'),
]
IPA_WEIGHT_SEED = 5


def ipa_config(hidden, num_layers, num_classes, **extra):
    return Cfg(dict(type='ipatransformer', node_feat_dim=hidden, n_heads=16, num_layers=num_layers,
                    num_classes=num_classes, **extra))


def make_ipa_inputs(hidden, n_nodes, n_lig, seed, gen_mode='denovo'):
    """Composed node arrays of the D3FG encoder in the layout compose_context produces ([protein | ligand] per graph):
    (x [N,3], o [N,3] so3 vectors, h [N,hidden], batch_idx, lig_flag, gen_flag)."""
    rs = np.random.RandomState(seed)
    xs, os_, hs, bs, ligs, gens = [], [], [], [], [], []
    for g, (n, nl) in enumerate(zip(n_nodes, n_lig)):
        x = rs.normal(0.0, 6.0, size=(n, 3))
        x[n - nl:] = rs.normal(0.0, 1.5, size=(nl, 3))
        xs.append(x)
        os_.append(rs.normal(0.0, 0.6, size=(n, 3)))
        hs.append(rs.normal(0.0, 1.0, size=(n, hidden)))
        bs.append(np.full(n, g))
        lig = np.zeros(n, dtype=bool)
        lig[n - nl:] = True
        gen = lig.copy()
        if gen_mode == 'partial':
            gen[n - nl: n - nl + (2 * nl) // 3] = False
        ligs.append(lig)
        gens.append(gen)
    cat = lambda a, dt: torch.from_numpy(np.concatenate(a, 0).astype(dt))
    return (cat(xs, np.float32), cat(os_, np.float32), cat(hs, np.float32), cat(bs, np.int64), cat(ligs, bool), cat(gens, bool))


# ---- D3FG sampler -----------------------------------------------------------------------------------------------------------
# schedule tables (betas ... Y) and the fixed angular-encoding frequencies are not weights
D3FG_SKIP = ('pos_scheduler.', 'rot_scheduler.', 'type_scheduler.', 'context_embedder.residue_emb.dihed_embed.')


def d3fg_config(num_steps=1000, hidden=256, num_layers=9, num_fgtype=28):
    """configs/denovo/train/d3fg_fg.yml:1-28 (+ num_fgtype: fg_only mode, configuration.py:6-10, 65).  The encoder type
    is spelled 'ipatransformer', the name the reference's factory accepts (both spellings build the same module here)."""
    return Cfg(dict(
        type='difffg', num_fgtype=num_fgtype,
        encoder=dict(type='ipatransformer', node_feat_dim=hidden, n_heads=16, num_layers=num_layers),
        generator=dict(pos_schedule=dict(type='sigmoid', beta_start=1.e-7, beta_end=2.e-3),
                       rot_schedule=dict(type='cosine', cosine_s=0.01), fg_schedule=dict(type='cosine', cosine_s=0.01),
                       num_diffusion_timesteps=num_steps, time_sampler='symmetric'),
        embedder=dict(type='fg', emb_dim=hidden, fg=dict(type='linear'), residue=dict(type='frame'))))


def _random_so3vec(rs, n):
    """so3 vectors of rotations uniform on SO(3) (unit quaternions from normalised Gaussians)."""
    q = rs.normal(size=(n, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    q[q[:, 0] < 0] *= -1
    v = q[:, 1:]
    s = np.linalg.norm(v, axis=1, keepdims=True)
    theta = 2 * np.arctan2(s[:, 0], q[:, 0])
    return v / np.maximum(s, 1e-12) * theta[:, None]


def make_fg_batch(n_res, n_fg, seed=2024, gen_mode='denovo', num_fgtype=28):
    """Flat D3FG sampling batch with the reference's keys (difffg.py:175-197): per graph ``n_res`` residues with
    non-degenerate N / CA / C backbones (15 heavy-atom slots, side chains of random length), ragged chains with gaps in
    the residue numbering, and ``n_fg`` functional groups with Gaussian centres, random types and orientations uniform
    on SO(3).  gen_mode 'partial': the first third of every graph's FGs is fixed context (no ligand_gen_flag)."""
    rs = np.random.RandomState(seed)
    n_res, n_fg = list(n_res), list(n_fg)
    assert len(n_res) == len(n_fg)
    keys = ('pp', 'pm', 'aa', 'rnb', 'cnb', 'nch', 'lp', 'lo', 'lt', 'gen', 'bl', 'br')
    acc = {k: [] for k in keys}
    for g, (nr, nf) in enumerate(zip(n_res, n_fg)):
        ca = np.cumsum(rs.normal(0.0, 2.2, size=(nr, 3)), axis=0)
        ca -= ca.mean(0, keepdims=True)
        pos = np.zeros((nr, 15, 3))
        mask = np.zeros((nr, 15), dtype=bool)
        for d, length in ((0, 1.46), (2, 1.52), (3, 2.4)):          # N, C, O around CA
            u = rs.normal(size=(nr, 3))
            pos[:, d] = ca + length * u / np.linalg.norm(u, axis=1, keepdims=True)
        pos[:, 1] = ca
        mask[:, :4] = True
        n_side = rs.randint(0, 11, size=nr)
        for r in range(nr):
            pos[r, 4:4 + n_side[r]] = ca[r] + rs.normal(0.0, 1.5, size=(n_side[r], 3))
            mask[r, 4:4 + n_side[r]] = True
        acc['pp'].append(pos)
        acc['pm'].append(mask)
        acc['aa'].append(rs.randint(0, 20, size=nr))
        acc['rnb'].append(1 + np.cumsum(rs.choice([1, 1, 1, 1, 2], size=nr)))
        chains = 2 if nr >= 8 and g % 2 == 0 else 1
        acc['cnb'].append((np.arange(nr) >= nr // 2).astype(np.int64) if chains == 2 else np.zeros(nr, dtype=np.int64))
        acc['nch'].append([chains])
        lp = np.zeros((nf, 15, 3))
        lp[:, 1] = rs.normal(0.0, 1.0, size=(nf, 3))
        acc['lp'].append(lp)
        acc['lo'].append(_random_so3vec(rs, nf))
        acc['lt'].append(rs.randint(0, num_fgtype, size=nf))
        gflag = np.ones(nf, dtype=bool)
        if gen_mode == 'partial':
            gflag[: nf // 3] = False
        acc['gen'].append(gflag)
        acc['bl'].append(np.full(nf, g))
        acc['br'].append(np.full(nr, g))
    cat = lambda k, dt: torch.from_numpy(np.concatenate(acc[k], 0).astype(dt))
    n_l, n_p = int(sum(n_fg)), int(sum(n_res))
    batch = {
        'ligand_pos_heavyatom': cat('lp', np.float32), 'ligand_o_fg': cat('lo', np.float32),
        'ligand_type_fg': cat('lt', np.int64),
        'protein_pos_heavyatom': cat('pp', np.float32), 'protein_mask_heavyatom': cat('pm', np.bool_),
        'protein_aa': cat('aa', np.int64), 'protein_type_fg': cat('aa', np.int64),      # fg_only: type_fg = aa (_base.py:17-27)
        'protein_res_nb': cat('rnb', np.int64), 'protein_chain_nb': cat('cnb', np.int64),
        'protein_num_chains': cat('nch', np.int64),
        'ligand_lig_flag': torch.ones(n_l, dtype=torch.bool), 'protein_lig_flag': torch.zeros(n_p, dtype=torch.bool),
        'ligand_type_fg_batch': cat('bl', np.int64), 'protein_type_fg_batch': cat('br', np.int64),
    }
    if gen_mode == 'partial':
        batch['ligand_gen_flag'] = cat('gen', np.bool_)
    return batch


def make_d3fg_noise(num_steps, n_fg, num_classes=28, seed=7):
    """Injected draws of one D3FG.sample call: positions N(0,1) [T,n,3]; rotation {'dir': N(0,1) [T,n,3], 'bin_u' /
    'in_u': U[0,1) [T,n], 'gauss': N(0,1) [T,n]}; Gumbel uniforms U[0,1) [T,n,K]."""
    rs = np.random.RandomState(seed)
    f = lambda a: torch.from_numpy(a.astype(np.float32))
    pos = f(rs.normal(size=(num_steps, n_fg, 3)))
    rot = {'dir': f(rs.normal(size=(num_steps, n_fg, 3))), 'bin_u': f(rs.random_sample(size=(num_steps, n_fg))),
           'in_u': f(rs.random_sample(size=(num_steps, n_fg))), 'gauss': f(rs.normal(size=(num_steps, n_fg)))}
    return pos, rot, f(rs.random_sample(size=(num_steps, n_fg, num_classes)))


# (name, residues per graph, FGs per graph, data seed, gen mode); T = 20, hidden 256, 9 layers, 28 classes
D3FG_CASES = [
    ('denovo_ragged', [46, 30, 21], [7, 5, 4], 41, 'denovo'),
    ('partial', [38, 26], [6, 6], 42, 'partial'),
    ('below_k', [15], [4], 43, 'denovo'),                 # 19 nodes: fewer than k + 1 = 33
]
D3FG_STEPS, D3FG_WEIGHT_SEED, D3FG_NOISE_SEED = 20, 6, 8
