"""Device-agnostic torch restatement of the reference's D3FG sampling loop (``D3FG.sample`` as written).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Functional style on the reference's own state-dict keys.  Pinned to the
live reference by tests/golden/make_golden_f5.py, which asserts oracle == reference at every state.

Reference code followed (``/root/reference``):
  repo/models/diffusion/difffg.py:174-246                  D3FG.sample (difffg_v2 has the same sample)
  repo/modules/context_emb.py:24-135                       FGContextEmbedder (fg 'linear', residue 'frame', no time emb)
  repo/modules/embs/res_emb.py:16-96                       AngularEncoding, PerResidueEncoder
  repo/models/utils/geometry.py:32-75, 100-119, 271-365   construct_3d_basis, global_to_local, dihedrals
  repo/models/utils/topology.py:5-24                       consecutive / terminus flags
  repo/models/diffusion/diffusion_scheduler.py:144-165     CTNVPScheduler.backward_remove_noise (type='score')
  repo/models/diffusion/diffusion_scheduler.py:558-574     RotVPScheduler.backward_remove_noise
  repo/models/diffusion/diffusion_scheduler.py:367-441     TypeVPScheduler.backward_remove_noise
  repo/models/utils/so3.py:10-146                          log / exp maps, ApproxAngularDistribution.sample

The multinomial draw.  ApproxAngularDistribution.sample draws the histogram bin with torch.multinomial(Y[t, :-1]).
This project defines the draw as an inverse CDF of one uniform u per row (``multinomial_bin``):
    cdf = cumsum(Y[t, :-1].double());   bin = first index with cdf[bin] > (double)u * cdf[-1]
Bins of zero weight are never chosen, so the distribution is torch.multinomial's (the same way oracle/graph_ops.py
defines PyG's semantics); the CUDA kernel searches the same float64 table, so bins are bit-exact.

Random numbers per step, in the reference's order: pos [n,3] (randn_like), rotation axis [n,3] (randn), bin uniform
[n] (replaces multinomial), offset inside the bin [n] (rand_like), Gaussian branch [n] (randn_like), Gumbel [n,K]
(rand_like); all injected here.
"""
import math

import torch
import torch.nn.functional as F

from .diffusion import compose, type_reverse_step
from .diffusion_bp import pos_reverse_step_score
from .ipa import ipatransformer_forward, rotation_to_so3vec, so3vec_to_rotation

N_FG_EMB_EXTRA = 21        # FGContextEmbedder.num_classes = num_fgtype + num_aa_types (21)
N_AA = 20                  # residue_emb input: one_hot(aa, len(aa_name_number))
BB_N, BB_CA, BB_C = 0, 1, 2


def construct_3d_basis(center, p1, p2):
    nrm = lambda v: v / (torch.linalg.norm(v, ord=2, dim=-1, keepdim=True) + 1e-6)
    e1 = nrm(p1 - center)
    v2 = p2 - center
    e2 = nrm(v2 - (e1 * v2).sum(dim=-1, keepdim=True) * e1)
    e3 = torch.cross(e1, e2, dim=-1)
    return torch.stack([e1, e2, e3], dim=-1)


def dihedral(p0, p1, p2, p3):
    v0, v1, v2 = p2 - p1, p0 - p1, p3 - p2
    u1, u2 = torch.cross(v0, v1, dim=-1), torch.cross(v0, v2, dim=-1)
    n1 = u1 / torch.linalg.norm(u1, dim=-1, keepdim=True)
    n2 = u2 / torch.linalg.norm(u2, dim=-1, keepdim=True)
    sgn = torch.sign((torch.cross(v1, v2, dim=-1) * v0).sum(-1))
    return torch.nan_to_num(sgn * torch.acos((n1 * n2).sum(-1).clamp(min=-0.999999, max=0.999999)))


def per_residue_encoder(sd, p, aa, res_nb, chain_nb, pos, mask):
    """PerResidueEncoder.forward (res_emb.py:56-96) over the flat residue list."""
    N = aa.shape[0]
    mask_res = mask[:, BB_CA]
    R = construct_3d_basis(pos[:, BB_CA], pos[:, BB_C], pos[:, BB_N])
    crd = torch.einsum('nji,naj->nai', R, pos - pos[:, BB_CA][:, None])           # R^T (q - t)
    crd = torch.where(mask[:, :, None], crd, torch.zeros_like(crd))
    crd_feat = torch.zeros(N, 22, 15, 3, dtype=pos.dtype, device=pos.device)
    crd_feat[torch.arange(N, device=pos.device), aa] = crd
    consec = ((res_nb[1:] - res_nb[:-1]).abs() == 1) & (chain_nb[1:] == chain_nb[:-1]) & mask_res[:-1]
    n_term = torch.cat([torch.ones(1, dtype=torch.bool, device=pos.device), ~consec])
    c_term = torch.cat([~consec, torch.ones(1, dtype=torch.bool, device=pos.device)])
    pN, pCA, pC = pos[:, BB_N], pos[:, BB_CA], pos[:, BB_C]
    z = torch.zeros(1, dtype=pos.dtype, device=pos.device)
    omega = torch.cat([z, dihedral(pCA[:-1], pC[:-1], pN[1:], pCA[1:])])
    phi = torch.cat([z, dihedral(pC[:-1], pN[1:], pCA[1:], pC[1:])])
    psi = torch.cat([dihedral(pN[:-1], pCA[:-1], pC[:-1], pN[1:]), z])
    dmask = torch.stack([~n_term, ~n_term, ~c_term], dim=-1)
    ang = (torch.stack([omega, phi, psi], dim=-1) * dmask)[:, :, None]                 # [N, 3, 1]
    fb = sd[p + 'dihed_embed.freq_bands']
    code = torch.cat([ang, torch.sin(ang * fb), torch.cos(ang * fb)], dim=-1)         # [N, 3, 13]
    feat = torch.cat([sd[p + 'aatype_embed.weight'][aa], crd_feat.reshape(N, -1), (code * dmask[:, :, None]).reshape(N, -1)], -1)
    for i in (0, 2, 4):
        feat = F.relu(F.linear(feat, sd[p + f'mlp.{i}.weight'], sd[p + f'mlp.{i}.bias']))
    out = F.linear(feat, sd[p + 'mlp.6.weight'], sd[p + 'mlp.6.bias'])
    return out * mask_res[:, None]


def chain_offsets(batch):
    """difffg.py:188-192: chain ids made distinct across graphs (graphs are contiguous)."""
    br = batch['protein_type_fg_batch']
    return batch['protein_chain_nb'] + batch['protein_num_chains'].cumsum(0)[br] - 1


def fg_context(sd, batch, c_lig, num_fgtype, prefix='context_embedder.'):
    """FGContextEmbedder.forward -> (o_rec, h_lig, h_rec)."""
    lin = lambda name, x: F.linear(x, sd[prefix + name + '.weight'], sd[prefix + name + '.bias'])
    K_emb = num_fgtype + N_FG_EMB_EXTRA
    x_rec = batch['protein_pos_heavyatom']
    o_rec = rotation_to_so3vec(construct_3d_basis(x_rec[:, BB_CA], x_rec[:, BB_C], x_rec[:, BB_N]))
    h_lig = lin('ligand_fg_emb', F.one_hot(c_lig.argmax(-1), num_classes=K_emb).float())       # re-one-hot, :95-102
    h_rec = lin('protein_fg_emb', F.one_hot(batch['protein_type_fg'], num_classes=K_emb).float())
    aa = F.one_hot(batch['protein_aa'], num_classes=N_AA).float().argmax(-1)
    h_aa = per_residue_encoder(sd, prefix + 'residue_emb.', aa, batch['protein_res_nb'], chain_offsets(batch), x_rec,
                               batch['protein_mask_heavyatom'])
    h_lig = h_lig + lin('ligand_indicator', batch['ligand_lig_flag'].float().unsqueeze(-1))
    h_rec = h_rec + h_aa + lin('ligand_indicator', batch['protein_lig_flag'].float().unsqueeze(-1))
    return o_rec, h_lig, h_rec


def inverse_cdf(sd, prefix='rot_scheduler.angular_distrib_inv.'):
    return torch.cumsum(sd[prefix + 'Y'][:, :-1].double(), dim=1)


def multinomial_bin(cdf_rows, u):
    """The project's definition of torch.multinomial(prob, 1): first bin with cdf > u * total (float64)."""
    target = u.double() * cdf_rows[:, -1]
    idx = torch.searchsorted(cdf_rows, target[:, None], right=True).squeeze(-1)
    return idx.clamp(max=cdf_rows.shape[1] - 1)


def rot_reverse_step(sd, o_pred, o_t, t_idx, gen_flag, rot_dir, bin_u, in_u, gauss, cdf=None,
                     prefix='rot_scheduler.angular_distrib_inv.'):
    """RotVPScheduler.backward_remove_noise with random_normal_so3 / ApproxAngularDistribution.sample.
    Returns (o_next, bin index per row)."""
    n = o_pred.shape[0]
    cdf = inverse_cdf(sd, prefix) if cdf is None else cdf
    u = F.normalize(rot_dir, dim=-1)
    b = multinomial_bin(cdf[t_idx].expand(n, -1).contiguous(), bin_u)
    X = sd[prefix + 'X'][t_idx]
    samples_hist = X[b] + in_u * (X[b + 1] - X[b])
    sd_t = sd[prefix + 'stddevs'][t_idx].expand(n)
    samples_gauss = (sd_t * 2 + gauss * sd_t).abs() % math.pi
    theta = torch.where(sd[prefix + 'approx_flag'][t_idx].expand(n), samples_gauss, samples_hist)
    e = u * theta[:, None]
    if not t_idx > 1:
        e = torch.zeros_like(e)
    o_next = rotation_to_so3vec(so3vec_to_rotation(e) @ so3vec_to_rotation(o_pred))
    return torch.where(gen_flag[:, None].expand_as(o_next), o_next, o_t), b


def denoise(sd, batch, x_lig, c_lig, o_lig, num_fgtype, k=32):
    """context embedder -> compose -> IPATransformer; ligand rows of (eps_pos, o_pred, logits)."""
    lig_flag, rec_flag = batch['ligand_lig_flag'], batch['protein_lig_flag']
    gen_lig = batch.get('ligand_gen_flag', lig_flag)
    gen_rec = batch.get('protein_gen_flag', torch.zeros_like(rec_flag))
    o_rec, h_lig, h_rec = fg_context(sd, batch, c_lig, num_fgtype)
    sort_idx, batch_idx, _ = compose(batch['ligand_type_fg_batch'], batch['protein_type_fg_batch'])
    cat = lambda r, l: torch.cat([r, l], 0)[sort_idx]
    x = cat(batch['protein_pos_heavyatom'][:, BB_CA], x_lig)
    lig = cat(rec_flag, lig_flag)
    eps, _, o_next, _, logits = ipatransformer_forward(sd, x, cat(o_rec, o_lig), cat(h_rec, h_lig), batch_idx, lig,
                                                       cat(gen_rec, gen_lig), prefix='denoiser.', k=k)
    return eps[lig], o_next[lig], logits[lig]


def sample(sd, batch, num_steps, pos_noise, rot_noise, type_uniform, num_fgtype=28, k=32, stop_after=None):
    """D3FG.sample with injected noise.  Returns traj t -> (x, c, o) with keys T-1 ... -1."""
    x = batch['ligand_pos_heavyatom'][:, BB_CA].float()
    c = F.one_hot(batch['ligand_type_fg'], num_classes=num_fgtype).float()
    o = batch['ligand_o_fg'].float()
    gen = batch.get('ligand_gen_flag', batch['ligand_lig_flag'])
    cdf = inverse_cdf(sd)
    traj = {num_steps - 1: (x, c, o)}
    for done, t in enumerate(reversed(range(num_steps))):
        x, c, o = traj[t]
        eps, o_pred, logits = denoise(sd, batch, x, c, o, num_fgtype, k=k)
        x_next = pos_reverse_step_score(sd, eps, x, t, gen, pos_noise[t])
        o_next, _ = rot_reverse_step(sd, o_pred, o, t, gen, rot_noise['dir'][t], rot_noise['bin_u'][t],
                                     rot_noise['in_u'][t], rot_noise['gauss'][t], cdf=cdf)
        c_next, _ = type_reverse_step(sd, logits, c, t, gen, type_uniform[t], num_fgtype)
        traj[t - 1] = (x_next, c_next, o_next)
        if stop_after is not None and done + 1 >= stop_after:
            break
    return traj
