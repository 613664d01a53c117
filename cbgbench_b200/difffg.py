"""B200 drop-in for the reference's ``D3FG`` model (registered as ``difffg`` and ``difffg_v2``), sampling path.

Mirrors /root/reference repo/models/diffusion/difffg.py:32-63 (constructor, sub-module names => state-dict keys) and
:174-246 (``sample(batch) -> traj``); both registered classes have the same ``sample``.  Per step ONE C-ABI call
(``cbg_d3fg_step_f32``): composed ligand FG rows -> IPA encoder (csrc/ipa.cu) -> fused reverse step (position, SO(3)
orientation, FG type; csrc/d3fg.cu).  What does not change over the T steps is computed once per batch by
``FGContextEmbedderB200.static_features``: the residue frames and their so3 vectors, the protein rows of h (FG
embedding + residue-frame encoder + indicator) and the ligand bias row.

Random numbers: per step ``randn_like`` [n,3] (positions), ``randn`` [n,3] (rotation axis), ``rand`` [n] (histogram
bin, see below), ``rand_like`` [n] (offset inside the bin), ``randn_like`` [n] (Gaussian branch), ``rand_like`` [n,K]
(Gumbel), in the reference's order, or injected.  The reference draws the bin with ``torch.multinomial``; here the bin
is the inverse CDF of a uniform (include/cbg_b200.h), so a seeded run is reproducible but is not the reference's random
stream.
"""
import ctypes as C

import torch
from torch import nn
import torch.nn.functional as F

from . import _lib
from .modules import _NoTorchPath, _Workspace, cfg_get, get_e3_gnn, graph_ptr_from_batch
from .schedulers import CTNVPTables, RotVPTables, TypeVPTables
from .targetdiff import register_model

N_AA = 20                 # len(aa_name_number), repo/utils/protein/constants.py:32-41 (input width of residue_emb)
N_AA_TYPES = 21           # num_aa_types = len(AA) incl. UNK (constants.py:45-75)
MAX_AA_TYPES, MAX_ATOMS = 22, 15      # PerResidueEncoder defaults (res_emb.py:42)
BB_N, BB_CA, BB_C = 0, 1, 2           # BBHeavyAtom


# ---- residue frames (geometry.py:32-75, 100-119, 271-288, 327-365; topology.py:5-24) -------------------------------------
def _normalize(v, eps=1e-6):
    return v / (torch.linalg.norm(v, ord=2, dim=-1, keepdim=True) + eps)


def residue_basis(ca, c, n):
    """construct_3d_basis: columns e1 (CA->C), e2 (CA->N orthogonalised), e3 = e1 x e2."""
    e1 = _normalize(c - ca)
    v2 = n - ca
    e2 = _normalize(v2 - (e1 * v2).sum(dim=-1, keepdim=True) * e1)
    e3 = torch.cross(e1, e2, dim=-1)
    return torch.cat([e1.unsqueeze(-1), e2.unsqueeze(-1), e3.unsqueeze(-1)], dim=-1)


def rotation_to_so3vec(R):
    """log map (so3.py:10-31, 60-63), no-grad branch (min_cos = -1)."""
    trace = R[..., range(3), range(3)].sum(-1)
    cos_t = ((trace - 1) / 2).clamp_min(min=-1.0)
    sin_t = torch.sqrt(1 - cos_t ** 2)
    theta = torch.acos(cos_t)
    logR = ((theta + 1e-8) / (2 * sin_t + 2e-8))[..., None, None] * (R - R.transpose(-1, -2))
    return torch.stack([logR[..., 1, 2], logR[..., 2, 0], logR[..., 0, 1]], dim=-1)


def _dihedral(p0, p1, p2, p3):
    v0, v1, v2 = p2 - p1, p0 - p1, p3 - p2
    u1 = torch.cross(v0, v1, dim=-1)
    n1 = u1 / torch.linalg.norm(u1, dim=-1, keepdim=True)
    u2 = torch.cross(v0, v2, dim=-1)
    n2 = u2 / torch.linalg.norm(u2, dim=-1, keepdim=True)
    sgn = torch.sign((torch.cross(v1, v2, dim=-1) * v0).sum(-1))
    return torch.nan_to_num(sgn * torch.acos((n1 * n2).sum(-1).clamp(min=-0.999999, max=0.999999)))


def backbone_dihedrals(pos, chain_nb, res_nb, mask):
    """(omega, phi, psi) [N,3] and their masks over the flat residue list (consecutive = same chain, |d res_nb| = 1)."""
    consec = ((res_nb[1:] - res_nb[:-1]).abs() == 1) & (chain_nb[1:] == chain_nb[:-1]) & mask[:-1]
    n_term = F.pad(~consec, pad=(1, 0), value=1)
    c_term = F.pad(~consec, pad=(0, 1), value=1)
    pN, pCA, pC = pos[:, BB_N], pos[:, BB_CA], pos[:, BB_C]
    omega = F.pad(_dihedral(pCA[:-1], pC[:-1], pN[1:], pCA[1:]), pad=(1, 0), value=0)
    phi = F.pad(_dihedral(pC[:-1], pN[1:], pCA[1:], pC[1:]), pad=(1, 0), value=0)
    psi = F.pad(_dihedral(pN[:-1], pCA[:-1], pC[:-1], pN[1:]), pad=(0, 1), value=0)
    m = torch.stack([~n_term, ~n_term, ~c_term], dim=-1)
    return torch.stack([omega, phi, psi], dim=-1) * m, m


class AngularEncodingW(nn.Module):
    """Buffer of AngularEncoding (res_emb.py:16-37): frequencies 1..3 and 1/1..1/3."""

    def __init__(self, num_funcs=3):
        super().__init__()
        self.register_buffer('freq_bands', torch.tensor([i + 1. for i in range(num_funcs)] +
                                                        [1. / (i + 1) for i in range(num_funcs)], dtype=torch.float32))


class PerResidueEncoderB200(_NoTorchPath):
    """Parameters of PerResidueEncoder (res_emb.py:40-96): aa embedding, local-frame atom coordinates placed by aa type,
    backbone dihedrals, a 4-layer MLP.  ``encode`` is the once-per-batch torch computation of static_features."""

    def __init__(self, feat_dim):
        super().__init__()
        self.aatype_embed = nn.Embedding(MAX_AA_TYPES, feat_dim)
        self.dihed_embed = AngularEncodingW()
        infeat = feat_dim + MAX_AA_TYPES * MAX_ATOMS * 3 + 3 * (1 + 4 * 3)
        self.mlp = nn.Sequential(nn.Linear(infeat, feat_dim * 2), nn.ReLU(), nn.Linear(feat_dim * 2, feat_dim), nn.ReLU(),
                                 nn.Linear(feat_dim, feat_dim), nn.ReLU(), nn.Linear(feat_dim, feat_dim))

    def encode(self, aa, res_nb, chain_nb, pos, mask):
        """PerResidueEncoder.forward in the dtype of ``pos``."""
        N = aa.shape[0]
        mask_res = mask[:, BB_CA]
        R = residue_basis(pos[:, BB_CA], pos[:, BB_C], pos[:, BB_N])
        q = pos.reshape(N, -1, 3).transpose(-1, -2)
        crd = torch.matmul(R.transpose(-1, -2), q - pos[:, BB_CA].unsqueeze(-1)).transpose(-1, -2).reshape(pos.shape)
        crd = torch.where(mask[:, :, None].expand_as(crd), crd, torch.zeros_like(crd))
        place = aa[:, None, None, None] == torch.arange(MAX_AA_TYPES, device=aa.device)[None, :, None, None]
        crd_feat = torch.where(place, crd[:, None].expand(N, MAX_AA_TYPES, MAX_ATOMS, 3), 0.0).reshape(N, -1)
        dih, dmask = backbone_dihedrals(pos, chain_nb, res_nb, mask_res)
        x = dih[:, :, None].unsqueeze(-1)
        fb = self.dihed_embed.freq_bands.to(pos.dtype)
        code = torch.cat([x, torch.sin(x * fb), torch.cos(x * fb)], dim=-1)
        dihed_feat = (code.reshape(N, 3, -1) * dmask[:, :, None]).reshape(N, -1)
        y = torch.cat([self.aatype_embed.weight.to(pos.dtype)[aa], crd_feat, dihed_feat], dim=-1)
        for i, layer in enumerate(self.mlp[::2]):
            y = F.linear(y, layer.weight.to(pos.dtype), layer.bias.to(pos.dtype))
            y = F.relu(y) if i < 3 else y
        return y * mask_res[:, None]


class FGContextEmbedderB200(nn.Module):
    """Parameter container for FGContextEmbedder (context_emb.py:24-135) with fg.type 'linear' and residue.type 'frame'
    (the shipped d3fg configs), no time / vec embedding."""

    def __init__(self, cfg, hidden_dim=None):
        super().__init__()
        self.num_fgtype = cfg_get(cfg, 'num_fgtype', 50)
        self.num_classes = self.num_fgtype + N_AA_TYPES
        self.emb_dim = emb_dim = cfg_get(cfg, 'emb_dim', 128)
        unsupported = []
        if cfg_get(cfg, 'time', None) is not None or cfg_get(cfg, 'vec', None) is not None:
            unsupported.append('time / vec embeddings (no shipped D3FG config uses them)')
        fg, res = cfg_get(cfg, 'fg', None), cfg_get(cfg, 'residue', None)
        if fg is None or cfg_get(fg, 'type') != 'linear':
            unsupported.append("fg.type must be 'linear'")
        if res is None or cfg_get(res, 'type') != 'frame':
            # the reference's 'linear' residue embedder is an nn.Linear, which FGContextEmbedder calls with 5 arguments
            unsupported.append("residue.type must be 'frame'")
        if hidden_dim is not None and emb_dim != hidden_dim:
            unsupported.append(f'emb_dim={emb_dim} must equal the encoder node_feat_dim={hidden_dim}')
        if unsupported:
            raise NotImplementedError('FGContextEmbedderB200: unsupported configuration: ' + ', '.join(unsupported))
        self.ligand_fg_emb = nn.Linear(self.num_classes, emb_dim)
        self.protein_fg_emb = nn.Linear(self.num_classes, emb_dim)
        self.residue_emb = PerResidueEncoderB200(emb_dim)
        self.ligand_indicator = nn.Linear(1, emb_dim)

    @torch.no_grad()
    def static_features(self, x_rec, v_rec, aa_rec, res_nb, chain_nb, mask_atom_rec, rec_flag):
        """The step-invariant part of FGContextEmbedder.forward, once per batch: (o_rec [N_rec,3], h_rec [N_rec,H],
        lig_bias [H] = ligand_indicator(1)).  ``chain_nb`` already carries the per-graph offsets (difffg.py:188-192).
        Computed in float64 and rounded once: the GEMM algorithm the library picks depends on the batch size, and in
        float64 its summation order does not reach the fp32 result, so a pocket gets the same rows alone or in a batch."""
        x64 = x_rec.double()
        lin = lambda m, x: F.linear(x, m.weight.double(), m.bias.double())
        o_rec = rotation_to_so3vec(residue_basis(x64[:, BB_CA], x64[:, BB_C], x64[:, BB_N]))
        h_rec = lin(self.protein_fg_emb, F.one_hot(v_rec, num_classes=self.num_classes).double())
        aa = F.one_hot(aa_rec, num_classes=N_AA).argmax(-1)
        h_aa = self.residue_emb.encode(aa, res_nb, chain_nb, x64, mask_atom_rec)
        # + t_emb_rec: zeros without a time embedding (context_emb.py:92-93)
        h_rec = h_rec + h_aa + lin(self.ligand_indicator, rec_flag.double().unsqueeze(-1))
        lig_bias = self.ligand_indicator(torch.ones(1, 1, device=x_rec.device)).reshape(-1)
        return o_rec.float().contiguous(), h_rec.float().contiguous(), lig_bias.contiguous()


class D3FGB200(nn.Module):
    """B200 drop-in for D3FG (difffg.py:32-246), sampling only."""

    def __init__(self, cfg):
        super().__init__()
        self.cfg = cfg
        gen = cfg.generator
        T = self.num_diffusion_timesteps = gen.num_diffusion_timesteps
        if not (cfg_get(gen, 'denoise_structure', True) and cfg_get(gen, 'denoise_atom', True)):
            raise NotImplementedError('denoise_structure / denoise_atom = False is not implemented')
        self.num_classes = cfg.num_fgtype
        ps, rs, fs = gen.pos_schedule, gen.rot_schedule, gen.fg_schedule
        self.pos_scheduler = CTNVPTables(T, beta_start=ps.beta_start, beta_end=ps.beta_end, type=ps.type)
        self.rot_scheduler = RotVPTables(T, type=rs.type, cosine_s=rs.cosine_s)
        self.type_scheduler = TypeVPTables(T, num_classes=self.num_classes, type=fs.type, cosine_s=fs.cosine_s)
        cfg.embedder.num_fgtype = cfg.num_fgtype
        self.context_embedder = FGContextEmbedderB200(cfg.embedder, hidden_dim=cfg_get(cfg.encoder, 'node_feat_dim', 128))
        self.denoiser = get_e3_gnn(cfg.encoder, num_classes=self.num_classes)
        self._ws = _Workspace()
        self._plan_generation = 0
        self._cdf_key, self._cdf = None, None
        self.last_launches = 0

    def forward(self, batch):
        raise NotImplementedError(f'{type(self).__name__} is a forward-only sampling build: the training / '
                                  'validation losses of the reference models are out of scope (DESIGN.md)')

    def check_state(self, state):
        if state.get('generation') != self._plan_generation:
            raise RuntimeError('stale sampling state: prepare() was called again on this model (its device workspace now '
                               'belongs to the newer batch); finish one batch before preparing the next, or use a second model')

    def rot_tables(self, device):
        """(float64 inverse-CDF table [T, 8191], bin edges [T, 8192]) on ``device``; the CDF is summed on the CPU once
        per set of table values."""
        inv = self.rot_scheduler.angular_distrib_inv
        key = (str(device), inv.Y.data_ptr(), inv.Y._version, inv.X.data_ptr(), inv.X._version)
        if self._cdf_key != key:
            self._cdf = (self.rot_scheduler.inverse_cdf().to(device).contiguous(),
                         inv.X.detach().to(device, torch.float32).contiguous(),
                         inv.stddevs.detach().cpu().tolist(), inv.approx_flag.detach().cpu().tolist())
            self._cdf_key = key
        return self._cdf

    def step_coef(self, t, stddevs, approx):
        ps, ts = self.pos_scheduler, self.type_scheduler
        tm1 = max(t - 1, 0)
        return _lib.D3fgCoef(
            alpha_cumprod=float(ps.host_table('alphas_cumprod')[t]), beta=float(ps.host_table('betas')[t]),
            pos_nonzero=0.0 if t == 0 else 1.0, rot_stddev=stddevs[t], rot_approx=1 if approx[t] else 0,
            rot_nonzero=1.0 if t > 1 else 0.0, rot_row=t,
            log_alphas_cumprod_prev=float(ts.host_table('log_alphas_cumprod_v')[tm1]),
            log_one_minus_alphas_cumprod_prev=float(ts.host_table('log_one_minus_alphas_cumprod_v')[tm1]),
            log_alpha=float(ts.host_table('log_alphas_v')[t]),
            log_one_minus_alpha=float(ts.host_table('log_one_minus_alphas_v')[t]))

    @torch.no_grad()
    def prepare(self, batch, device=None):
        """Move the batch to the device, compute the step-invariant features, compose_context (common.py:189-214) and
        build the plan.  Reads the reference's keys (difffg.py:175-197)."""
        dev = torch.device(device) if device is not None else next(self.parameters()).device
        if dev.type != 'cuda':
            raise RuntimeError(f'{type(self).__name__}.sample needs the model on a CUDA device (no CPU fallback)')
        g = lambda k, d=None: batch.get(k, d) if hasattr(batch, 'get') else (batch[k] if k in batch else d)
        to = lambda t: t.to(dev, non_blocking=True)
        x_lig = to(batch['ligand_pos_heavyatom'][:, BB_CA]).float().contiguous()
        o_lig = to(batch['ligand_o_fg']).float().contiguous()
        v_lig = to(batch['ligand_type_fg']).long()
        x_rec = to(batch['protein_pos_heavyatom']).float()
        lig_flag = to(batch['ligand_lig_flag']).bool()
        rec_flag = to(batch['protein_lig_flag']).bool()
        gl, gr = g('ligand_gen_flag', None), g('protein_gen_flag', None)
        gen_lig = to(gl).bool() if gl is not None else lig_flag
        gen_rec = to(gr).bool() if gr is not None else torch.zeros_like(rec_flag)
        bl = to(batch['ligand_type_fg_batch']).long()
        br = to(batch['protein_type_fg_batch']).long()
        if br.numel() > 1 and not bool((br[1:] >= br[:-1]).all()):
            raise ValueError('protein_type_fg_batch must be sorted')
        chain_nb = to(batch['protein_chain_nb']).long() + to(batch['protein_num_chains']).long().cumsum(0)[br] - 1
        o_rec, h_rec, lig_bias = self.context_embedder.static_features(
            x_rec, to(batch['protein_type_fg']).long(), to(batch['protein_aa']).long(), to(batch['protein_res_nb']).long(),
            chain_nb, to(batch['protein_mask_heavyatom']).bool(), rec_flag)
        n_lig, n_rec = x_lig.shape[0], x_rec.shape[0]
        N, H, K = n_lig + n_rec, self.denoiser.hidden_dim, self.num_classes
        sort_idx = torch.sort(torch.cat([br, bl], 0), stable=True).indices
        inv = torch.empty_like(sort_idx)
        inv[sort_idx] = torch.arange(N, device=dev)
        lig_node = inv[n_rec:].to(torch.int32).contiguous()
        if n_lig > 1 and not bool((lig_node[1:] > lig_node[:-1]).all()):
            raise ValueError('ligand_type_fg_batch must be sorted')
        gptr, B, max_n = graph_ptr_from_batch(torch.cat([br, bl], 0)[sort_idx])
        x_nodes = torch.cat([x_rec[:, BB_CA], x_lig], 0)[sort_idx].contiguous()
        o_nodes = torch.cat([o_rec, o_lig], 0)[sort_idx].contiguous()
        h_static = torch.cat([h_rec, torch.zeros(n_lig, H, device=dev)], 0)[sort_idx].contiguous()
        lig_nodes = torch.cat([rec_flag, lig_flag], 0)[sort_idx].to(torch.uint8).contiguous()
        gen_nodes = torch.cat([gen_rec, gen_lig], 0)[sort_idx].to(torch.uint8).contiguous()
        gen_lig8 = gen_lig.to(torch.uint8).contiguous()
        emb = self.context_embedder.ligand_fg_emb
        fg_wt = emb.weight.detach()[:, :K].t().contiguous().float()
        fg_b = emb.bias.detach().float().contiguous()
        cdf, rot_x, stddevs, approx = self.rot_tables(dev)
        L = _lib.lib()
        ws_ptr, ws_have = self._ws.get(L.cbg_d3fg_workspace_bytes(N, H, K), dev)
        den = self.denoiser
        blob = den.packed_blob(dev)
        plan = _lib.D3fgPlan(
            blob=blob.data_ptr(), hidden=H, num_sublayers=den.num_layers * den.num_x2h, num_blocks=den.num_blocks,
            num_classes=K, k=den.cut_off, graph_ptr=gptr.data_ptr(), n_graphs=B, max_graph_nodes=max_n, n_nodes=N,
            lig_flag=lig_nodes.data_ptr(), gen_flag=gen_nodes.data_ptr(), lig_node=lig_node.data_ptr(), n_lig=n_lig,
            gen_lig=gen_lig8.data_ptr(), fg_wt=fg_wt.data_ptr(), fg_b=fg_b.data_ptr(), lig_bias=lig_bias.data_ptr(),
            h_static=h_static.data_ptr(), x=x_nodes.data_ptr(), o=o_nodes.data_ptr(), rot_cdf=cdf.data_ptr(),
            rot_x=rot_x.data_ptr(), n_bins=cdf.shape[1], workspace=ws_ptr, workspace_bytes=ws_have)
        keep = dict(blob=blob, gptr=gptr, lig_nodes=lig_nodes, gen_nodes=gen_nodes, lig_node=lig_node, gen_lig8=gen_lig8,
                    fg_wt=fg_wt, fg_b=fg_b, lig_bias=lig_bias, h_static=h_static, x_nodes=x_nodes, o_nodes=o_nodes,
                    cdf=cdf, rot_x=rot_x)
        self._plan_generation += 1
        return dict(plan=plan, keep=keep, device=dev, generation=self._plan_generation, x_lig=x_lig, o_lig=o_lig,
                    c_lig=F.one_hot(v_lig, num_classes=K).float().contiguous(), batch_idx_lig=bl, n_lig=n_lig, n_nodes=N,
                    n_graphs=B, stddevs=stddevs, approx=approx)

    @torch.no_grad()
    def run_steps(self, state, t_seq, slots, pos_noise=None, rot_noise=None, type_uniform=None, outs=None):
        """Enqueue the reverse steps ``t_seq`` (descending t): one ``cbg_d3fg_step_f32`` call each.  ``slots(t)`` gives
        the (x, c, o) views of trajectory slot t: slot t+1 is the state entering step t, slot t its result.  ``outs``
        (dict) receives per step the ligand rows of the encoder's eps_pos / logits / o_pred."""
        self.check_state(state)
        dev, n, plan, K = state['device'], state['n_lig'], state['plan'], self.num_classes
        v_scratch = torch.empty(n, dtype=torch.int64, device=dev)
        L = _lib.lib()
        st = _lib.stream_ptr(dev)
        launches0 = L.cbg_launch_count()
        inj = lambda src, t: src[t].to(dev, torch.float32).contiguous()
        with torch.cuda.device(dev):
            for t in t_seq:
                x_t, c_t, o_t = slots(t + 1)
                x_n, c_n, o_n = slots(t)
                if pos_noise is None:
                    pn = torch.randn_like(x_t)
                else:
                    pn = inj(pos_noise, t)
                if rot_noise is None:
                    r_dir = torch.randn((n, 3), device=dev)
                    r_bin = torch.rand((n,), device=dev)
                    r_in = torch.rand_like(r_bin)
                    r_g = torch.randn_like(r_bin)
                else:
                    r_dir, r_bin, r_in, r_g = (inj(rot_noise[k], t) for k in ('dir', 'bin_u', 'in_u', 'gauss'))
                tu = torch.rand_like(c_t) if type_uniform is None else inj(type_uniform, t)
                o3 = None
                if outs is not None:
                    o3 = outs[t] = (torch.empty((n, 3), device=dev), torch.empty((n, K), device=dev),
                                    torch.empty((n, 3), device=dev))
                coef = self.step_coef(t, state['stddevs'], state['approx'])
                _lib.check(L.cbg_d3fg_step_f32(
                    C.byref(plan), C.byref(coef), x_t.data_ptr(), c_t.data_ptr(), o_t.data_ptr(), pn.data_ptr(),
                    r_dir.data_ptr(), r_bin.data_ptr(), r_in.data_ptr(), r_g.data_ptr(), tu.data_ptr(), x_n.data_ptr(),
                    c_n.data_ptr(), o_n.data_ptr(), v_scratch.data_ptr(), *([a.data_ptr() for a in o3] if o3 else [None] * 3),
                    st))
        self.last_launches = L.cbg_launch_count() - launches0

    @torch.no_grad()
    def sample(self, batch, pos_noise=None, rot_noise=None, type_uniform=None, num_steps=None, traj_mode='full', outs=None):
        """D3FG.sample (difffg.py:174-246).  Returns ``traj``: {t: (xc_lig [n,3], c_lig [n,K] one-hot, o_lig [n,3],
        batch_idx_lig)} with keys T-1 ... -1; entries >= 0 on the CPU and key -1 on the device like the reference.  The
        reference's per-step D2H copy is replaced by one device trajectory buffer and a single copy at the end.

        ``pos_noise[t]`` [n,3], ``rot_noise`` = {'dir': [T,n,3], 'bin_u', 'in_u', 'gauss': [T,n]} and
        ``type_uniform[t]`` [n,K] inject the random numbers; ``num_steps`` stops early; ``traj_mode='final'`` keeps only
        traj[t_last] and traj[-1]; ``outs`` (dict) receives the encoder outputs per step."""
        T, K = self.num_diffusion_timesteps, self.num_classes
        state = self.prepare(batch)
        dev, n = state['device'], state['n_lig']
        W = n * (6 + K)
        buf = torch.empty((T + 1, W), dtype=torch.float32, device=dev)      # slot: x [n,3] | o [n,3] | c [n,K]

        def split(row):
            return row[:3 * n].view(n, 3), row[6 * n:].view(n, K), row[3 * n:6 * n].view(n, 3)

        x0, c0, o0 = split(buf[T])
        x0.copy_(state['x_lig'])
        c0.copy_(state['c_lig'])
        o0.copy_(state['o_lig'])
        t_seq = list(reversed(range(T)))
        if num_steps is not None:
            t_seq = t_seq[:num_steps]
        self.run_steps(state, t_seq, lambda t: split(buf[t]), pos_noise, rot_noise, type_uniform, outs)
        bl = state['batch_idx_lig']
        t_last = t_seq[-1]
        bl_cpu = bl.cpu()
        traj = {}
        host = buf[t_last + 1:].cpu() if traj_mode == 'full' else buf[t_last + 1:t_last + 2].cpu()
        for t in (range(t_last, T) if traj_mode == 'full' else [t_last]):
            x, c, o = split(host[t - t_last])
            traj[t] = (x, c, o, bl_cpu)
        x, c, o = split(buf[t_last].clone())
        traj[t_last - 1] = (x, c, o, bl)
        return traj


register_model('difffg')(D3FGB200)
register_model('difffg_v2')(D3FGB200)
