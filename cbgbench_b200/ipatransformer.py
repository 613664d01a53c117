"""Host-side mirror of the D3FG encoder ``IPATransformer`` (SURVEY.md section 8 row f4), backed by libcbg_b200.so.

Drop-in target: /root/reference repo/modules/e3nn/itatransformer.py:14-145 (factory ``get_e3_gnn`` with
``cfg.type == 'ipatransformer'``, repo/modules/e3nn/__init__.py:15; the shipped config names it 'itatransformer',
configs/denovo/train/d3fg_fg.yml:4, which the reference factory rejects - both spellings are accepted here).
Same constructor argument, same ``forward(x, o, h, batch_idx, lig_flag, gen_flag) -> (eps_pos, h, o_next, R_next, c)``
signature, same state-dict keys.  The sub-modules only hold parameters; the arithmetic runs in csrc/ipa.cu
(``cbg_ipa_forward_f32``) - there is no PyTorch fallback.
"""
import math

import torch
from torch import nn

from . import _lib
from .modules import (GaussianSmearing, MLP, ShiftedSoftplus, _NoTorchPath, _Workspace, cfg_get, graph_ptr_from_batch,
                      N_HEADS, N_RBF)

MAX_CLASSES = 32      # CBG_IPA_MAXCLS (csrc/cbg_kernels.cuh): D3FG's fg_only mode has 28 FG types


class X2HAttentionW(_NoTorchPath):
    """Parameters of x2h_attention.py:8-41 at hidden width ``hidden`` (ew_net_type='global', out_fc=False)."""

    def __init__(self, hidden, edge_feat_dim=4, num_r_gaussian=N_RBF):
        super().__init__()
        kv_in = hidden * 2 + edge_feat_dim + num_r_gaussian * 4
        self.distance_expansion = GaussianSmearing(num_r_gaussian)
        self.hk_func = MLP(kv_in, hidden, hidden)
        self.hv_func = MLP(kv_in, hidden, hidden)
        self.hq_func = MLP(hidden, hidden, hidden)


class InvAttentionLayer(_NoTorchPath):
    """itatransformer.py:147-188: num_x2h x X2HAttention, no coordinate update."""

    def __init__(self, hidden, num_x2h=1):
        super().__init__()
        self.x2h_layers = nn.ModuleList([X2HAttentionW(hidden) for _ in range(num_x2h)])


def _field_maps(hidden):
    L = _lib.lib()
    head = {L.cbg_ipa_head_field_name(f).decode(): (L.cbg_ipa_head_field_offset(hidden, f), L.cbg_ipa_head_field_size(hidden, f))
            for f in range(L.cbg_ipa_head_fields())}
    layer = {L.cbg_ipa_layer_field_name(f).decode(): (L.cbg_ipa_layer_field_offset(hidden, f), L.cbg_ipa_layer_field_size(hidden, f))
             for f in range(L.cbg_ipa_layer_fields())}
    return head, layer


def pack_ipa_blob(sd, hidden, num_layers, num_x2h, num_classes):
    """Reference-keyed state dict -> flat fp32 blob: [global block of the denoiser layout (edge gate) | head block |
    num_layers * num_x2h layer blocks] (field table: cbg_ipa_*_field_* of include/cbg_b200.h).  fp64 staging; the first
    Linear of the edge MLPs is split into node planes / RBF / type parts exactly like the 128-wide denoiser
    (modules.py: pack_denoiser_blob); it is NOT centred here (the generic kernels subtract the LayerNorm mean)."""
    L = _lib.lib()
    lay = _lib.blob_layout()
    head_f, layer_f = _field_maps(hidden)
    g0 = lay['global_floats']
    hf, lf = L.cbg_ipa_head_floats(hidden), L.cbg_ipa_layer_floats(hidden)
    n_sub = num_layers * num_x2h
    blob = torch.zeros(g0 + hf + n_sub * lf, dtype=torch.float64)
    t = lambda k: sd[k].detach().to('cpu', torch.float64)

    def put(base, fmap, name, value):
        off, size = fmap[name]
        v = value.reshape(-1)
        assert v.numel() <= size, (name, v.numel(), size)
        blob[base + off: base + off + v.numel()] = v

    def rbf_field(offset_buf, extra=None):
        o = offset_buf.detach().to('cpu', torch.float64)
        v = torch.zeros(32, dtype=torch.float64)
        v[:N_RBF] = o
        v[20] = -0.5 / float(o[1] - o[0]) ** 2
        if extra is not None:
            v[21] = extra
        return v

    g = lay['global']
    put(0, g, 'GATE_W0T', t('dist_emb.1.net.0.weight').t().contiguous())
    put(0, g, 'GATE_B0', t('dist_emb.1.net.0.bias'))
    put(0, g, 'GATE_LN', torch.cat([t('dist_emb.1.net.1.weight'), t('dist_emb.1.net.1.bias')]))
    put(0, g, 'GATE_W1', t('dist_emb.1.net.3.weight').reshape(-1))
    put(0, g, 'GATE_RBF', rbf_field(sd['dist_emb.0.offset'], float(sd['dist_emb.1.net.3.bias'].reshape(-1)[0])))
    for tag, net in (('ROT', 'eps_rot_net'), ('CRD', 'eps_crd_net')):
        put(g0, head_f, f'{tag}_W0T', t(f'{net}.0.weight').t().contiguous())
        put(g0, head_f, f'{tag}_B0', t(f'{net}.0.bias'))
        put(g0, head_f, f'{tag}_W1T', t(f'{net}.2.weight').t().contiguous())
        put(g0, head_f, f'{tag}_B1', t(f'{net}.2.bias'))
        put(g0, head_f, f'{tag}_W2', t(f'{net}.4.weight'))
        put(g0, head_f, f'{tag}_B2', t(f'{net}.4.bias'))
    put(g0, head_f, 'CLS_W0T', t('classifier.0.weight').t().contiguous())
    put(g0, head_f, 'CLS_B0', t('classifier.0.bias'))
    assert t('classifier.2.weight').shape == (num_classes, hidden) and num_classes <= MAX_CLASSES
    put(g0, head_f, 'CLS_W1', t('classifier.2.weight'))
    put(g0, head_f, 'CLS_B1', t('classifier.2.bias'))
    inv = 1.0 / math.sqrt(hidden // N_HEADS)
    H = hidden
    for l in range(num_layers):
        for s in range(num_x2h):
            base = g0 + hf + (l * num_x2h + s) * lf
            sp = f'blocks.{l}.x2h_layers.{s}.'
            w0k, w0v = t(sp + 'hk_func.net.0.weight'), t(sp + 'hv_func.net.0.weight')       # [H, 4 + 80 + 2H]
            split = lambda w0: (w0[:, 4:84].reshape(H, 4, N_RBF).permute(1, 2, 0).contiguous(),   # Wrf [t][m][f]
                                w0[:, 0:4].t().contiguous(),                                      # c   [t][f]
                                w0[:, 84:84 + H].t().contiguous(),                                # W_i^T [k][n]
                                w0[:, 84 + H:84 + 2 * H].t().contiguous())                        # W_j^T
            wrf_k, c_k, wi_k, wj_k = split(w0k)
            wrf_v, c_v, wi_v, wj_v = split(w0v)
            wq0_t = t(sp + 'hq_func.net.0.weight').t().contiguous()
            put(base, layer_f, 'NODE_WT', torch.cat([wj_k, wj_v, wi_k, wi_v, wq0_t], dim=1))      # [H k][5H n]
            put(base, layer_f, 'NODE_B', torch.cat([torch.zeros(2 * H, dtype=torch.float64), t(sp + 'hk_func.net.0.bias'),
                                                    t(sp + 'hv_func.net.0.bias'), t(sp + 'hq_func.net.0.bias')]))
            put(base, layer_f, 'Q_LN', torch.cat([t(sp + 'hq_func.net.1.weight'), t(sp + 'hq_func.net.1.bias')]))
            put(base, layer_f, 'Q_W1T', (t(sp + 'hq_func.net.3.weight') * inv).t().contiguous())
            put(base, layer_f, 'Q_B1', t(sp + 'hq_func.net.3.bias') * inv)
            put(base, layer_f, 'K_WRF', wrf_k)
            put(base, layer_f, 'K_C', c_k)
            put(base, layer_f, 'K_LN', torch.cat([t(sp + 'hk_func.net.1.weight'), t(sp + 'hk_func.net.1.bias')]))
            put(base, layer_f, 'K_W1T', t(sp + 'hk_func.net.3.weight').t().contiguous())
            put(base, layer_f, 'V_WRF', wrf_v)
            put(base, layer_f, 'V_C', c_v)
            put(base, layer_f, 'V_LN', torch.cat([t(sp + 'hv_func.net.1.weight'), t(sp + 'hv_func.net.1.bias')]))
            put(base, layer_f, 'V_W1T', t(sp + 'hv_func.net.3.weight').t().contiguous())
            put(base, layer_f, 'V_B1', t(sp + 'hv_func.net.3.bias'))
            put(base, layer_f, 'RBF', rbf_field(sd[sp + 'distance_expansion.offset']))
    return blob.to(torch.float32)


class IPATransformerB200(nn.Module):
    """B200 drop-in for the reference's ``IPATransformer`` (itatransformer.py:14-145)."""

    def __init__(self, cfg):
        super().__init__()
        self.cfg = cfg
        self.num_classes = cfg_get(cfg, 'num_classes', None)
        self.num_blocks = cfg_get(cfg, 'num_blocks', 1)
        self.num_layers = cfg_get(cfg, 'num_layers', 6)
        self.hidden_dim = cfg_get(cfg, 'node_feat_dim', 128)
        self.n_heads = cfg_get(cfg, 'n_heads', 16)
        self.cutoff_mode = cfg_get(cfg, 'cutoff_mode', 'knn')
        self.cut_off = int(cfg_get(cfg, 'k', 32))
        self.r_max = float(cfg_get(cfg, 'r_max', 10.0))
        self.num_r_gaussian = cfg_get(cfg, 'num_r_gaussian', 20)
        self.num_x2h = cfg_get(cfg, 'num_x2h', 1)
        unsupported = []
        if self.hidden_dim not in (128, 256):
            unsupported.append('node_feat_dim must be 128 or 256')
        if self.n_heads != N_HEADS:
            unsupported.append('n_heads != 16')
        if cfg_get(cfg, 'ew_type', 'global') != 'global':
            unsupported.append("ew_type != 'global'")
        if cfg_get(cfg, 'act_fn', 'relu') != 'relu' or not cfg_get(cfg, 'norm', True):
            unsupported.append('act_fn/norm')
        if cfg_get(cfg, 'x2h_out_fc', False):
            unsupported.append('x2h_out_fc')
        if cfg_get(cfg, 'dist_emb_type', 'gaussian_exp') != 'gaussian_exp':
            unsupported.append('dist_emb_type')
        if self.cutoff_mode != 'knn':      # the reference's radius branch reads an undefined name (itatransformer.py:89-90)
            unsupported.append(f'cutoff_mode={self.cutoff_mode}')
        if not (1 <= self.cut_off <= 32):
            unsupported.append('k outside [1,32]')
        if self.num_classes is None or not (1 <= self.num_classes <= MAX_CLASSES):
            unsupported.append(f'num_classes must be in [1,{MAX_CLASSES}]')
        if unsupported:
            raise NotImplementedError('IPATransformerB200: unsupported configuration: ' + ', '.join(unsupported))
        H = self.hidden_dim
        self.dist_emb = nn.Sequential(GaussianSmearing(self.num_r_gaussian), MLP(self.num_r_gaussian, 1, self.num_r_gaussian * 8))
        self.blocks = nn.ModuleList([InvAttentionLayer(H, self.num_x2h) for _ in range(self.num_layers)])
        self.classifier = nn.Sequential(nn.Linear(H, H), ShiftedSoftplus(), nn.Linear(H, self.num_classes))
        self.eps_rot_net = nn.Sequential(nn.Linear(H, 2 * H), nn.ReLU(), nn.Linear(2 * H, H), nn.ReLU(), nn.Linear(H, 3))
        self.eps_crd_net = nn.Sequential(nn.Linear(H, 2 * H), nn.ReLU(), nn.Linear(2 * H, H), nn.ReLU(), nn.Linear(H, 3))
        self._blob = None
        self._blob_key = None
        self._ws = _Workspace()

    def packed_blob(self, device):
        key = (str(device),) + tuple((t.data_ptr(), t._version) for t in self.state_dict(keep_vars=True).values())
        if self._blob is None or key != self._blob_key:
            self._blob = pack_ipa_blob(dict(self.state_dict()), self.hidden_dim, self.num_layers, self.num_x2h,
                                       self.num_classes).to(device)
            self._blob_key = key
        return self._blob

    @torch.no_grad()
    def forward(self, x, o, h, batch_idx, lig_flag, gen_flag):
        if not x.is_cuda:
            raise RuntimeError('IPATransformerB200 runs on a CUDA device only (no CPU fallback)')
        dev = x.device
        L = _lib.lib()
        N, H = x.shape[0], self.hidden_dim
        if h.shape != (N, H) or o.shape != (N, 3):
            raise ValueError(f'expected h [{N},{H}] and o [{N},3]')
        x32 = x.detach().to(torch.float32).contiguous()
        o32 = o.detach().to(torch.float32).contiguous()
        h32 = h.detach().to(torch.float32).contiguous()
        gptr, B, max_n = graph_ptr_from_batch(batch_idx)
        lig8 = lig_flag.to(torch.uint8).contiguous()
        gen8 = gen_flag.to(torch.uint8).contiguous()
        blob = self.packed_blob(dev)
        eps_pos = torch.empty((N, 3), dtype=torch.float32, device=dev)
        h_out = torch.empty_like(h32)
        o_next = torch.empty((N, 3), dtype=torch.float32, device=dev)
        r_next = torch.empty((N, 3, 3), dtype=torch.float32, device=dev)
        c = torch.empty((N, self.num_classes), dtype=torch.float32, device=dev)
        ws_ptr, ws_have = self._ws.get(L.cbg_ipa_workspace_bytes(N, H), dev)
        with torch.cuda.device(dev):
            _lib.check(L.cbg_ipa_forward_f32(
                blob.data_ptr(), H, self.num_layers * self.num_x2h, self.num_blocks, self.num_classes,
                x32.data_ptr(), o32.data_ptr(), h32.data_ptr(), gptr.data_ptr(), B, max_n, lig8.data_ptr(), gen8.data_ptr(),
                N, self.cut_off, eps_pos.data_ptr(), h_out.data_ptr(), o_next.data_ptr(), r_next.data_ptr(), c.data_ptr(),
                ws_ptr, ws_have, _lib.stream_ptr(dev)))
        return eps_pos, h_out, o_next, r_next, c
