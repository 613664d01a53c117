"""ctypes binding of libcbg_b200.so (the C-ABI declared in include/cbg_b200.h).

There is no CPU fallback: if the library is missing the import of any compute entry point
raises, and every call with a non-zero return code raises RuntimeError with the library's
message (the reference's error convention is Python exceptions, SURVEY.md section 8b).
"""
import ctypes as C
import os

from .build import LIB_PATH

_lib = None
DEFAULT_EDGE_IMPL = 6      # library default of cbg_set_edge_impl (csrc/edge.cu: g_edge_impl)


class SamplePlan(C.Structure):
    _fields_ = [
        ('blob', C.c_void_p), ('num_layers', C.c_int32), ('num_classes', C.c_int32),
        ('emb_wt', C.c_void_p), ('h_lig_bias', C.c_void_p), ('h_static', C.c_void_p),
        ('graph_ptr', C.c_void_p), ('n_graphs', C.c_int32), ('max_graph_nodes', C.c_int32),
        ('n_nodes', C.c_int64), ('lig_node', C.c_void_p), ('n_lig', C.c_int32),
        ('gen_lig', C.c_void_p), ('gen_node', C.c_void_p), ('n_gen', C.c_int32),
        ('mode', C.c_int32), ('k', C.c_int32), ('r_max', C.c_float),
        ('workspace', C.c_void_p), ('workspace_bytes', C.c_size_t),
        ('rcache', C.c_void_p), ('rcache_bytes', C.c_size_t), ('prune', C.c_int32), ('static_lists', C.c_int32),
    ]


class StepCoef(C.Structure):
    _fields_ = [
        ('pos_c0', C.c_float), ('pos_ct', C.c_float), ('pos_logvar', C.c_float), ('pos_nonzero', C.c_float),
        ('log_alphas_cumprod_prev', C.c_float), ('log_one_minus_alphas_cumprod_prev', C.c_float),
        ('log_alpha', C.c_float), ('log_one_minus_alpha', C.c_float),
    ]


class SbddCoef(C.Structure):
    _fields_ = [('a', C.c_float), ('b', C.c_float), ('s', C.c_float), ('mode', C.c_int32)]


class BpCoef(C.Structure):
    _fields_ = [('alpha_cumprod', C.c_float), ('beta', C.c_float), ('nonzero', C.c_float), ('change_prob', C.c_float)]


class D3fgPlan(C.Structure):
    _fields_ = [
        ('blob', C.c_void_p), ('hidden', C.c_int32), ('num_sublayers', C.c_int32), ('num_blocks', C.c_int32),
        ('num_classes', C.c_int32), ('k', C.c_int32), ('graph_ptr', C.c_void_p), ('n_graphs', C.c_int32),
        ('max_graph_nodes', C.c_int32), ('n_nodes', C.c_int64), ('lig_flag', C.c_void_p), ('gen_flag', C.c_void_p),
        ('lig_node', C.c_void_p), ('n_lig', C.c_int32), ('gen_lig', C.c_void_p), ('fg_wt', C.c_void_p), ('fg_b', C.c_void_p),
        ('lig_bias', C.c_void_p), ('h_static', C.c_void_p), ('x', C.c_void_p), ('o', C.c_void_p), ('rot_cdf', C.c_void_p),
        ('rot_x', C.c_void_p), ('n_bins', C.c_int32), ('workspace', C.c_void_p), ('workspace_bytes', C.c_int64),
    ]


class D3fgCoef(C.Structure):
    _fields_ = [
        ('alpha_cumprod', C.c_float), ('beta', C.c_float), ('pos_nonzero', C.c_float),
        ('rot_stddev', C.c_float), ('rot_approx', C.c_int32), ('rot_nonzero', C.c_float), ('rot_row', C.c_int32),
        ('log_alphas_cumprod_prev', C.c_float), ('log_one_minus_alphas_cumprod_prev', C.c_float),
        ('log_alpha', C.c_float), ('log_one_minus_alpha', C.c_float),
    ]


_P, _I32, _I64, _F, _SZ = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list every symbol of include/cbg_b200.h
SIGNATURES = {
    'cbg_version': (_I32, []),
    'cbg_last_error': (C.c_char_p, []),
    'cbg_launch_count': (_I64, []),
    'cbg_set_edge_impl': (_I32, [_I32, _I32]),
    'cbg_selftest_umma_f16': (_I32, [_P, _P, _P, _I32, _P]),
    'cbg_debug_x2h_trace': (_I32, [_P, _I32]),
    'cbg_debug_node_gemm_trace': (_I32, [_P]),
    'cbg_set_option': (_I32, [C.c_char_p, _I32]),
    'cbg_profile_num_families': (_I32, []),
    'cbg_profile_family_name': (C.c_char_p, [_I32]),
    'cbg_profile_enable': (_I32, [_I32]),
    'cbg_profile_collect': (_I32, [_P, _P]),
    'cbg_blob_global_floats': (_I64, []),
    'cbg_blob_layer_floats': (_I64, []),
    'cbg_blob_num_fields': (_I32, [_I32]),
    'cbg_blob_field_name': (C.c_char_p, [_I32, _I32]),
    'cbg_blob_field_offset': (_I64, [_I32, _I32]),
    'cbg_blob_field_size': (_I64, [_I32, _I32]),
    'cbg_rcache_bytes': (_I64, [_I64, _I32]),
    'cbg_workspace_bytes': (_I64, [_I64, _I64]),
    'cbg_build_neighbors_f32': (_I32, [_P, _P, _I32, _I64, _I32, _I32, _I32, _F, _P, _P, _SZ, _P]),
    'cbg_edge_gate_f32': (_I32, [_P, _P, _P, _I64, _P, _P, _SZ, _P]),
    'cbg_denoiser_forward_f32': (_I32, [_P, _I32, _I32, _P, _P, _P, _I32, _I32, _P, _P, _P, _I32, _P, _I32,
                                        _I64, _I32, _I32, _F, _I32, _P, _P, _P, _P, _SZ, _P]),
    'cbg_denoiser_forward_host_f32': (_I32, [_P, _I64, _I64, _I32, _I32, _P, _P, _P, _I32, _P, _P, _I64,
                                             _I32, _I32, _F, _P, _P, _P]),
    'cbg_node_proj_f32': (_I32, [_P, _I32, _I32, _P, _P, _I32, _I64, _P, _P]),
    'cbg_sample_begin_f32': (_I32, [C.POINTER(SamplePlan), _P, _P, _P, _P]),
    'cbg_sample_prune_counts_host': (_I32, [C.POINTER(SamplePlan), _P, _P]),
    'cbg_sample_step_f32': (_I32, [C.POINTER(SamplePlan), C.POINTER(StepCoef), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'cbg_sample_step_graph_f32': (_I32, [C.POINTER(SamplePlan), C.POINTER(StepCoef), _P, _P, _P, _P, _P, _P, _P, _P]),
    'cbg_sample_step_graph_nodes': (_I64, [C.POINTER(SamplePlan), _P]),
    'cbg_sbdd_step_f32': (_I32, [C.POINTER(SamplePlan), C.POINTER(SbddCoef), _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'cbg_bp_step_f32': (_I32, [C.POINTER(SamplePlan), _P, _I32, C.POINTER(BpCoef), _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'cbg_pocket_stats_f32': (_I32, [_P, _P, _I32, _P, _P, _I32, _P, _P, _P]),
    'cbg_sample_ligand_sizes': (_I32, [_P, _P, _I32, _I32, _P, _P, _P, _P, _P, _P]),
    'cbg_build_batch_f32': (_I32, [_P, _P]),
    'cbg_ipa_head_floats': (_I64, [_I32]),
    'cbg_ipa_layer_floats': (_I64, [_I32]),
    'cbg_ipa_head_fields': (_I32, []),
    'cbg_ipa_layer_fields': (_I32, []),
    'cbg_ipa_head_field_name': (C.c_char_p, [_I32]),
    'cbg_ipa_layer_field_name': (C.c_char_p, [_I32]),
    'cbg_ipa_head_field_offset': (_I64, [_I32, _I32]),
    'cbg_ipa_head_field_size': (_I64, [_I32, _I32]),
    'cbg_ipa_layer_field_offset': (_I64, [_I32, _I32]),
    'cbg_ipa_layer_field_size': (_I64, [_I32, _I32]),
    'cbg_ipa_workspace_bytes': (_I64, [_I64, _I32]),
    'cbg_ipa_forward_f32': (_I32, [_P, _I32, _I32, _I32, _I32, _P, _P, _P, _P, _I32, _I32, _P, _P, _I64, _I32,
                                   _P, _P, _P, _P, _P, _P, _I64, _P]),
    'cbg_d3fg_workspace_bytes': (_I64, [_I64, _I32, _I32]),
    'cbg_d3fg_step_f32': (_I32, [C.POINTER(D3fgPlan), C.POINTER(D3fgCoef)] + [_P] * 17),
    'cbg_d3fg_reverse_f32': (_I32, [C.POINTER(D3fgCoef), _P, _P, _I32] + [_P] * 13 + [_I32, _I32] + [_P] * 6),
    'cbg_reverse_step_f32': (_I32, [C.POINTER(StepCoef), _P, _P, _P, _P, _P, _P, _P, _I32, _I32, _P, _P, _P, _P]),
}


def lib():
    """Load the shared library (once). Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} is missing: build it with `python -m cbgbench_b200.build` '
                '(or __graft_entry__.build()). cbgbench_b200 has no CPU / PyTorch fallback.')
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().cbg_last_error()
        raise RuntimeError(f'cbg_b200 error {rc}: {msg.decode() if msg else "?"}')


def blob_layout():
    """{'global': {name: (offset, size)}, 'layer': {...}, 'global_floats': n, 'layer_floats': n}"""
    L = lib()
    out = {'global_floats': L.cbg_blob_global_floats(), 'layer_floats': L.cbg_blob_layer_floats()}
    for sec, key in ((0, 'global'), (1, 'layer')):
        d = {}
        for i in range(L.cbg_blob_num_fields(sec)):
            d[L.cbg_blob_field_name(sec, i).decode()] = (L.cbg_blob_field_offset(sec, i), L.cbg_blob_field_size(sec, i))
        out[key] = d
    return out


def profile_collect():
    """{family: (total_ms, launches)} since cbg_profile_enable(1); clears the recorded events."""
    L = lib()
    n = L.cbg_profile_num_families()
    ms = (C.c_double * n)()
    cnt = (C.c_int64 * n)()
    check(L.cbg_profile_collect(ms, cnt))
    return {L.cbg_profile_family_name(i).decode(): (ms[i], cnt[i]) for i in range(n)}


def ptr(t):
    """Device/host pointer of a contiguous tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), 'cbg_b200 needs contiguous tensors'
    return t.data_ptr()


def stream_ptr(device):
    import torch
    return torch.cuda.current_stream(device).cuda_stream
