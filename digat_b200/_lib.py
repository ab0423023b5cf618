"""ctypes binding of libdigat_sm100.so (include/digat_sm100.h).  There is no fallback: if the library is missing,
or the device is not sm_100, every compute entry point raises RuntimeError."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('DIGAT_SM100_LIB') or os.path.join(_HERE, 'libdigat_sm100.so')   # (override: kernel experiments)

c_void_p, c_int, c_int64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64

# name -> argument ctypes (all return int).  Must list EVERY symbol declared in include/digat_sm100.h.
SIGNATURES = {
    'digat_abi_version': [],
    'digat_device_check': [c_void_p],
    'digat_linear_f32': [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                         c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    'digat_gemm_f32_small': [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    'digat_split_tf32': [c_void_p, c_void_p, c_void_p, c_int64, c_void_p],
    'digat_linear_tf32x3': [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                            c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    'digat_linear_bf16': [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                          c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p],
    'digat_linear_tf32x3_splitk': [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                   c_int64, c_void_p],
    'digat_debug_set_layer_mode': [c_int],
    'digat_graph_layer_fwd': [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                              c_void_p, ctypes.c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                              c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    'digat_build_graph_csr': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p],
    'digat_gat_layer_fwd': [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
    'digat_graph_layer_supports_row_active': [c_int, c_int, c_int],
    'digat_compact_lists': [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    'digat_news_active_rows': [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p],
    'digat_user_active_rows': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_int,
                               c_void_p],
    'digat_attention_pool_fwd': [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                 c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
    'digat_news_gate_fwd': [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
    'digat_topic_segment_fwd': [c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    'digat_gather_rows_i32': [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p],
    'digat_gather_sag_i32': [c_void_p, c_int64, c_void_p, c_int, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p],
    'digat_build_user_nodes': [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                               c_void_p, c_void_p],
    'digat_graph_layer_bwd': [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, ctypes.c_float, c_void_p,
                              c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p],
    'digat_graph_layer_bwd_csr': [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  ctypes.c_float, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                  c_int, c_void_p],
    'digat_graph_layer_csr_training_supported': [c_int, c_int],
    'digat_graph_layer_bwd_csr_parts': [],
    'digat_gat_layer_train_fwd': [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                  ctypes.c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    'digat_gat_layer_bwd_csr': [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                ctypes.c_float, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p],
    'digat_grad_sumsq': [c_void_p, c_int64, c_void_p, c_void_p, c_void_p],
    'digat_adam_clip_step': [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p] + [ctypes.c_float] * 6
                            + [c_void_p],
    'digat_attention_pool_bwd': [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                 c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
    'digat_news_gate_bwd': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
    'digat_topic_segment_bwd': [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                c_int, c_int, c_int, c_int, c_int, c_void_p],
    'digat_reduce_workspace_floats': [c_int, c_int, c_int, c_void_p],
    'digat_linear_wgrad': [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
    'digat_colsum': [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p],
    'digat_transpose_f32': [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p],
    'digat_groupsum': [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    'digat_logits': [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
    'digat_add_inplace': [c_void_p, c_void_p, c_int64, c_void_p],
    'digat_build_user_graphs': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p],
    'digat_sag_bfs': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                      ctypes.c_double, c_void_p, c_void_p],
    'digat_msa_attention_fwd': [c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_int, c_int, c_void_p],
    'digat_additive_pool_fwd': [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_int,
                                c_void_p],
    'digat_msa_attention_bwd': [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_int, c_int,
                                c_void_p],
    'digat_additive_pool_bwd': [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                c_int, c_void_p, c_int64, c_int, c_int, c_int, c_void_p],
    'digat_scatter_add_rows': [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p],
    'digat_rank_impressions': [c_void_p, c_void_p, c_void_p, c_int64, c_void_p],
    'digat_impression_metrics': [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p],
}

_lib = None
_device_ok = {}


def load():
    """Loads the shared library (no GPU needed) and binds every entry point."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError('libdigat_sm100.so not found at %s -- build it with `python -c "import __graft_entry__ as g; '
                               'g.build()"` (there is no CPU/PyTorch fallback)' % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = c_int
        lib.digat_last_error.argtypes = []
        lib.digat_last_error.restype = ctypes.c_char_p
        _lib = lib
    return _lib


def last_error() -> str:
    return load().digat_last_error().decode(errors='replace')


def require_device(device_index: int):
    """Raises unless the given CUDA device is an sm_100 part (checked once per device)."""
    if _device_ok.get(device_index):
        return
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError('digat_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
    with torch.cuda.device(device_index):
        rc = load().digat_device_check(None)
    if rc != 0:
        raise RuntimeError('digat_device_check failed: ' + last_error())
    _device_ok[device_index] = True


_NON_KERNEL = ('digat_graph_layer_supports_row_active', 'digat_graph_layer_csr_training_supported', 'digat_graph_layer_bwd_csr_parts', 'digat_abi_version', 'digat_device_check', 'digat_debug_set_layer_mode',
               'digat_reduce_workspace_floats')
_launches = 0
_profile = None      # list of (name, args, start_event, end_event) while bench.py's per-kernel pass is running


def reset_launch_count():
    global _launches
    _launches = 0


def launch_count() -> int:
    """Kernel launches issued through the C ABI since the last reset (every compute entry point = 1 launch)."""
    return _launches


def start_profile():
    global _profile
    _profile = []
    return _profile


def stop_profile():
    """-> [(entry point, args, milliseconds)]; call after torch.cuda.synchronize()."""
    global _profile
    rec, _profile = _profile or [], None
    return [(n, a, s.elapsed_time(e)) for (n, a, s, e) in rec]


def call(name, *args):
    global _launches
    if _profile is not None:
        import torch
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        rc = getattr(load(), name)(*args)
        e.record()
        _profile.append((name, args, s, e))
    else:
        rc = getattr(load(), name)(*args)
    if name not in _NON_KERNEL:
        _launches += 1
    if rc != 0:
        raise RuntimeError('%s failed (%d): %s' % (name, rc, last_error()))
