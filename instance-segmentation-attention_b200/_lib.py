"""ctypes binding of libisa_sm100.so (the C-ABI declared in include/isa_b200.h).

There is no fallback: if the library is missing or a call fails, the op raises.
Mirrors the reference's lazily-loaded native module idiom
(/root/reference/code/lib/archs/modules/sru/sru_functional.py:13-37).
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libisa_sm100.so")

_lock = threading.Lock()
_lib = None

c_void_p = ctypes.c_void_p
c_int = ctypes.c_int
c_float = ctypes.c_float
c_size_t = ctypes.c_size_t
c_uint64 = ctypes.c_uint64
c_double = ctypes.c_double
c_longlong = ctypes.c_longlong

# name -> (restype, argtypes); kept in the order of include/isa_b200.h
SIGNATURES = {
    "isa_last_error": (ctypes.c_char_p, []),
    "isa_version": (c_int, []),
    "isa_num_sms": (c_int, [ctypes.POINTER(c_int)]),
    "isa_selftest_fma_rate": (c_int, [c_int, c_int, c_float, c_void_p, ctypes.POINTER(c_float)]),
    "isa_selftest_tmem_ld_rate": (c_int, [c_int, c_int, c_float, c_void_p, ctypes.POINTER(c_float)]),
    "isa_selftest_grid_barrier": (c_int, [c_int, c_int, c_int, c_int, c_void_p, ctypes.POINTER(c_float)]),
    # discriminative loss
    "isa_disc_loss_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int, c_int]),
    "isa_disc_loss_plan": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int, ctypes.POINTER(c_int)]),
    "isa_disc_loss_fwd": (c_int, [c_void_p, c_void_p, c_int, c_void_p,
                                  c_int, c_int, c_int, c_int, c_int,
                                  c_float, c_float, c_int, c_int,
                                  c_float, c_float, c_float, c_float,
                                  c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_size_t, c_void_p]),
    "isa_disc_loss_bwd": (c_int, [c_void_p, c_void_p, c_int, c_void_p,
                                  c_int, c_int, c_int, c_int, c_int,
                                  c_float, c_float, c_int, c_int,
                                  c_float, c_float, c_float, c_float,
                                  c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_onehot_to_labels": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int,
                                     c_void_p, c_void_p, c_void_p, c_void_p]),
    "isa_label_fg_count": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_void_p]),
    # clustering
    "isa_kmeans_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "isa_kmeans_fit": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_double,
                               c_int, c_void_p, c_void_p,
                               c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_size_t, c_void_p]),
    "isa_fg_compact_workspace_bytes": (c_size_t, [c_int]),
    "isa_fg_compact": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                               c_void_p, c_void_p, c_void_p, c_void_p,
                               c_void_p, c_size_t, c_void_p]),
    "isa_scatter_labels_upsample": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                            c_void_p, c_void_p, c_void_p, c_void_p]),
    # dense attention
    "isa_attention_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "isa_attention_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float,
                                  c_void_p, c_void_p, c_int, c_float, c_uint64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_attention_probs": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float,
                                    c_void_p, c_void_p, c_int, c_float, c_uint64, c_void_p, c_void_p]),
    "isa_attention_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                  c_int, c_int, c_int, c_int, c_int, c_float,
                                  c_void_p, c_void_p, c_int, c_float, c_uint64,
                                  c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    # ReNet GRU scan
    "isa_gru_scan_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                 c_int, c_longlong, c_longlong, c_longlong,
                                 c_void_p, c_void_p, c_void_p]),
    "isa_gru_scan_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                 c_int, c_longlong, c_longlong, c_longlong,
                                 c_void_p, c_void_p, c_void_p]),
    # masked spatial softmaxes, SE primitives, readout, local attention
    "isa_masked_softmax_hw_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "isa_masked_softmax_hw_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int,
                                          c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_masked_softmax_hw_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                          c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_row_dot_workspace_bytes": (c_size_t, [c_int, c_int]),
    "isa_row_dot": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_row_affine": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "isa_mask_bn_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "isa_mask_bn_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_float,
                                c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_mask_bn_bwd": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_float, c_int, c_int, c_int,
                                c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_readout_fwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "isa_readout_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "isa_local_attention_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                        c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "isa_local_attention_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                        c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "isa_bias_act_workspace_bytes": (c_size_t, [c_int]),
    "isa_bias_act_fwd": (c_int, [c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p]),
    "isa_bias_act_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "isa_add_layernorm_workspace_bytes": (c_size_t, [c_longlong, c_int]),
    "isa_add_layernorm_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "isa_add_layernorm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_int,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_pixel_heads_fwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int,
                                    c_longlong, c_int, c_void_p]),
    "isa_pixel_heads_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int,
                                    c_longlong, c_int, c_void_p]),
    "isa_pixel_heads_wgrad_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "isa_pixel_heads_wgrad": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_longlong, c_int,
                                      c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_maxpool2x2_fwd": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "isa_maxpool2x2_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_longlong, c_void_p, c_void_p]),
    # instance-count tail
    "isa_count_head_workspace_bytes": (c_size_t, [c_int, c_longlong, c_int]),
    "isa_count_head_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_int, c_int,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_count_head_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_longlong, c_int, c_int,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_adadelta_workspace_bytes": (c_size_t, []),
    "isa_adadelta_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_float, c_float, c_float, c_float, c_float,
                                  c_void_p, c_void_p, c_size_t, c_void_p]),
    # ReNet projection GEMMs
    "isa_renet_proj_workspace_bytes": (c_size_t, [c_int, c_int]),
    "isa_renet_proj_fwd": (c_int, [c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_renet_proj_dx": (c_int, [c_void_p, c_void_p, c_longlong, c_int, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_renet_proj_wgrad_workspace_bytes": (c_size_t, [c_longlong, c_int, c_int]),
    "isa_renet_proj_wgrad": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_int, c_longlong, c_int, c_int,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    # fused semantic-head losses
    "isa_seg_losses_workspace_bytes": (c_size_t, [c_int, c_int, c_longlong]),
    "isa_seg_losses_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_longlong, c_int, c_float, c_int,
                                   c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_seg_losses_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_longlong, c_int, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_size_t, c_void_p]),
    "isa_onehot_argmax": (c_int, [c_void_p, c_int, c_int, c_int, c_longlong, c_void_p, c_void_p]),
    # evaluation
    "isa_sbd_workspace_bytes": (c_size_t, [c_int]),
    "isa_sbd": (c_int, [c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_size_t, c_void_p]),
}


class IsaError(RuntimeError):
    pass


# kernels launched per C-ABI call (memsets and copies not counted); used by bench.py's gpu_launches
KERNELS_PER_CALL = {
    "isa_disc_loss_fwd": 2, "isa_disc_loss_bwd": 2, "isa_onehot_to_labels": 1, "isa_label_fg_count": 1,
    "isa_kmeans_fit": 5, "isa_fg_compact": 3, "isa_scatter_labels_upsample": 3,
    "isa_attention_fwd": 2, "isa_attention_probs": 1, "isa_attention_bwd": 3,
    "isa_gru_scan_fwd": 1, "isa_gru_scan_bwd": 1,
    "isa_masked_softmax_hw_fwd": 2, "isa_masked_softmax_hw_bwd": 3, "isa_row_dot": 2, "isa_row_affine": 1,
    "isa_mask_bn_fwd": 5, "isa_mask_bn_bwd": 2,
    "isa_readout_fwd": 1, "isa_readout_bwd": 1, "isa_local_attention_fwd": 1, "isa_local_attention_bwd": 2,
    "isa_bias_act_fwd": 1, "isa_bias_act_bwd": 2, "isa_add_layernorm_fwd": 1, "isa_add_layernorm_bwd": 2,
    "isa_pixel_heads_fwd": 1, "isa_pixel_heads_bwd": 1, "isa_pixel_heads_wgrad": 2,
    "isa_maxpool2x2_fwd": 1, "isa_maxpool2x2_bwd": 1, "isa_count_head_fwd": 2, "isa_count_head_bwd": 1, "isa_adadelta_step": 2,
    "isa_renet_proj_fwd": 2, "isa_renet_proj_dx": 2, "isa_renet_proj_wgrad": 2,
    "isa_seg_losses_fwd": 1, "isa_seg_losses_bwd": 1, "isa_onehot_argmax": 1, "isa_sbd": 2,
}


class CallTimer(object):
    """Opt-in per-entry-point timing with CUDA events recorded on the launching stream (the stream the
    kernels are enqueued on); used by bench.py for the roofline numbers.  Off by default: zero overhead."""

    def __init__(self):
        self.enabled = False
        self.records = {}   # name -> list of (start_event, end_event, meta)
        self.counts = {}

    def reset(self):
        self.records = {}
        self.counts = {}

    def summary(self):
        """-> {name: (n_calls, total_ms)}; synchronises."""
        import torch
        torch.cuda.synchronize()
        out = {}
        for name, evs in self.records.items():
            out[name] = (len(evs), sum(s.elapsed_time(e) for s, e, _ in evs))
        return out


TIMER = CallTimer()


class _TimedFn(object):
    def __init__(self, name, fn):
        self.name, self.fn = name, fn

    def __call__(self, *args):
        if not TIMER.enabled or self.name not in KERNELS_PER_CALL:
            return self.fn(*args)
        import torch
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        stream = torch.cuda.current_stream()
        s.record(stream)
        rc = self.fn(*args)
        e.record(stream)
        TIMER.records.setdefault(self.name, []).append((s, e, None))
        TIMER.counts[self.name] = TIMER.counts.get(self.name, 0) + 1
        return rc


class _LibProxy(object):
    def __init__(self, lib):
        self._lib = lib
        for name in SIGNATURES:
            setattr(self, name, _TimedFn(name, getattr(lib, name)))


def load():
    """Loads the shared library once; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise IsaError(
                "libisa_sm100.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `python instance-segmentation-attention_b200/build.py`. There is no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        _lib = _LibProxy(lib)
    return _lib


def check(rc, what):
    if rc != 0:
        msg = load().isa_last_error()
        raise IsaError("%s failed (rc=%d): %s" % (what, rc, msg.decode() if msg else "?"))


def ptr(t):
    """Device (or host) address of a contiguous torch tensor, or NULL for None."""
    if t is None:
        return None
    assert t.is_contiguous(), "tensor handed to the C-ABI must be contiguous"
    return t.data_ptr()


def stream_ptr(device=None):
    import torch
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t, name):
    if not t.is_cuda:
        raise IsaError("%s must be a CUDA tensor: the sm_100a kernels have no CPU fallback" % name)
