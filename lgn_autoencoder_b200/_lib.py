"""ctypes binding of liblgae_b200.so (C ABI declared in include/lgae_b200.h).

There is no CPU fallback: every op of this package needs the CUDA library; if it is missing the import of
the product modules fails loudly."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LGAE_B200_LIB") or os.path.join(HERE, "liblgae_b200.so")   # env override: developer A/B builds

MAX_LEVELS = 8
MAX_LINEAR = 12
MAX_CHANNELS = 8

LATENT_MODES = {"mean": 0, "average": 0, "min&max": 1, "min": 2, "max": 3, "sum": 4, "mix": 5}
# CGMLP activations (LGAE_ACT_*): the names of the reference's get_activation_fn table
ACTIVATIONS = {"leakyrelu": 0, "relu": 1, "elu": 2, "sigmoid": 3, "logsigmoid": 4, "tanh": 5, "atan": 6}


class LgaeModelDesc(C.Structure):
    _fields_ = [
        ("is_decoder", C.c_int32),
        ("n_levels", C.c_int32),
        ("n_particles", C.c_int32),
        ("n_basis", C.c_int32),
        ("channels", C.c_int32 * (MAX_LEVELS + 1)),
        ("has_mlp", C.c_int32),
        ("mlp_hidden", C.c_int32),
        ("mlp_width", C.c_int32 * MAX_LEVELS),
        ("latent_mode", C.c_int32),
        ("tau_s", C.c_int32),
        ("tau_v", C.c_int32),
        ("mlp_activation", C.c_int32),
        ("n_params", C.c_int64),
        ("off_in00", C.c_int64),
        ("off_in11", C.c_int64),
        ("off_rad_a", C.c_int64 * MAX_LEVELS),
        ("off_rad_b", C.c_int64 * MAX_LEVELS),
        ("off_rad_c", C.c_int64 * MAX_LEVELS),
        ("off_rad_w0", C.c_int64 * MAX_LEVELS),
        ("off_rad_b0", C.c_int64 * MAX_LEVELS),
        ("off_rad_w1", C.c_int64 * MAX_LEVELS),
        ("off_rad_b1", C.c_int64 * MAX_LEVELS),
        ("off_mix00", C.c_int64 * MAX_LEVELS),
        ("off_mix11", C.c_int64 * MAX_LEVELS),
        ("off_mlp_w", (C.c_int64 * MAX_LINEAR) * MAX_LEVELS),
        ("off_mlp_b", (C.c_int64 * MAX_LINEAR) * MAX_LEVELS),
        ("off_lat00", C.c_int64),
        ("off_lat11", C.c_int64),
        ("off_graph00", C.c_int64),
        ("off_graph11", C.c_int64),
        ("off_out00", C.c_int64),
        ("off_out11", C.c_int64),
        ("input_scale", C.c_double),
        ("maxdim", C.c_int32),   # 0 / 2: maxdim 2; 3: maxdim 3 (forward entry points only)
        ("off_mix20", C.c_int64 * MAX_LEVELS),
        ("off_mix02", C.c_int64 * MAX_LEVELS),
        ("off_mix22", C.c_int64 * MAX_LEVELS),
    ]


CG_MAX_OUT = 16


class LgaeCgPairDesc(C.Structure):
    _fields_ = [
        ("d1", C.c_int32),
        ("d2", C.c_int32),
        ("channels", C.c_int32),
        ("n_out", C.c_int32),
        ("n_comp", C.c_int32),
        ("n_terms", C.c_int32),
        ("out_d", C.c_int32 * CG_MAX_OUT),
        ("out_comp0", C.c_int32 * CG_MAX_OUT),
        ("out_ctotal", C.c_int32 * CG_MAX_OUT),
        ("out_coffset", C.c_int32 * CG_MAX_OUT),
    ]


CG_MAX_PARTS = 8


class LgaeCgMultiDesc(C.Structure):
    _fields_ = [
        ("channels", C.c_int32),
        ("n_node", C.c_int32),
        ("n_edge", C.c_int32),
        ("n_out", C.c_int32),
        ("n_comp", C.c_int32),
        ("n_terms", C.c_int32),
        ("node_d", C.c_int32 * CG_MAX_PARTS),
        ("edge_d", C.c_int32 * CG_MAX_PARTS),
        ("out_d", C.c_int32 * CG_MAX_OUT),
        ("out_ctotal", C.c_int32 * CG_MAX_OUT),
    ]


_P = C.c_void_p
_D = C.POINTER(LgaeModelDesc)
_CG = C.POINTER(LgaeCgPairDesc)

_PROTOS = {
    "lgae_version": (C.c_int, []),
    "lgae_error_string": (C.c_char_p, [C.c_int]),
    "lgae_last_cuda_error": (C.c_char_p, []),
    "lgae_device_sm_count": (C.c_int, []),
    "lgae_launch_count": (C.c_int64, []),
    "lgae_timing_enable": (None, [C.c_int32]),
    "lgae_timing_report": (C.c_int, [C.c_char_p, C.c_int32]),
    "lgae_workspace_doubles": (C.c_int64, [_D, C.c_int32]),
    "lgae_workspace_offset": (C.c_int64, [_D, C.c_int32, C.c_int32, C.c_int32]),
    "lgae_partials_doubles": (C.c_int64, [_D, C.c_int32]),
    "lgae_backward_tiled_scratch_doubles": (C.c_int64, [_D, C.c_int32]),
    "lgae_encoder_forward": (C.c_int, [_D, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P]),
    "lgae_encoder_backward": (C.c_int, [_D, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_double, _P, _P]),
    "lgae_decoder_forward": (C.c_int, [_D, _P, _P, C.c_int32, _P, _P, _P, _P]),
    "lgae_decoder_backward": (C.c_int, [_D, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_double, _P, _P]),
    "lgae_encoder_backward_tiled": (C.c_int, [_D, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_double, _P, _P]),
    "lgae_encoder_backward_p4": (C.c_int, [_D, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_double, _P, _P, _P, _P]),
    "lgae_encoder_backward_tiled_p4": (C.c_int, [_D, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_double, _P, _P, _P, _P]),
    "lgae_encoder_input_grad_scratch_doubles": (C.c_int64, [_D, C.c_int32]),
    "lgae_decoder_backward_tiled": (C.c_int, [_D, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_double, _P, _P]),
    "lgae_train_step_partials_doubles": (C.c_int64, [_D, _D, C.c_int32]),
    "lgae_train_step": (C.c_int, [_D, _D, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, C.c_int64, _P,
                                  C.c_double, C.c_int32, C.c_int32, _P]),
    "lgae_aux_stream": (C.c_void_p, []),
    "lgae_train_step_host": (C.c_int, [_D, _D, _P, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                       C.c_int64, _P, C.c_double, C.c_int32, C.c_int32, _P]),
    "lgae_train_step_tiled_scratch_doubles": (C.c_int64, [_D, _D, C.c_int32]),
    "lgae_train_step_tiled": (C.c_int, [_D, _D, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                        C.c_int64, _P, C.c_double, C.c_int32, C.c_int32, _P]),
    "lgae_train_step_tiled_host": (C.c_int, [_D, _D, _P, _P, _P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                             _P, _P, C.c_int64, _P, C.c_double, C.c_int32, C.c_int32, _P]),
    "lgae_chamfer": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "lgae_anomaly_scores": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "lgae_normalize_p4": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P]),
    "lgae_normalize_p4_backward": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "lgae_chamfer_target_grad": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P]),
    "lgae_l1": (C.c_int, [_P, C.c_int64, C.c_double, _P, _P, _P]),
    "lgae_level_forward": (C.c_int, [_D, C.c_int32, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    "lgae_level_backward": (C.c_int, [_D, C.c_int32, _P, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "lgae_mlp_pack_doubles": (C.c_int64, [_D, C.c_int32]),
    "lgae_mlp_forward": (C.c_int, [_D, C.c_int32, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "lgae_mlp_backward": (C.c_int, [_D, C.c_int32, _P, _P, C.c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "lgae_cg_product_forward": (C.c_int, [_CG, _P, _P, _P, _P, C.c_int64, C.c_int32, _P, _P]),
    "lgae_cg_product_backward": (C.c_int, [_CG, _P, _P, _P, _P, C.c_int64, C.c_int32, _P, _P, _P, C.c_int32, C.c_int32, _P]),
    "lgae_cg_aggregate_multi_forward": (C.c_int, [C.POINTER(LgaeCgMultiDesc), _P, _P, _P, _P, C.c_int64, C.c_int32, _P, _P]),
    "lgae_cg_aggregate_multi_backward": (C.c_int, [C.POINTER(LgaeCgMultiDesc), _P, _P, _P, _P, C.c_int64, C.c_int32, _P, _P, _P, _P]),
    "lgae_mix_partials_doubles": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "lgae_mix_forward": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "lgae_mix_backward": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "lgae_scalar_irrep_forward": (C.c_int, [_P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "lgae_scalar_irrep_backward": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P]),
    "lgae_radial_functions_forward": (C.c_int, [_P, _P, C.c_int64, C.c_int64, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, C.c_int32,
                                                _P]),
    "lgae_radial_functions_partials_doubles": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32, C.c_int32]),
    "lgae_radial_functions_backward": (C.c_int, [_P, _P, C.c_int64, C.c_int64, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, C.c_int32,
                                                 _P, _P, _P, _P]),
    "lgae_linear_forward": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_double, _P, _P]),
    "lgae_linear_partials_doubles": (C.c_int64, [C.c_int64, C.c_int32, C.c_int32]),
    "lgae_linear_backward": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_double, _P, _P, _P, _P, _P]),
    "lgae_peer_signal_bytes": (C.c_int64, []),
    "lgae_peer_allreduce": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int64, _P, _P, _P, _P]),
    "lgae_adam_step": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P, _P, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                 _P, _P]),
    "lgae_rmsprop_step": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P, _P, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double,
                                    C.c_double, _P]),
}

EXPORTED_SYMBOLS = tuple(_PROTOS)

_lib = None


def load():
    """Load the shared library (once) and attach prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: the LGAE B200 kernels are not built. Run `python -m lgn_autoencoder_b200.build` "
            "(needs nvcc); there is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc == 0:
        return
    lib = load()
    msg = lib.lgae_error_string(rc).decode()
    if rc == -3:
        msg += ": " + lib.lgae_last_cuda_error().decode()
    if rc == -2:
        raise NotImplementedError(f"lgae_b200 {what}: {msg}")
    raise RuntimeError(f"lgae_b200 {what}: {msg}")


def ptr(t):
    """Device pointer of a (contiguous) tensor, or NULL."""
    return None if t is None else t.data_ptr()


def kernel_timings(fn, reps: int = 1):
    """Run fn() `reps` times with per-kernel event timing on; returns {kernel name: (launches, mean ms per launch)}."""
    lib = load()
    lib.lgae_timing_enable(1)
    try:
        for _ in range(reps):
            fn()
        buf = C.create_string_buffer(1 << 16)
        n = lib.lgae_timing_report(buf, len(buf))
        if n < 0:
            check(n, "timing_report")
    finally:
        lib.lgae_timing_enable(0)
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.rsplit(" ", 2)
        out[name] = (int(n), float(ms) / int(n))
    return out


def launch_count() -> int:
    return int(load().lgae_launch_count())
