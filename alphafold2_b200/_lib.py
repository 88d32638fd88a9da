"""ctypes binding of libaf2b200.so (include/af2b200.h).  No torch extension, no pybind: the C ABI is the
drop-in boundary.  There is deliberately NO fallback: if the library is missing or the device is not
sm_100, every op raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# AF2_LIB_PATH: A/B builds of the same library on one box (tools/gpu_ab.sh); never a different implementation
LIB_PATH = os.environ.get("AF2_LIB_PATH") or os.path.join(_HERE, "csrc", "libaf2b200.so")

_lib = None

vp, ll, ci, cf = C.c_void_p, C.c_longlong, C.c_int, C.c_float


class FFWeights(C.Structure):
    _fields_ = [("ln_gamma", vp), ("ln_beta", vp), ("w1", vp), ("b1", vp), ("w2", vp), ("b2", vp), ("bn", ci),
                ("w_cat", vp), ("b_cat", vp), ("w_ext", vp)]


class AttnWeights(C.Structure):
    _fields_ = [("ln_gamma", vp), ("ln_beta", vp), ("w_qkv", vp), ("w_gate", vp), ("b_gate", vp),
                ("w_out", vp), ("b_out", vp), ("w_edge", vp), ("w_cat", vp), ("b_cat", vp), ("w_ext", vp)]


class TriMulWeights(C.Structure):
    _fields_ = [("ln_gamma", vp), ("ln_beta", vp), ("w_left", vp), ("b_left", vp), ("w_right", vp),
                ("b_right", vp), ("w_ogate", vp), ("b_ogate", vp), ("on_gamma", vp), ("on_beta", vp),
                ("w_out", vp), ("b_out", vp), ("bn", ci), ("w_cat", vp), ("b_cat", vp),
                ("w_ext", vp), ("w_ext_out", vp)]


class OuterWeights(C.Structure):
    _fields_ = [("ln_gamma", vp), ("ln_beta", vp), ("w_lr", vp), ("b_lr", vp), ("w_out", vp), ("b_out", vp),
                ("w_cat", vp), ("b_cat", vp), ("w_ext", vp), ("w_ext_out", vp)]


class FFWeightsStrict(C.Structure):
    _fields_ = [("ln_gamma", vp), ("ln_beta", vp), ("w1", vp), ("b1", vp), ("w2", vp), ("b2", vp)]


class AttnWeightsStrict(C.Structure):
    _fields_ = [("ln_gamma", vp), ("ln_beta", vp), ("w_qkvg", vp), ("b_qkvg", vp), ("w_out", vp), ("b_out", vp), ("w_edge", vp)]


class TriMulWeightsStrict(C.Structure):
    _fields_ = [("ln_gamma", vp), ("ln_beta", vp), ("w5", vp), ("b5", vp), ("on_gamma", vp), ("on_beta", vp),
                ("w_out", vp), ("b_out", vp)]


class OuterWeightsStrict(C.Structure):
    _fields_ = [("ln_gamma", vp), ("ln_beta", vp), ("w_lr", vp), ("b_lr", vp), ("w_out", vp), ("b_out", vp)]


_SIGNATURES = {
    "af2_last_error": (C.c_char_p, []),
    "af2_abi_version": (ci, []),
    "af2_check_device": (ci, []),
    "af2_set_proj_mode": (None, [ci]),
    "af2_set_ff_fused": (None, [ci]),
    "af2_debug_proj_trace": (ci, [C.POINTER(C.c_longlong)]),
    "af2_debug_attn_trace": (ci, [C.POINTER(C.c_longlong)]),
    "af2_launch_count": (C.c_ulonglong, []),
    "af2_profile_enable": (None, [ci]),
    "af2_profile_read": (ll, [ci, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "af2_feed_forward": (ci, [C.POINTER(FFWeights), vp, ll, ci, ci, vp, ll, vp]),
    "af2_feed_forward_workspace": (ll, [ll, ci, ci]),
    "af2_axial_attention": (ci, [C.POINTER(AttnWeights), vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, vp, ll, vp]),
    "af2_axial_attention_ex": (ci, [C.POINTER(AttnWeights), vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, ci, vp, ll, vp]),
    "af2_axial_attention_workspace": (ll, [ci, ci, ci, ci, ci, ci, ci]),
    "af2_triangle_multiply": (ci, [C.POINTER(TriMulWeights), vp, vp, ci, ci, ci, ci, vp, ll, vp]),
    "af2_triangle_multiply_workspace": (ll, [ci, ci, ci]),
    "af2_outer_mean": (ci, [C.POINTER(OuterWeights), vp, vp, vp, ci, ci, ci, ci, cf, vp, ll, vp]),
    "af2_outer_mean_workspace": (ll, [ci, ci, ci, ci]),
    "af2_pair_bias": (ci, [vp, vp, vp, ci, ci, ci, ci, vp]),
    "af2_axial_attention_prebias": (ci, [C.POINTER(AttnWeights), vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, vp, ll, vp]),
    "af2_triangle_project": (ci, [C.POINTER(TriMulWeights), vp, vp, ll, ci, ci, vp, vp, ll, vp, vp, ll, vp]),
    "af2_triangle_project_workspace": (ll, [ll, ci]),
    "af2_triangle_contract": (ci, [C.POINTER(TriMulWeights), vp, vp, ll, vp, ll, ll, ci, vp, ci, ci, ci, ci, ci, vp, ll, vp]),
    "af2_triangle_contract_workspace": (ll, [ci, ci, ci]),
    "af2_outer_project": (ci, [C.POINTER(OuterWeights), vp, vp, ll, ci, ci, vp, ll, vp, ll, vp]),
    "af2_outer_project_workspace": (ll, [ll, ci]),
    "af2_outer_contract": (ci, [C.POINTER(OuterWeights), vp, vp, ll, vp, ll, ll, ci, vp, ci, ci, ci, ci, ci, cf, vp, ll, vp]),
    "af2_outer_contract_workspace": (ll, [ci, ci, ci]),
    "af2_rotary": (ci, [vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, vp]),
    "af2_layernorm_bf16": (ci, [vp, vp, vp, vp, ll, ci, cf, vp]),
    "af2_gemm_bf16_f32": (ci, [vp, ll, ll, vp, ll, ll, vp, ll, ll, ci, ci, ci, ci, ci, vp]),
    # strict precision mode (split-bf16 x3 operands)
    "af2_feed_forward_strict": (ci, [C.POINTER(FFWeightsStrict), vp, ll, ci, ci, vp, ll, vp]),
    "af2_feed_forward_strict_workspace": (ll, [ll, ci, ci]),
    "af2_axial_attention_strict": (ci, [C.POINTER(AttnWeightsStrict), vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, ci, vp, ll, vp]),
    "af2_axial_attention_strict_workspace": (ll, [ci, ci, ci, ci, ci, ci, ci]),
    "af2_triangle_multiply_strict": (ci, [C.POINTER(TriMulWeightsStrict), vp, vp, ci, ci, ci, ci, vp, ll, vp]),
    "af2_triangle_multiply_strict_workspace": (ll, [ci, ci, ci]),
    "af2_outer_mean_strict": (ci, [C.POINTER(OuterWeightsStrict), vp, vp, vp, ci, ci, ci, ci, cf, vp, ll, vp]),
    "af2_outer_mean_strict_workspace": (ll, [ci, ci, ci, ci]),
    "af2_embed_pair_init_workspace": (ll, [ci, ci, ci]),
    "af2_embed_pair_init": (ci, [vp, vp, vp, ci, vp, vp, vp, vp, vp, ci, vp, vp, vp, ci, ci, ci, ci, vp, ll, vp]),
    "af2_distogram_head": (ci, [vp, vp, vp, vp, vp, vp, ci, ci, ci, ci, vp]),
    "af2_l2_persist": (ci, [vp, ll, cf, vp]),
    "af2_split_bf16": (ci, [vp, vp, ll, ci, vp]),
    "af2_gemm_split_f32": (ci, [vp, vp, vp, ll, ci, ci, ci, ci, vp]),
    # peer-memory exchange of the sharded trunk
    "af2_peer_ctrl_bytes": (ci, []),
    "af2_peer_can_access": (ci, [ci, ci]),
    "af2_peer_alloc": (ci, [ll, C.POINTER(vp)]),
    "af2_peer_free": (ci, [vp]),
    "af2_peer_export": (ci, [vp, vp]),
    "af2_peer_open": (ci, [vp, C.POINTER(vp)]),
    "af2_peer_close": (ci, [vp]),
    "af2_peer_error": (ci, [vp]),
    "af2_peer_exchange": (ci, [vp, ll, ll, vp, ll, ll, ci, ll, ci, ci, ci, vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def load():
    """Load the shared library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). alphafold2_b200 has no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(code: int):
    if code != 0:
        msg = load().af2_last_error().decode("utf-8", "replace")
        if code == -1:
            raise ValueError(f"af2b200: {msg}")
        raise RuntimeError(f"af2b200 (code {code}): {msg}")
