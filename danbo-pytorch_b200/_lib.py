"""ctypes binding of libdanbo_b200.so (include/danbo_b200.h).  No fallback: a missing library raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_PATH = os.path.join(_HERE, "libdanbo_b200.so")
_lib = None
ABI_VERSION = 5          # danbo_version() of the header this binding was written against

c_p = ctypes.c_void_p
c_i = ctypes.c_int
c_f = ctypes.c_float

_SIGNATURES = {
    "danbo_version": [],
    "danbo_nearfar": [c_p, c_i, c_i, c_p, c_i, c_p, c_i, c_i, c_p, c_p, c_i, c_i, c_f, c_f, c_p, c_p, c_p, c_i, c_p, c_p, c_p],
    "danbo_sample_mask": [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_p],
    "danbo_field_agg": [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_p],
    "danbo_agg_frag_bytes": [],
    "danbo_pair_logits_set_blocks": [c_i],
    "danbo_pack_agg_frags": [c_p, c_p, c_p],
    "danbo_ray_bias": [c_p, c_i, c_i, c_p, c_p, c_i, c_p, c_p, c_p, c_p],
    "danbo_mlp_workspace_bytes": [c_p, c_p, c_p],
    "danbo_mlp_set_pack_empty": [c_i],
    "danbo_mlp_empty_rows": [c_p, c_i, c_p, c_p, c_i, c_p],
    "danbo_mlp_set_cta_pair": [c_i],
    "danbo_graph_net_fwd": [c_p, c_i, c_p, c_p, c_p, c_p],
    "danbo_graph_net_bwd": [c_i, c_p, c_p, c_p, c_p, c_p, c_p],
    "danbo_graph_net_bwd_pose": [c_p, c_i, c_p, c_p, c_p, c_p, c_p],
    "danbo_pose_fwd": [c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_i, c_i, c_p, c_p, c_f, c_f, c_f, c_p, c_p, c_p, c_p, c_p],
    "danbo_pose_bwd": [c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_f, c_f, c_p, c_p, c_p,
                       c_p],
    "danbo_pose_kp2d": [c_p, c_p, c_p, c_i, c_f, c_f, c_p, c_p, c_p],
    "danbo_train_loss": [c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_i, c_i, c_i, c_f, c_f, c_p, c_p, c_p, c_p, c_i, c_f, c_p, c_p, c_f,
                         c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "danbo_adam_step": [c_p, c_p, c_p, c_p, ctypes.c_longlong, c_p, c_f, c_f, c_f, c_p, c_i, c_p],
    "danbo_anerf_workspace_bytes": [c_i, c_p, c_p, c_p, c_p],
    "danbo_anerf_pack_weights": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "danbo_anerf_ray_encode": [c_p, c_i, c_i, c_p, c_i, c_i, c_p, c_p, c_i, c_p, c_p, c_p, c_p],
    "danbo_anerf_embed": [c_p, c_i, c_i, c_p, c_i, c_p, c_i, c_i, c_p, c_p, c_f, c_p, c_p, c_p],
    "danbo_anerf_mlp": [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_i, c_i, c_p, c_p],
    "danbo_anerf_save_bytes": [c_i, c_p],
    "danbo_anerf_mlp_save": [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_i, c_i, c_p, c_p],
    "danbo_anerf_untile": [c_p, ctypes.c_longlong, c_i, c_i, c_p, c_p],
    "danbo_anerf_embed_bwd": [c_p, c_i, c_i, c_i, c_p, c_p, c_i, c_i, c_p, c_p, c_f, c_p, c_p, c_p, c_p],
    "danbo_pack_mlp_weights": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "danbo_mlp_forward": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_i, c_i, c_i, c_p],
    "danbo_mlp_forward_trace": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_i, c_i, c_i, c_p, c_p],
    "danbo_mlp_forward_save": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_i, c_i, c_p, c_p, c_i, c_p],
    "danbo_composite_bwd": [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_f, c_p, c_p, c_p, c_p],
    "danbo_merge_composite_bwd": [c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "danbo_mlp_head_bwd": [c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p],
    "danbo_gemm_dgrad": [c_p, c_i, c_i, c_p, c_i, c_p, c_i, c_p, c_i, c_i, c_i, c_i, c_p, c_i, c_p],
    "danbo_gemm_wgrad": [c_p, c_i, c_p, c_i, c_i, c_p, c_i, c_p, c_i, c_i, c_i, c_p],
    "danbo_colsum": [c_p, c_i, c_p, c_p, c_i, c_i, c_p],
    "danbo_ray_bias_bwd": [c_p, c_i, c_i, c_p, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_p],
    "danbo_view_root_bwd": [c_p, c_i, c_i, c_p, c_i, c_i, c_p, c_p, c_p, c_p],
    "danbo_field_agg_bwd": [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_i, c_i, c_p],
    "danbo_field_agg_bwd_pts": [c_p, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_i, c_i, c_p],
    "danbo_mlp_bwd_workspace": [c_i, c_p, c_p, c_p, c_p, c_p, c_p],
    "danbo_pack_mlp_dgrad": [c_p, c_p, c_p, c_p, c_p],
    "danbo_mlp_dgrad": [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_i, c_p, c_p, c_p, c_i, c_p],
    "danbo_mlp_wgrad": [c_p, c_p, c_p, c_i, c_p, c_i, c_p, c_i, c_p, c_p, c_p, c_p, c_p],
    "danbo_composite_resample": [c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_f, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p],
    "danbo_merge_composite": [c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "danbo_merge_composite_parts": [c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_p, c_p, c_p, c_p, c_p,
                                    c_p, c_p, c_p, c_i, c_p, c_p],
}

EXPORTS = tuple(_SIGNATURES)


def path():
    return _PATH


def load():
    """Load the library once; raise loudly if it has not been built (python -m danbo_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_PATH):
            raise RuntimeError(f"{_PATH} is missing: build it with `python __graft_entry__.py build` "
                               "(there is no CPU fallback for the DANBO hot path)")
        lib = ctypes.CDLL(_PATH)
        for name, argtypes in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = argtypes
            fn.restype = ctypes.c_int
        got = lib.danbo_version()
        if got != ABI_VERSION:
            raise RuntimeError(f"{_PATH} has ABI version {got}, this binding expects {ABI_VERSION}: rebuild it with "
                               "`python __graft_entry__.py build`")
        if os.environ.get("DANBO_PAIR_LOGITS_BLOCKS", ""):       # tuning aid: resident blocks per SM of the mma agg net
            lib.danbo_pair_logits_set_blocks(int(os.environ["DANBO_PAIR_LOGITS_BLOCKS"]))
        if os.environ.get("DANBO_MLP_CTA_PAIR", "") == "0":      # debugging aid: single-CTA MLP kernel variant
            lib.danbo_mlp_set_cta_pair(0)
        _lib = lib
    return _lib


def check(code, what):
    if code != 0:
        raise RuntimeError(f"{what} failed with code {code}" + (" (cudaError)" if code > 0 else " (invalid argument)"))
