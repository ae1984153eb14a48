"""ctypes binding of libxvb200.so (C ABI: include/xvb200.h).  No fallback: if the shared library
is missing or a call fails, an exception is raised."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libxvb200.so")

RELU, BN, SIGMOID, TANH = 1, 2, 4, 8


class TdnnArgs(C.Structure):
    """xvb_tdnn_args_t (include/xvb200.h)."""
    _fields_ = [("x_hi", C.c_void_p), ("x_lo", C.c_void_p), ("ldx", C.c_int64),
                ("x2_hi", C.c_void_p), ("x2_lo", C.c_void_p), ("ldx2", C.c_int64),
                ("w_hi", C.c_void_p), ("w_lo", C.c_void_p),
                ("bias", C.c_void_p), ("bn_scale", C.c_void_p), ("bn_shift", C.c_void_p),
                ("row_bias", C.c_void_p), ("utt_bias", C.c_void_p), ("ld_utt_bias", C.c_int64),
                ("flags", C.c_int), ("context_host", C.POINTER(C.c_int)), ("ntaps", C.c_int),
                ("y_hi", C.c_void_p), ("y_lo", C.c_void_p), ("ldy", C.c_int64),
                ("y_f32", C.c_void_p), ("ldyf", C.c_int64),
                ("B", C.c_int), ("T", C.c_int), ("Cin", C.c_int), ("Cout", C.c_int),
                ("pool_partial", C.c_void_p), ("x_batch_stride", C.c_int64), ("lengths", C.c_void_p)]
MAX_TAPS = 16


class XvbError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "asv_subtools_b200: native library {} not found -- build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (make -C asv_subtools_b200/csrc). "
            "There is no Python/CPU fallback.".format(LIB_PATH))
    return C.CDLL(LIB_PATH)


lib = _load()

_p = C.c_void_p
_i = C.c_int
_i64 = C.c_int64
_f = C.c_float
_ip = C.POINTER(C.c_int)

# name -> (restype, argtypes); every symbol declared in include/xvb200.h must appear here
SIGNATURES = {
    "xvb_version": (_i, []),
    "xvb_last_error": (C.c_char_p, []),
    "xvb_device_check": (_i, []),
    "xvb_split_f32": (_i, [_p, _i64, _i, _i64, _p, _p, _i64, _p]),
    "xvb_packed_weight_elems": (_i64, [_i, _i, _i]),
    "xvb_pack_tdnn_weight": (_i, [_p, _i, _i, _i, _i, _ip, _i, _p, _p, _p]),
    "xvb_tdnn_affine": (_i, [_p, _p, _i64, _p, _p, _p, _p, _p, _i, _ip, _i, _p, _p, _i64, _p, _i64, _i, _i, _i, _i, _p]),
    "xvb_tdnn_affine_simt": (_i, [_p, _i64, _p, _i, _i, _p, _p, _p, _i, _ip, _i, _p, _i64, _i, _i, _i, _i, _p]),
    "xvb_stats_pool": (_i, [_p, _i64, _i, _i, _i, _f, _p, _p, _p, _i64, _p]),
    "xvb_stats_pool_ex": (_i, [_p, _i64, _i, _i, _i, _f, _i, _p, _p, _p, _i64, _p]),
    "xvb_tdnn_affine_ex": (_i, [_p, _p]),
    "xvb_split_frames": (_i, [_p, _i, _i, _i, _p, _p, _i64, _i, _i, _p]),
    "xvb_pool_partial_blocks": (_i, [_i, _i, _ip]),
    "xvb_pool_finalize": (_i, [_p, _i, _i, _i, _i, _i, _f, _i, _p, _p, _p, _i64, _p]),
    "xvb_extractor_set_fused_pooling": (_i, [_p, _i]),
    "xvb_plane_mean": (_i, [_p, _p, _i64, _i, _i, _i, _p, _p, _p, _i64, _p]),
    "xvb_res2net_block": (_i, [_p, _p, _i64, _p, _p, _p, _p, _p, _i, _i, _p, _p, _i64, _i, _i, _p]),
    "xvb_copy_rows": (_i, [_p, _i64, _p, _i64, _i64, _i64, _p]),
    "xvb_se_apply": (_i, [_p, _p, _i64, _p, _p, _i64, _p, _p, _p, _i64, _p, _p, _i64, _i, _i, _i, _p]),
    "xvb_attn_stats_pool": (_i, [_p, _i64, _p, _i64, _i, _i, _i, _f, _p, _p, _p, _i64, _p]),
    "xvb_vad_energy": (_i, [_p, _p, _i, _i, _f, _f, _i, _f, _p, _p, _p]),
    "xvb_cmn": (_i, [_p, _p, _i, _i, _i, _p, _p]),
    "xvb_select_frames": (_i, [_p, _p, _p, _p, _i, _i, _p, _p]),
    "xvb_center_length_norm": (_i, [_p, _p, _p, _i64, _i, _p]),
    "xvb_column_mean": (_i, [_p, _i64, _i, _p, _p]),
    "xvb_cosine_trials": (_i, [_p, _p, _i, _p, _p, _i64, _p, _p]),
    "xvb_speaker_mean": (_i, [_p, _i, _p, _p, _i, _p, _p]),
    "xvb_ipc_alloc": (_i, [_p, C.c_size_t]),
    "xvb_ipc_free": (_i, [_p]),
    "xvb_ipc_export": (_i, [_p, _p]),
    "xvb_ipc_open": (_i, [_p, _p]),
    "xvb_ipc_close": (_i, [_p]),
    "xvb_scatter_rows": (_i, [_p, _i64, _i, _p, _i, _i64, _i64, _p]),
    "xvb_extractor_set_gather": (_i, [_p, _p, _i, _i64, _i64]),
    "xvb_ecapa_set_gather": (_i, [_p, _p, _i, _i64, _i64]),
    "xvb_lde_pool": (_i, [_p, _i64, _i, _i, _i, _p, _i, _p, _p, _p, _p, _p, _i64, _p]),
    "xvb_small_affine": (_i, [_p, _i64, _p, _i, _i, _i, _p, _p, _p, _i, _p, _i64, _p, _p, _i64, _p]),
    "xvb_attn_head_stats_pool": (_i, [_p, _i64, _i, _p, _i64, _i, _i, _i, _i, _i, _f, _i, _p, _p, _p, _i64, _p]),
    "xvb_attn_head_stats_pool_prior": (_i, [_p, _i64, _i, _p, _i64, _i, _i, _i, _i, _i, _f, _i, _p, _p, _i, _p, _p, _p, _i64, _p]),
    "xvb_topn_mean_std": (_i, [_p, _i64, _i64, _i, _i, _p, _p, _p]),
    "xvb_topn_mean_std_ddof": (_i, [_p, _i64, _i64, _i, _i, _i, _p, _p, _p]),
    "xvb_snorm_trials": (_i, [_p, _p, _p, _i64, _p, _p, _p, _p, _p, _p]),
    "xvb_bilinear_trials": (_i, [_p, _p, _i, _p, _p, _i64, _p, _p, _p, _p]),
    "xvb_project": (_i, [_p, _i64, _i, _p, _i, _p, _p]),
    "xvb_cosine_matrix": (_i, [_p, _i64, _p, _i64, _i, _p, _i64, _p]),
    "xvb_plda_terms": (_i, [_p, _i64, _i, _p, _p, _p, _p]),
    "xvb_plda_matrix": (_i, [_p, _i64, _p, _i64, _i, _p, _p, _p, _p, _i64, _p]),
    "xvb_topn_indices": (_i, [_p, _i64, _i64, _i, _i, _p, _p]),
    "xvb_snorm_cross_trials": (_i, [_p, _p, _p, _i64, _p, _i64, _p, _i64, _p, _p, _i, _p, _p]),
    "xvb_matmul_nt": (_i, [_p, _i64, _p, _i64, _i, _p, _p, _p, _i64, _p]),
    "xvb_center_rows_transposed": (_i, [_p, _p, _p, _p, _i64, _i, _p, _i64, _p]),
    "xvb_plda_em_rows": (_i, [_p, _p, _p, _p, _i, _i, _p, _p, _i64, _p]),
    "xvb_plda_normalize_rows": (_i, [_p, _p, _p, _i64, _i, _i, _p]),
    "xvb_plda_llr_operands": (_i, [_p, _p, _p, _i64, _i, _i, _p, _p, _p]),
    "xvb_trial_histogram": (_i, [_p, _i64, _p, _p, _i64, _p, _i, _p, _p, _i, _i, _i, _f, _f, _i, _p, _p]),
    "xvb_extractor_create": (_i, [C.POINTER(_p), _i]),
    "xvb_extractor_add_frame_layer": (_i, [_p, _i, _ip, _i, _p, _p, _p, _p, _i]),
    "xvb_extractor_add_segment_layer": (_i, [_p, _i, _p, _p, _p, _p, _i]),
    "xvb_extractor_finalize": (_i, [_p, _f]),
    "xvb_extractor_embed_dim": (_i, [_p]),
    "xvb_extractor_extract": (_i, [_p, _p, _i, _i, _p, _p]),
    "xvb_extractor_extract_host": (_i, [_p, _p, _i, _i, _p, _p]),
    "xvb_extractor_submit_host": (_i, [_p, _p, _i, _i, _p, _i, _p]),
    "xvb_extractor_wait": (_i, [_p, _i]),
    "xvb_extractor_extract_shard": (_i, [_p, _p, C.c_int64, _i, _i, _p, _p]),
    "xvb_extractor_extract_shard_host": (_i, [_p, _p, C.c_int64, _i, _i, _p, _p]),
    "xvb_extractor_extract_ragged": (_i, [_p, _p, _p, _i, _p, _p]),
    "xvb_extractor_extract_ragged_shard_host": (_i, [_p, _p, _p, _i64, _i, _i64, _p, _p]),
    "xvb_ragged_plan": (_i, [_p, _i64, _i, _i64, _p, _p, _p]),
    "xvb_extractor_set_profiling": (_i, [_p, _i]),
    "xvb_extractor_kernel_times": (_i, [_p, C.POINTER(C.c_float), _i]),
    "xvb_extractor_last_launches": (_i, [_p]),
    "xvb_extractor_debug_f32": (_p, [_p, _i]),
    "xvb_extractor_destroy": (None, [_p]),
    "xvb_fbank_default_opts": (None, [_p]),
    "xvb_fbank_create": (_i, [C.POINTER(_p), _p]),
    "xvb_fbank_dim": (_i, [_p]),
    "xvb_fbank_num_frames": (_i64, [_p, _i64]),
    "xvb_fbank_compute": (_i, [_p, _p, _p, _p, _i, _i64, _p, _p]),
    "xvb_fbank_destroy": (None, [_p]),
    "xvb_ecapa_create": (_i, [C.POINTER(_p), _i, _i, _i, _i, _i]),
    "xvb_ecapa_set_layer": (_i, [_p, C.c_char_p, _i, _i, _ip, _i, _p, _p, _p, _p, _i]),
    "xvb_ecapa_finalize": (_i, [_p]),
    "xvb_ecapa_embed_dim": (_i, [_p]),
    "xvb_ecapa_feat_dim": (_i, [_p]),
    "xvb_ecapa_extract": (_i, [_p, _p, _i, _i, _p, _p]),
    "xvb_ecapa_extract_host": (_i, [_p, _p, _i, _i, _p, _p]),
    "xvb_ecapa_extract_shard": (_i, [_p, _p, C.c_int64, _i, _i, _p, _p]),
    "xvb_ecapa_extract_shard_host": (_i, [_p, _p, C.c_int64, _i, _i, _p, _p]),
    "xvb_ecapa_last_launches": (_i, [_p]),
    "xvb_ecapa_save": (_i, [_p, C.c_char_p]),
    "xvb_ecapa_load": (_i, [C.POINTER(_p), C.c_char_p]),
    "xvb_ecapa_destroy": (None, [_p]),
    "xvb_extractor_load": (_i, [C.POINTER(_p), C.c_char_p]),
    "xvb_extractor_feat_dim": (_i, [C.c_char_p]),
    "xvb_ark_reader_open": (_i, [C.POINTER(_p), C.c_char_p]),
    "xvb_ark_reader_next": (_i, [_p, C.POINTER(C.c_char_p), _ip, _ip, C.POINTER(C.POINTER(C.c_float))]),
    "xvb_ark_reader_close": (None, [_p]),
    "xvb_ark_writer_open": (_i, [C.POINTER(_p), C.c_char_p]),
    "xvb_ark_writer_put_vector": (_i, [_p, C.c_char_p, _p, _i]),
    "xvb_ark_writer_close": (_i, [_p]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here == the .so does not export what the header declares
    _fn.restype = _res
    _fn.argtypes = _args


class FbankOpts(C.Structure):
    """xvb_fbank_opts_t"""
    _fields_ = [(n, C.c_float) for n in ("sample_frequency", "frame_length_ms", "frame_shift_ms", "preemphasis_coefficient",
                                         "low_freq", "high_freq", "energy_floor", "cepstral_lifter", "blackman_coeff")] + \
               [(n, C.c_int) for n in ("num_mel_bins", "num_ceps", "use_energy", "raw_energy", "remove_dc_offset",
                                       "use_log_fbank", "use_power", "htk_compat", "window_type")]


def last_error():
    return lib.xvb_last_error().decode("utf-8", "replace")


def check(rc, what=""):
    if rc != 0:
        raise XvbError("{} failed (rc={}): {}".format(what or "libxvb200 call", rc, last_error()))


def int_array(values):
    arr = (C.c_int * len(values))(*[int(v) for v in values])
    return arr
