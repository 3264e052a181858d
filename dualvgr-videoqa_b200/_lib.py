"""ctypes binding of libdualvgr_b200.so (C ABI: include/dualvgr_b200.h).

The library is the product: if it is missing this module raises at import time — there is no CPU or PyTorch
fallback for any op it exports."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdualvgr_b200.so")


class DvgrError(RuntimeError):
    pass


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(or tools/build_lib.sh). There is no fallback path.")

lib = ctypes.CDLL(LIB_PATH)

c_void_p, c_int, c_ll, c_float = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float


class Operand(ctypes.Structure):
    _fields_ = [("ptr", c_void_p), ("major", c_int), ("ndim", c_int), ("dims", c_ll * 4), ("strides", c_ll * 4)]


class GemmArgs(ctypes.Structure):
    _fields_ = [
        ("A", Operand), ("B", Operand),
        ("M", c_int), ("N", c_int), ("K", c_int), ("batch", c_int),
        ("a_c0", c_int * 4), ("a_c2", c_int * 4), ("a_c3", c_int * 4),
        ("b_c0", c_int * 4), ("b_c2", c_int * 4), ("b_c3", c_int * 4),
        ("k_inner", c_int), ("a_c2_step", c_int * 4), ("b_c2_step", c_int * 4),
        ("C", c_void_p), ("ldc", c_ll), ("c_batch", c_ll),
        ("out_f32", c_int), ("act", c_int), ("beta", c_int),
        ("bias", c_void_p), ("bias_batch", c_ll), ("row_map", c_void_p),
        ("bn", c_int), ("max_ctas", c_int), ("ksplit", c_int), ("tile_counter", c_void_p),
    ]


class LstmArgs(ctypes.Structure):
    _fields_ = [
        ("S", c_int), ("H", c_int), ("T", c_int), ("ndir", c_int), ("s", c_int),
        ("gates", c_void_p), ("whh", c_void_p), ("h_hist", c_void_p), ("c_hist", c_void_p),
        ("h_last", c_void_p), ("h_last_ld", c_ll), ("seq_len", c_void_p),
        ("seq_out", c_void_p), ("seq_out_ld", c_ll),
        ("dc", c_void_p), ("dh_last", c_void_p), ("dh_last_ld", c_ll), ("dh_seq", c_void_p), ("dh_carry", c_void_p),
        ("max_ctas", c_int),
    ]


class LstmSeqArgs(ctypes.Structure):
    _fields_ = [("lstm", LstmArgs), ("x", c_void_p), ("x_ld", c_ll), ("K1", c_int), ("wih", c_void_p), ("wih_ld", c_ll),
                ("bias", c_void_p), ("sync", c_void_p)]


lib.dvgr_last_error.restype = ctypes.c_char_p
lib.dvgr_abi_version.restype = c_int
lib.dvgr_launch_count.restype = c_ll
lib.dvgr_set_seed_offset.argtypes = [c_void_p]
lib.dvgr_set_seed_offset.restype = None


def check(rc, what=""):
    if rc != 0:
        raise DvgrError(f"{what}: {lib.dvgr_last_error().decode()}")


def launch_count():
    return int(lib.dvgr_launch_count())


def _sig(name, argtypes):
    fn = getattr(lib, name)
    fn.argtypes = argtypes
    fn.restype = c_int
    return fn


gemm = _sig("dvgr_gemm", [ctypes.POINTER(GemmArgs), c_void_p])
gemm_reference = _sig("dvgr_gemm_reference",
                      [c_void_p, c_ll, c_ll, c_void_p, c_ll, c_ll, c_void_p, c_ll, c_int, c_int, c_int, c_void_p])
class WgradProblem(ctypes.Structure):
    _fields_ = [("dy", c_void_p), ("ld_dy", c_ll), ("x", c_void_p), ("ld_x", c_ll), ("M", c_int), ("rows", c_int),
                ("cols", c_int), ("out", c_void_p), ("ldc", c_ll)]


wgrad_grouped = _sig("dvgr_wgrad_grouped", [ctypes.POINTER(WgradProblem), c_int, c_void_p])
lstm_step_fwd = _sig("dvgr_lstm_step_fwd", [ctypes.POINTER(LstmArgs), c_void_p])
lstm_step_bwd = _sig("dvgr_lstm_step_bwd", [ctypes.POINTER(LstmArgs), c_void_p])
lstm_seq_fwd = _sig("dvgr_lstm_seq_fwd", [ctypes.POINTER(LstmSeqArgs), c_void_p])
lstm_seq_sync_words = _sig("dvgr_lstm_seq_sync_words", [c_int, c_int])
lstm_seq_bwd = _sig("dvgr_lstm_seq_bwd", [ctypes.POINTER(LstmArgs), c_void_p, c_void_p, c_void_p])


class GatGraph(ctypes.Structure):
    _fields_ = [("wh", c_void_p), ("gate", c_void_p), ("avec", c_void_p), ("out", c_void_p), ("out_f32", c_void_p),
                ("dout", c_void_p), ("dout_f32", c_void_p), ("dwh", c_void_p), ("dgate", c_void_p),
                ("davec", c_void_p), ("drop_stream", ctypes.c_uint)]


class GatArgs(ctypes.Structure):
    _fields_ = [("graphs", GatGraph * 4), ("n_graphs", c_int), ("B", c_int), ("N", c_int), ("D", c_int),
                ("heads", c_int), ("ld_wh", c_ll), ("ld_out", c_ll), ("adj", c_void_p), ("slope", c_float),
                ("p_att", c_float), ("p_out", c_float), ("seed", ctypes.c_ulonglong)]


P = c_void_p
c_ull, c_uint = ctypes.c_ulonglong, ctypes.c_uint
gat_attn_fwd = _sig("dvgr_gat_attn_fwd", [ctypes.POINTER(GatArgs), P])
gat_attn_bwd = _sig("dvgr_gat_attn_bwd", [ctypes.POINTER(GatArgs), P])
qattn_fwd = _sig("dvgr_qattn_fwd", [P, P, P, P, P, c_ll, c_int, c_int, c_int, c_int, P, P, P, P, P, c_ll, P])
qattn_bwd = _sig("dvgr_qattn_bwd", [P, c_ll, P, P, P, P, c_ll, c_int, c_int, c_int, c_int, P, P, P, P, P, P, c_int, P, P, P])
gate_fwd = _sig("dvgr_gate_fwd", [P, P, P, c_ll, c_int, c_int, c_int, P, P, P])
gate_bwd = _sig("dvgr_gate_bwd", [P, P, P, c_ll, c_int, c_int, c_int, P, P, P, P, P, P, P, P, P, P])
view_attn_fwd = _sig("dvgr_view_attn_fwd", [P, P, P, P, c_ll, c_int, P, P, P, P])
view_attn_bwd_blocks = _sig("dvgr_view_attn_bwd_blocks", [c_ll])
view_attn_bwd = _sig("dvgr_view_attn_bwd", [P, P, P, P, P, P, c_ll, c_int, P, P, P, P])
mfb_fwd = _sig("dvgr_mfb_fwd", [P, P, P, c_ll, c_int, P])
mfb_bwd = _sig("dvgr_mfb_bwd", [P, P, P, P, P, c_ll, c_int, P])
readout_fwd = _sig("dvgr_readout_fwd", [P, P, P, P, c_int, c_int, c_int, P, P, c_ll, P])
readout_bwd = _sig("dvgr_readout_bwd", [P, c_ll, P, P, P, P, c_int, c_int, c_int, P, P, P, P, P])
bn_fwd = _sig("dvgr_bn_fwd", [P, c_int, c_int, c_int, P, P, P, P, c_int, c_float, c_float, P, P, P, P])
bn_bwd = _sig("dvgr_bn_bwd", [P, P, c_int, c_int, c_int, P, P, P, c_int, P, P, P, P])
cross_entropy_ex = _sig("dvgr_cross_entropy_ex", [P, P, c_int, c_int, c_float, P, P, c_int, c_ll, P, P])
accuracy_counters = _sig("dvgr_accuracy_counters", [P, P, c_int, c_int, P, P, c_ll, P, c_int, c_int, P, P, P])
bn_stats = _sig("dvgr_bn_stats", [P, c_int, c_int, c_int, P, P])
bn_fwd_ex = _sig("dvgr_bn_fwd_ex", [P, c_int, c_int, c_int, P, P, P, P, c_int, c_float, c_float, P, P, P, P, c_int, P])
bn_bwd_ex = _sig("dvgr_bn_bwd_ex", [P, P, c_int, c_int, c_int, P, P, P, c_int, P, P, P, P, c_int, c_int, P])
cross_entropy = _sig("dvgr_cross_entropy", [P, P, c_int, c_int, c_float, P, P, c_ll, P, P])


class PairJob(ctypes.Structure):
    _fields_ = [("x", c_void_p), ("y", c_void_p), ("dx", c_void_p), ("dy", c_void_p), ("loss_part", c_void_p),
                ("loss_col", c_int), ("loss_ld", c_int), ("mode", c_int), ("accumulate_x", c_int),
                ("accumulate_y", c_int), ("coef", c_float)]


lib.dvgr_pair_loss_workspace.argtypes = [c_int, c_int, c_int, c_int]
lib.dvgr_pair_loss_workspace.restype = c_ll
pair_loss_multi = _sig("dvgr_pair_loss_multi", [ctypes.POINTER(PairJob), c_int, c_int, c_int, c_int, P, P])
lib.dvgr_aux_loss_workspace.argtypes = [c_int, c_int, c_int]
lib.dvgr_aux_loss_workspace.restype = c_ll
aux_loss_unit = _sig("dvgr_aux_loss_unit", [P, P, P, P, c_float, c_float, c_int, c_int, c_int, P, P, P, P, P, P, P])
aux_loss_unit_ex = _sig("dvgr_aux_loss_unit_ex", [P, P, P, P, c_float, c_float, c_int, c_int, c_int, P, P, P, P, P, P, c_int, P])
prep_features = _sig("dvgr_prep_features", [P, P, c_ll, c_int, c_int, c_int, c_int, c_float, c_ull, c_uint, P])
prep_features_ex = _sig("dvgr_prep_features_ex", [P, c_int, P, c_ll, c_int, c_int, c_int, c_int, c_float, c_ull, c_uint, P])
prep_features_gather = _sig("dvgr_prep_features_gather", [P, c_int, c_ll, c_int, P, c_int, P, c_int, c_int, c_int, c_int,
                                                           c_float, c_ull, c_uint, P, P])
cast_rows = _sig("dvgr_cast_rows", [P, c_ll, P, c_ll, c_int, c_int, c_int, c_int, P])
dropout = _sig("dvgr_dropout", [P, P, c_ll, c_float, c_ull, c_uint, P])
act_bwd = _sig("dvgr_act_bwd", [P, P, P, c_ll, c_int, c_int, c_float, c_ull, c_uint, P])
add = _sig("dvgr_add", [P, P, c_ll, P])
PP = ctypes.POINTER(c_void_p)
dropout_multi = _sig("dvgr_dropout_multi", [PP, PP, ctypes.POINTER(c_uint), c_int, c_ll, c_float, c_ull, P])
gat_input_bwd = _sig("dvgr_gat_input_bwd", [PP, ctypes.POINTER(c_uint), c_int, c_int, PP, PP, c_ll, c_float, c_ull, P])
PLL, PI, PF = ctypes.POINTER(c_ll), ctypes.POINTER(c_int), ctypes.POINTER(c_void_p)
cast_rows_grouped = _sig("dvgr_cast_rows_grouped", [PP, PLL, PP, PI, PI, c_int, c_ll, c_int, c_int, P])
lstm_pack_bias = _sig("dvgr_lstm_pack_bias", [PP, PP, c_int, c_int, P, P])
lstm_pack_dh = _sig("dvgr_lstm_pack_dh", [P, c_ll, c_int, P, c_ll, c_int, c_int, c_int, c_int, c_int, P, P, P])
split3 = _sig("dvgr_split3", [P, c_ll, c_int, c_int, P, c_ll, P])
finalize_loss = _sig("dvgr_finalize_loss", [P, P, c_int, PP, c_int, P, P])
embed_fwd = _sig("dvgr_embed_fwd", [P, P, c_int, c_int, c_int, c_int, P, P, c_float, c_ull, c_uint, P])
embed_bwd = _sig("dvgr_embed_bwd", [P, P, P, P, c_int, c_int, c_int, c_int, P, c_float, c_ull, c_uint, P])
view_attn_fwd_multi = _sig("dvgr_view_attn_fwd_multi", [P, P, P, P, c_ll, c_int, c_int, P, P, P, P])
view_attn_bwd_multi = _sig("dvgr_view_attn_bwd_multi", [P, P, P, P, P, P, c_ll, c_int, c_int, P, P, P, P])


class Seg(ctypes.Structure):
    _fields_ = [("dst", c_void_p), ("src", c_void_p), ("n", c_int)]


scatter = _sig("dvgr_scatter", [ctypes.POINTER(Seg), c_int, c_int, P])
lib.dvgr_colsum_workspace.argtypes = [c_ll, c_int]
lib.dvgr_colsum_workspace.restype = c_ll
colsum = _sig("dvgr_colsum", [P, c_int, c_ll, c_ll, c_int, P, P, c_int, c_float, P])
class ColsumProblem(ctypes.Structure):
    _fields_ = [("in_", c_void_p), ("in_is_f32", c_int), ("ld", c_ll), ("R", c_ll), ("C", c_int), ("out", c_void_p),
                ("perm_H", c_int), ("out2", c_void_p)]


colsum_grouped = _sig("dvgr_colsum_grouped", [ctypes.POINTER(ColsumProblem), c_int, P])
colsum_batched = _sig("dvgr_colsum_batched", [P, c_int, c_ll, c_ll, c_ll, c_int, c_int, P, P, c_ll, c_int, c_float, P])
sumsq_blocks = _sig("dvgr_sumsq_blocks", [])
sumsq = _sig("dvgr_sumsq", [P, c_ll, P, P, P])
adam_step = _sig("dvgr_adam_step", [P, P, P, P, c_ll, c_float, c_float, c_float, c_float, c_int, c_float, P, c_float, P, P, P])


class Lstm32Args(ctypes.Structure):
    _fields_ = [("S", c_int), ("H", c_int), ("T", c_int), ("ndir", c_int), ("s", c_int),
                ("gates", c_void_p), ("rec", c_void_p), ("h", c_void_p), ("c_hist", c_void_p), ("h_planes", c_void_p),
                ("hprev_t", c_void_p), ("seq_out", c_void_p), ("seq_out_ld", c_ll), ("h_last", c_void_p), ("h_last_ld", c_ll),
                ("seq_len", c_void_p), ("dh", c_void_p), ("dc", c_void_p), ("dgate_planes", c_void_p),
                ("dh_last", c_void_p), ("dh_last_ld", c_ll), ("dh_seq", c_void_p), ("dh_seq_ld", c_ll), ("dgates", c_void_p)]


lstm32_cell_fwd = _sig("dvgr_lstm32_cell_fwd", [ctypes.POINTER(Lstm32Args), P])
lstm32_cell_bwd = _sig("dvgr_lstm32_cell_bwd", [ctypes.POINTER(Lstm32Args), P])

# fp32-activation variants (fp32 mode, DESIGN.md): the same sources compiled a second time with act_t = float export every
# entry point below under the suffix _f32 with an identical signature (every bf16 activation pointer is a float pointer)
F32_VARIANTS = ["gat_attn_fwd", "gat_attn_bwd", "qattn_fwd", "qattn_bwd", "gate_fwd", "gate_bwd", "view_attn_fwd",
                "view_attn_bwd", "mfb_fwd", "mfb_bwd", "readout_fwd", "readout_bwd", "bn_fwd_ex", "bn_bwd_ex",
                "prep_features_ex", "prep_features_gather", "dropout", "act_bwd", "add", "embed_fwd", "embed_bwd"]
for _n in F32_VARIANTS:
    globals()[_n + "_f32"] = _sig("dvgr_" + _n + "_f32", list(globals()[_n].argtypes))


def variant(name, f32):
    """The entry point `name` for bf16 (f32 False) or fp32 activations."""
    return globals()[name + "_f32"] if f32 else globals()[name]


EXPORTED = [
    "dvgr_last_error", "dvgr_abi_version", "dvgr_launch_count", "dvgr_set_seed_offset", "dvgr_gemm", "dvgr_gemm_reference", "dvgr_wgrad_grouped",
    "dvgr_lstm_step_fwd", "dvgr_lstm_step_bwd", "dvgr_lstm_seq_fwd", "dvgr_lstm_seq_sync_words", "dvgr_lstm_seq_bwd", "dvgr_gat_attn_fwd", "dvgr_gat_attn_bwd", "dvgr_qattn_fwd",
    "dvgr_qattn_bwd", "dvgr_gate_fwd", "dvgr_gate_bwd", "dvgr_view_attn_fwd", "dvgr_view_attn_bwd_blocks",
    "dvgr_view_attn_bwd", "dvgr_mfb_fwd", "dvgr_mfb_bwd", "dvgr_readout_fwd", "dvgr_readout_bwd", "dvgr_bn_fwd",
    "dvgr_bn_bwd", "dvgr_cross_entropy", "dvgr_pair_loss_workspace", "dvgr_pair_loss_multi", "dvgr_aux_loss_workspace", "dvgr_aux_loss_unit", "dvgr_aux_loss_unit_ex", "dvgr_prep_features", "dvgr_prep_features_ex", "dvgr_prep_features_gather", "dvgr_cast_rows", "dvgr_dropout",
    "dvgr_act_bwd", "dvgr_add", "dvgr_scatter", "dvgr_colsum_workspace", "dvgr_colsum", "dvgr_colsum_batched", "dvgr_colsum_grouped", "dvgr_sumsq_blocks", "dvgr_sumsq",
    "dvgr_adam_step", "dvgr_dropout_multi", "dvgr_gat_input_bwd", "dvgr_embed_fwd", "dvgr_embed_bwd",
    "dvgr_view_attn_fwd_multi", "dvgr_view_attn_bwd_multi", "dvgr_cast_rows_grouped", "dvgr_lstm_pack_bias",
    "dvgr_lstm_pack_dh", "dvgr_finalize_loss", "dvgr_bn_stats", "dvgr_bn_fwd_ex", "dvgr_bn_bwd_ex", "dvgr_cross_entropy_ex", "dvgr_accuracy_counters", "dvgr_split3", "dvgr_lstm32_cell_fwd", "dvgr_lstm32_cell_bwd",
] + ["dvgr_" + _n + "_f32" for _n in F32_VARIANTS]
