"""ctypes binding of the C ABI declared in ``include/fragnet_b200.h``.

The product path has NO CPU fallback: if the library cannot be loaded the import of any module that
needs a kernel fails loudly here.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

_vp, _i64, _i32, _sz, _u64, _f32 = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_uint64, C.c_float

# name -> (restype, argtypes).  Mirrors include/fragnet_b200.h one to one (tests check the export list).
SIGNATURES = {
    "fnb_version": (C.c_int, []),
    "fnb_error_string": (C.c_char_p, [C.c_int]),
    "fnb_launch_count": (_u64, []),
    "fnb_scratch_bytes": (_sz, []),
    "fnb_csr_workspace_bytes": (_sz, [_i64, _i64]),
    "fnb_csr_build": (C.c_int, [_vp, _vp, _i64, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    "fnb_gather_rows": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "fnb_segment_offsets": (C.c_int, [_vp, _i64, _i64, _vp, _vp]),
    "fnb_narrow_index": (C.c_int, [_vp, _i64, _vp, _vp]),
    "fnb_proj_fwd": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _i32, _vp]),
    "fnb_proj_bwd": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _i32, _vp, _vp]),
    "fnb_node_scalars": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _i32, _vp, _vp]),
    "fnb_attn_by_source": (C.c_int, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "fnb_segment_sum": (C.c_int, [_vp, _vp, _i64, _vp, _vp, _i64, _vp, _i32, _i32, _i32, _vp, _vp]),
    "fnb_segment_gather": (C.c_int, [_vp, _i64, _vp, _i64, _vp, _vp, _vp]),
    "fnb_dropout_relu_fwd": (C.c_int, [_vp, _vp, _i64, _f32, _i32, _i32, _u64, _u64, _vp]),
    "fnb_dropout_relu_bwd": (C.c_int, [_vp, _vp, _vp, _i64, _f32, _i32, _vp]),
    "fnb_adam_step": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _f32, _i64, _vp]),
    "fnb_widen_batch": (C.c_int, [_vp, _i32, _vp]),
    "fnb_allreduce_adam_step": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _f32, _f32, _f32, _f32, _f32, _i64, C.c_uint32, _vp,
                                          _vp]),
    "fnb_allreduce_adam_runs": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _vp, _i32, _f32, _f32, _f32, _f32, _f32, C.c_uint32,
                                          _vp, _vp]),
    "fnb_gat_fwd_tiled": (C.c_int, [_vp, _vp, _vp]),
    "fnb_gat_bwd_tiled": (C.c_int, [_vp, _vp, _vp]),
    "fnb_gat_bwd_tiled_marked": (C.c_int, [_vp, _vp, _vp, _vp]),
    "fnb_edge_table_bwd_fused": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp]),
    "fnb_batch_plan_bytes": (_sz, [_vp]),
    "fnb_batch_plan_build": (C.c_int, [_vp, _vp, _sz, _vp, _vp]),
    "fnb_encoder_workspace_bytes": (_sz, [_vp, _vp, _vp]),
    "fnb_encoder_bwd_workspace_bytes": (_sz, [_vp, _vp, _vp]),
    "fnb_encoder_rng_span": (_u64, [_vp, _vp, _vp]),
    "fnb_encoder_forward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp]),
    "fnb_encoder_backward": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp, _sz, _vp, _vp]),
    "fnb_pretrain_heads_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "fnb_pretrain_heads_bwd_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "fnb_pretrain_heads_forward": (C.c_int, [_vp, _vp, _i32, _vp, _sz, _vp, _vp]),
    "fnb_pretrain_heads_backward": (C.c_int, [_vp, _vp, _vp, _i32, _vp, _sz, _vp, _sz, _vp, _vp]),
    "fnb_mse_sum_loss": (C.c_int, [_vp, _i32, _vp, _vp, _vp]),
    "fnb_pretrain_step_workspace_bytes": (_sz, [_vp]),
    "fnb_pretrain_step_rng_span": (_u64, [_vp]),
    "fnb_pretrain_step": (C.c_int, [_vp, _vp, _sz, _vp, _vp]),
    "fnb_pretrain_plan_prefetch": (C.c_int, [_vp, _vp, _sz, _vp]),
    "fnb_finetune_step_workspace_bytes": (_sz, [_vp]),
    "fnb_finetune_step_rng_span": (_u64, [_vp]),
    "fnb_finetune_step": (C.c_int, [_vp, _vp, _sz, _vp, _vp]),
    "fnb_arena_workspace_bytes": (_sz, [_i64, _i32]),
    "fnb_arena_assemble": (C.c_int, [_vp, _i64, _i64, _vp, _i32, _vp, _i32, _vp, _sz, _vp, _vp]),
}


# C structs of include/fragnet_b200.h (native alignment, same field order)
class CGraph(C.Structure):
    _fields_ = [("n_nodes", _i64), ("n_edges", _i64), ("n_real_edges", _i64),
                ("rowptr", _vp), ("col", _vp), ("row", _vp), ("eid", _vp), ("slot_of_eid", _vp),
                ("rrowptr", _vp), ("rslot", _vp), ("rdst", _vp), ("edge_attr", _vp)]


class CPostAct(C.Structure):
    _fields_ = [("p", _f32), ("training", _i32), ("relu", _i32), ("seed", _u64), ("offset", _u64)]


class CGatFwdArgs(C.Structure):
    _fields_ = [("h", _vp), ("S", _vp), ("edge_mode", _i32), ("edge_table", _vp), ("We", _vp), ("be", _vp),
                ("alpha_e", _vp), ("alpha_stride", _i32), ("out", _vp), ("y", _vp), ("post", CPostAct),
                ("p_saved", _vp), ("mask_lo", _i64), ("mask_hi", _i64), ("next_alpha_e", _vp),
                ("next_alpha_stride", _i32), ("next_Se", _vp)]


class CGatBwdArgs(C.Structure):
    _fields_ = [("h", _vp), ("dout", _vp), ("p_saved", _vp), ("edge_mode", _i32), ("We", _vp), ("be", _vp),
                ("alpha", _vp), ("alpha_stride", _i32), ("off_t", _i32), ("off_e", _i32), ("off_s", _i32),
                ("dz", _vp), ("dSt", _vp), ("dh", _vp), ("d_alpha", _vp), ("d_bias", _vp), ("dWe", _vp), ("dbe", _vp),
                ("scratch", _vp)]

class CArenaKind(C.Structure):
    _fields_ = [("counts", _vp), ("prefix", _vp)]


class CArenaJob(C.Structure):
    _fields_ = [("src", _vp), ("dst", _vp), ("kind", C.c_int32), ("offset_kind", C.c_int32), ("width", C.c_int32),
                ("mode", C.c_int32)]


class CPeerSet(C.Structure):
    _fields_ = [("grads", _vp * 8), ("flags", _vp * 8), ("world", C.c_int32), ("rank", C.c_int32)]


class CAdamRun(C.Structure):
    _fields_ = [("first", _i64), ("end", _i64), ("step", _i64)]


MAX_ADAM_RUNS = 16


class CWidenJob(C.Structure):
    _fields_ = [("src", _vp), ("dst", _vp), ("n", C.c_int64), ("mode", C.c_int32)]


WIDEN_U8_F32, WIDEN_I32_I64, WIDEN_MAX_JOBS = 0, 1, 16
ARENA_COPY32, ARENA_INDEX, ARENA_FILL = 0, 1, 2
ARENA_MAX_KINDS, ARENA_MAX_JOBS = 24, 32
ABI_VERSION = 13
EDGE_NONE, EDGE_AFFINE1, EDGE_AFFINE6, EDGE_TABLE = 0, 1, 2, 3
PRECISION_FP32, PRECISION_TF32, PRECISION_TF32X3 = 0, 1, 2

_lib = None


def library_path() -> str:
    return _build.LIB_PATH


def load():
    """Load (building first if the in-tree library is missing or stale and nvcc is present)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.LIB_PATH
    if _build.nvcc_path() is not None:
        path = _build.build()
    if not os.path.isfile(path):
        raise RuntimeError(
            f"fragnet_b200: kernel library {path} is missing and nvcc is not available to build it. "
            "There is no CPU fallback; run `python -c 'import __graft_entry__ as g; g.build()'` first.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here == ABI / header mismatch: fail loudly
        fn.restype, fn.argtypes = res, args
    if lib.fnb_version() != ABI_VERSION:
        raise RuntimeError(f"fragnet_b200: ABI version mismatch ({lib.fnb_version()} != {ABI_VERSION})")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().fnb_error_string(rc).decode()
        raise RuntimeError(f"fragnet_b200.{what} failed: {msg} (code {rc})")


PARAM_FIELDS = ("Wb", "bb", "Wfb", "bfb", "We_b", "be_b", "We_fb", "be_fb", "Wa", "ba", "a_b", "a", "f", "f_a_b")


class CLayerParams(C.Structure):
    _fields_ = [(n, _vp) for n in PARAM_FIELDS] + [
        ("K_atom", _i32), ("K_bond", _i32), ("K_fbond", _i32), ("run_frag_block", _i32), ("want_attention", _i32),
        ("bond_mask", _i64), ("frag_bond_mask", _i64), ("atom_mask", _i64), ("atom_mask_list", _vp),
        ("n_atom_mask", _i64), ("bond_mask_rows", _vp), ("n_bond_mask_rows", _i64), ("fbond_mask_rows", _vp),
        ("n_fbond_mask_rows", _i64)]


class CLayerGrads(C.Structure):
    _fields_ = [(n, _vp) for n in PARAM_FIELDS]


class CBatchPlan(C.Structure):
    _fields_ = [("bond", CGraph), ("atom", CGraph), ("fbond", CGraph), ("frag", CGraph),
                ("pool_rowptr", _vp), ("pool_col", _vp), ("a2f", _vp), ("n_atoms", _i64), ("n_frags", _i64),
                ("mol_atom_ptr", _vp), ("mol_frag_ptr", _vp), ("batch32", _vp), ("frag_batch32", _vp),
                ("n_graphs", _i64), ("status", _vp)]


class CBatchInputs(C.Structure):
    _fields_ = [(n, _vp) for n in ("edge_index", "frag_index", "atom_to_frag_ids", "edge_index_bonds_graph",
                                   "edge_index_fbonds", "batch", "frag_batch", "edge_attr_bonds",
                                   "edge_attr_fbonds")] + \
               [(n, _i64) for n in ("n_atoms", "n_frags", "n_bonds", "n_bond_edges", "n_fbond_nodes", "n_fbond_edges",
                                    "n_graphs")]


class CEncoderOpts(C.Structure):
    _fields_ = [("n_layers", _i32), ("post_act", _i32), ("drop_p", _f32), ("training", _i32), ("seed", _u64),
                ("offset", _u64), ("precision", _i32), ("save_for_backward", _i32), ("need_dx_atoms", _i32),
                ("need_dx_bond", _i32), ("need_dx_fbond", _i32), ("first_trained_layer", _i32), ("pool_frags", _i32),
                ("skip_fbond", _i32)]


class CEncoderIO(C.Structure):
    _fields_ = [(n, _vp) for n in ("x_atoms", "x_bond", "x_fbond", "out_atoms", "out_frags", "out_bond", "out_fbond",
                                   "attn_atoms", "attn_frags", "attn_bonds", "attn_fbonds", "g_atoms", "g_frags",
                                   "g_bond", "g_fbond", "dx_atoms", "dx_bond", "dx_fbond", "frag_table",
                                   "d_frag_table")]


MLP3_FIELDS = ("W0", "b0", "W1", "b1", "W2", "b2")


class CMlp3(C.Structure):          # fnb_mlp3_params and fnb_mlp3_grads share one layout
    _fields_ = [(n, _vp) for n in MLP3_FIELDS]


class CPretrainHeadParams(C.Structure):   # fnb_pretrain_head_params / fnb_pretrain_head_grads
    _fields_ = [("Wr", _vp), ("br", _vp), ("bl", CMlp3), ("ba", CMlp3), ("da", CMlp3), ("fc", CMlp3)]


class CPretrainHeadIO(C.Structure):
    _fields_ = [(n, _vp) for n in ("x_atoms", "x_frags", "edge_feat", "edge_index", "mol_atom_ptr", "mol_frag_ptr",
                                   "batch32", "frag_batch32")] + \
               [(n, _i64) for n in ("n_atoms", "n_frags", "n_edges", "n_graphs")] + \
               [(n, _vp) for n in ("bond_length", "bond_angle", "dihedral", "energy", "g_bond_angle", "g_dihedral",
                                   "g_energy", "g_atoms", "g_frags", "g_edge")]


class CMseTerm(C.Structure):
    _fields_ = [("pred", _vp), ("target", _vp), ("n", _i64), ("weight", _f32), ("grad", _vp)]


class CPretrainStepArgs(C.Structure):
    _fields_ = [("batch", CBatchInputs)] + \
               [(n, _vp) for n in ("x_atoms", "x_bond", "x_fbond", "t_bond_angle", "t_dihedral", "t_energy")] + \
               [("n_layers", _i32), ("layers", _vp), ("layer_grads", _vp), ("heads", _vp), ("head_grads", _vp),
                ("drop_p", _f32), ("training", _i32), ("seed", _u64), ("offset", _u64), ("precision", _i32),
                ("backward", _i32)] + \
               [(n, _vp) for n in ("loss", "bond_length", "bond_angle", "dihedral", "energy", "plan_arena")]


ACT_NONE, ACT_RELU, ACT_CELU, ACT_SILU, ACT_GELU, ACT_SELU, ACT_RELU6, ACT_LEAKYRELU = range(8)
MLP_MAX_LAYERS = 8
LOSS_MSE, LOSS_BCE_MASKED = 0, 1
VARIANT_GAT2, VARIANT_LITE, VARIANT_EDGE = 0, 1, 2


class CMlpLayer(C.Structure):
    _fields_ = [(n, _vp) for n in ("W", "b", "dW", "db")] + [("in_dim", _i32), ("out_dim", _i32), ("p_in", _f32),
                                                               ("p_out", _f32), ("act", _i32)]


class CFinetuneStepArgs(C.Structure):
    _fields_ = [("batch", CBatchInputs)] + \
               [(n, _vp) for n in ("x_atoms", "x_bond", "x_fbond", "target")] + \
               [("n_layers", _i32), ("layers", _vp), ("layer_grads", _vp), ("n_head_layers", _i32), ("head", _vp),
                ("loss_kind", _i32), ("drop_p", _f32), ("training", _i32), ("seed", _u64), ("offset", _u64),
                ("precision", _i32), ("backward", _i32)] + \
               [(n, _vp) for n in ("loss", "predictions", "plan_arena")] + [("first_trained_layer", _i32)] + \
               [("variant", _i32)] + [(n, _vp) for n in ("cnx_attr", "W_cnx", "b_cnx", "dW_cnx", "db_cnx")]
