"""ctypes binding of libb200prover.so (C ABI in include/b200prover.h).

The library is built in-tree by `__graft_entry__.build()` / `make -C renegade_b200/csrc`.
There is no CPU fallback: if the shared library is missing, or no CUDA device is visible, the
calls below raise — they never route to the oracle or to any host implementation.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200_LIB_PATH: developer knob to load an alternative build of the same library (tuning experiments)
LIB_PATH = os.environ.get("B200_LIB_PATH") or os.path.join(_HERE, "libb200prover.so")

# every symbol include/b200prover.h declares (tests/test_abi.py checks this list against the
# header and against the built library)
EXPORTS = [
    "b200_init", "b200_shutdown", "b200_last_error", "b200_version", "b200_kernel_launches", "b200_launch_host_ns", "b200_graph_launches", "b200_ctx_use_graphs",
    "b200_srs_parse_ptau", "b200_bases_load", "b200_bases_load_device", "b200_bases_free",
    "b200_bases_len", "b200_bases_plan",
    "b200_msm", "b200_msm_device", "b200_msm_batch_device", "b200_msm_timing", "b200_msm_timing_totals", "b200_msm_tuning", "b200_g1_sum_affine",
    "b200_ntt", "b200_ntt_device", "b200_ntt_last_ms", "b200_domain_generator",
    "b200_splitmix_fr_device", "b200_known_dlog_bases_device",
    "b200_selftest_field", "b200_field_op",
    "b200_plonk_preprocess", "b200_pk_verifying_key", "b200_pk_num_inputs", "b200_pk_log_n", "b200_pk_free", "b200_plonk_prove", "b200_plonk_link", "b200_plonk_verify", "b200_plonk_verify_link", "b200_plonk_batch_verify", "b200_pairing_check", "b200_plonk_last_timings", "b200_keccak256",
    "b200_fr_vec_op", "b200_fr_batch_inverse_device", "b200_fr_poly_eval_device", "b200_fr_poly_div_linear_device",
    "b200_poseidon2_hash_batch", "b200_poseidon2_permute_batch", "b200_poseidon2_merkle_root_batch", "b200_poseidon2_csprng_batch",
    "b200_pool_create", "b200_pool_destroy", "b200_pool_workers", "b200_pool_ctx", "b200_pool_submit_prove",
    "b200_pool_submit_link", "b200_pool_submit_bundle", "b200_pool_wait", "b200_pool_wait_all", "b200_pool_stats",
    "b200_box_create", "b200_box_destroy", "b200_box_devices", "b200_box_pool", "b200_box_srs_load", "b200_box_srs_free",
    "b200_box_preprocess", "b200_box_pk_verifying_key", "b200_box_pk_free", "b200_box_submit_prove", "b200_box_submit_bundle",
    "b200_box_wait", "b200_box_ticket_device",
    "b200_shard_range", "b200_multi_init", "b200_nccl_unique_id", "b200_multi_init_rank", "b200_multi_shutdown",
    "b200_nccl_version", "b200_multi_world", "b200_multi_local_devices", "b200_multi_ctx", "b200_multi_rank",
    "b200_multi_bases_load", "b200_multi_bases_known_dlog", "b200_multi_bases_free", "b200_multi_bases_len",
    "b200_multi_bases_shard", "b200_multi_bases_plan", "b200_multi_msm", "b200_multi_msm_local",
    "b200_mpc_prep_size", "b200_mpc_prep_load", "b200_mpc_prep_dealer", "b200_mpc_prep_free", "b200_mpc_prove", "b200_mpc_link",
    "b200_mpc_local_group_create", "b200_mpc_local_group_transport", "b200_mpc_local_group_destroy", "b200_mpc_last_stats",
    "b200_mpc_prep_load_auth", "b200_mpc_prep_dealer_auth", "b200_mpc_dealer_share_auth", "b200_mpc_prove_auth",
    "b200_mpc_link_auth",
]


class B200Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libb200prover error {code}: {msg}")
        self.code = code


_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no CPU fallback for the proving path)")
    lib = C.CDLL(LIB_PATH)
    vp, sz, i32, u64, u32 = C.c_void_p, C.c_size_t, C.c_int, C.c_uint64, C.c_uint
    lib.b200_last_error.restype = C.c_char_p
    lib.b200_version.restype = C.c_char_p
    lib.b200_kernel_launches.restype = C.c_uint64
    lib.b200_kernel_launches.argtypes = []
    lib.b200_launch_host_ns.restype = C.c_uint64
    lib.b200_launch_host_ns.argtypes = []
    lib.b200_graph_launches.restype = C.c_uint64
    lib.b200_graph_launches.argtypes = []
    lib.b200_ctx_use_graphs.restype = C.c_int
    lib.b200_ctx_use_graphs.argtypes = [C.c_void_p, C.c_int]
    lib.b200_init.argtypes = [i32, C.POINTER(vp)]
    lib.b200_shutdown.argtypes = [vp]
    lib.b200_shutdown.restype = None
    lib.b200_srs_parse_ptau.argtypes = [vp, sz, C.POINTER(vp), C.POINTER(sz)]
    lib.b200_bases_load.argtypes = [vp, vp, sz, i32, i32, C.POINTER(vp)]
    lib.b200_bases_load_device.argtypes = [vp, vp, sz, i32, C.POINTER(vp)]
    lib.b200_bases_free.argtypes = [vp, vp]
    lib.b200_bases_free.restype = None
    lib.b200_bases_len.argtypes = [vp]
    lib.b200_bases_len.restype = sz
    lib.b200_bases_plan.argtypes = [vp, C.POINTER(i32 * 4)]
    lib.b200_bases_plan.restype = None
    lib.b200_msm.argtypes = [vp, vp, sz, vp, sz, i32, vp, C.POINTER(i32)]
    lib.b200_msm_device.argtypes = [vp, vp, sz, vp, sz, i32, vp, C.POINTER(i32)]
    lib.b200_msm_batch_device.argtypes = [vp, vp, sz, vp, sz, sz, u32, i32, vp, vp]
    lib.b200_msm_timing_totals.argtypes = [vp, i32, C.POINTER(C.c_double * 3)]
    lib.b200_msm_timing.argtypes = [vp, i32, C.POINTER(C.c_float * 4)]
    lib.b200_msm_tuning.argtypes = [vp, i32]
    lib.b200_ntt_last_ms.argtypes = [vp, C.POINTER(C.c_float)]
    lib.b200_g1_sum_affine.argtypes = [vp, vp, sz, vp, C.POINTER(i32)]
    lib.b200_ntt.argtypes = [vp, vp, u32, i32, i32]
    lib.b200_ntt_device.argtypes = [vp, vp, u32, i32, i32, u32, sz]
    lib.b200_domain_generator.argtypes = [vp, u32, vp]
    lib.b200_splitmix_fr_device.argtypes = [vp, u64, sz, sz, i32, vp]
    lib.b200_known_dlog_bases_device.argtypes = [vp, u64, sz, sz, vp]
    lib.b200_selftest_field.argtypes = [vp, u64, sz, C.POINTER(u64)]
    lib.b200_field_op.argtypes = [vp, i32, i32, vp, vp, sz, vp]
    lib.b200_plonk_preprocess.argtypes = [vp, vp, u32, sz, vp, vp, vp, C.POINTER(vp)]
    lib.b200_pk_verifying_key.argtypes = [vp, vp, vp]
    lib.b200_pk_num_inputs.argtypes = [vp]
    lib.b200_pk_num_inputs.restype = sz
    lib.b200_pk_log_n.argtypes = [vp]
    lib.b200_pk_log_n.restype = u32
    lib.b200_pk_free.argtypes = [vp, vp]
    lib.b200_pk_free.restype = None
    lib.b200_plonk_prove.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    lib.b200_plonk_link.argtypes = [vp, vp, vp, sz, vp, sz, vp, vp, u32, sz, sz, vp, vp]
    lib.b200_plonk_verify.argtypes = [u32, sz, vp, vp, vp, vp, vp, vp, vp, C.POINTER(i32)]
    lib.b200_plonk_verify_link.argtypes = [vp, vp, u32, sz, sz, vp, vp, vp, C.POINTER(i32)]
    lib.b200_plonk_batch_verify.argtypes = [vp, vp, sz, vp, sz, vp, sz, vp, vp, C.POINTER(i32), vp, vp, C.POINTER(sz)]
    lib.b200_pairing_check.argtypes = [vp, vp, sz, C.POINTER(i32)]
    lib.b200_plonk_last_timings.argtypes = [vp, C.POINTER(C.c_float * 8)]
    lib.b200_fr_vec_op.argtypes = [vp, i32, vp, vp, i32, sz, vp]
    lib.b200_fr_batch_inverse_device.argtypes = [vp, vp, sz]
    lib.b200_fr_poly_eval_device.argtypes = [vp, vp, sz, vp, vp]
    lib.b200_fr_poly_div_linear_device.argtypes = [vp, vp, sz, vp, vp]
    lib.b200_poseidon2_hash_batch.argtypes = [vp, vp, sz, sz, vp]
    lib.b200_poseidon2_permute_batch.argtypes = [vp, vp, sz]
    lib.b200_poseidon2_merkle_root_batch.argtypes = [vp, vp, vp, vp, sz, u32, vp]
    lib.b200_poseidon2_csprng_batch.argtypes = [vp, vp, vp, sz, sz, vp]
    lib.b200_pool_create.argtypes = [i32, u32, C.POINTER(vp)]
    lib.b200_pool_destroy.argtypes = [vp]
    lib.b200_pool_destroy.restype = None
    lib.b200_pool_workers.argtypes = [vp]
    lib.b200_pool_workers.restype = u32
    lib.b200_pool_ctx.argtypes = [vp, u32]
    lib.b200_pool_ctx.restype = vp
    lib.b200_pool_submit_prove.argtypes = [vp, vp, vp, vp, sz, vp, vp, vp, C.POINTER(u64)]
    lib.b200_pool_submit_link.argtypes = [vp, vp, vp, sz, vp, sz, vp, vp, u32, sz, sz, vp, C.POINTER(u64)]
    lib.b200_pool_submit_bundle.argtypes = [vp, vp, vp, sz, vp, sz, C.POINTER(u64)]
    lib.b200_pool_wait.argtypes = [vp, u64]
    lib.b200_pool_wait_all.argtypes = [vp]
    lib.b200_pool_stats.argtypes = [vp, C.POINTER(u64 * 4)]
    lib.b200_box_create.argtypes = [C.POINTER(i32), i32, u32, C.POINTER(vp)]
    lib.b200_box_destroy.argtypes = [vp]
    lib.b200_box_destroy.restype = None
    lib.b200_box_devices.argtypes = [vp]
    lib.b200_box_pool.argtypes = [vp, i32]
    lib.b200_box_pool.restype = vp
    lib.b200_box_srs_load.argtypes = [vp, vp, sz, i32, i32, C.POINTER(vp)]
    lib.b200_box_srs_free.argtypes = [vp, vp]
    lib.b200_box_srs_free.restype = None
    lib.b200_box_preprocess.argtypes = [vp, vp, u32, sz, vp, vp, vp, C.POINTER(vp)]
    lib.b200_box_pk_verifying_key.argtypes = [vp, vp, vp]
    lib.b200_box_pk_free.argtypes = [vp, vp]
    lib.b200_box_pk_free.restype = None
    lib.b200_box_submit_prove.argtypes = [vp, vp, vp, vp, sz, vp, vp, vp, C.POINTER(u64)]
    lib.b200_box_submit_bundle.argtypes = [vp, vp, vp, vp, sz, vp, sz, C.POINTER(u64)]
    lib.b200_box_wait.argtypes = [vp, u64]
    lib.b200_box_ticket_device.argtypes = [vp, u64]
    lib.b200_shard_range.argtypes = [sz, i32, i32, C.POINTER(sz), C.POINTER(sz)]
    lib.b200_shard_range.restype = None
    lib.b200_multi_init.argtypes = [C.POINTER(i32), i32, C.POINTER(vp)]
    lib.b200_nccl_unique_id.argtypes = [vp]
    lib.b200_multi_init_rank.argtypes = [i32, i32, i32, vp, C.POINTER(vp)]
    lib.b200_multi_shutdown.argtypes = [vp]
    lib.b200_multi_shutdown.restype = None
    lib.b200_nccl_version.argtypes = [C.POINTER(i32)]
    lib.b200_multi_world.argtypes = [vp]
    lib.b200_multi_local_devices.argtypes = [vp]
    lib.b200_multi_ctx.argtypes = [vp, i32]
    lib.b200_multi_ctx.restype = vp
    lib.b200_multi_rank.argtypes = [vp, i32]
    lib.b200_multi_bases_load.argtypes = [vp, vp, sz, i32, i32, C.POINTER(vp)]
    lib.b200_multi_bases_known_dlog.argtypes = [vp, u64, sz, i32, C.POINTER(vp)]
    lib.b200_multi_bases_free.argtypes = [vp, vp]
    lib.b200_multi_bases_free.restype = None
    lib.b200_multi_bases_len.argtypes = [vp]
    lib.b200_multi_bases_len.restype = sz
    lib.b200_multi_bases_shard.argtypes = [vp, i32, C.POINTER(sz), C.POINTER(sz)]
    lib.b200_multi_bases_plan.argtypes = [vp, i32, C.POINTER(i32 * 4)]
    lib.b200_multi_msm.argtypes = [vp, vp, vp, sz, i32, vp, C.POINTER(i32)]
    lib.b200_multi_msm_local.argtypes = [vp, vp, C.POINTER(vp), i32, i32, vp, C.POINTER(i32)]
    lib.b200_mpc_prep_size.argtypes = [vp, C.POINTER(sz), C.POINTER(sz)]
    lib.b200_mpc_prep_load.argtypes = [vp, vp, vp, vp, vp, vp, C.POINTER(vp)]
    lib.b200_mpc_prep_dealer.argtypes = [vp, vp, u64, i32, i32, C.POINTER(vp)]
    lib.b200_mpc_prep_free.argtypes = [vp, vp]
    lib.b200_mpc_prep_free.restype = None
    lib.b200_mpc_prove.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.b200_mpc_link.argtypes = [vp, vp, vp, vp, sz, vp, sz, vp, vp, u32, sz, sz, vp, vp]
    lib.b200_mpc_local_group_create.argtypes = [i32, u32, C.POINTER(vp)]
    lib.b200_mpc_local_group_transport.argtypes = [vp, i32, vp]
    lib.b200_mpc_local_group_destroy.argtypes = [vp]
    lib.b200_mpc_local_group_destroy.restype = None
    lib.b200_mpc_last_stats.argtypes = [vp, C.POINTER(C.c_double * 4)]
    lib.b200_mpc_prep_load_auth.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(vp)]
    lib.b200_mpc_prep_dealer_auth.argtypes = [vp, vp, u64, i32, i32, vp, C.POINTER(vp)]
    lib.b200_mpc_dealer_share_auth.argtypes = [vp, u64, i32, i32, vp, sz, vp, vp]
    lib.b200_mpc_prove_auth.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.b200_mpc_link_auth.argtypes = [vp, vp, vp, vp, vp, vp, sz, vp, vp, sz, vp, vp, u32, sz, sz, vp, vp]
    lib.b200_keccak256.argtypes = [C.c_char_p, sz, vp]
    lib.b200_keccak256.restype = None
    for name in EXPORTS:
        fn = getattr(lib, name)  # raises AttributeError if a declared symbol is not exported
        if fn.restype is C.c_int and name not in ("b200_last_error", "b200_version"):
            pass
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise B200Error(rc, (load().b200_last_error() or b"").decode(errors="replace"))
