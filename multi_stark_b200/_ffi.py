"""ctypes binding of include/msgpu.h. The signatures below are the whole ABI; tests/test_abi.py checks
that every symbol the header declares is exported by the built library."""
import ctypes as C
import os

from . import build as _build

_LIB = None

c_u64p = C.POINTER(C.c_uint64)
c_u8p = C.POINTER(C.c_uint8)
c_u32p = C.POINTER(C.c_uint32)
c_vpp = C.POINTER(C.c_void_p)

SIGNATURES = {
    "msgpu_ctx_create": (C.c_int, [C.c_int, C.c_void_p, c_vpp]),
    "msgpu_ctx_destroy": (None, [C.c_void_p]),
    "msgpu_last_error": (C.c_char_p, []),
    "msgpu_sync": (C.c_int, [C.c_void_p]),
    "msgpu_stream": (C.c_void_p, [C.c_void_p]),
    "msgpu_launch_count": (C.c_uint64, [C.c_void_p]),
    "msgpu_profile_begin": (C.c_int, [C.c_void_p]),
    "msgpu_profile_end": (C.c_int, [C.c_void_p, C.c_char_p, C.c_size_t]),
    "msgpu_malloc": (C.c_int, [C.c_void_p, C.c_size_t, c_vpp]),
    "msgpu_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "msgpu_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "msgpu_host_alloc": (C.c_int, [C.c_size_t, c_vpp]),
    "msgpu_host_free": (C.c_int, [C.c_void_p]),
    "msgpu_upload_canonical": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "msgpu_blake3_hash": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "msgpu_dft_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msgpu_dft_batch_bitrev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msgpu_idft_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msgpu_coset_lde_batch_bitrev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64,
                                               C.c_void_p]),
    "msgpu_lde_from_shifted_coefficients": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                                      C.c_void_p]),
    "msgpu_dft_batch_bitrev_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msgpu_coset_lde_batch_bitrev_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                                   C.c_uint64, C.c_void_p]),
    "msgpu_lde_from_shifted_coefficients_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32,
                                                          C.c_void_p]),
    "msgpu_commit": (C.c_int, [C.c_void_p, c_vpp, c_u64p, c_u64p, C.c_uint64, C.c_uint32, c_vpp, C.c_void_p]),
    "msgpu_upload_begin": (C.c_int, [C.c_void_p, c_vpp, c_u64p, c_u64p, C.c_uint64, c_vpp]),
    "msgpu_commit_upload": (C.c_int, [C.c_void_p, C.c_uint32, C.c_int, c_vpp, C.c_int, c_vpp, C.c_void_p]),
    "msgpu_upload_free": (None, [C.c_void_p]),
    "msgpu_commit_dev": (C.c_int, [C.c_void_p, c_vpp, c_u64p, c_u64p, C.c_uint64, C.c_uint32, c_vpp, C.c_void_p]),
    "msgpu_commit_ldes_dev": (C.c_int, [C.c_void_p, c_vpp, c_u64p, c_u64p, C.c_uint64, C.c_int, c_vpp, C.c_void_p]),
    "msgpu_commit_local_dev": (C.c_int, [C.c_void_p, c_vpp, c_u64p, c_u64p, C.c_uint64, C.c_uint32, C.c_int, c_vpp]),
    "msgpu_pdata_num_classes": (C.c_uint64, [C.c_void_p]),
    "msgpu_pdata_class_digests": (C.c_int, [C.c_void_p, C.c_uint64, c_u64p, c_vpp]),
    "msgpu_tree_from_digests": (C.c_int, [C.c_void_p, C.c_uint64, c_u64p, c_vpp, c_vpp, C.c_void_p]),
    "msgpu_pdata_max_height": (C.c_uint64, [C.c_void_p]),
    "msgpu_pdata_root": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_pdata_digests": (C.c_int, [C.c_void_p, c_vpp, c_u64p]),
    "msgpu_pdata_from_parts": (C.c_int, [C.c_void_p, C.c_uint64, c_vpp, c_u64p, C.c_uint64, C.c_uint64, c_vpp, c_vpp, C.c_void_p]),
    "msgpu_mmcs_commit": (C.c_int, [C.c_void_p, c_vpp, c_u64p, c_u64p, C.c_uint64, c_vpp, C.c_void_p]),
    "msgpu_pdata_free": (None, [C.c_void_p]),
    "msgpu_pdata_num_matrices": (C.c_uint64, [C.c_void_p]),
    "msgpu_pdata_matrix": (C.c_int, [C.c_void_p, C.c_uint64, c_vpp, c_u64p, c_u64p]),
    "msgpu_pdata_read_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msgpu_pdata_num_layers": (C.c_uint64, [C.c_void_p]),
    "msgpu_pdata_layer_len": (C.c_uint64, [C.c_void_p, C.c_uint64]),
    "msgpu_pdata_read_layer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "msgpu_open_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "msgpu_open_batch_multi": (C.c_int, [C.c_void_p, c_vpp, c_u32p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "msgpu_program_create": (C.c_int, [C.c_void_p, C.c_void_p, c_vpp]),
    "msgpu_program_free": (None, [C.c_void_p]),
    "msgpu_stage2_trace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "msgpu_claims_accumulator": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p,
                                           C.c_void_p]),
    "msgpu_claims_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_uint64, c_vpp, C.c_void_p]),
    "msgpu_claims_prefetch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, c_vpp]),
    "msgpu_claims_digest": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "msgpu_claims_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msgpu_claims_free": (None, [C.c_void_p]),
    "msgpu_quotient": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p,
                                 C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, c_vpp, C.c_void_p]),
    "msgpu_shifted_quotient_slices": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msgpu_open_begin": (C.c_int, [C.c_void_p, C.c_uint64, c_vpp, c_u64p, c_u64p, C.c_uint32, c_vpp, c_u64p]),
    "msgpu_open_values": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_open_reduce": (C.c_int, [C.c_void_p, C.c_void_p, c_u64p, c_u32p]),
    "msgpu_open_read_input": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, c_u64p]),
    "msgpu_open_input_dev": (C.c_int, [C.c_void_p, C.c_uint64, c_vpp, c_u64p]),
    "msgpu_open_add_input": (C.c_int, [C.c_void_p, C.c_uint64, c_vpp]),
    "msgpu_fri_current_len": (C.c_int, [C.c_void_p, c_u64p]),
    "msgpu_fri_commit_round": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_fri_fold": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_fri_read_current": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_fri_commit_phase": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msgpu_fri_num_layers": (C.c_uint64, [C.c_void_p]),
    "msgpu_fri_layer_pdata": (C.c_void_p, [C.c_void_p, C.c_uint64]),
    "msgpu_open_free": (None, [C.c_void_p]),
    "msgpu_measure_int_peak": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "msgpu_blake3_compress_raw": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msgpu_pack_column_blocks_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msgpu_interleave_column_blocks_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]),
    "msgpu_quotient_values_shard": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                              C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msgpu_extract_columns_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msgpu_quotient_finish": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p]),
    "msgpu_open_begin_shard": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msgpu_open_sums": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_open_finish_values": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_pdata_placeholder": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msgpu_ext_add_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "msgpu_ext_add_scalar_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "msgpu_host_register": (C.c_int, [C.c_void_p, C.c_size_t]),
    "msgpu_host_unregister": (C.c_int, [C.c_void_p]),
    "msgpu_ctx_set_option": (C.c_int, [C.c_void_p, C.c_int, C.c_uint64]),
    "msgpu_arena_in_use": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "msgpu_selectors_on_coset": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msgpu_commit_ldes_blocks_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p,
                                               C.c_int, C.c_void_p, C.c_void_p]),
    "msgpu_memcpy_d2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "msgpu_peers_create": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "msgpu_peers_segment_create": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p]),
    "msgpu_peers_segment_open": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_peers_segment_open_local": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msgpu_peers_num_segments": (C.c_uint64, [C.c_void_p]),
    "msgpu_peers_alloc": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p]),
    "msgpu_peers_free_block": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64]),
    "msgpu_peers_ptr": (C.c_void_p, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_int32]),
    "msgpu_peers_barrier": (C.c_int, [C.c_void_p]),
    "msgpu_peers_put": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64]),
    "msgpu_peers_put_root": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "msgpu_peers_check": (C.c_int, [C.c_void_p]),
    "msgpu_peers_pack_push": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint64]),
    "msgpu_peers_pull_interleave": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msgpu_peers_destroy": (None, [C.c_void_p]),
}


class MsgpuError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("msgpu error %d: %s" % (code, message))
        self.code = code
        self.message = message


def lib_path():
    return _build.LIB


def lib():
    """Loads libmsgpu.so, building it with nvcc first if the sources are newer. Raises if that fails."""
    global _LIB
    if _LIB is not None:
        return _LIB
    if _build.needs_build():
        if not os.path.exists(_build.NVCC):
            if not os.path.exists(_build.LIB):
                raise MsgpuError(-3, "libmsgpu.so is not built and nvcc is not available")
        else:
            _build.build()
    L = C.CDLL(_build.LIB)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)  # AttributeError here = the library does not export the ABI
        fn.restype = res
        fn.argtypes = args
    _LIB = L
    return L


def check(code):
    if code != 0:
        raise MsgpuError(code, (lib().msgpu_last_error() or b"").decode("utf-8", "replace"))


def host_error(code, extra=""):
    """MsgpuError(code) carrying libmshost.so's last error message, followed by `extra` (a communicator's errors) if given."""
    message = (host_lib().msh_last_error() or b"").decode("utf-8", "replace")
    return MsgpuError(code, message + " " + extra if extra else message)


# ---- libmshost.so: host-side protocol layer (system assembly, workloads, prove driver) ---------------
_HOST = None
HOST_SIGNATURES = {
    "msh_last_error": (C.c_char_p, []),
    "msh_system_create": (C.c_void_p, [C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "msh_system_create_from_graphs": (C.c_void_p, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32,
                                                   C.c_uint32, C.c_uint32, C.c_uint32]),
    "msh_system_free": (None, [C.c_void_p]),
    "msh_system_num_circuits": (C.c_uint32, [C.c_void_p]),
    "msh_circuit_info": (None, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "msh_circuit_graph": (C.c_void_p, [C.c_void_p, C.c_uint32]),
    "msh_circuit_preprocessed": (None, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "msh_u32add_workload": (None, [C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msh_u32add_workload_seeded": (None, [C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "msh_rowshard_commit": (C.c_int, [C.c_void_p, c_vpp, c_u64p, c_u64p, C.c_uint64, C.c_int, C.c_void_p]),
    "msh_rowshard_shardable": (C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64]),
    "msh_rowshard_peer_memory": (C.c_int, [C.c_void_p]),
    "msh_rowshard_peer_bytes": (C.c_uint64, [C.c_void_p]),
    "msh_rowshard_prover_create": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "msh_dist_prover_create": (C.c_void_p, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]),
    "msh_fib_trace": (None, [C.c_uint64, C.c_void_p]),
    "msh_wide_trace": (None, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msh_wide_trace_block": (None, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_void_p]),
    "msh_prover_create": (C.c_void_p, [C.c_void_p, C.c_void_p]),
    "msh_prover_free": (None, [C.c_void_p]),
    "msh_prover_inject_stage1": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msh_prover_preprocessed_commit": (C.c_int, [C.c_void_p, C.c_void_p]),
    "msh_prove": (C.c_int, [C.c_void_p, c_vpp, c_u64p, c_u64p, c_u64p, C.c_uint64, C.c_uint64, c_vpp, c_u64p, C.POINTER(C.c_double)]),
    "msh_bytes_free": (None, [C.c_void_p]),
    "msh_last_transcript": (C.c_uint64, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p]),
    "msh_challenger_create": (C.c_void_p, [C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]),
    "msh_challenger_free": (None, [C.c_void_p]),
    "msh_challenger_observe_digest": (None, [C.c_void_p, C.c_void_p]),
    "msh_challenger_observe_values": (None, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "msh_challenger_sample_ext": (None, [C.c_void_p, C.c_void_p]),
    "msh_pcs_open": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, c_vpp, c_u64p, c_u64p, c_vpp, c_u64p, C.POINTER(C.c_double)]),
}


def host_lib():
    global _HOST
    if _HOST is not None:
        return _HOST
    lib()  # builds both libraries if needed and loads libmsgpu first
    H = C.CDLL(_build.HOST_LIB)
    for name, (res, args) in HOST_SIGNATURES.items():
        fn = getattr(H, name)
        fn.restype = res
        fn.argtypes = args
    _HOST = H
    return H
