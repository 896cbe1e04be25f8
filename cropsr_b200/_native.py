"""ctypes binding of libcropsr_b200.so (include/cropsr_b200.h).

There is no CPU fallback: if the shared library is missing this module raises
at import time, and if no CUDA device is usable every compute call raises
``CropsrError`` with the library's message.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# CROPSR_B200_LIB: another build of the same library (kernel experiments, tools/variants.sh)
LIB_PATH = os.environ.get("CROPSR_B200_LIB") or os.path.join(_HERE, "libcropsr_b200.so")

ABI_VERSION = 11

CRP_SCAN_DEFAULT = 0
CRP_SCAN_NO_SCORE = 1
CRP_SCAN_LOGISTIC = 2
CRP_SCAN_EXTRAS = 4

CRP_CLASS_CANONICAL = 0
CRP_CLASS_PAIR = 1
CRP_CLASS_SINGLE = 2

PACKED_IRREGULAR = 1 << 30
PACKED_TRUNCATED = 1 << 31
PACKED_UNSCORED = 1 << 62

OFFTARGET_NO_COUNT = 0xFFFFFFFF     # counts of a candidate without a protospacer (crp_offtarget_count_candidates)
OFFTARGET_NO_SCORE = 0xFFFFFFFFFFFFFFFF   # score of a candidate without a protospacer (crp_offtarget_score_candidates)
OFFTARGET_SCORE_SETS = 1351         # CRP_OT_SCORE_SETS: mismatch-position sets of size <= 3


class SegmentDesc(C.Structure):
    """crp_segment_desc"""
    _fields_ = [("token_id", C.c_uint32), ("token", C.c_void_p), ("token_len", C.c_uint64),
                ("begin", C.c_uint64), ("end", C.c_uint64)]


class PrimerParams(C.Structure):
    """crp_primer_params: the CLI flags -e -s -l -m -x -M -X -D of the reference's prmrdsgn2.py (:26-54)"""
    _fields_ = [("e", C.c_uint32), ("s", C.c_uint32), ("l", C.c_uint32), ("m", C.c_double), ("x", C.c_double),
                ("M", C.c_double), ("X", C.c_double), ("D", C.c_double)]


class CropsrError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libcropsr_b200 error {code}: {message}")
        self.code = code


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `make -C {os.path.join(_HERE, 'csrc')}` "
        "(or __graft_entry__.build()).  cropsr_b200 has no CPU fallback.")

lib = C.CDLL(LIB_PATH)

_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)
_u64p = C.POINTER(C.c_uint64)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_vpp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); mirrors include/cropsr_b200.h one to one
SIGNATURES = {
    "crp_init": (C.c_int, [C.c_int]),
    "crp_shutdown": (C.c_int, []),
    "crp_last_error": (C.c_char_p, []),
    "crp_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "crp_abi_version": (C.c_int, []),
    "crp_tile_size": (C.c_int, []),
    "crp_checked_build": (C.c_int, []),
    "crp_host_alloc": (C.c_int, [_vpp, C.c_uint64]),
    "crp_host_free": (C.c_int, [C.c_void_p]),
    "crp_genome_new": (C.c_int, [_vpp]),
    "crp_genome_add_segment": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64]),
    "crp_genome_add_fasta_record": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64, C.c_uint32, C.c_int]),
    "crp_genome_token_length": (C.c_int, [C.c_void_p, C.c_uint32, _u64p]),
    "crp_genome_fetch_token": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64]),
    "crp_genome_release_tokens": (C.c_int, [C.c_void_p]),
    "crp_genome_commit": (C.c_int, [C.c_void_p]),
    "crp_genome_num_segments": (C.c_int, [C.c_void_p, _u32p]),
    "crp_genome_num_positions": (C.c_int, [C.c_void_p, _u64p]),
    "crp_genome_free": (C.c_int, [C.c_void_p]),
    "crp_scan_score": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, _vpp]),
    "crp_result_totals": (C.c_int, [C.c_void_p, _u64p, _u64p]),
    "crp_result_segment_counts": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_result_device_counts": (C.c_int, [C.c_void_p, _vpp]),
    "crp_result_fetch": (C.c_int, [C.c_void_p, C.c_char, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_result_free": (C.c_int, [C.c_void_p]),
    "crp_scan_segments": (C.c_int, [C.c_uint32, C.c_void_p, C.c_int, C.c_uint32, C.c_uint64,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, _f32p]),
    "crp_result_extras": (C.c_int, [C.c_void_p, C.c_uint32, C.c_char, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_result_annotate": (C.c_int, [C.c_void_p, C.c_uint32, C.c_char, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_result_extras_strand": (C.c_int, [C.c_void_p, C.c_char, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_result_annotate_strand": (C.c_int, [C.c_void_p, C.c_char, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_genome_other_runs": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p, _u64p]),
    "crp_primer_windows": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(PrimerParams),
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_legacy_ids": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.c_uint64, C.c_void_p]),
    "crp_format_rows": (C.c_int, [C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                  C.c_int, C.c_void_p, C.c_uint64, _u64p]),
    "crp_logistic": (C.c_int, [C.c_uint64, C.c_void_p, C.c_void_p]),
    "crp_rs1_score": (C.c_int, [C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_rescore": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_genome_timing": (C.c_int, [C.c_void_p, _f32p, _f32p]),
    "crp_result_timing": (C.c_int, [C.c_void_p, _f32p]),
    "crp_launch_count": (C.c_int, [_u64p]),
    "crp_perf_report": (C.c_int, [C.c_void_p, C.c_uint64, _u64p]),
    "crp_debug_set_times": (C.c_int, [C.c_void_p]),
    "crp_device_synchronize": (C.c_int, []),
    "crp_flush_l2": (C.c_int, []),
    "crp_comm_unique_id": (C.c_int, [C.c_void_p]),
    "crp_comm_init": (C.c_int, [C.c_int, C.c_int, C.c_void_p]),
    "crp_comm_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "crp_comm_set_exchange": (C.c_int, [C.c_int]),
    "crp_comm_exchange_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_char_p)]),
    "crp_comm_barrier": (C.c_int, []),
    "crp_comm_max_f64": (C.c_int, [C.c_void_p, C.c_uint32]),
    "crp_comm_sum_f64": (C.c_int, [C.c_void_p, C.c_uint32]),
    "crp_comm_shutdown": (C.c_int, []),
    "crp_comm_allgather_u64": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "crp_link_probe": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint32, _f32p]),
    "crp_scan_score_sharded": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32, _vpp]),
    "crp_result_gathered_counts": (C.c_int, [C.c_void_p, C.c_void_p]),
    "crp_result_timing_detail": (C.c_int, [C.c_void_p, _f32p, _f32p, _u32p]),
    "crp_rs1_preactivation": (C.c_int, [C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "crp_offtarget_new": (C.c_int, [_vpp]),
    "crp_offtarget_add_genome": (C.c_int, [C.c_void_p, C.c_void_p]),
    "crp_offtarget_num_sites": (C.c_int, [C.c_void_p, _u64p]),
    "crp_offtarget_fetch_sites": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, _u64p]),
    "crp_offtarget_count_candidates": (C.c_int, [C.c_void_p, C.c_void_p, C.c_char, C.c_uint32, C.c_void_p]),
    "crp_offtarget_count_keys": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p]),
    "crp_offtarget_new_with_loci": (C.c_int, [_vpp]),
    "crp_offtarget_fetch_loci": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, _u64p]),
    "crp_offtarget_list_candidates": (C.c_int, [C.c_void_p, C.c_void_p, C.c_char, C.c_uint32, C.c_uint64, C.c_void_p,
                                                C.c_void_p, C.c_void_p]),
    "crp_offtarget_list_keys": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "crp_offtarget_score_candidates": (C.c_int, [C.c_void_p, C.c_void_p, C.c_char, C.c_uint32, C.c_void_p, C.c_void_p]),
    "crp_offtarget_score_keys": (C.c_int, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "crp_offtarget_new_pam": (C.c_int, [_vpp, C.c_char_p, C.c_int]),
    "crp_offtarget_timing": (C.c_int, [C.c_void_p, _f32p, _f32p, _u64p]),
    "crp_offtarget_free": (C.c_int, [C.c_void_p]),
}
COMM_ID_BYTES = 128

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)       # AttributeError here = library/header mismatch
    _fn.restype = _res
    _fn.argtypes = _args

if lib.crp_abi_version() != ABI_VERSION:
    raise ImportError(f"{LIB_PATH}: ABI version {lib.crp_abi_version()} != binding {ABI_VERSION}; rebuild")


def check(rc):
    if rc != 0:
        raise CropsrError(rc, lib.crp_last_error().decode("utf-8", "replace"))
