"""ctypes binding of libgavisunk_b200.so (the C ABI declared in include/gavisunk_b200.h).

There is no CPU fallback: if the shared library has not been built (``python -c "import
__graft_entry__ as g; g.build()"`` or ``make -C gavisunk_b200/csrc``) loading raises, and every
compute entry point fails when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GVS_LIB_PATH") or os.path.join(_HERE, "libgavisunk_b200.so")  # (the variable: kernel experiments only)

u8p, u32p, u64p, i32p, i64p, f64p = (C.POINTER(t) for t in (C.c_uint8, C.c_uint32, C.c_uint64, C.c_int32, C.c_int64, C.c_double))
vp = C.c_void_p

# name -> (restype, argtypes); mirrors include/gavisunk_b200.h one to one
PROTOTYPES = {
    "gvs_create": (vp, [C.c_int, C.c_int]),
    "gvs_destroy": (None, [vp]),
    "gvs_last_error": (C.c_char_p, [vp]),
    "gvs_version": (C.c_char_p, []),
    "gvs_set_stream": (C.c_int, [vp, vp]),
    "gvs_sync": (C.c_int, [vp]),
    "gvs_set_profiling": (C.c_int, [vp, C.c_int]),
    "gvs_stage_ms": (C.c_int, [vp, C.c_int, C.POINTER(C.c_float)]),
    "gvs_launch_count": (C.c_uint64, [vp]),
    "gvs_host_alloc": (C.c_int, [C.c_uint64, C.POINTER(vp)]),
    "gvs_host_free": (None, [vp]),
    "gvs_db_load_loc": (C.c_int, [vp, vp, C.c_uint64, vp, vp, vp, vp, C.c_uint64, C.c_uint32]),
    "gvs_db_build": (C.c_int, [vp, vp, vp, C.c_uint32, C.c_int]),
    "gvs_set_probe_variant": (C.c_int, [vp, C.c_int]),
    "gvs_set_db_passes": (C.c_int, [vp, C.c_int]),
    "gvs_db_size": (C.c_int, [vp, u64p, u64p]),
    "gvs_db_export": (C.c_int, [vp, vp, vp, vp, vp, vp]),
    "gvs_reads_set": (C.c_int, [vp, vp, vp, C.c_uint64, vp, vp, C.c_uint32, C.c_int]),
    "gvs_reads_set_packed": (C.c_int, [vp, vp, vp, C.c_uint64, vp, vp, C.c_uint32, C.c_int]),
    "gvs_set_copy_pipeline": (C.c_int, [vp, C.c_uint64, C.c_uint32]),
    "gvs_set_host_pack": (C.c_int, [vp, C.c_int, C.c_int]),
    "gvs_copy_stats": (C.c_int, [vp, u64p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "gvs_reads_meta": (C.c_int, [vp, vp, C.c_uint64, vp, vp, C.c_uint32]),
    "gvs_rows_set": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp, C.c_uint64, C.c_uint32]),
    "gvs_match": (C.c_int, [vp, u64p]),
    "gvs_rows_get": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp]),
    "gvs_diag_filter": (C.c_int, [vp, vp, vp, u64p, u64p]),
    "gvs_diag_filter_haps": (C.c_int, [vp, vp, vp, C.c_int, u64p, u64p]),
    "gvs_read_haps": (C.c_int, [vp, u64p]),
    "gvs_read_haps_get": (C.c_int, [vp] * 9),
    "gvs_best_get": (C.c_int, [vp, vp, vp, vp, vp]),
    "gvs_filter_best": (C.c_int, [vp, vp, u64p]),
    "gvs_contigs_set": (C.c_int, [vp, vp, vp, C.c_uint32]),
    "gvs_group_hist":(C.c_int, [vp, C.c_int, C.POINTER(vp)]),
    "gvs_hist_mode": (C.c_int, [vp, i64p]),
    "gvs_bad_groups": (C.c_int, [vp, i64p, u64p]),
    "gvs_bad_get": (C.c_int, [vp, vp]),
    "gvs_bad_set": (C.c_int, [vp, vp, vp, C.c_uint64, u64p]),
    "gvs_groups_count": (C.c_int, [vp, u64p]),
    "gvs_groups_get": (C.c_int, [vp, vp, vp, vp]),
    "gvs_batches_begin": (C.c_int, [vp]),
    "gvs_batch_stash": (C.c_int, [vp, u64p]),
    "gvs_batches_bind": (C.c_int, [vp, u64p, u64p]),
    "gvs_validate": (C.c_int, [vp, C.c_uint32, u64p]),
    "gvs_pairs_get": (C.c_int, [vp, vp, vp, vp, vp]),
    "gvs_validate_stats": (C.c_int, [vp, u64p]),
    "gvs_components_local": (C.c_int, [vp, C.POINTER(vp)]),
    "gvs_components_merge_all": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32]),
    "gvs_placements": (C.c_int, [vp, u64p, C.POINTER(vp)]),
    "gvs_placements_get": (C.c_int, [vp, vp, vp, vp, vp, vp, vp]),
    "gvs_support": (C.c_int, [vp, vp, u64p]),
    "gvs_support_get": (C.c_int, [vp, vp, vp, vp, vp]),
    "gvs_spans": (C.c_int, [vp, C.c_uint32, C.c_uint32, u64p, C.POINTER(vp)]),
    "gvs_spans_get": (C.c_int, [vp] * 9),
    "gvs_discordance": (C.c_int, [vp, vp, u64p]),
    "gvs_discordance_get": (C.c_int, [vp] * 7),
    "gvs_intervals": (C.c_int, [vp, u64p]),
    "gvs_intervals_get": (C.c_int, [vp, vp, vp, vp]),
    "gvs_intervals_set": (C.c_int, [vp, vp, vp, vp, C.c_uint64, C.c_uint32]),
    "gvs_gaps": (C.c_int, [vp, vp, u64p, u64p]),
    "gvs_gaps_get": (C.c_int, [vp, vp, vp, vp, vp]),
    "gvs_gap_evidence": (C.c_int, [vp, C.c_uint32, u64p]),
    "gvs_gap_evidence_get": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "gvs_junction_screen": (C.c_int, [vp, C.c_uint32, u64p, u64p]),
    "gvs_junctions": (C.c_int, [vp, u64p]),
    "gvs_junctions_get": (C.c_int, [vp] * 14),
    "gvs_strand_switches": (C.c_int, [vp, C.c_uint32, u64p]),
    "gvs_strand_switches_get": (C.c_int, [vp] * 17),
    "gvs_sunk_depth": (C.c_int, [vp, C.c_int, C.POINTER(vp)]),
    "gvs_sunk_depth_get": (C.c_int, [vp] * 4),
    "gvs_depth_runs": (C.c_int, [vp, vp, u64p]),
    "gvs_depth_runs_get": (C.c_int, [vp] * 7),
    "gvs_allele_support": (C.c_int, [vp, C.c_int, C.POINTER(vp)]),
    "gvs_allele_support_get": (C.c_int, [vp] * 5),
    "gvs_allele_runs": (C.c_int, [vp, vp, u64p]),
    "gvs_allele_runs_get": (C.c_int, [vp] * 6),
    "gvs_covprob_table": (C.c_int, [vp, vp, vp, C.c_uint32, C.c_double, C.c_double, vp]),
    "gvs_covprob_gaps": (C.c_int, [vp, vp, vp, C.c_uint64, vp, vp, vp, C.c_uint64, vp, vp, vp]),
    "gvs_slop": (C.c_int, [vp, vp, vp, vp, C.c_uint64, vp, C.c_uint32, C.c_int64]),
    "gvs_synth_assembly": (C.c_int, [vp, vp, vp, C.c_uint32, C.c_double, C.c_double, C.c_uint64]),
    "gvs_synth_reads_plan": (C.c_int, [vp, vp, C.c_uint32, C.c_uint32, C.c_uint64, C.c_double, C.c_double,
                                       C.c_uint32, C.c_uint32, C.c_uint64, vp, u64p]),
    "gvs_synth_reads_fill": (C.c_int, [vp, vp, vp, vp, C.c_uint64]),
}



class FastxStruct(C.Structure):
    """struct gvs_fastx of include/gavisunk_b200.h"""
    _fields_ = [("impl", C.c_void_p), ("seq", C.c_void_p), ("read_off", C.c_void_p), ("names", C.c_void_p),
                ("name_off", C.c_void_p), ("chunk_first", C.c_void_p), ("n_reads", C.c_uint64), ("total_bases", C.c_uint64),
                ("n_files", C.c_uint32), ("pinned", C.c_int), ("words", C.c_void_p), ("n_words", C.c_uint64)]


PROTOTYPES["gvs_fastx_read"] = (C.c_int, [C.POINTER(C.c_char_p), C.c_uint32, C.c_int, C.c_int, C.POINTER(FastxStruct), C.c_char_p,
                                          C.c_uint64])
PROTOTYPES["gvs_fastx_free"] = (None, [C.POINTER(FastxStruct)])
PROTOTYPES["gvs_fastx_pack"] = (C.c_int, [C.POINTER(FastxStruct), C.c_int, C.c_int])
PROTOTYPES["gvs_pack_2bit"] = (C.c_int, [vp, C.c_uint64, vp, C.c_int])
PROTOTYPES["gvs_fastx_read_packed"] = (C.c_int, [C.POINTER(C.c_char_p), C.c_uint32, C.c_int, C.c_int, C.c_uint64, C.POINTER(FastxStruct),
                                                 C.c_char_p, C.c_uint64])


class ColStruct(C.Structure):
    """struct gvs_col of include/gavisunk_b200.h"""
    _fields_ = [("kind", C.c_int32), ("k", C.c_int32), ("data", C.c_void_p), ("names", C.c_void_p), ("name_off", C.c_void_p),
                ("prefix", C.c_char), ("sep", C.c_char)]


PROTOTYPES["gvs_format_rows"] = (C.c_int64, [C.POINTER(ColStruct), C.c_uint32, C.c_uint64, vp, C.c_uint64, vp, C.c_uint64, C.c_int])

GVS_E_KEYERROR = -3
STAGES = {"probe": 0, "emit": 1, "diag": 2, "hist": 3, "validate": 4, "intervals": 5, "dbbuild": 6, "components": 7, "mode": 8,
          "bad": 9, "merge": 10, "support": 11, "evidence": 12, "screen": 13,
          "junctions": 14, "discordance": 15, "readhaps": 16, "switches": 17, "depth": 18,
          "alleles": 19}

_lib = None


class GavisunkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libgavisunk_b200 error {code}: {msg}")
        self.code = code


class GavisunkKeyError(GavisunkError, KeyError):
    """GVS_E_KEYERROR: the reference raises KeyError at this point (kmerpos_annot3.nim:90 for a db k-mer
    without a .loc row, covprob.py:118,130 for a gap without a group / beyond the table); callers may
    catch it as either."""

    def __str__(self):  # KeyError.__str__ would repr() the message
        return RuntimeError.__str__(self)


def load():
    """Load the shared library (once) and attach prototypes.  Raises if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA extension first (python -c 'import __graft_entry__ as g; "
            "g.build()').  gavisunk_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
