"""ctypes binding of libdigb200.so (include/dig_b200.h).

There is deliberately no CPU fallback: if the shared library is missing or a call fails,
an exception is raised.
"""
import ctypes
import os

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# DIG_LIB_PATH selects another build of the same library (developer probes: tools/probe_lb.py --timing)
LIB_PATH = os.environ.get("DIG_LIB_PATH") or os.path.join(_PKG_DIR, "libdigb200.so")

_c = ctypes
_P = _c.c_void_p
_I64 = _c.c_int64
_I = _c.c_int
_U64 = _c.c_uint64
_D = _c.c_double

# name -> (restype, argtypes); mirrors include/dig_b200.h one to one
SIGNATURES = {
    "dig_version": (_I, []),
    "dig_last_error": (_c.c_char_p, []),
    "dig_device_sm_count": (_I, []),
    "dig_packed_words": (_I64, [_I64]),
    "dig_nmask_words": (_I64, [_I64]),
    "dig_pack_genome": (_I, [_P, _I64, _P, _P, _P, _P]),
    "dig_scan_workspace_bytes": (_I64, [_I64]),
    "dig_count_contexts": (_I, [_P, _P, _I64, _P, _P, _P, _P, _P, _P, _I64, _I, _I, _P, _P, _P, _P]),
    "dig_count_contexts_fused53": (_I, [_P, _P, _I64, _P, _P, _P, _P, _P, _I64, _P, _P, _P, _P, _P, _P]),
    "dig_narrow_counts_u16": (_I, [_P, _I64, _P, _P, _P]),
    "dig_peer_broadcast": (_I, [_P, _I64, _P, _I, _P]),
    "dig_nmask_fill_runs": (_I, [_P, _I64, _P, _I64, _I64, _P]),
    "dig_nmask_summary": (_I, [_P, _I64, _I64, _P, _P]),
    "dig_tabulate_capacity": (_I64, [_I64]),
    "dig_tabulate_elements_workspace_bytes": (_I64, [_I64]),
    "dig_tabulate_genes_workspace_bytes": (_I64, [_I64]),
    "dig_synth_genome": (_I, [_P, _I64, _I64, _U64, _I, _P]),
    "dig_mutation_contexts": (_I, [_P, _P, _I64, _P, _P, _P, _P, _P, _I64, _I, _I, _P, _P]),
    "dig_substitution_counts": (_I, [_P, _P, _I64, _I, _I, _P, _P]),
    "dig_count_hits": (_I, [_P, _P, _P, _P, _I64, _P, _P, _I64, _P, _P]),
    "dig_tabulate_elements": (_I, [_P, _P, _P, _P, _I64, _P, _P, _P, _P, _I64, _P, _P, _P, _I64, _I64, _P,
                                   _I64, _I64, _I64, _P, _P, _I, _P]),
    "dig_site_counts": (_I, [_P, _P, _I64, _I64, _I, _P, _P]),
    "dig_tabulate_genes": (_I, [_P, _P, _P, _I64, _P, _P, _I64, _I64, _I64, _P, _P, _P, _P]),
    "dig_element_transfer": (_I, [_P, _P, _P, _P, _P, _I64, _I64, _I, _P, _P, _P, _P, _P, _P, _P, _I64, _I, _P,
                                  _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "dig_nb_pvalue_greater_midp": (_I, [_P, _P, _P, _I64, _P, _P]),
    "dig_nb_burden_test": (_I, [_P, _P, _P, _P, _I64, _P, _P, _P]),
    "dig_fisher_combine2": (_I, [_P, _P, _I64, _P, _P]),
    "dig_sequence_freq": (_I, [_P, _P, _I, _P, _P]),
    "dig_size_ratio": (_I, [_P, _P, _I64, _P, _P]),
    "dig_gene_scale_sums": (_I, [_P, _P, _P, _P, _P, _P, _I64, _I64, _P, _P]),
    "dig_gene_burden_test": (_I, [_P, _P, _P, _P, _P, _P, _I64, _P, _D, _D, _P, _P]),
    "dig_gene_dnds_sel": (_I, [_P, _P, _P, _P, _I64, _P, _P]),
    "dig_selection_coefficient": (_I, [_P, _P, _P, _P, _P, _I64, _P, _P, _P]),
    "dig_window_denominators": (_I, [_P, _P, _I64, _P, _P, _P]),
    "dig_site_test": (_I, [_P, _P, _P, _P, _P, _I64, _I64, _I, _P, _P, _P, _P, _P, _P, _P, _D, _P, _P, _P, _P, _P]),
    "dig_region_prob_norm": (_I, [_P, _P, _I64, _I, _P, _P]),
    "dig_position_obs": (_I, [_P, _I64, _P, _P, _P, _P, _P, _I64, _I, _I, _I, _P, _I64, _P, _P]),
    "dig_position_test": (_I, [_P, _P, _I64, _P, _P, _P, _P, _P, _I64, _I, _I, _P, _P, _P, _P, _I, _P, _P, _P, _P,
                               _P, _P, _P]),
    "dig_nb_pvalue_exact": (_I, [_P, _P, _P, _I64, _P, _P]),
    "dig_nb_pvalue_variant": (_I, [_I, _P, _P, _P, _P, _I64, _P, _P]),
    "dig_loglik": (_I, [_I, _P, _P, _P, _I64, _P, _P]),
    "dig_gene_llr_test": (_I, [_I, _P, _P, _P, _P, _P, _P, _I64, _P, _P]),
    "dig_element_region_counts": (_I, [_P, _P, _P, _P, _P, _I64, _I64, _I, _P, _P, _P, _I64, _I, _P, _P, _P, _P]),
    "dig_element_psum": (_I, [_P, _P, _P, _I64, _P, _P, _P]),
    "dig_overlap_count": (_I, [_P, _P, _P, _I64, _P, _P, _I64, _P, _P]),
    "dig_overlap_fill": (_I, [_P, _P, _P, _I64, _P, _P, _I64, _P, _P, _P, _P]),
    "dig_cds_substitution_table": (_I, [_P, _P, _I64, _P, _P, _I, _P, _P, _P, _P, _P, _I64, _P, _I, _P, _I, _P, _P,
                                        _P, _P]),
    "dig_annotate_snvs": (_I, [_P, _P, _I64, _P, _P, _I, _P, _P, _P, _P, _P, _I64, _P, _I, _P, _I, _P, _P, _P, _P,
                               _I64, _P, _P, _P]),
    "dig_codon_sites": (_I, [_P, _P, _I64, _P, _P, _I, _P, _P, _P, _P, _P, _I64, _P, _I64, _P, _P, _P, _P, _P, _P, _P]),
    "dig_codon_transfer": (_I, [_P, _P, _P, _I64, _P, _P, _P, _I64, _I64, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "dig_snv_codons": (_I, [_P, _P, _P, _P, _P, _I64, _P, _P, _P, _P, _P, _P, _P, _I64, _P, _P, _P, _P]),
}



class ScanOpts(ctypes.Structure):
    """dig_scan_opts of include/dig_b200.h."""
    _fields_ = [("workspace_d", _c.c_void_p), ("workspace_bytes", _c.c_int64), ("variant", _c.c_int32),
                ("totals_limit_kb", _c.c_uint32), ("tile_window", _c.c_int64), ("n_peer_counts3", _c.c_int32),
                ("nsum_offset_words", _c.c_int32), ("peer_counts3_d", _c.c_void_p * 8), ("mc_counts3_d", _c.c_void_p)]


SCAN_AUTO, SCAN_PER_BASE, SCAN_HEX = 0, 1, 3

_lib = None

# kernels launched per successful call (memsets not counted); summed into `launch_count` so that
# bench.py can report how many of OUR kernels ran inside a timed region
KERNELS_PER_CALL = {
    "dig_pack_genome": 1, "dig_count_contexts": 1, "dig_count_contexts_fused53": 1, "dig_synth_genome": 1, "dig_mutation_contexts": 1,
    "dig_substitution_counts": 1, "dig_count_hits": 1, "dig_tabulate_elements": 3, "dig_tabulate_genes": 2, "dig_site_counts": 1,
    "dig_element_transfer": 1, "dig_nb_pvalue_greater_midp": 1, "dig_nb_burden_test": 1, "dig_fisher_combine2": 1,
    "dig_sequence_freq": 1, "dig_size_ratio": 1, "dig_gene_scale_sums": 1, "dig_gene_burden_test": 2,
    "dig_window_denominators": 1, "dig_site_test": 1, "dig_gene_dnds_sel": 1, "dig_selection_coefficient": 1, "dig_region_prob_norm": 1, "dig_position_obs": 1, "dig_position_test": 1, "dig_nb_pvalue_exact": 1,
    "dig_nb_pvalue_variant": 1, "dig_loglik": 1, "dig_gene_llr_test": 1, "dig_overlap_count": 1, "dig_overlap_fill": 1,
    "dig_element_region_counts": 1, "dig_element_psum": 1, "dig_narrow_counts_u16": 1, "dig_peer_broadcast": 1, "dig_nmask_fill_runs": 1,
    "dig_nmask_summary": 1, "dig_cds_substitution_table": 1, "dig_annotate_snvs": 1, "dig_codon_sites": 1,
    "dig_codon_transfer": 1, "dig_snv_codons": 1,
}
launch_count = 0


class DigError(RuntimeError):
    pass


def load():
    """Load libdigb200.so; raises if it has not been built (python -m digdriver_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DigError(
            "libdigb200.so not found at %s: the CUDA extension is required (no CPU fallback). "
            "Build it with `python -m digdriver_b200.build`." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)        # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().dig_last_error()
        raise DigError("%s failed with code %d: %s" % (what or "libdigb200 call", rc, (msg or b"").decode()))


def call(name, *args):
    """Call an int-returning entry point and raise on a non-zero status."""
    global launch_count
    fn = getattr(load(), name)
    check(fn(*args), name)
    launch_count += KERNELS_PER_CALL.get(name, 0)
