"""ctypes binding of include/phmm_b200.h. Fails loudly when the extension is missing: there is no fallback."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libphmm_b200.so")

PHMM_OK, PHMM_ERR_INVALID, PHMM_ERR_CUDA, PHMM_ERR_BAND, PHMM_ERR_SHORT_HAPLOTYPE, PHMM_ERR_NOMEM = 0, -1, -2, -3, -4, -5
SPACE_HOST, SPACE_DEVICE = 0, 1

EXPORTS = ["phmm_version", "phmm_default_config", "phmm_create", "phmm_destroy", "phmm_last_error", "phmm_launch_count",
           "phmm_last_dp_kernel_ms", "phmm_last_dp_cells", "phmm_align_scores", "phmm_align_traceback", "phmm_align_reads", "phmm_align_pairs", "phmm_genotype_likelihoods", "phmm_populate", "phmm_populate_templates", "phmm_populate_regions", "phmm_populate_regions_ex",
           "phmm_error_model_create", "phmm_error_model_create_custom", "phmm_error_model_destroy", "phmm_error_model_last_error",
           "phmm_reset_haplotypes", "phmm_tandem_repeats", "phmm_wait_event", "phmm_engine_stream", "phmm_reserve_sms", "phmm_host_alloc", "phmm_host_free",
           "phmm_populate_ld", "phmm_device_alloc", "phmm_device_free", "phmm_ipc_export", "phmm_ipc_open", "phmm_ipc_close"]


class Config(C.Structure):
    _fields_ = [("max_indel_error", C.c_int32), ("use_int_scores", C.c_int32), ("use_mapping_quality", C.c_int32),
                ("mapping_quality_cap", C.c_int32), ("mapping_quality_cap_trigger", C.c_int32),
                ("use_flank_state", C.c_int32), ("nuc_prior", C.c_int32), ("disable_naive_shortcut", C.c_int32),
                ("map_positions", C.c_int32)]


class Haplotypes(C.Structure):
    _fields_ = [("n", C.c_int32), ("off", C.c_void_p), ("seq", C.c_void_p), ("snv_mask_fwd", C.c_void_p),
                ("snv_prior_fwd", C.c_void_p), ("snv_mask_rev", C.c_void_p), ("snv_prior_rev", C.c_void_p),
                ("gap_open", C.c_void_p), ("gap_extend", C.c_void_p), ("begin", C.c_void_p)]


class Reads(C.Structure):
    _fields_ = [("n", C.c_int32), ("off", C.c_void_p), ("bases", C.c_void_p), ("quals", C.c_void_p),
                ("mapq", C.c_void_p), ("reverse", C.c_void_p), ("begin", C.c_void_p)]


class Positions(C.Structure):
    _fields_ = [("off", C.c_void_p), ("pos", C.c_void_p)]


class FlankState(C.Structure):
    _fields_ = [("has_flank", C.c_int32), ("lhs_flank", C.c_int64), ("rhs_flank", C.c_int64)]


class Regions(C.Structure):
    _fields_ = [("n", C.c_int32), ("hap_first", C.c_void_p), ("read_first", C.c_void_p), ("flank", C.c_void_p)]


class RegionTemplates(C.Structure):
    _fields_ = [("template_first", C.c_void_p), ("template_off", C.c_void_p)]


_lib = None


def load():
    """Load libphmm_b200.so (building it first if the sources are newer). Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build
        _build.build()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("octopus_b200: CUDA extension %s is missing and could not be built" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.phmm_version.restype = C.c_char_p
    lib.phmm_default_config.argtypes = [C.POINTER(Config)]
    lib.phmm_create.restype = C.c_int
    lib.phmm_create.argtypes = [C.POINTER(C.c_void_p), C.c_int]
    lib.phmm_destroy.argtypes = [C.c_void_p]
    lib.phmm_last_error.restype = C.c_char_p
    lib.phmm_last_error.argtypes = [C.c_void_p]
    lib.phmm_launch_count.restype = C.c_int64
    lib.phmm_launch_count.argtypes = [C.c_void_p, C.c_int]
    lib.phmm_last_dp_kernel_ms.restype = C.c_double
    lib.phmm_last_dp_kernel_ms.argtypes = [C.c_void_p]
    lib.phmm_last_dp_cells.restype = C.c_int64
    lib.phmm_last_dp_cells.argtypes = [C.c_void_p]
    lib.phmm_align_scores.restype = C.c_int
    lib.phmm_align_scores.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(Haplotypes), C.POINTER(Reads),
                                      C.c_void_p, C.c_int64, C.c_void_p, C.c_int]
    lib.phmm_align_traceback.restype = C.c_int
    lib.phmm_align_traceback.argtypes = [C.c_void_p, C.c_int, C.c_char_p, C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_char_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                         C.c_char_p, C.c_char_p]
    lib.phmm_align_reads.restype = C.c_int
    lib.phmm_align_reads.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Haplotypes), C.POINTER(Reads), C.c_void_p, C.c_int64,
                                     C.POINTER(Positions), C.POINTER(FlankState), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                     C.c_void_p, C.c_int]
    lib.phmm_align_pairs.restype = C.c_int
    lib.phmm_align_pairs.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Haplotypes), C.POINTER(Reads), C.c_void_p, C.c_void_p, C.c_int64,
                                     C.POINTER(FlankState), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int]
    lib.phmm_genotype_likelihoods.restype = C.c_int
    lib.phmm_genotype_likelihoods.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int]
    lib.phmm_populate.restype = C.c_int
    lib.phmm_populate.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Haplotypes), C.POINTER(Reads),
                                  C.POINTER(Positions), C.POINTER(FlankState), C.c_void_p, C.c_void_p, C.c_int]
    lib.phmm_populate_regions.restype = C.c_int
    lib.phmm_populate_regions.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Haplotypes), C.POINTER(Reads), C.POINTER(Regions),
                                          C.c_void_p, C.c_void_p, C.c_int]
    lib.phmm_populate_regions_ex.restype = C.c_int
    lib.phmm_populate_regions_ex.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Haplotypes), C.POINTER(Reads), C.POINTER(Regions),
                                             C.POINTER(RegionTemplates), C.POINTER(Positions), C.c_void_p, C.c_void_p, C.c_int]
    lib.phmm_populate_templates.restype = C.c_int
    lib.phmm_populate_templates.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Haplotypes), C.POINTER(Reads), C.c_void_p, C.c_int32,
                                            C.POINTER(Positions), C.POINTER(FlankState), C.c_void_p, C.c_void_p, C.c_int]
    lib.phmm_populate_ld.restype = C.c_int
    lib.phmm_populate_ld.argtypes = [C.c_void_p, C.POINTER(Config), C.POINTER(Haplotypes), C.POINTER(Reads),
                                     C.POINTER(Positions), C.POINTER(FlankState), C.c_void_p, C.c_int64, C.c_void_p]
    lib.phmm_device_alloc.restype = C.c_int
    lib.phmm_device_alloc.argtypes = [C.c_int, C.c_size_t, C.POINTER(C.c_void_p)]
    lib.phmm_device_free.restype = C.c_int
    lib.phmm_device_free.argtypes = [C.c_void_p]
    lib.phmm_ipc_export.restype = C.c_int
    lib.phmm_ipc_export.argtypes = [C.c_void_p, C.c_char_p]
    lib.phmm_ipc_open.restype = C.c_int
    lib.phmm_ipc_open.argtypes = [C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]
    lib.phmm_ipc_close.restype = C.c_int
    lib.phmm_ipc_close.argtypes = [C.c_void_p]
    lib.phmm_wait_event.restype = C.c_int
    lib.phmm_wait_event.argtypes = [C.c_void_p, C.c_void_p]
    lib.phmm_reserve_sms.restype = C.c_int
    lib.phmm_reserve_sms.argtypes = [C.c_void_p, C.c_int]
    lib.phmm_engine_stream.restype = C.c_void_p
    lib.phmm_engine_stream.argtypes = [C.c_void_p]
    lib.phmm_host_alloc.restype = C.c_void_p
    lib.phmm_host_alloc.argtypes = [C.c_size_t]
    lib.phmm_host_free.argtypes = [C.c_void_p]
    lib.phmm_error_model_create.restype = C.c_int
    lib.phmm_error_model_create.argtypes = [C.POINTER(C.c_void_p), C.c_char_p]
    lib.phmm_error_model_create_custom.restype = C.c_int
    lib.phmm_error_model_create_custom.argtypes = [C.POINTER(C.c_void_p), C.c_char_p]
    lib.phmm_error_model_destroy.argtypes = [C.c_void_p]
    lib.phmm_error_model_last_error.restype = C.c_char_p
    lib.phmm_reset_haplotypes.restype = C.c_int
    lib.phmm_reset_haplotypes.argtypes = [C.c_void_p, C.c_int32] + [C.c_void_p] * 9 + [C.c_int32]
    lib.phmm_tandem_repeats.restype = C.c_int
    lib.phmm_tandem_repeats.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32]
    _lib = lib
    return lib
