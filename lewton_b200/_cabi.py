"""ctypes binding of lewton_b200/liblewton_b200.so (declarations mirror include/lewton_b200.h).

There is no CPU fallback: if the library cannot be loaded the import raises, and every compute
entry point fails with LWB_ERR_NO_DEVICE when no sm_100 GPU is usable.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# LWB_LIB selects an alternative build of the same ABI (kernel tuning variants, see profiles/)
SO_PATH = os.environ.get("LWB_LIB") or os.path.join(_HERE, "liblewton_b200.so")

MAX_POSTS, MAX_CHANNELS, MAX_COUPLING, MAX_SUBMAPS, MAX_MODES = 65, 255, 256, 16, 64
OK, ERR_BAD_FORMAT, ERR_BUFFER, ERR_MISMATCH, ERR_INVALID, ERR_CUDA, ERR_NO_DEVICE = range(7)
FLOOR_TYPE_ZERO, FLOOR_TYPE_ONE = 0, 1
FLOOR_UNUSED, FLOOR_ONE, FLOOR_DENSE = 0, 1, 2
OUT_F32_PLANAR, OUT_I16_PLANAR, OUT_F32_INTERLEAVED, OUT_I16_INTERLEAVED = 0, 1, 2, 3
ENTRY_SPECTRUM, ENTRY_RESIDUE, ENTRY_VQ = 0, 1, 2
MEM_HOST, MEM_DEVICE = 0, 1

vp, u8p, fp, u32p = C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_float), C.POINTER(C.c_uint32)


class TablesRef(C.Structure):
    _fields_ = [("a", fp), ("b", fp), ("c", fp), ("window", fp), ("bitrev", u32p)]


class FloorDesc(C.Structure):
    _fields_ = [("floor_type", C.c_uint8), ("floor1_multiplier", C.c_uint8), ("floor1_values", C.c_uint8),
                ("reserved", C.c_uint8), ("floor1_x_list", C.c_uint32 * MAX_POSTS)]


class MappingDesc(C.Structure):
    _fields_ = [("coupling_steps", C.c_uint16), ("submaps", C.c_uint8), ("reserved", C.c_uint8),
                ("magnitudes", C.c_uint8 * MAX_COUPLING), ("angles", C.c_uint8 * MAX_COUPLING),
                ("mux", C.c_uint8 * (MAX_CHANNELS + 1)), ("submap_floors", C.c_uint8 * MAX_SUBMAPS)]


class ModeDesc(C.Structure):
    _fields_ = [("blockflag", C.c_uint8), ("mapping", C.c_uint8)]


class CodebookDesc(C.Structure):
    _fields_ = [("dimensions", C.c_uint16), ("reserved", C.c_uint16), ("entries", C.c_uint32), ("vq", fp)]


class ResidueDesc(C.Structure):
    _fields_ = [("residue_type", C.c_uint8), ("reserved", C.c_uint8 * 3), ("partition_size", C.c_uint32)]


class VqRun(C.Structure):
    _fields_ = [("pos", C.c_uint16), ("first", C.c_uint16), ("book", C.c_uint8), ("pass_kind", C.c_uint8), ("aux", C.c_uint8),
                ("count", C.c_uint8)]


class SetupDesc(C.Structure):
    _fields_ = [("audio_channels", C.c_uint8), ("blocksize_0", C.c_uint8), ("blocksize_1", C.c_uint8),
                ("reserved", C.c_uint8), ("tables", TablesRef * 2),
                ("n_floors", C.c_uint32), ("floors", C.POINTER(FloorDesc)),
                ("n_mappings", C.c_uint32), ("mappings", C.POINTER(MappingDesc)),
                ("n_modes", C.c_uint32), ("modes", C.POINTER(ModeDesc)),
                ("n_codebooks", C.c_uint32), ("codebooks", C.POINTER(CodebookDesc)),
                ("n_residues", C.c_uint32), ("residues", C.POINTER(ResidueDesc))]


class Packet(C.Structure):
    _fields_ = [("mode_number", C.c_uint8), ("prev_window_flag", C.c_uint8), ("next_window_flag", C.c_uint8),
                ("reserved", C.c_uint8), ("floor_kind", u8p), ("floor1_y", u32p), ("dense_floor", fp),
                ("residue", fp)]


class Chain(C.Structure):
    _fields_ = [("stream", vp), ("n_packets", C.c_uint32), ("mode_numbers", u8p),
                ("prev_window_flags", u8p), ("next_window_flags", u8p),
                ("coeff_offset", C.c_uint64), ("packet_index", C.c_uint64), ("out_offset", C.c_uint64),
                ("out_stride", C.c_uint64), ("n_samples", C.c_uint32), ("packets_done", C.c_uint32),
                ("status", C.c_int32)]


class BatchIo(C.Structure):
    _fields_ = [("entry", C.c_int), ("memory", C.c_int), ("coeffs", vp), ("dense_floor", vp),
                ("floor_kind", vp), ("floor1_y", vp), ("out_format", C.c_int), ("pcm", vp),
                ("vq_runs", vp), ("vq_run_offsets", vp), ("vq_entries", vp), ("vq_entry_offsets", vp), ("floor_memory", C.c_int)]


# name -> (restype, argtypes); every symbol include/lewton_b200.h declares
SYMBOLS = {
    "lwb_abi_version": (C.c_int, []),
    "lwb_device_count": (C.c_int, []),
    "lwb_ctx_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "lwb_ctx_destroy": (None, [vp]),
    "lwb_ctx_synchronize": (C.c_int, [vp]),
    "lwb_last_error": (C.c_char_p, [vp]),
    "lwb_ctx_cuda_stream": (vp, [vp]),
    "lwb_ctx_launch_count": (C.c_uint64, [vp]),
    "lwb_ctx_long_launch_count": (C.c_uint64, [vp]),
    "lwb_host_alloc": (vp, [C.c_size_t]),
    "lwb_bind_host_to_device": (C.c_int, [C.c_int]),
    "lwb_host_free": (None, [vp]),
    "lwb_device_alloc": (C.c_int, [vp, C.c_size_t, C.POINTER(vp)]),
    "lwb_device_free": (None, [vp, vp]),
    "lwb_memcpy_h2d": (C.c_int, [vp, vp, vp, C.c_size_t]),
    "lwb_memcpy_d2h": (C.c_int, [vp, vp, vp, C.c_size_t]),
    "lwb_tables_generate": (C.c_int, [C.c_int, vp, vp, vp, vp, vp]),
    "lwb_setup_create": (C.c_int, [vp, C.POINTER(SetupDesc), C.POINTER(vp)]),
    "lwb_setup_destroy": (None, [vp]),
    "lwb_stream_open": (C.c_int, [vp, vp, C.POINTER(vp)]),
    "lwb_stream_destroy": (None, [vp]),
    "lwb_stream_reset": (C.c_int, [vp]),
    "lwb_stream_is_empty": (C.c_int, [vp]),
    "lwb_stream_clone": (C.c_int, [vp, C.POINTER(vp)]),
    "lwb_stream_state_len": (C.c_uint32, [vp]),
    "lwb_stream_export_state": (C.c_int, [vp, vp]),
    "lwb_stream_import_state": (C.c_int, [vp, vp, C.c_uint32]),
    "lwb_decoded_sample_count": (C.c_int, [vp, C.c_uint8, C.c_int, C.c_int, C.POINTER(C.c_uint32)]),
    "lwb_decode_packet": (C.c_int, [vp, C.POINTER(Packet), C.c_int, vp, C.c_size_t, C.POINTER(C.c_size_t)]),
    "lwb_decode_spectrum": (C.c_int, [vp, C.c_uint8, C.c_int, C.c_int, vp, C.c_int, vp, C.c_size_t,
                                      C.POINTER(C.c_size_t)]),
    "lwb_decode_chains": (C.c_int, [vp, C.POINTER(Chain), C.c_size_t, C.POINTER(BatchIo)]),
    "lwb_plan_create": (C.c_int, [vp, C.POINTER(Chain), C.c_size_t, C.POINTER(BatchIo), C.POINTER(vp)]),
    "lwb_plan_execute": (C.c_int, [vp]),
    "lwb_plan_destroy": (None, [vp]),
    "lwb_debug_packet_taps": (C.c_int, [vp, C.POINTER(Packet), vp, vp, vp]),
}

_lib = None


def lib():
    """Load the shared library (raises if it is missing: there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc required; lewton_b200 has no CPU fallback)")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib
