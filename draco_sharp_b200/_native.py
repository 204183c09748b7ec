"""ctypes bindings of libdracob200.so (include/dracob200.h) and of the synthetic generator.

The bindings are 1:1 with the C# P/Invoke declarations in csharp/DracoBatchDecoder.cs: same
entry points, same blittable structs.  Nothing here imports the CPU oracle.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DCB_LIB") or os.path.join(HERE, "libdracob200.so")
SYNTH_PATH = os.path.join(HERE, "synth", "libdrcsynth.so")

DCB_DUMP_SYMBOLS = 1
DCB_DUMP_QINTS = 2
DCB_ORDER_ENTRIES = 0
DCB_ORDER_POINTS = 1
DCB_FACES_NONE = 0
DCB_FACES_ARENA = 1

ERR = {
    0: "DCB_OK", -1: "DCB_ERR_EOF", -2: "DCB_ERR_MAGIC", -3: "DCB_ERR_UNSUPPORTED", -4: "DCB_ERR_SCHEME",
    -5: "DCB_ERR_BITLEN", -6: "DCB_ERR_TABLE", -7: "DCB_ERR_RANS_INIT", -8: "DCB_ERR_PRED", -9: "DCB_ERR_WRAP",
    -10: "DCB_ERR_QUANT", -11: "DCB_ERR_ATTR", -12: "DCB_ERR_TAG", -13: "DCB_ERR_NUM_SYMBOLS", -14: "DCB_ERR_MAPS",
    -15: "DCB_ERR_CONNECTIVITY", -100: "DCB_ERR_ARG", -101: "DCB_ERR_NO_DEVICE", -102: "DCB_ERR_CUDA",
    -103: "DCB_ERR_OOM", -104: "DCB_ERR_STATE",
}
DCB_ERR_NO_DEVICE = -101


class BufferInfo(C.Structure):
    _fields_ = [
        ("status", C.c_int32), ("geometry_type", C.c_int32), ("encoder_method", C.c_int32),
        ("version_major", C.c_int32), ("version_minor", C.c_int32), ("flags", C.c_int32),
        ("n_points", C.c_uint32), ("n_attr_decoders", C.c_int32), ("n_attrs", C.c_int32),
        ("needs_connectivity", C.c_int32), ("device", C.c_int32), ("reserved", C.c_int32),
        ("attr_section_off", C.c_uint64),
    ]


class AttrInfo(C.Structure):
    _fields_ = [
        ("att_type", C.c_int32), ("data_type", C.c_int32), ("num_components", C.c_int32), ("normalized", C.c_int32),
        ("unique_id", C.c_uint32), ("seq_decoder_type", C.c_int32), ("decoder_id", C.c_int32),
        ("pred_method", C.c_int32), ("transform", C.c_int32), ("scheme", C.c_int32), ("precision_bits", C.c_int32),
        ("n_entries", C.c_uint32), ("out_bytes", C.c_uint64), ("out_off", C.c_uint64), ("dbg_off", C.c_uint64),
        ("xf_a", C.c_int32), ("xf_b", C.c_int32), ("q_min", C.c_float * 4), ("q_range", C.c_float),
        ("q_bits", C.c_int32), ("resolved", C.c_int32),
    ]


class FaceInfo(C.Structure):
    _fields_ = [
        ("out_off", C.c_uint64), ("out_bytes", C.c_uint64), ("n_faces", C.c_uint64), ("source", C.c_int32),
        ("reserved", C.c_int32),
    ]


class LaunchStats(C.Structure):
    _fields_ = [
        ("n_launches", C.c_int32), ("n_streams", C.c_int32), ("n_waves", C.c_int32), ("lanes_per_warp", C.c_int32),
        ("smem_per_stream", C.c_uint64), ("ms_total", C.c_float), ("ms_dominant", C.c_float),
        ("ms_raw", C.c_float), ("ms_tag", C.c_float), ("ms_par", C.c_float), ("ms_para", C.c_float),
        ("algo_bytes_dominant", C.c_uint64), ("dominant_name", C.c_char * 96),
    ]


class SynthSpec(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("n_points", C.c_uint32), ("pos_bits", C.c_int32), ("rho_num", C.c_int32),
        ("rho_den", C.c_int32), ("scheme", C.c_int32), ("normal_bits", C.c_int32), ("colors", C.c_int32),
        ("color_step", C.c_int32), ("reserved", C.c_int32),
    ]


class SynthTruth(C.Structure):
    _fields_ = [
        ("pos_q", C.c_void_p), ("nrm_st", C.c_void_p), ("rgb", C.c_void_p),
        ("scheme", C.c_int32 * 3), ("sums", C.c_uint64 * 3),
    ]


# every symbol include/dracob200.h declares: (name, restype, argtypes)
_P = C.c_void_p
EXPORTS = [
    ("dcb_version", C.c_int, []),
    ("dcb_device_count", C.c_int, []),
    ("dcb_error_string", C.c_char_p, [C.c_int]),
    ("dcb_create", C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(_P)]),
    ("dcb_destroy", None, [_P]),
    ("dcb_set_stream", C.c_int, [_P, C.c_int, _P]),
    ("dcb_set_limits", C.c_int, [_P, C.c_uint64, C.c_uint64]),
    ("dcb_index", C.c_int, [_P, C.POINTER(_P), C.POINTER(C.c_uint64), C.c_int, C.POINTER(_P)]),
    ("dcb_index_arena", C.c_int, [_P, _P, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int, C.POINTER(_P)]),
    ("dcb_get_buffer_info", C.c_int, [_P, C.c_int, C.POINTER(BufferInfo)]),
    ("dcb_get_attr_info", C.c_int, [_P, C.c_int, C.c_int, C.POINTER(AttrInfo)]),
    ("dcb_batch_out_bytes", C.c_uint64, [_P]),
    ("dcb_batch_dbg_bytes", C.c_uint64, [_P]),
    ("dcb_batch_in_bytes", C.c_uint64, [_P]),
    ("dcb_batch_points", C.c_uint64, [_P]),
    ("dcb_batch_algo_bytes", C.c_uint64, [_P]),
    ("dcb_set_attr_section", C.c_int, [_P, C.c_int, C.c_uint64, C.c_uint32]),
    ("dcb_set_mesh_maps", C.c_int, [_P, C.c_int, C.c_int, _P, _P, C.c_uint64, _P, C.c_uint64, _P, C.c_uint64]),
    ("dcb_host_connectivity", C.c_int, [_P, C.c_int]),
    ("dcb_mesh_faces", C.c_int, [_P, C.c_int, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    ("dcb_mesh_map", C.c_int, [_P, C.c_int, C.c_int, C.c_int, _P, C.c_uint64, C.POINTER(C.c_uint64)]),
    ("dcb_index_finish", C.c_int, [_P, _P]),
    ("dcb_set_output_order", C.c_int, [_P, C.c_int]),
    ("dcb_set_mesh_faces", C.c_int, [_P, C.c_int, _P, C.c_uint64]),
    ("dcb_set_face_output", C.c_int, [_P, C.c_int]),
    ("dcb_get_face_info", C.c_int, [_P, C.c_int, C.POINTER(FaceInfo)]),
    ("dcb_decode", C.c_int, [_P, _P, _P, _P, C.c_uint32]),
    ("dcb_decode_scatter", C.c_int, [_P, _P, C.POINTER(_P), C.c_int, C.c_uint32]),
    ("dcb_upload", C.c_int, [_P, _P]),
    ("dcb_decode_resident", C.c_int, [_P, _P, _P, _P, C.c_uint32]),
    ("dcb_download", C.c_int, [_P, _P, _P, _P]),
    ("dcb_device_out", _P, [_P, C.c_int]),
    ("dcb_sync", C.c_int, [_P]),
    ("dcb_status", C.c_int, [_P, C.c_int]),
    ("dcb_batch_free", None, [_P]),
    ("dcb_last_stats", C.c_int, [_P, C.POINTER(LaunchStats)]),
]

_lib = None
_synth = None


def lib():
    """The product library.  Raises if it has not been built: there is no Python/CPU fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libdracob200.so is missing (%s): build it with `python -m draco_sharp_b200.build`; "
                "there is no CPU fallback" % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, res, args in EXPORTS:
            f = getattr(l, name)
            f.restype = res
            f.argtypes = args
        _lib = l
    return _lib


def synth():
    global _synth
    if _synth is None:
        if not os.path.exists(SYNTH_PATH):
            raise RuntimeError("libdrcsynth.so is missing: python -m draco_sharp_b200.build")
        s = C.CDLL(SYNTH_PATH)
        s.synth_cloud.restype = C.c_int64
        s.synth_cloud.argtypes = [C.POINTER(SynthSpec), _P, C.c_uint64, C.POINTER(SynthTruth)]
        s.synth_batch.restype = C.c_int64
        s.synth_batch.argtypes = [C.POINTER(SynthSpec), C.c_uint32, C.c_int, _P, C.c_uint64, _P, _P, _P, _P]
        s.synth_grid_topology.restype = C.c_int64
        s.synth_grid_topology.argtypes = [C.c_uint32, C.c_uint32, _P, _P, _P, _P]
        s.synth_grid_mesh.restype = C.c_int64
        s.synth_grid_mesh.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, C.c_uint64,
                                      C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), _P, C.POINTER(C.c_int32)]
        s.synth_word_checksum.restype = C.c_uint64
        s.synth_word_checksum.argtypes = [_P, C.c_uint64]
        _synth = s
    return _synth


class DracoError(RuntimeError):
    def __init__(self, code, what=""):
        self.code = code
        msg = lib().dcb_error_string(code).decode() if _lib is not None else ""
        super().__init__("%s (%s)%s" % (ERR.get(code, str(code)), msg, (": " + what) if what else ""))


def check(code, what=""):
    if code != 0:
        raise DracoError(code, what)
