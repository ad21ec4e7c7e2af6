"""ctypes binding of include/sigmap_b200.h (the C ABI of libsigmap_b200.so).

The library is built in-tree by ``sigmap_b200/csrc/Makefile`` (``__graft_entry__.build()``)
into ``sigmap_b200/lib/libsigmap_b200.so``.  There is no Python or CPU fallback: if the
shared object is missing, importing this module raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SIGMAP_B200_LIB", os.path.join(_HERE, "lib", "libsigmap_b200.so"))
if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `make -C sigmap_b200/csrc` "
        "(or `python -c 'import __graft_entry__ as g; g.build()'`); there is no fallback path"
    )
lib = C.CDLL(LIB_PATH)

SMB_OK = 0
SMB_CHUNK = 4000
SMB_DIM = 6
SMB_MAX_HITS = 5000

u8p = C.POINTER(C.c_uint8)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
i16p = C.POINTER(C.c_int16)
f32p = C.POINTER(C.c_float)
charpp = C.POINTER(C.c_char_p)


class Params(C.Structure):
    """smb_params: the reference CLI's mapping knobs (sigmap.cc:1380-1419)."""

    _fields_ = [
        ("search_radius", C.c_float),
        ("step_size", C.c_int32),
        ("max_num_chunks", C.c_int32),
        ("min_num_anchors", C.c_int32),
        ("min_num_anchors_output", C.c_int32),
        ("stop_mapping", C.c_float),
        ("stop_mapping_output", C.c_float),
        ("stop_mapping_mean", C.c_float),
        ("stop_mapping_mean_output", C.c_float),
    ]


class Mapping(C.Structure):
    """smb_mapping: one PAF row's numeric content."""

    _fields_ = [
        ("mapped", C.c_uint32),
        ("read_len", C.c_uint32),
        ("q_start", C.c_uint32),
        ("q_end", C.c_uint32),
        ("strand_plus", C.c_uint32),
        ("contig", C.c_uint32),
        ("t_start", C.c_uint32),
        ("frag_len", C.c_uint32),
        ("mapq", C.c_uint32),
        ("chunks", C.c_uint32),
        ("n_chains", C.c_uint32),
        ("cm", C.c_uint32),
        ("s1", C.c_float),
        ("s2", C.c_float),
        ("sm", C.c_float),
        ("ad", C.c_float),
        ("at", C.c_float),
        ("aq", C.c_float),
        ("num_events", C.c_uint32),
        ("flags", C.c_uint32),
    ]


class Chain(C.Structure):
    _fields_ = [
        ("score", C.c_float),
        ("contig", C.c_uint32),
        ("start", C.c_uint32),
        ("end", C.c_uint32),
        ("n_anchors", C.c_uint32),
        ("mapq", C.c_uint32),
        ("dir", C.c_uint32),
    ]


class Anchor(C.Structure):
    _fields_ = [("target", C.c_uint32), ("query", C.c_uint32), ("dist", C.c_float)]


class Stats(C.Structure):
    _fields_ = [
        ("samples", C.c_uint64),
        ("raw_events", C.c_uint64),
        ("events", C.c_uint64),
        ("queries", C.c_uint64),
        ("hits", C.c_uint64),
        ("anchors", C.c_uint64),
        ("capped_queries", C.c_uint64),
        ("chunks", C.c_uint64),
        ("steps", C.c_uint64),
        ("launches", C.c_uint64),
        ("ms_events", C.c_double),
        ("ms_search", C.c_double),
        ("ms_sort", C.c_double),
        ("ms_chain", C.c_double),
        ("ms_filter", C.c_double),
        ("ms_total", C.c_double),
        ("search_launches", C.c_uint64),
        ("h2d_bytes", C.c_uint64),
        ("d2h_bytes", C.c_uint64),
        ("linked", C.c_uint64),
        ("seg_sort_steps", C.c_uint64),
        ("exchanges", C.c_uint64),
        ("part_sort_steps", C.c_uint64),
        ("overflow_queries", C.c_uint64),
        ("sync_points", C.c_uint64),
        ("ms_stream_stage", C.c_double),
        ("pending", C.c_uint64),
    ]


class Fasta(C.Structure):
    _fields_ = [("n", C.c_uint32), ("names", charpp), ("seqs", charpp), ("lengths", u32p)]


class Reads(C.Structure):
    _fields_ = [
        ("n", C.c_size_t),
        ("names", charpp),
        ("read_off", u64p),
        ("raw", i16p),
        ("digitisation", f32p),
        ("range", f32p),
        ("offset", f32p),
    ]


class CloudPart(C.Structure):
    _fields_ = [
        ("n_values", C.c_size_t),
        ("n_runs", C.c_size_t),
        ("n_points_total", C.c_uint64),
        ("pos", u64p),
        ("val", f32p),
        ("own", u8p),
        ("run_off", u64p),
        ("run_first", u64p),
    ]


class BuildStats(C.Structure):
    _fields_ = [
        ("points", C.c_uint64),
        ("tiles", C.c_uint64),
        ("tiles_rewalked", C.c_uint64),
        ("tiles_unconverged", C.c_uint64),
        ("tiles_redone", C.c_uint64),
        ("tile", C.c_uint64),
        ("strands", C.c_uint32),
        ("strands_serial_mean", C.c_uint32),
    ] + [(f"ms_{k}", C.c_double) for k in ("upload", "census", "levels", "zsums", "select", "scatter", "index")]


# name -> (restype, argtypes); every symbol include/sigmap_b200.h declares
PROTOTYPES = {
    "smb_default_params": (None, [C.POINTER(Params)]),
    "smb_device_count": (C.c_int, []),
    "smb_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "smb_destroy": (None, [C.c_void_p]),
    "smb_last_error": (C.c_char_p, [C.c_void_p]),
    "smb_stats_reset": (None, [C.c_void_p]),
    "smb_stats_get": (C.c_int, [C.c_void_p, C.POINTER(Stats)]),
    "smb_timer_start": (C.c_int, [C.c_void_p]),
    "smb_timer_stop": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "smb_set_limits": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint64]),
    "smb_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p]),
    "smb_index_load": (C.c_int, [C.c_void_p, C.c_char_p]),
    "smb_index_set_points": (C.c_int, [C.c_void_p, u64p, f32p, C.c_size_t]),
    "smb_index_set_contigs": (C.c_int, [C.c_void_p, u32p, C.c_uint32]),
    "smb_index_num_points": (C.c_uint64, [C.c_void_p]),
    "smbh_assign_contigs": (C.c_int, [u32p, C.c_uint32, C.c_uint32, u32p]),
    "smb_shard_local_group": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint32]),
    "smb_shard_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "smb_shard_nccl_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_char_p]),
    "smb_shard_rank": (C.c_int, [C.c_void_p]),
    "smb_shard_world": (C.c_int, [C.c_void_p]),
    "smb_index_set_points_sharded": (C.c_int, [C.c_void_p, u64p, f32p, C.c_size_t, u32p,
                                               C.c_uint32]),
    "smb_index_set_points_part": (C.c_int, [C.c_void_p, C.POINTER(CloudPart), C.c_uint32]),
    "smbh_build_point_cloud_part": (C.c_int, [charpp, u32p, C.c_uint32, f32p, u32p, C.c_uint32,
                                              C.POINTER(CloudPart)]),
    "smbh_cloud_part_free": (None, [C.POINTER(CloudPart)]),
    "smb_index_num_contigs": (C.c_uint32, [C.c_void_p]),
    "smb_index_broadcast": (C.c_int, [C.c_void_p, C.c_int]),
    "smb_point_cloud_build": (C.c_int, [C.c_void_p, charpp, u32p, C.c_uint32, f32p, C.POINTER(u64p),
                                        C.POINTER(f32p), C.POINTER(C.c_size_t)]),
    "smb_point_cloud_build_part": (C.c_int, [C.c_void_p, charpp, u32p, C.c_uint32, f32p, u32p, C.c_uint32,
                                             C.POINTER(CloudPart)]),
    "smb_index_build": (C.c_int, [C.c_void_p, charpp, u32p, C.c_uint32, f32p, u32p]),
    "smb_index_build_stats": (C.c_int, [C.c_void_p, C.POINTER(BuildStats)]),
    "smb_map_reads": (C.c_int, [C.c_void_p, i16p, u64p, f32p, f32p, f32p, C.c_size_t,
                                C.POINTER(Params), C.POINTER(Mapping)]),
    "smb_map_reads_device": (C.c_int, [C.c_void_p, C.c_void_p, u64p, u32p, f32p, f32p, f32p, C.c_size_t,
                                       C.POINTER(Params), C.POINTER(Mapping), C.c_void_p]),
    "smb_reads_upload": (C.c_int, [C.c_void_p, i16p, u64p, f32p, f32p, f32p, C.c_size_t]),
    "smb_map_uploaded": (C.c_int, [C.c_void_p, C.POINTER(Params), C.POINTER(Mapping)]),
    "smb_stage_raw_to_pa": (C.c_int, [C.c_void_p, i16p, C.c_size_t, C.c_float, C.c_float,
                                      C.c_float, f32p, C.POINTER(C.c_size_t)]),
    "smb_stage_events": (C.c_int, [C.c_void_p, f32p, C.c_size_t, f32p, u32p]),
    "smb_stage_detect": (C.c_int, [C.c_void_p, f32p, f32p, f32p, u32p, u32p, f32p, u32p]),
    "smb_stage_radius": (C.c_int, [C.c_void_p, f32p, C.c_size_t, C.c_float, u64p, u64p, f32p,
                                   C.c_uint64]),
    "smb_batch_create": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]),
    "smb_batch_destroy": (None, [C.c_void_p]),
    "smb_batch_reset": (C.c_int, [C.c_void_p]),
    "smb_batch_generate_chains": (C.c_int, [C.c_void_p, u32p, C.c_uint32, f32p, u32p,
                                            C.POINTER(Params)]),
    "smb_batch_chain_count": (C.c_int, [C.c_void_p, C.c_uint32, u32p]),
    "smb_batch_get_chains": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(Chain), C.c_uint32]),
    "smb_batch_get_anchors": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.POINTER(Anchor),
                                        C.c_uint32]),
    "smb_stream_open": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(Params)]),
    "smb_stream_begin_read": (C.c_int, [C.c_void_p, C.c_uint32, C.c_float, C.c_float, C.c_float]),
    "smb_stream_round": (C.c_int, [C.c_void_p, u32p, C.c_uint32, i16p, u32p, u8p,
                                   C.POINTER(Mapping)]),
    "smb_stream_close": (C.c_int, [C.c_void_p]),
    "smbh_format_paf": (C.c_int, [C.POINTER(Mapping), C.c_char_p, C.c_char_p, C.c_uint32,
                                  C.c_double, C.c_char_p, C.c_size_t]),
    "smbh_pore_model_load": (C.c_int, [C.c_char_p, f32p, f32p]),
    "smbh_fasta_load": (C.c_int, [C.c_char_p, C.POINTER(Fasta)]),
    "smbh_fasta_free": (None, [C.POINTER(Fasta)]),
    "smbh_fasta_write": (C.c_int, [C.c_char_p, charpp, charpp, u32p, C.c_uint32]),
    "smbh_build_point_cloud": (C.c_size_t, [charpp, u32p, C.c_uint32, f32p, u64p, f32p]),
    "smbh_build_point_cloud_alloc": (C.c_int, [charpp, u32p, C.c_uint32, f32p, C.POINTER(u64p), C.POINTER(f32p),
                                              C.POINTER(C.c_size_t)]),
    "smbh_pt_write": (C.c_int, [C.c_char_p, u64p, f32p, C.c_size_t, C.c_int, C.c_int]),
    "smbh_pt_read": (C.c_int, [C.c_char_p, C.POINTER(u64p), C.POINTER(f32p),
                               C.POINTER(C.c_size_t), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "smbh_si_write": (C.c_int, [C.c_char_p, f32p, C.c_size_t, C.c_int, C.c_int]),
    "smbh_free": (None, [C.c_void_p]),
    "smbh_blow5_write": (C.c_int, [C.c_char_p, charpp, i16p, u64p, C.c_size_t, C.c_double,
                                   C.c_double, C.c_double, C.c_double]),
    "smbh_blow5_read": (C.c_int, [C.c_char_p, C.POINTER(Reads)]),
    "smbh_reads_free": (None, [C.POINTER(Reads)]),
    "smbh_last_error": (C.c_char_p, []),
    "smbh_sim_reference": (C.c_int, [C.c_uint64, u32p, C.c_uint32, charpp]),
    "smbh_sim_reads": (C.c_int, [C.c_uint64, charpp, u32p, C.c_uint32, f32p, f32p, C.c_uint64,
                                 C.c_uint64, C.c_uint32, C.c_uint32, C.c_float, u64p, i16p, u32p]),
}

MISSING = []
for _name, (_res, _args) in PROTOTYPES.items():
    try:
        _fn = getattr(lib, _name)
    except AttributeError:
        MISSING.append(_name)
        continue
    _fn.restype = _res
    _fn.argtypes = _args


def ptr(a, typ):
    """numpy array -> typed ctypes pointer (None passes NULL)."""
    if a is None:
        return None
    return a.ctypes.data_as(typ)
