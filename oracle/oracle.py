"""ctypes bindings of the CPU oracle.  TEST INFRASTRUCTURE ONLY.

`Port`  = oracle/liboracle.so, the plain-C restatement (oracle/sigmap_oracle.c).
`Ref`   = oracle/_ref/libsigmap_ref_stage.so, the unmodified reference objects behind
          oracle/ref_harness.cc (present where oracle/Makefile built it; travels to the GPU
          box with the snapshot).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module; nothing under sigmap_b200/ does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "liboracle.so")
REF_SO = os.path.join(HERE, "_ref", "libsigmap_ref_stage.so")
REF_BIN = os.path.join(HERE, "_ref", "sigmap_ref")

u32p, u64p, f32p, i16p = (C.POINTER(t) for t in (C.c_uint32, C.c_uint64, C.c_float, C.c_int16))


def _p(a, t):
    return None if a is None else a.ctypes.data_as(t)


def build(ref=True):
    """make the port (always) and the reference build (if /root/reference is mounted)."""
    subprocess.run(["make", "-s", "-C", HERE, "port"], check=True)
    if ref and os.path.isdir(os.environ.get("SIGMAP_REF", "/root/reference")):
        subprocess.run(["make", "-s", "-j8", "-C", HERE, "ref"], check=True)


class Anchor(C.Structure):
    _fields_ = [("target", C.c_uint32), ("query", C.c_uint32), ("dist", C.c_float)]


class Chain(C.Structure):
    _fields_ = [("score", C.c_float), ("contig", C.c_uint32), ("start", C.c_uint32),
                ("end", C.c_uint32), ("n_anchors", C.c_uint32), ("mapq", C.c_uint32),
                ("dir", C.c_uint32), ("anchors", C.POINTER(Anchor))]


class ChainList(C.Structure):
    _fields_ = [("chains", C.POINTER(Chain)), ("n", C.c_size_t), ("cap", C.c_size_t)]


class Params(C.Structure):
    _fields_ = [("search_radius", C.c_float), ("step", C.c_int), ("max_num_chunks", C.c_int),
                ("stop_min_anchors", C.c_int), ("output_min_anchors", C.c_int),
                ("stop_ratio", C.c_float), ("output_ratio", C.c_float),
                ("stop_mean_ratio", C.c_float), ("output_mean_ratio", C.c_float)]


class Mapping(C.Structure):
    _fields_ = [("mapped", C.c_int), ("read_len", C.c_uint32), ("q_start", C.c_uint32),
                ("q_end", C.c_uint32), ("strand_plus", C.c_uint32), ("contig", C.c_uint32),
                ("t_start", C.c_uint32), ("frag_len", C.c_uint32), ("mapq", C.c_uint32),
                ("chunks", C.c_uint32), ("n_chains", C.c_uint32), ("cm", C.c_uint32),
                ("s1", C.c_float), ("s2", C.c_float), ("sm", C.c_float), ("ad", C.c_float),
                ("at", C.c_float), ("aq", C.c_float), ("num_events", C.c_uint32)]


class ChainCounters(C.Structure):
    """orc_chain_counters: what the chaining met (sigmap_oracle.h)."""
    _fields_ = [(n, C.c_uint64) for n in (
        "max_query_hits", "max_bucket_anchors", "walks_band", "walks_skips", "walks_target_gap", "longest_walk",
        "deep_link_ranges", "traceback_hit_used", "end_ties", "primary_ties")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}

    def add(self, other):
        """fold another read's counters into these (sums; the maxima keep the larger)"""
        for n, _ in self._fields_:
            a, b = getattr(self, n), getattr(other, n)
            setattr(self, n, max(a, b) if n in ("max_query_hits", "max_bucket_anchors", "longest_walk") else a + b)


def chains_to_py(n, get_chain, get_anchors):
    out = []
    for i in range(n):
        c = get_chain(i)
        c["anchors"] = get_anchors(i, c["n_anchors"])
        out.append(c)
    return out


class Port:
    """The C restatement."""

    def __init__(self):
        if not os.path.exists(PORT_SO):
            build(ref=False)
        L = self.lib = C.CDLL(PORT_SO)
        L.orc_raw_to_pa.restype = C.c_size_t
        L.orc_raw_to_pa.argtypes = [i16p, C.c_size_t, C.c_double, C.c_double, C.c_double, f32p]
        L.orc_detect_events.restype = C.c_size_t
        L.orc_detect_events.argtypes = [f32p, C.c_size_t, f32p, f32p, u64p, C.POINTER(C.c_size_t),
                                        f32p, u64p, u64p]
        L.orc_generate_events.restype = C.c_size_t
        L.orc_generate_events.argtypes = [f32p, C.c_size_t, f32p]
        L.orc_radius_search.restype = C.c_size_t
        L.orc_radius_search.argtypes = [f32p, C.c_size_t, f32p, C.c_float, u64p, f32p, C.c_size_t]
        L.orc_generate_chains.restype = None
        L.orc_generate_chains.argtypes = [u64p, f32p, C.c_size_t, f32p, C.c_size_t, C.c_uint32,
                                          C.c_int, C.c_float, C.c_size_t, C.POINTER(ChainList)]
        L.orc_generate_chains_counted.restype = None
        L.orc_generate_chains_counted.argtypes = L.orc_generate_chains.argtypes + [C.POINTER(ChainCounters)]
        L.orc_chain_from_hits.restype = None
        L.orc_chain_from_hits.argtypes = [u64p, u32p, C.c_size_t, u64p, u64p, f32p, C.c_float,
                                          C.c_size_t, C.POINTER(ChainList)]
        L.orc_chain_list_free.argtypes = [C.POINTER(ChainList)]
        L.orc_default_params.argtypes = [C.POINTER(Params)]
        L.orc_streaming_map.restype = None
        L.orc_streaming_map.argtypes = [u64p, f32p, C.c_size_t, C.c_size_t, u32p, f32p, C.c_size_t,
                                        C.POINTER(Params), C.POINTER(Mapping)]
        L.orc_streaming_map_counted.restype = None
        L.orc_streaming_map_counted.argtypes = L.orc_streaming_map.argtypes + [C.POINTER(ChainCounters)]
        L.orc_format_paf.restype = C.c_int
        L.orc_format_paf.argtypes = [C.POINTER(Mapping), C.c_char_p, C.c_char_p, C.c_uint32,
                                     C.c_double, C.c_char_p, C.c_size_t]
        L.orc_build_point_cloud.restype = C.c_size_t
        L.orc_build_point_cloud.argtypes = [C.POINTER(C.c_char_p), u32p, C.c_size_t, f32p, u64p, f32p]

    def default_params(self):
        p = Params()
        self.lib.orc_default_params(C.byref(p))
        return p

    def raw_to_pa(self, raw, digitisation, offset, range_):
        raw = np.ascontiguousarray(raw, np.int16)
        out = np.zeros(len(raw), np.float32)
        n = self.lib.orc_raw_to_pa(_p(raw, i16p), len(raw), digitisation, offset, range_, _p(out, f32p))
        return out[:n].copy()

    def detect_events(self, x):
        x = np.ascontiguousarray(x, np.float32)
        n = len(x)
        t1, t2 = np.zeros(n + 1, np.float32), np.zeros(n + 1, np.float32)
        peaks = np.zeros(2 * n + 2, np.uint64)
        means = np.zeros(n + 2, np.float32)
        starts, lengths = np.zeros(n + 2, np.uint64), np.zeros(n + 2, np.uint64)
        npk = C.c_size_t()
        ne = self.lib.orc_detect_events(_p(x, f32p), n, _p(t1, f32p), _p(t2, f32p), _p(peaks, u64p),
                                        C.byref(npk), _p(means, f32p), _p(starts, u64p),
                                        _p(lengths, u64p))
        return dict(tstat1=t1, tstat2=t2, peaks=peaks[:npk.value].copy(), means=means[:ne].copy(),
                    starts=starts[:ne].copy(), lengths=lengths[:ne].copy())

    def generate_events(self, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.zeros(len(x) + 2, np.float32)
        n = self.lib.orc_generate_events(_p(x, f32p), len(x), _p(out, f32p))
        return out[:n].copy()

    def radius_search(self, vals, q, radius=0.08, cap=1 << 20):
        vals = np.ascontiguousarray(vals, np.float32)
        q = np.ascontiguousarray(q, np.float32)
        idx, d2 = np.zeros(cap, np.uint64), np.zeros(cap, np.float32)
        n = self.lib.orc_radius_search(_p(vals, f32p), len(vals), _p(q, f32p), radius, _p(idx, u64p),
                                       _p(d2, f32p), cap)
        assert n <= cap
        return idx[:n].copy(), d2[:n].copy()

    def new_chain_list(self):
        return ChainList(None, 0, 0)

    def generate_chains(self, pos, vals, features, query_offset, chain_list, step=2, radius=0.08,
                        n_targets=1, counters=None):
        """`counters`: a ChainCounters to add this chunk's counts to"""
        pos = np.ascontiguousarray(pos, np.uint64)
        vals = np.ascontiguousarray(vals, np.float32)
        features = np.ascontiguousarray(features, np.float32)
        self.lib.orc_generate_chains_counted(_p(pos, u64p), _p(vals, f32p), len(pos),
                                             _p(features, f32p), len(features), query_offset, step,
                                             radius, n_targets, C.byref(chain_list),
                                             None if counters is None else C.byref(counters))
        return self.chains_py(chain_list)

    def chain_from_hits(self, pos, query_pos, hit_off, hit_idx, hit_d2, chain_list, radius=0.08,
                        n_targets=1):
        pos = np.ascontiguousarray(pos, np.uint64)
        query_pos = np.ascontiguousarray(query_pos, np.uint32)
        hit_off = np.ascontiguousarray(hit_off, np.uint64)
        hit_idx = np.ascontiguousarray(hit_idx, np.uint64)
        hit_d2 = np.ascontiguousarray(hit_d2, np.float32)
        self.lib.orc_chain_from_hits(_p(pos, u64p), _p(query_pos, u32p), len(query_pos),
                                     _p(hit_off, u64p), _p(hit_idx, u64p), _p(hit_d2, f32p), radius,
                                     n_targets, C.byref(chain_list))
        return self.chains_py(chain_list)

    @staticmethod
    def chains_py(cl):
        out = []
        for i in range(cl.n):
            c = cl.chains[i]
            out.append(dict(score=np.float32(c.score), contig=c.contig, start=c.start, end=c.end,
                            n_anchors=c.n_anchors, mapq=c.mapq, dir=c.dir,
                            anchors=[(c.anchors[a].target, c.anchors[a].query,
                                      np.float32(c.anchors[a].dist)) for a in range(c.n_anchors)]))
        return out

    def free_chain_list(self, cl):
        self.lib.orc_chain_list_free(C.byref(cl))

    def streaming_map(self, pos, vals, n_targets, contig_len, pa, params=None, counters=None):
        """`counters`: a ChainCounters to add the read's counts to"""
        pos = np.ascontiguousarray(pos, np.uint64)
        vals = np.ascontiguousarray(vals, np.float32)
        contig_len = np.ascontiguousarray(contig_len, np.uint32)
        pa = np.ascontiguousarray(pa, np.float32)
        p = params or self.default_params()
        m = Mapping()
        self.lib.orc_streaming_map_counted(_p(pos, u64p), _p(vals, f32p), len(pos), n_targets,
                                           _p(contig_len, u32p), _p(pa, f32p), len(pa), C.byref(p),
                                           C.byref(m), None if counters is None else C.byref(counters))
        return m

    def format_paf(self, m, read_name, contig_name, contig_len, mt_ms=0.0):
        buf = C.create_string_buffer(2048)
        self.lib.orc_format_paf(C.byref(m), read_name.encode(), contig_name.encode(), contig_len,
                                mt_ms, buf, 2048)
        return buf.value.decode()

    def build_point_cloud(self, seqs, level_mean):
        lens = np.array([len(s) for s in seqs], np.uint32)
        bufs = [C.create_string_buffer(bytes(s), len(s) + 1) for s in seqs]
        ptrs = (C.c_char_p * len(seqs))(*[C.cast(b, C.c_char_p) for b in bufs])
        level_mean = np.ascontiguousarray(level_mean, np.float32)
        n = self.lib.orc_build_point_cloud(ptrs, _p(lens, u32p), len(seqs), _p(level_mean, f32p),
                                           None, None)
        pos, val = np.zeros(n, np.uint64), np.zeros(n, np.float32)
        self.lib.orc_build_point_cloud(ptrs, _p(lens, u32p), len(seqs), _p(level_mean, f32p),
                                       _p(pos, u64p), _p(val, f32p))
        return pos, val


class Ref:
    """The unmodified reference behind oracle/ref_harness.cc."""

    @staticmethod
    def available():
        return os.path.exists(REF_SO) and os.path.exists(REF_BIN)

    def __init__(self):
        L = self.lib = C.CDLL(REF_SO)
        L.ref_raw_to_pa.restype = C.c_size_t
        L.ref_raw_to_pa.argtypes = [i16p, C.c_size_t, C.c_double, C.c_double, C.c_double, f32p]
        L.ref_generate_events.restype = C.c_size_t
        L.ref_generate_events.argtypes = [f32p, C.c_size_t, f32p, f32p, C.c_size_t]
        L.ref_detect_events.restype = C.c_size_t
        L.ref_detect_events.argtypes = [f32p, C.c_size_t, f32p, f32p, u64p, C.POINTER(C.c_size_t),
                                        f32p, u64p, u64p, C.c_size_t]
        L.ref_index_load.restype = C.c_void_p
        L.ref_index_load.argtypes = [C.c_char_p]
        L.ref_index_free.argtypes = [C.c_void_p]
        L.ref_index_num_points.restype = C.c_size_t
        L.ref_index_num_points.argtypes = [C.c_void_p]
        L.ref_index_points.argtypes = [C.c_void_p, u64p, f32p]
        L.ref_radius_search.restype = C.c_size_t
        L.ref_radius_search.argtypes = [C.c_void_p, f32p, C.c_float, u64p, f32p, C.c_size_t]
        L.ref_chain_state_new.restype = C.c_void_p
        L.ref_chain_state_free.argtypes = [C.c_void_p]
        L.ref_chain_state_clear.argtypes = [C.c_void_p]
        L.ref_generate_chains.restype = C.c_size_t
        L.ref_generate_chains.argtypes = [C.c_void_p, C.c_void_p, f32p, C.c_size_t, C.c_uint32,
                                          C.c_int, C.c_float, C.c_size_t]
        L.ref_chain_count.restype = C.c_size_t
        L.ref_chain_count.argtypes = [C.c_void_p]
        L.ref_chain_get.argtypes = [C.c_void_p, C.c_size_t, f32p, u32p]
        L.ref_chain_anchors.argtypes = [C.c_void_p, C.c_size_t, u32p, u32p, f32p]

    def raw_to_pa(self, raw, digitisation, offset, range_):
        raw = np.ascontiguousarray(raw, np.int16)
        out = np.zeros(len(raw), np.float32)
        n = self.lib.ref_raw_to_pa(_p(raw, i16p), len(raw), digitisation, offset, range_, _p(out, f32p))
        return out[:n].copy()

    def generate_events(self, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.zeros(len(x) + 2, np.float32)
        n = self.lib.ref_generate_events(_p(x, f32p), len(x), _p(out, f32p), None, len(out))
        return out[:n].copy()

    def detect_events(self, x):
        x = np.ascontiguousarray(x, np.float32)
        n = len(x)
        t1, t2 = np.zeros(n + 1, np.float32), np.zeros(n + 1, np.float32)
        cap = 2 * n + 2
        peaks, means = np.zeros(cap, np.uint64), np.zeros(cap, np.float32)
        starts, lengths = np.zeros(cap, np.uint64), np.zeros(cap, np.uint64)
        npk = C.c_size_t()
        ne = self.lib.ref_detect_events(_p(x, f32p), n, _p(t1, f32p), _p(t2, f32p), _p(peaks, u64p),
                                        C.byref(npk), _p(means, f32p), _p(starts, u64p),
                                        _p(lengths, u64p), cap)
        return dict(tstat1=t1, tstat2=t2, peaks=peaks[:npk.value].copy(), means=means[:ne].copy(),
                    starts=starts[:ne].copy(), lengths=lengths[:ne].copy())

    def index_load(self, prefix):
        return self.lib.ref_index_load(prefix.encode())

    def index_free(self, h):
        self.lib.ref_index_free(h)

    def radius_search(self, h, q, radius=0.08, cap=1 << 20):
        q = np.ascontiguousarray(q, np.float32)
        idx, d2 = np.zeros(cap, np.uint64), np.zeros(cap, np.float32)
        n = self.lib.ref_radius_search(h, _p(q, f32p), radius, _p(idx, u64p), _p(d2, f32p), cap)
        assert n <= cap
        return idx[:n].copy(), d2[:n].copy()

    def chain_state_new(self):
        return self.lib.ref_chain_state_new()

    def chain_state_free(self, s):
        self.lib.ref_chain_state_free(s)

    def generate_chains(self, h, state, features, query_offset, step=2, radius=0.08, n_targets=1):
        features = np.ascontiguousarray(features, np.float32)
        n = self.lib.ref_generate_chains(h, state, _p(features, f32p), len(features), query_offset,
                                         step, radius, n_targets)
        out = []
        for i in range(n):
            sc = C.c_float()
            o7 = np.zeros(7, np.uint32)
            self.lib.ref_chain_get(state, i, C.byref(sc), _p(o7, u32p))
            na = int(o7[6])
            t, q, d = np.zeros(na, np.uint32), np.zeros(na, np.uint32), np.zeros(na, np.float32)
            self.lib.ref_chain_anchors(state, i, _p(t, u32p), _p(q, u32p), _p(d, f32p))
            out.append(dict(score=np.float32(sc.value), contig=int(o7[0]), start=int(o7[1]),
                            end=int(o7[2]), n_anchors=int(o7[3]), mapq=int(o7[4]), dir=int(o7[5]),
                            anchors=list(zip(t.tolist(), q.tolist(), d.tolist()))))
        return out

    @staticmethod
    def cli(args, **kw):
        """Run the reference CLI (oracle/_ref/sigmap_ref)."""
        return subprocess.run([REF_BIN] + list(args), capture_output=True, text=True, **kw)
