"""Python face of the B200 mapping engine: a thin mirror of the reference's operator
interface for the hot path, on top of the C ABI (include/sigmap_b200.h).

Reference interface mirrored (names kept so parity tests read like the reference's code):
  SpatialIndex::Load                      spatial_index.cc:132   -> Mapper.Load / load_index
  Sigmap::GenerateEvents                  sigmap.cc:1048         -> Mapper.GenerateEvents
  index->radiusSearch                     spatial_index.cc:366   -> Mapper.radiusSearch
  SpatialIndex::GenerateChains            spatial_index.cc:276   -> ChainBatch.GenerateChains
  Sigmap::StreamingMap (per-read body)    sigmap.cc:630-866      -> Mapper.StreamingMap
All compute happens in libsigmap_b200.so on the GPU; this module only marshals numpy arrays.
There is no CPU fallback: constructing a Mapper without a CUDA device raises.
"""
import collections.abc
import ctypes as C

import numpy as np

from . import _ffi as F
from .host import format_paf  # noqa: F401  (re-exported)

CHUNK = F.SMB_CHUNK


class SigmapError(RuntimeError):
    pass


def default_params(**overrides):
    p = F.Params()
    F.lib.smb_default_params(C.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise AttributeError(f"smb_params has no field {k}")
        setattr(p, k, v)
    return p


def full_read_params(**overrides):
    """CLI equivalent: --max-num-chunks 100000 --stop-mapping 1e30 --stop-mapping-mean 1e30
    --min-num-anchors 2000000000 (every chunk of every read is consumed; SURVEY.md 8d)."""
    kw = dict(max_num_chunks=100000, stop_mapping=1e30, stop_mapping_mean=1e30,
              min_num_anchors=2000000000)
    kw.update(overrides)
    return default_params(**kw)


class Rows(collections.abc.Sequence):
    """The smb_mapping rows of a mapping call: a read-only sequence over the ctypes array the
    library filled (no per-row Python work inside the call: 100 000 rows cost 45 ms as a list)."""

    __slots__ = ("_arr", "_n")

    def __init__(self, arr, n):
        self._arr, self._n = arr, n

    def __len__(self):
        return self._n

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self._arr[k] for k in range(*i.indices(self._n))]
        if i < 0:
            i += self._n
        if not 0 <= i < self._n:
            raise IndexError(i)
        return self._arr[i]


class Mapper:
    def __init__(self, device=0):
        self._ctx = C.c_void_p()
        rc = F.lib.smb_create(C.byref(self._ctx), device)
        if rc != 0:
            msg = F.lib.smb_last_error(None).decode()
            self._ctx = None
            raise SigmapError(f"smb_create failed ({rc}): {msg}")
        self.device = device
        self.contig_lengths = None

    def close(self):
        if self._ctx:
            F.lib.smb_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise SigmapError(f"{what} failed ({rc}): {F.lib.smb_last_error(self._ctx).decode()}")

    # ------------------------------------------------------------------ index
    def load_index(self, prefix):
        self._check(F.lib.smb_index_load(self._ctx, prefix.encode()), "smb_index_load")

    Load = load_index

    def set_index(self, pos, val):
        pos = np.ascontiguousarray(pos, np.uint64)
        val = np.ascontiguousarray(val, np.float32)
        self._check(F.lib.smb_index_set_points(self._ctx, F.ptr(pos, F.u64p), F.ptr(val, F.f32p),
                                               len(pos)), "smb_index_set_points")

    def set_index_sharded(self, pos, val, contig_owner):
        """Contig-sharded index: keep only the windows of contigs with contig_owner[c] == this
        context's shard rank (join a group first: shard.ContigShardGroup / shard.nccl_join)."""
        pos = np.ascontiguousarray(pos, np.uint64)
        val = np.ascontiguousarray(val, np.float32)
        owner = np.ascontiguousarray(contig_owner, np.uint32)
        self._check(F.lib.smb_index_set_points_sharded(self._ctx, F.ptr(pos, F.u64p),
                                                       F.ptr(val, F.f32p), len(pos),
                                                       F.ptr(owner, F.u32p), len(owner)),
                    "smb_index_set_points_sharded")

    def set_index_part(self, part, n_contigs):
        """Contig-sharded index from this rank's own part of the cloud
        (host.build_point_cloud_part with this context's shard rank)."""
        self._check(F.lib.smb_index_set_points_part(self._ctx, C.byref(part.c), n_contigs),
                    "smb_index_set_points_part")

    def build_index(self, ref, level_mean, owner=None):
        """Build the device index from the reference sequences on this GPU (smb_index_build): the
        index set_index builds from host.build_point_cloud, with no point cloud in host memory.
        owner: contig -> shard rank table; this context's shard only (join a group first).
        Sets the contig lengths too."""
        level_mean = np.ascontiguousarray(level_mean, np.float32)
        own = None if owner is None else np.ascontiguousarray(owner, np.uint32)
        self._check(F.lib.smb_index_build(self._ctx, ref.seq_ptrs, F.ptr(ref.lengths, F.u32p), ref.n,
                                          F.ptr(level_mean, F.f32p), F.ptr(own, F.u32p)), "smb_index_build")
        self.set_contigs(ref.lengths)

    def point_cloud(self, ref, level_mean):
        """(pos uint64[n], val float32[n]) built on this GPU: equal to host.build_point_cloud."""
        level_mean = np.ascontiguousarray(level_mean, np.float32)
        pp, vp, n = F.u64p(), F.f32p(), C.c_size_t()
        self._check(F.lib.smb_point_cloud_build(self._ctx, ref.seq_ptrs, F.ptr(ref.lengths, F.u32p), ref.n,
                                                F.ptr(level_mean, F.f32p), C.byref(pp), C.byref(vp),
                                                C.byref(n)), "smb_point_cloud_build")
        try:
            pos = np.ctypeslib.as_array(pp, (max(n.value, 1),))[:n.value].copy()
            val = np.ctypeslib.as_array(vp, (max(n.value, 1),))[:n.value].copy()
        finally:
            F.lib.smbh_free(pp)
            F.lib.smbh_free(vp)
        return pos, val

    def point_cloud_part(self, ref, level_mean, owner, rank):
        """Shard `rank`'s part of the point cloud built on this GPU: equal to
        host.build_point_cloud_part (a host.CloudPart)."""
        from .host import CloudPart
        level_mean = np.ascontiguousarray(level_mean, np.float32)
        owner = np.ascontiguousarray(owner, np.uint32)
        c = F.CloudPart()
        self._check(F.lib.smb_point_cloud_build_part(self._ctx, ref.seq_ptrs, F.ptr(ref.lengths, F.u32p), ref.n,
                                                     F.ptr(level_mean, F.f32p), F.ptr(owner, F.u32p), rank,
                                                     C.byref(c)), "smb_point_cloud_build_part")
        return CloudPart(c)

    def build_stats(self):
        """Tiles and per-stage device milliseconds of the last device cloud build."""
        s = F.BuildStats()
        self._check(F.lib.smb_index_build_stats(self._ctx, C.byref(s)), "smb_index_build_stats")
        return {k: getattr(s, k) for k, _ in F.BuildStats._fields_}

    def broadcast_index(self, root=0):
        """Read-sharded runs: receive (or, on `root`, send) the device index over NVLink instead of
        building it on every rank.  Collective over the joined group; contig lengths travel too."""
        self._check(F.lib.smb_index_broadcast(self._ctx, root), "smb_index_broadcast")
        n = F.lib.smb_index_num_contigs(self._ctx)
        if self.contig_lengths is None or len(self.contig_lengths) != n:
            self.contig_lengths = None  # the caller sets them with set_contigs() for PAF formatting

    @property
    def shard_rank(self):
        return F.lib.smb_shard_rank(self._ctx)

    @property
    def shard_world(self):
        return F.lib.smb_shard_world(self._ctx)

    def set_contigs(self, lengths):
        lengths = np.ascontiguousarray(lengths, np.uint32)
        self.contig_lengths = lengths
        self._check(F.lib.smb_index_set_contigs(self._ctx, F.ptr(lengths, F.u32p), len(lengths)),
                    "smb_index_set_contigs")

    @property
    def num_points(self):
        return F.lib.smb_index_num_points(self._ctx)

    def set_limits(self, max_batch_chunks=0, max_batch_anchors=0):
        self._check(F.lib.smb_set_limits(self._ctx, max_batch_chunks, max_batch_anchors),
                    "smb_set_limits")

    def set_option(self, name, value):
        """Run-time switch (an SMB_<NAME> environment variable without the prefix): A/B
        measurements, and tests that have to reach the fallback paths."""
        self._check(F.lib.smb_set_option(self._ctx, str(name).encode(), str(value).encode()),
                    "smb_set_option")

    def timer_start(self):
        self._check(F.lib.smb_timer_start(self._ctx), "smb_timer_start")

    def timer_stop(self):
        ms = C.c_double()
        self._check(F.lib.smb_timer_stop(self._ctx, C.byref(ms)), "smb_timer_stop")
        return ms.value

    # ------------------------------------------------------------------ stats
    def stats_reset(self):
        F.lib.smb_stats_reset(self._ctx)

    def stats(self):
        s = F.Stats()
        self._check(F.lib.smb_stats_get(self._ctx, C.byref(s)), "smb_stats_get")
        return {k: getattr(s, k) for k, _ in F.Stats._fields_}

    # ------------------------------------------------------------------ whole path
    def upload_reads(self, reads):
        self._check(F.lib.smb_reads_upload(self._ctx, F.ptr(reads.raw, F.i16p),
                                           F.ptr(reads.read_off, F.u64p),
                                           F.ptr(reads.digitisation, F.f32p),
                                           F.ptr(reads.range, F.f32p), F.ptr(reads.offset, F.f32p),
                                           reads.n), "smb_reads_upload")
        self._n_uploaded = reads.n

    def map_uploaded(self, params=None):
        params = params or default_params()
        out = (F.Mapping * max(self._n_uploaded, 1))()
        self._check(F.lib.smb_map_uploaded(self._ctx, C.byref(params), out), "smb_map_uploaded")
        return Rows(out, self._n_uploaded)

    def map_reads(self, reads, params=None):
        """Raw host reads in, PAF rows out (host<->device copies included)."""
        params = params or default_params()
        out = (F.Mapping * max(reads.n, 1))()
        self._check(F.lib.smb_map_reads(self._ctx, F.ptr(reads.raw, F.i16p),
                                        F.ptr(reads.read_off, F.u64p),
                                        F.ptr(reads.digitisation, F.f32p), F.ptr(reads.range, F.f32p),
                                        F.ptr(reads.offset, F.f32p), reads.n, C.byref(params), out),
                    "smb_map_reads")
        return Rows(out, reads.n)

    StreamingMap = map_reads

    def map_device(self, raw, read_start, read_len, digitisation, range_, offset, params=None,
                   stream=None):
        """Map reads whose samples are already in device memory (smb_map_reads_device): raw is a
        contiguous torch.int16 CUDA tensor on this mapper's device, of any shape, read as flat
        elements; read r is raw.view(-1)[read_start[r] : read_start[r] + read_len[r]].  The samples
        are not copied, and raw is not written.  The per-read tables are host arrays (or tensors).
        The call's device work is ordered after what is queued on `stream` (a torch.cuda.Stream or
        a cudaStream_t handle; default: the device's current torch stream).  Returns the rows
        map_reads returns for the same samples."""
        import torch
        if not isinstance(raw, torch.Tensor):
            raise SigmapError(f"map_device: raw must be a torch tensor, not {type(raw).__name__}")
        if raw.dtype != torch.int16:
            raise SigmapError(f"map_device: raw must be torch.int16, not {raw.dtype}")
        if raw.device != torch.device("cuda", self.device):
            raise SigmapError(f"map_device: raw is on {raw.device}, this mapper runs on cuda:{self.device}")
        if not raw.is_contiguous():
            raise SigmapError("map_device: raw must be contiguous")

        def table(x, dtype):
            if isinstance(x, torch.Tensor):
                x = x.cpu().numpy()
            return np.ascontiguousarray(x, dtype).reshape(-1)

        start, length = table(read_start, np.uint64), table(read_len, np.uint32)
        dig, rng, off = table(digitisation, np.float32), table(range_, np.float32), table(offset, np.float32)
        n = len(start)
        if not len(length) == len(dig) == len(rng) == len(off) == n:
            raise SigmapError("map_device: read_start, read_len, digitisation, range_ and offset "
                              "must have one entry per read")
        if n and int((start + length).max()) > raw.numel():
            raise SigmapError(f"map_device: a read ends past the {raw.numel()} elements of raw")
        if stream is None:
            stream = torch.cuda.current_stream(raw.device)
        handle = stream.cuda_stream if isinstance(stream, torch.cuda.Stream) else int(stream)
        params = params or default_params()
        out = (F.Mapping * max(n, 1))()
        self._check(F.lib.smb_map_reads_device(self._ctx, raw.data_ptr(), F.ptr(start, F.u64p),
                                               F.ptr(length, F.u32p), F.ptr(dig, F.f32p), F.ptr(rng, F.f32p),
                                               F.ptr(off, F.f32p), n, C.byref(params), out, handle),
                    "smb_map_reads_device")
        return Rows(out, n)

    def map_device_padded(self, batch, lengths, digitisation, range_, offset, params=None,
                          stream=None):
        """map_device over the rows of a padded [n, stride] batch: read r is batch[r, :lengths[r]]."""
        if batch.dim() != 2:
            raise SigmapError(f"map_device_padded: batch must be [n, stride], not {list(batch.shape)}")
        n, stride = batch.shape
        read_start = np.arange(n, dtype=np.uint64) * np.uint64(stride)
        return self.map_device(batch, read_start, lengths, digitisation, range_, offset, params, stream)

    def paf_lines(self, reads, rows, contig_names, mt_ms=0.0):
        out = []
        for name, m in zip(reads.names, rows):
            cn = contig_names[m.contig] if m.mapped else ""
            cl = int(self.contig_lengths[m.contig]) if m.mapped else 0
            out.append(format_paf(m, name, cn, cl, mt_ms))
        return out

    # ------------------------------------------------------------------ stage hooks
    def raw_to_pa(self, raw, digitisation, offset, range_):
        raw = np.ascontiguousarray(raw, np.int16)
        out = np.zeros(max(len(raw), 1), np.float32)
        n = C.c_size_t()
        self._check(F.lib.smb_stage_raw_to_pa(self._ctx, F.ptr(raw, F.i16p), len(raw), digitisation,
                                              offset, range_, F.ptr(out, F.f32p), C.byref(n)),
                    "smb_stage_raw_to_pa")
        return out[:n.value].copy()

    def GenerateEvents(self, pa_chunks):
        """pa_chunks: (n_chunks, 4000) float32 pA -> list of per-chunk feature arrays."""
        pa = np.ascontiguousarray(pa_chunks, np.float32).reshape(-1, CHUNK)
        n = pa.shape[0]
        feats = np.zeros((max(n, 1), CHUNK), np.float32)
        cnt = np.zeros(max(n, 1), np.uint32)
        self._check(F.lib.smb_stage_events(self._ctx, F.ptr(pa, F.f32p), n, F.ptr(feats, F.f32p),
                                           F.ptr(cnt, F.u32p)), "smb_stage_events")
        return [feats[i, :cnt[i]].copy() for i in range(n)]

    def detect_events(self, pa_chunk):
        pa = np.ascontiguousarray(pa_chunk, np.float32)
        assert pa.shape == (CHUNK,)
        t1, t2 = np.zeros(CHUNK + 1, np.float32), np.zeros(CHUNK + 1, np.float32)
        peaks, means = np.zeros(CHUNK, np.uint32), np.zeros(CHUNK, np.float32)
        npk, nev = C.c_uint32(), C.c_uint32()
        self._check(F.lib.smb_stage_detect(self._ctx, F.ptr(pa, F.f32p), F.ptr(t1, F.f32p),
                                           F.ptr(t2, F.f32p), F.ptr(peaks, F.u32p), C.byref(npk),
                                           F.ptr(means, F.f32p), C.byref(nev)), "smb_stage_detect")
        return dict(tstat1=t1, tstat2=t2, peaks=peaks[:npk.value].copy(), means=means[:nev.value].copy())

    def radiusSearch(self, queries, radius=0.08, cap=None):
        """queries: (nq, 6).  -> (hit_off[nq+1], hit_idx, hit_d2), hits sorted by point index."""
        q = np.ascontiguousarray(queries, np.float32).reshape(-1, F.SMB_DIM)
        nq = q.shape[0]
        cap = cap or max(1 << 20, nq * 4096)
        off = np.zeros(nq + 1, np.uint64)
        idx, d2 = np.zeros(cap, np.uint64), np.zeros(cap, np.float32)
        self._check(F.lib.smb_stage_radius(self._ctx, F.ptr(q, F.f32p), nq, radius, F.ptr(off, F.u64p),
                                           F.ptr(idx, F.u64p), F.ptr(d2, F.f32p), cap),
                    "smb_stage_radius")
        n = int(off[-1])
        return off, idx[:n].copy(), d2[:n].copy()

    def ChainBatch(self, n_slots):
        return ChainBatch(self, n_slots)

    # ------------------------------------------------------------------ streaming
    def stream_open(self, n_channels, params=None):
        params = params or default_params()
        self._check(F.lib.smb_stream_open(self._ctx, n_channels, C.byref(params)), "smb_stream_open")

    def stream_begin_read(self, channel, digitisation, range_, offset):
        self._check(F.lib.smb_stream_begin_read(self._ctx, channel, digitisation, range_, offset),
                    "smb_stream_begin_read")

    def stream_round(self, channels, sample_lists):
        channels = np.ascontiguousarray(channels, np.uint32)
        off = np.zeros(len(channels) + 1, np.uint32)
        off[1:] = np.cumsum([len(s) for s in sample_lists])
        samples = (np.concatenate(sample_lists).astype(np.int16) if len(sample_lists)
                   else np.zeros(0, np.int16))
        return self.stream_round_arrays(channels, samples, off)

    def stream_round_arrays(self, channels, samples, off):
        """One round from pre-packed host arrays: channels u32[n], samples i16[off[n]], off u32[n+1]
        -> (stop decisions u8[n], provisional rows: a ctypes array of Mapping, rows [0, n) valid).
        This is the call whose duration is the per-chunk latency of read-until mode
        (submit -> decision), so nothing per-row happens on the Python side."""
        n = len(channels)
        dec = np.zeros(max(n, 1), np.uint8)
        maps = (F.Mapping * max(n, 1))()
        self._check(F.lib.smb_stream_round(self._ctx, F.ptr(channels, F.u32p), n,
                                           F.ptr(samples, F.i16p), F.ptr(off, F.u32p),
                                           F.ptr(dec, F.u8p), maps), "smb_stream_round")
        return dec[:n], maps

    def stream_close(self):
        self._check(F.lib.smb_stream_close(self._ctx), "smb_stream_close")


class ChainBatch:
    """n_slots independent `std::vector<SignalAnchorChain> chains` states on the device."""

    def __init__(self, mapper, n_slots):
        self.m = mapper
        self._b = C.c_void_p()
        mapper._check(F.lib.smb_batch_create(mapper._ctx, n_slots, C.byref(self._b)), "smb_batch_create")

    def close(self):
        if self._b:
            F.lib.smb_batch_destroy(self._b)
            self._b = None

    def reset(self):
        self.m._check(F.lib.smb_batch_reset(self._b), "smb_batch_reset")

    def GenerateChains(self, slots, feature_list, params=None):
        """GenerateChains(features, num_events[slot], step, radius, n_contigs, chains[slot]) for
        each (slot, features) pair; num_events advances as in sigmap.cc:666."""
        params = params or default_params()
        slots = np.ascontiguousarray(slots, np.uint32)
        off = np.zeros(len(slots) + 1, np.uint32)
        off[1:] = np.cumsum([len(f) for f in feature_list])
        feats = (np.concatenate(feature_list).astype(np.float32) if len(feature_list)
                 else np.zeros(0, np.float32))
        feats = np.ascontiguousarray(feats, np.float32)
        self.m._check(F.lib.smb_batch_generate_chains(self._b, F.ptr(slots, F.u32p), len(slots),
                                                      F.ptr(feats, F.f32p), F.ptr(off, F.u32p),
                                                      C.byref(params)), "smb_batch_generate_chains")

    def chains(self, slot):
        n = C.c_uint32()
        self.m._check(F.lib.smb_batch_chain_count(self._b, slot, C.byref(n)), "smb_batch_chain_count")
        recs = (F.Chain * max(n.value, 1))()
        self.m._check(F.lib.smb_batch_get_chains(self._b, slot, recs, n.value), "smb_batch_get_chains")
        out = []
        for i in range(n.value):
            c = recs[i]
            an = (F.Anchor * max(c.n_anchors, 1))()
            self.m._check(F.lib.smb_batch_get_anchors(self._b, slot, i, an, c.n_anchors),
                          "smb_batch_get_anchors")
            out.append(dict(score=np.float32(c.score), contig=c.contig, start=c.start, end=c.end,
                            n_anchors=c.n_anchors, mapq=c.mapq, dir=c.dir,
                            anchors=[(an[a].target, an[a].query, np.float32(an[a].dist))
                                     for a in range(c.n_anchors)]))
        return out
