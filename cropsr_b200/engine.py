"""Python face of the C ABI: device, packed genome shard, candidate streams.

Everything that computes happens in libcropsr_b200.so on the GPU; this module
only owns handles, numpy output buffers and index arithmetic.
"""
import ctypes as C

import numpy as np

from . import _native as N
from ._native import CropsrError, check, lib

_device = None

SEGMENT_ALIGN = 128   # crp_genome_add_segment: seg_begin granularity
TILE = lib.crp_tile_size()   # positions per scan tile (csrc/cropsr_b200.cu kTile)


def init(device=0):
    """Bind this process to one GPU (one process per GPU)."""
    global _device
    if _device is not None and _device != device:
        raise CropsrError(-3, f"already initialised on device {_device}")
    check(lib.crp_init(int(device)))
    _device = int(device)
    return _device


def bind_host_near(device=0):
    """Pin the calling process to the CPUs of the NUMA node the GPU hangs off, so that the pinned
    staging buffers it allocates next (first touch) and its copies stay on that node's memory and
    PCIe root.  One process per GPU: with eight ranks on a two-socket host the host side of the
    end-to-end path is otherwise what limits it.  Best effort: returns the node, or None (no
    nvidia-smi / sysfs, single node, cgroup without those CPUs) without touching anything."""
    import os
    import subprocess
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(int(device))],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not bus:
            return None
        dom, rest = bus.split(":", 1)
        with open(f"/sys/bus/pci/devices/{dom[-4:]}:{rest}/numa_node") as f:
            node = int(f.read())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return node
    except Exception:
        return None


def shutdown():
    global _device
    check(lib.crp_shutdown())
    _device = None


def device_count():
    n = C.c_int(0)
    check(lib.crp_device_count(C.byref(n)))
    return n.value


def perf_report():
    """dict of the library's counters since init (crp_perf_report)"""
    import json
    buf = C.create_string_buffer(4096)
    need = C.c_uint64(0)
    check(lib.crp_perf_report(buf, len(buf), C.byref(need)))
    return json.loads(buf.value.decode())


def launch_count():
    n = C.c_uint64(0)
    check(lib.crp_launch_count(C.byref(n)))
    return n.value


def device_synchronize():
    check(lib.crp_device_synchronize())


def flush_l2():
    """Evict L2 (benchmarks, between timed scans)."""
    check(lib.crp_flush_l2())


# ---- one process per GPU: the NCCL communicator of the count all-gather (include/cropsr_b200.h) ----
def comm_unique_id():
    buf = (C.c_uint8 * N.COMM_ID_BYTES)()
    check(lib.crp_comm_unique_id(buf))
    return bytes(buf)


def comm_init(rank, world, unique_id):
    if _device is None:
        raise CropsrError(-3, "engine.init(device) comes first")
    assert len(unique_id) == N.COMM_ID_BYTES
    buf = (C.c_uint8 * N.COMM_ID_BYTES).from_buffer_copy(unique_id)
    check(lib.crp_comm_init(int(rank), int(world), buf))


def comm_info():
    r, w = C.c_int(0), C.c_int(1)
    check(lib.crp_comm_info(C.byref(r), C.byref(w)))
    return r.value, w.value


def comm_set_exchange(mode):
    """'fused' (the scan kernel exchanges the counts itself over peer memory) or 'nccl'; on every rank."""
    check(lib.crp_comm_set_exchange({"fused": 0, "nccl": 1}[mode]))


def comm_exchange_info():
    """(fused?, why not) of the sharded scans of this communicator"""
    f, why = C.c_int(0), C.c_char_p()
    check(lib.crp_comm_exchange_info(C.byref(f), C.byref(why)))
    return bool(f.value), (why.value or b"").decode()


def comm_barrier():
    check(lib.crp_comm_barrier())


def comm_max(values):
    v = np.ascontiguousarray(values, dtype=np.float64).copy()
    check(lib.crp_comm_max_f64(v.ctypes.data, v.size))
    return v


def comm_sum(values):
    v = np.ascontiguousarray(values, dtype=np.float64).copy()
    check(lib.crp_comm_sum_f64(v.ctypes.data, v.size))
    return v


def comm_allgather(values):
    """uint64[n] per rank -> uint64[world, n] on every rank (host in, host out)"""
    v = np.ascontiguousarray(values, dtype=np.uint64)
    _, world = comm_info()
    out = np.empty((world, v.size), dtype=np.uint64)
    check(lib.crp_comm_allgather_u64(v.ctypes.data, v.size, out.ctypes.data))
    return out


def link_probe(h2d_bytes, d2h_bytes, reps=5):
    """ms of one round of concurrent pinned H2D + D2H copies of these sizes (what the link allows)"""
    ms = C.c_float(0)
    check(lib.crp_link_probe(int(h2d_bytes), int(d2h_bytes), int(reps), C.byref(ms)))
    return ms.value


def comm_shutdown():
    check(lib.crp_comm_shutdown())


def logistic(x):
    """1 / (1 + np.exp(x)) on the device with numpy's own digits (CROPSR.py:313; csrc/npexp.cuh)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    check(lib.crp_logistic(x.size, x.ctypes.data, out.ctypes.data))
    return out


def rs1_score(rows, cls):
    """crp_rs1_score: rows (n, 30) uint8 ASCII, cls (n,) uint8 BLAS classes -> float64 scores."""
    rows = np.ascontiguousarray(rows, dtype=np.uint8)
    cls = np.ascontiguousarray(cls, dtype=np.uint8)
    out = np.empty(len(rows), dtype=np.float64)
    check(lib.crp_rs1_score(len(rows), rows.ctypes.data, cls.ctypes.data, out.ctypes.data))
    return out


def rs1_preactivation(rows, cls):
    """crp_rs1_preactivation: like rs1_score without the logistic (x of every row)."""
    rows = np.ascontiguousarray(rows, dtype=np.uint8)
    cls = np.ascontiguousarray(cls, dtype=np.uint8)
    out = np.empty(len(rows), dtype=np.float64)
    if len(rows):
        check(lib.crp_rs1_preactivation(len(rows), rows.ctypes.data, cls.ctypes.data, out.ctypes.data))
    return out


def _as_u8(token):
    """Token -> contiguous uint8 numpy view (str is encoded; must be ASCII)."""
    if isinstance(token, str):
        try:
            token = token.encode("ascii")
        except UnicodeEncodeError as e:
            raise ValueError("sequence tokens must be ASCII (the reference's rs1 scoring "
                             "raises on non-ASCII windows, CROPSR.py:458)") from e
    arr = np.frombuffer(token, dtype=np.uint8) if not isinstance(token, np.ndarray) else token
    if arr.dtype != np.uint8 or arr.ndim != 1:
        raise ValueError("token must be bytes-like or a 1-D uint8 array")
    return np.ascontiguousarray(arr)


class PinnedBuffer:
    """Page-locked host memory from crp_host_alloc, exposed as a numpy array."""

    def __init__(self, nbytes):
        self._ptr = C.c_void_p()
        check(lib.crp_host_alloc(C.byref(self._ptr), int(nbytes)))
        self.nbytes = int(nbytes)
        buf = (C.c_uint8 * max(self.nbytes, 1)).from_address(self._ptr.value)
        self.array = np.frombuffer(buf, dtype=np.uint8, count=self.nbytes)

    def view(self, dtype, count, offset=0):
        return self.array[offset:offset + count * np.dtype(dtype).itemsize].view(dtype)

    def free(self):
        if self._ptr:
            self.array = None
            check(lib.crp_host_free(self._ptr))
            self._ptr = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Arena:
    """Pinned host arrays for the candidate rows of both strands (crp_scan_segments)."""

    def __init__(self, capacity, scored=True, want=("pos", "packed", "x")):
        self.capacity = int(capacity)
        self.scored = scored
        self.want = tuple(want)
        self._bufs = []
        self.arrays = {}
        for strand in "+-":
            row = {}
            for name, dt in (("pos", np.uint32), ("packed", np.uint64), ("x", np.float64)):
                if (name != "pos" and not scored) or name not in self.want:
                    row[name] = None
                    continue
                b = PinnedBuffer(self.capacity * np.dtype(dt).itemsize)
                self._bufs.append(b)
                row[name] = b.view(dt, self.capacity)
            self.arrays[strand] = row

    def free(self):
        self.arrays = {}
        for b in self._bufs:
            b.free()
        self._bufs = []


def scan_segments(segments, guide_len=20, flags=N.CRP_SCAN_DEFAULT, arena=None, want=("pos", "packed", "x")):
    """Pipelined whole call: `segments` = [(token_id, token uint8 array (pinned for full speed),
    begin, end)].  Returns (arena, n_plus[], n_minus[], device_ms); rows of a strand are in
    arena.arrays[strand][name][:sum(counts)] in segment order.  If the arena is too small a
    larger one is allocated and the call repeated.  `want`: the columns that come back (a caller
    that formats its rows from the tokens -- the CSV writer -- leaves "packed" out: 12 instead of
    20 bytes per candidate over the link)."""
    if _device is None:
        init(0)
    scored = int(guide_len) == 20 and not (flags & N.CRP_SCAN_NO_SCORE)
    n = len(segments)
    descs = (N.SegmentDesc * max(n, 1))()
    keep = []
    for i, (tid, tok, a, b) in enumerate(segments):
        arr = _as_u8(tok)
        keep.append(arr)
        descs[i] = N.SegmentDesc(int(tid), arr.ctypes.data, len(arr), int(a), len(arr) if b is None else int(b))
    n_plus = np.zeros(max(n, 1), dtype=np.uint64)
    n_minus = np.zeros(max(n, 1), dtype=np.uint64)
    ms = C.c_float(0)
    if arena is None:
        total = sum((len(k) if b is None else b) - a for k, (_, _, a, b) in zip(keep, segments))
        arena = Arena(total // 12 + 4096, scored, want)
    for attempt in range(2):
        ptr = lambda a: a.ctypes.data if a is not None else None
        p, m = arena.arrays["+"], arena.arrays["-"]
        rc = lib.crp_scan_segments(n, descs, int(guide_len), int(flags), arena.capacity,
                                   ptr(p["pos"]), ptr(p["packed"]), ptr(p["x"]),
                                   ptr(m["pos"]), ptr(m["packed"]), ptr(m["x"]),
                                   n_plus.ctypes.data, n_minus.ctypes.data, C.byref(ms))
        if rc == -5 and attempt == 0:          # CRP_ERR_RANGE: arena too small, counts are valid
            arena.free()
            arena = Arena(int(max(n_plus.sum(), n_minus.sum())) + 1024, scored, want)
            continue
        check(rc)
        break
    return arena, n_plus[:n], n_minus[:n], ms.value


class Genome:
    """A genome shard: an ordered list of token segments packed into HBM."""

    def __init__(self):
        if _device is None:
            init(0)
        self._h = C.c_void_p()
        check(lib.crp_genome_new(C.byref(self._h)))
        self._keep = []          # host arrays that must outlive commit()
        self.segments = []       # (token_id, token_len, begin, end)
        self.committed = False

    def add_segment(self, token_id, token, begin=0, end=None):
        arr = _as_u8(token)
        end = len(arr) if end is None else int(end)
        check(lib.crp_genome_add_segment(self._h, int(token_id), arr.ctypes.data, len(arr), int(begin), end))
        self._keep.append(arr)
        self.segments.append((int(token_id), len(arr), int(begin), end))
        return len(self.segments) - 1

    def add_fasta_record(self, file_bytes, seq_off, seq_bytes, line_width, last, token_id=None):
        """One record of a plain multi-line FASTA file, ingested on the device: file_bytes is a
        uint8 array of the whole file, [seq_off, seq_off + seq_bytes) its sequence lines.
        Raises CropsrError(code -6) if the record is not plain (see include/cropsr_b200.h)."""
        arr = _as_u8(file_bytes)
        tid = len(self.segments) if token_id is None else int(token_id)
        check(lib.crp_genome_add_fasta_record(self._h, tid, arr.ctypes.data + int(seq_off), int(seq_bytes),
                                              int(line_width), int(bool(last))))
        self._keep.append(arr)
        n = C.c_uint64(0)
        check(lib.crp_genome_token_length(self._h, len(self.segments), C.byref(n)))
        self.segments.append((tid, n.value, 0, n.value))
        return len(self.segments) - 1

    def fetch_token(self, segment):
        """Token bytes of a device-ingested FASTA record (uint8 array, decoration included)."""
        n = self.segments[segment][1]
        out = np.empty(n, dtype=np.uint8)
        check(lib.crp_genome_fetch_token(self._h, int(segment), out.ctypes.data, n))
        return out

    def release_tokens(self):
        check(lib.crp_genome_release_tokens(self._h))

    def add_token(self, token, token_id=None):
        return self.add_segment(len(self.segments) if token_id is None else token_id, token)

    def commit(self):
        check(lib.crp_genome_commit(self._h))
        self._keep = []
        self.committed = True
        return self

    @property
    def num_positions(self):
        n = C.c_uint64(0)
        check(lib.crp_genome_num_positions(self._h, C.byref(n)))
        return n.value

    def timing(self):
        a, b = C.c_float(0), C.c_float(0)
        check(lib.crp_genome_timing(self._h, C.byref(a), C.byref(b)))
        return {"h2d_ms": a.value, "pack_ms": b.value}

    def scan(self, guide_len=20, flags=N.CRP_SCAN_DEFAULT):
        res = C.c_void_p()
        check(lib.crp_scan_score(self._h, int(guide_len), int(flags), C.byref(res)))
        return ScanResult(self, res, guide_len, flags)

    def scan_sharded(self, slots, guide_len=20, flags=N.CRP_SCAN_DEFAULT):
        """This rank's shard of a genome spread over the communicator: scan + NCCL all-gather of the
        per-segment counts (`slots` per rank and strand, the same on every rank).  Collective."""
        res = C.c_void_p()
        check(lib.crp_scan_score_sharded(self._h, int(guide_len), int(flags), int(slots), C.byref(res)))
        r = ScanResult(self, res, guide_len, flags)
        r.slots = int(slots)
        return r

    def rescore(self, segment, t, strand, cls):
        """x of the given candidates re-summed in BLAS class cls (see blas_order)."""
        segment = np.ascontiguousarray(segment, dtype=np.uint32)
        t = np.ascontiguousarray(t, dtype=np.uint32)
        strand = np.ascontiguousarray(strand, dtype="S1")
        cls = np.ascontiguousarray(cls, dtype=np.uint8)
        n = len(t)
        out = np.empty(n, dtype=np.float64)
        if n:
            check(lib.crp_rescore(self._h, n, segment.ctypes.data, t.ctypes.data, strand.ctypes.data,
                                  cls.ctypes.data, out.ctypes.data))
        return out

    def other_runs(self, segment, min_len=1):
        """Gap table of one segment: runs of bytes that are not ACGTacgt, at least min_len long.
        -> (start uint32[], length uint32[]) in token coordinates, ascending."""
        cap = 4096
        for _ in range(2):
            start = np.empty(cap, np.uint32)
            length = np.empty(cap, np.uint32)
            n = C.c_uint64(0)
            rc = lib.crp_genome_other_runs(self._h, int(segment), int(min_len), cap, start.ctypes.data, length.ctypes.data,
                                           C.byref(n))
            if rc == -5 and n.value > cap:
                cap = int(n.value)
                continue
            check(rc)
            return start[:n.value], length[:n.value]
        raise CropsrError(-5, "gap table: capacity negotiation failed")

    def free(self):
        if self._h:
            check(lib.crp_genome_free(self._h))
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _flank(flank):
    """The flank half-width as the library takes it (uint32): ValueError outside 0 <= flank < 2**32, which a
    ctypes uint32 would wrap silently (-1 -> 2**32 - 1, 2**32 + 200 -> 200)."""
    f = int(flank)
    if not 0 <= f < 1 << 32:
        raise ValueError(f"flank {flank}: 0 <= flank < 2**32 expected")
    return f


class ScanResult:
    """Two ordered candidate streams ('+', '-') resident in HBM."""

    def __init__(self, genome, handle, guide_len, flags):
        self.genome = genome
        self._h = handle
        self.guide_len = int(guide_len)
        self.flags = int(flags)
        self.scored = self.guide_len == 20 and not (flags & N.CRP_SCAN_NO_SCORE)
        a, b = C.c_uint64(0), C.c_uint64(0)
        check(lib.crp_result_totals(self._h, C.byref(a), C.byref(b)))
        self.n_plus, self.n_minus = a.value, b.value
        ns = len(genome.segments)
        self.seg_plus = np.zeros(ns, dtype=np.uint64)
        self.seg_minus = np.zeros(ns, dtype=np.uint64)
        if ns:
            check(lib.crp_result_segment_counts(self._h, self.seg_plus.ctypes.data, self.seg_minus.ctypes.data))
        # first candidate of every segment inside each strand stream
        self.off_plus = np.concatenate(([0], np.cumsum(self.seg_plus))).astype(np.uint64)
        self.off_minus = np.concatenate(([0], np.cumsum(self.seg_minus))).astype(np.uint64)

    def scan_ms(self):
        v = C.c_float(0)
        check(lib.crp_result_timing(self._h, C.byref(v)))
        return v.value

    def timing_detail(self):
        """dict(kernel_ms, total_ms (kernel + all-gather for a sharded scan), launches)"""
        a, b, n = C.c_float(0), C.c_float(0), C.c_uint32(0)
        check(lib.crp_result_timing_detail(self._h, C.byref(a), C.byref(b), C.byref(n)))
        return {"kernel_ms": a.value, "total_ms": b.value, "launches": n.value}

    def gathered_counts(self):
        """uint64[world, 2, slots]: every rank's per-segment counts ('+' then '-') of a sharded scan"""
        _, world = comm_info()
        out = np.empty((world, 2, self.slots), dtype=np.uint64)
        check(lib.crp_result_gathered_counts(self._h, out.ctypes.data))
        return out

    def device_counts_ptr(self):
        p = C.c_void_p()
        check(lib.crp_result_device_counts(self._h, C.byref(p)))
        return p.value

    def fetch(self, strand, first=0, count=None, out=None, want=("pos", "packed", "x")):
        """Copy [first, first+count) of one strand stream to host numpy arrays.
        Returns dict(pos=uint32[], packed=uint64[], x=float64[]); packed / x only
        exist for scored results.  `out` may supply preallocated (pinned) arrays."""
        total = self.n_plus if strand == "+" else self.n_minus
        count = total - first if count is None else count
        out = {} if out is None else out
        res = {}
        for name, dt in (("pos", np.uint32), ("packed", np.uint64), ("x", np.float64)):
            if name not in want or (name != "pos" and not self.scored):
                res[name] = None
                continue
            arr = out.get(name)
            if arr is None:
                arr = np.empty(count, dtype=dt)
            assert arr.dtype == dt and len(arr) >= count and arr.flags.c_contiguous
            res[name] = arr[:count]
        ptr = lambda a: a.ctypes.data if a is not None and len(a) else None
        check(lib.crp_result_fetch(self._h, strand.encode(), int(first), int(count),
                                   ptr(res["pos"]), ptr(res["packed"]), ptr(res["x"])))
        return res

    def extras(self, seg, strand, flank=200):
        """Opt-in side outputs of one segment's candidates (never in the parity CSV):
        dict(gc, flags, run: uint8[]; cut, flank_lo, flank_hi: uint32[]).  flank: 0 <= flank < 2**32."""
        flank = _flank(flank)
        n = int((self.seg_plus if strand == "+" else self.seg_minus)[seg])
        out = {k: np.empty(n, np.uint8) for k in ("gc", "flags", "run")}
        out.update({k: np.empty(n, np.uint32) for k in ("cut", "flank_lo", "flank_hi")})
        ptr = lambda a: a.ctypes.data if len(a) else None
        check(lib.crp_result_extras(self._h, int(seg), strand.encode(), flank, ptr(out["gc"]), ptr(out["flags"]),
                                    ptr(out["run"]), ptr(out["cut"]), ptr(out["flank_lo"]), ptr(out["flank_hi"])))
        return out

    def extras_strand(self, strand, flank=200):
        """extras() of every candidate of one strand stream (all segments), in stream order"""
        flank = _flank(flank)
        n = int(self.n_plus if strand == "+" else self.n_minus)
        out = {k: np.empty(n, np.uint8) for k in ("gc", "flags", "run")}
        out.update({k: np.empty(n, np.uint32) for k in ("cut", "flank_lo", "flank_hi")})
        ptr = lambda a: a.ctypes.data if len(a) else None
        check(lib.crp_result_extras_strand(self._h, strand.encode(), flank, ptr(out["gc"]), ptr(out["flags"]),
                                           ptr(out["run"]), ptr(out["cut"]), ptr(out["flank_lo"]), ptr(out["flank_hi"])))
        return out

    def annotate_strand(self, strand, iv_offset, start, end):
        """annotate() of a whole strand stream: intervals of segment s are [iv_offset[s], iv_offset[s+1])"""
        iv_offset = np.ascontiguousarray(iv_offset, dtype=np.uint64)
        start = np.ascontiguousarray(start, dtype=np.uint32)
        end = np.ascontiguousarray(end, dtype=np.uint32)
        n = int(self.n_plus if strand == "+" else self.n_minus)
        out = np.empty(n, np.int32)
        if n:
            check(lib.crp_result_annotate_strand(self._h, strand.encode(), iv_offset.ctypes.data,
                                                 start.ctypes.data if len(start) else None,
                                                 end.ctypes.data if len(end) else None, out.ctypes.data))
        return out

    def annotate(self, seg, strand, start, end):
        """Index of the innermost interval [start, end] (inclusive token coordinates,
        sorted by start) containing each candidate's cut site, -1 if none."""
        start = np.ascontiguousarray(start, dtype=np.uint32)
        end = np.ascontiguousarray(end, dtype=np.uint32)
        n = int((self.seg_plus if strand == "+" else self.seg_minus)[seg])
        out = np.empty(n, np.int32)
        if n:
            check(lib.crp_result_annotate(self._h, int(seg), strand.encode(), len(start),
                                          start.ctypes.data if len(start) else None,
                                          end.ctypes.data if len(end) else None, out.ctypes.data))
        return out

    def fetch_segment(self, seg, strand, **kw):
        off = self.off_plus if strand == "+" else self.off_minus
        return self.fetch(strand, int(off[seg]), int(off[seg + 1] - off[seg]), **kw)

    def free(self):
        if self._h:
            check(lib.crp_result_free(self._h))
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


_GUIDE_CODE = np.full(256, 255, dtype=np.uint8)
for _i, _c in enumerate(b"ATCG"):
    _GUIDE_CODE[_c] = _GUIDE_CODE[_c | 0x20] = _i


def guide_keys(guides):
    """20-base guides (ACGTacgt, the orientation followed by NGG in the genome) -> uint64 keys:
    base i (A0 T1 C2 G3) in bits 2i, 2i+1.  ValueError for anything else."""
    keys = np.zeros(len(guides), dtype=np.uint64)
    for n, g in enumerate(guides):
        b = np.frombuffer(g.encode("ascii") if isinstance(g, str) else bytes(g), dtype=np.uint8)
        code = _GUIDE_CODE[b]
        if len(b) != 20 or (code == 255).any():
            raise ValueError(f"guide {g!r}: 20 characters of ACGTacgt expected")
        keys[n] = int((code.astype(np.uint64) << (2 * np.arange(20, dtype=np.uint64))).sum())
    return keys


LIST_BATCH_SITES = 1 << 28       # site indices one listing call returns at most (1 GiB on the device and the host)

# MIT specificity score (Hsu et al. 2013) as CRISPOR's calcHitScore / calcMitGuideScore compute it: the per-position
# mismatch weights, position 0 PAM-distal
MIT_M = (0, 0, 0.014, 0, 0, 0.395, 0.317, 0, 0.389, 0.079, 0.445, 0.508, 0.613, 0.851, 0.732, 0.828, 0.615, 0.804,
         0.685, 0.583)
SCORE_SETS = N.OFFTARGET_SCORE_SETS
SCORE_ONE = 1 << 24              # fixed point of the weights: w = round(hit * 2**24)


def score_sets():
    """The mismatch-position sets of size <= 3 (ascending tuples) in rank order (include/cropsr_b200.h):
    {}, then {a} by a, {a<b} by (b, a), {a<b<c} by (c, b, a) -- colexicographic within a size."""
    from itertools import combinations
    return [c for d in range(4) for c in sorted(combinations(range(20), d), key=lambda c: c[::-1])]


def mit_hit(positions):
    """CRISPOR's calcHitScore of one site from its ascending mismatch positions, in its IEEE operation order.  The
    distance term uses the mean of CONSECUTIVE distances, as CRISPOR does (not the all-pairs mean of the paper)."""
    score1 = 1.0
    for p in positions:
        score1 *= 1 - MIT_M[p]
    n = len(positions)
    if n < 2:
        score2 = 1.0
    else:
        dists = [positions[i + 1] - positions[i] for i in range(n - 1)]
        score2 = 1.0 / (((19 - sum(dists) / len(dists)) / 19.0) * 4 + 1)
    score3 = 1.0 if n == 0 else 1.0 / (n ** 2)
    return score1 * score2 * score3 * 100


def mit_weights():
    """uint32[SCORE_SETS]: round(mit_hit(set) * 2**24) (half to even; the product is exact) in rank order"""
    return np.array([round(mit_hit(c) * SCORE_ONE) for c in score_sets()], dtype=np.uint32)


def mit_specificity(sums):
    """CRISPOR's calcMitGuideScore, int(round(100 / (100 + H) * 100)) with H = sum / 2**24, of score sums
    (score_candidates / score_guides with the MIT weights) -> uint64, NO_SCORE passed through"""
    sums = np.asarray(sums, dtype=np.uint64)
    ok = sums != np.uint64(N.OFFTARGET_NO_SCORE)
    h = sums[ok].astype(np.float64) / SCORE_ONE
    out = np.full(sums.shape, N.OFFTARGET_NO_SCORE, dtype=np.uint64)
    out[ok] = np.round(100 / (100 + h) * 100).astype(np.uint64)
    return out


def _weights(weights):
    w = mit_weights() if weights is None else np.ascontiguousarray(weights, dtype=np.uint32)
    if w.shape != (SCORE_SETS,):
        raise ValueError(f"weights: {SCORE_SETS} entries expected, got shape {w.shape}")
    return w


# PAM patterns N + two IUPAC letters (crp_offtarget_new_pam): the bases each letter stands for; N is refused there
PAM_LETTERS = {"A": "A", "C": "C", "G": "G", "T": "T", "R": "AG", "Y": "CT", "S": "CG", "W": "AT", "K": "GT",
               "M": "AC", "B": "CGT", "D": "AGT", "H": "ACT", "V": "ACG"}


def parse_pam(text):
    """A PAM pattern, upper case ('nag' -> 'NAG'): ValueError unless it is N followed by two of A C G T R Y S W K M B
    D H V (IUPAC letters for one to three bases)."""
    pam = str(text).upper()
    if len(pam) != 3 or pam[0] != "N" or pam[1] not in PAM_LETTERS or pam[2] not in PAM_LETTERS:
        raise ValueError(f"PAM pattern {text!r}: N followed by two of {''.join(PAM_LETTERS)} expected")
    return pam


def pams_overlap(a, b):
    """True if a base triple matches both patterns: N a2 a3 and N b2 b3 overlap iff a2, b2 and a3, b3 share a base"""
    a, b = parse_pam(a), parse_pam(b)
    return all(set(PAM_LETTERS[x]) & set(PAM_LETTERS[y]) for x, y in zip(a[1:], b[1:]))


def pam_has_own_site(pam):
    """True if a scan candidate's own site (its NGG) is a site of the pattern: G in letters 2 and 3.  Only then do
    its counts and score leave the site out."""
    pam = parse_pam(pam)
    return "G" in PAM_LETTERS[pam[1]] and "G" in PAM_LETTERS[pam[2]]


class OffTargetIndex:
    """The sites of one PAM pattern (NGG by default; both strands, case-insensitive) of one or more committed genomes,
    resident in HBM: counts of sites within 0 .. k <= 3 mismatches of every scan candidate or of arbitrary guides,
    their weighted scores, and with loci=True the sites themselves (semantics: include/cropsr_b200.h,
    csrc/offtarget.cuh)."""

    NO_COUNT = N.OFFTARGET_NO_COUNT
    NO_SCORE = N.OFFTARGET_NO_SCORE

    def __init__(self, genomes=(), loci=False, pam="NGG"):
        """loci=True: the index also keeps every site's locus (8 bytes per site more), which site_loci and the
        listings (list_candidates, list_guides) need.  pam: the PAM pattern (parse_pam) whose sites the index holds;
        a candidate's own site is left out of its counts and score only where pam_has_own_site(pam)."""
        self.pam = parse_pam(pam)
        if _device is None:
            init(0)
        self._h = C.c_void_p()
        self.loci = bool(loci)
        if self.pam == "NGG":
            check((lib.crp_offtarget_new_with_loci if self.loci else lib.crp_offtarget_new)(C.byref(self._h)))
        else:
            check(lib.crp_offtarget_new_pam(C.byref(self._h), self.pam.encode(), int(self.loci)))
        for g in genomes:
            self.add_genome(g)

    def add_genome(self, genome):
        check(lib.crp_offtarget_add_genome(self._h, genome._h))

    def num_sites(self):
        n = C.c_uint64(0)
        check(lib.crp_offtarget_num_sites(self._h, C.byref(n)))
        return n.value

    def sites(self):
        """uint64 keys of every site, in no particular order"""
        n = self.num_sites()
        out = np.empty(n, dtype=np.uint64)
        got = C.c_uint64(0)
        check(lib.crp_offtarget_fetch_sites(self._h, n, out.ctypes.data if n else None, C.byref(got)))
        return out

    def count_candidates(self, result, strand, k=3):
        """uint32[n_strand, k + 1]: sites at exactly d mismatches of every candidate of one strand stream
        (stream order, the candidate's own site not counted); rows of NO_COUNT where the candidate has
        no protospacer (cut off by the token end, or a byte outside ACGTacgt)."""
        n = int(result.n_plus if strand == "+" else result.n_minus)
        out = np.empty((n, int(k) + 1), dtype=np.uint32)
        check(lib.crp_offtarget_count_candidates(self._h, result._h, strand.encode(), int(k),
                                                 out.ctypes.data if n else None))
        return out

    def count_guides(self, guides, k=3):
        """uint32[len(guides), k + 1] for 20-base guides in the protospacer orientation; nothing subtracted"""
        keys = guide_keys(guides)
        out = np.empty((len(keys), int(k) + 1), dtype=np.uint32)
        if len(keys):
            check(lib.crp_offtarget_count_keys(self._h, len(keys), keys.ctypes.data, int(k), out.ctypes.data))
        return out

    def site_loci(self):
        """(genome, segment, t, strand) arrays in sites() order: the ordinal of the add_genome call that added
        the site's handle, the segment index in that handle, t in token coordinates, and 0 for '+' / 1 for '-'"""
        n = self.num_sites()
        loci = np.empty(n, dtype=np.uint64)
        got = C.c_uint64(0)
        check(lib.crp_offtarget_fetch_loci(self._h, n, loci.ctypes.data if n else None, C.byref(got)))
        return ((loci >> np.uint64(56) & np.uint64(0x7F)).astype(np.uint8),
                (loci >> np.uint64(32) & np.uint64(0xFFFFFF)).astype(np.uint32),
                (loci & np.uint64(0xFFFFFFFF)).astype(np.uint32),
                (loci >> np.uint64(63)).astype(np.uint8))

    def _list(self, n_rows, totals, call):
        """Batches of consecutive rows whose listings hold at most LIST_BATCH_SITES indices (a row above that
        goes alone): call(lo, hi, first, out) per batch -> (first [n_rows + 1] uint64, sites uint32)."""
        totals = np.asarray(totals, dtype=np.uint64)
        first = np.zeros(n_rows + 1, dtype=np.uint64)
        np.cumsum(totals, out=first[1:])
        sites = np.empty(int(first[-1]), dtype=np.uint32)
        lo = 0
        while lo < n_rows:
            hi = int(np.searchsorted(first, first[lo] + np.uint64(LIST_BATCH_SITES), side="right")) - 1
            hi = min(max(hi, lo + 1), n_rows)
            f = first[lo:hi + 1] - first[lo]
            out = sites[int(first[lo]):int(first[hi])]
            call(lo, hi, f, out)
            lo = hi
        return first, sites

    def list_candidates(self, result, strand, k=3, rows=None, counts=None):
        """The other sites within k mismatches of candidates of one strand stream -> (rows, first, sites):
        rows (uint32, ascending stream rows; default every row with a protospacer), first (uint64 [len(rows) + 1])
        and sites (uint32 indices into sites() / site_loci() order): row rows[i] lists sites[first[i]:first[i + 1]],
        in no particular order.  counts: count_candidates(result, strand, k), computed when not given."""
        if counts is None:
            counts = self.count_candidates(result, strand, k)
        counts = np.asarray(counts)
        if rows is None:
            rows = np.nonzero(counts[:, 0] != self.NO_COUNT)[0] if len(counts) else np.zeros(0, np.int64)
        rows = np.ascontiguousarray(rows, dtype=np.uint32)
        totals = counts[rows.astype(np.int64), :int(k) + 1].astype(np.uint64).sum(axis=1) if len(rows) else []

        def call(lo, hi, f, out):
            r = np.ascontiguousarray(rows[lo:hi])
            check(lib.crp_offtarget_list_candidates(self._h, result._h, strand.encode(), int(k), hi - lo, r.ctypes.data,
                                                    f.ctypes.data, out.ctypes.data if len(out) else None))
        first, sites = self._list(len(rows), totals, call)
        return rows, first, sites

    def list_guides(self, guides, k=3):
        """(first, sites) of 20-base guides in the protospacer orientation: guide i lists the sites within k
        mismatches, sites[first[i]:first[i + 1]]; nothing subtracted"""
        keys = guide_keys(guides)
        totals = self.count_guides(guides, k).astype(np.uint64).sum(axis=1) if len(keys) else []

        def call(lo, hi, f, out):
            kk = np.ascontiguousarray(keys[lo:hi])
            check(lib.crp_offtarget_list_keys(self._h, hi - lo, kk.ctypes.data, int(k), f.ctypes.data,
                                              out.ctypes.data if len(out) else None))
        return self._list(len(keys), totals, call)

    def score_candidates(self, result, strand, k=3, weights=None):
        """uint64[n_strand]: per candidate of one strand stream (stream order) the sum of weights[rank] over the
        sites its counts count (its own site not included), rank being that of the pair's mismatch-position set
        (score_sets order); NO_SCORE where the candidate has no protospacer.  weights: uint32[SCORE_SETS], each
        < 2**31 (default mit_weights(): sums of MIT hit scores * 2**24 over the sites within k mismatches)."""
        w = _weights(weights)
        n = int(result.n_plus if strand == "+" else result.n_minus)
        out = np.empty(n, dtype=np.uint64)
        check(lib.crp_offtarget_score_candidates(self._h, result._h, strand.encode(), int(k), w.ctypes.data,
                                                 out.ctypes.data if n else None))
        return out

    def score_guides(self, guides, k=3, weights=None):
        """uint64[len(guides)] for 20-base guides in the protospacer orientation; nothing subtracted"""
        w = _weights(weights)
        keys = guide_keys(guides)
        out = np.empty(len(keys), dtype=np.uint64)
        if len(keys):
            check(lib.crp_offtarget_score_keys(self._h, len(keys), keys.ctypes.data, int(k), w.ctypes.data,
                                               out.ctypes.data))
        return out

    def timing(self):
        """dict(ms_sites: every add_genome, ms_count and comparisons: the last count, list or score call)"""
        a, b, n = C.c_float(0), C.c_float(0), C.c_uint64(0)
        check(lib.crp_offtarget_timing(self._h, C.byref(a), C.byref(b), C.byref(n)))
        return {"ms_sites": a.value, "ms_count": b.value, "comparisons": n.value}

    def free(self):
        if self._h:
            check(lib.crp_offtarget_free(self._h))
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass
