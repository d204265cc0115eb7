"""Python surface of the ungapped X-drop seed extender (the reference's cudaextender module,
cudaextender/include/claraparabricks/genomeworks/cudaextender/{cudaextender,extender,utils}.hpp) over the gw-b200 C ABI.
pygenomeworks has no binding for it; the names follow the C++ API.

    ext = create_extender(score_matrix, xdrop_threshold=910, no_entropy=False)
    ext.extend_async(encode_sequence(query), encode_sequence(target), 3000, seed_pairs)   # host arrays
    ext.sync()
    ext.get_scored_segment_pairs()          # numpy structured array, SCORED_SEGMENT_PAIR_DTYPE

The device pointer form takes torch CUDA tensors (extend_async_device)."""
import ctypes as C

import numpy as np

from ._lib import E_BAD_ALLOC, check, last_error, lib

success = 0
invalid_operation = 1
invalid_input = 2
generic_error = 3

ungapped_xdrop = 0

# utils.hpp:36-44
A_NT, C_NT, G_NT, T_NT, L_NT, N_NT, X_NT, E_NT = range(8)
NUC = 8
NUC2 = NUC * NUC

# extender.hpp:36-53: SeedPair {query, target}; ScoredSegmentPair {SeedPair start_coord, length, score}
SEED_PAIR_DTYPE = np.dtype([("query_position_in_read", "<u4"), ("target_position_in_read", "<u4")])
SCORED_SEGMENT_PAIR_DTYPE = np.dtype([("query_position_in_read", "<u4"), ("target_position_in_read", "<u4"), ("length", "<i4"),
                                      ("score", "<i4")])

_ENCODE = np.full(256, X_NT, dtype=np.int8)
for _c, _v in ((b"A", A_NT), (b"C", C_NT), (b"G", G_NT), (b"T", T_NT), (b"&", E_NT), (b"n", N_NT), (b"N", N_NT), (b"a", L_NT),
               (b"c", L_NT), (b"g", L_NT), (b"t", L_NT)):
    _ENCODE[_c[0]] = _v

_ALLOC_FN = C.CFUNCTYPE(C.c_void_p, C.c_void_p, C.c_int64)
_FREE_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_int64)


def encode_sequence(seq):
    """utils.hpp encode_sequence: A C G T -> 0..3, a c g t -> 4, N n -> 5, & -> 7, anything else -> 6. Returns an int8 array."""
    b = seq.encode() if isinstance(seq, str) else bytes(seq)
    return _ENCODE[np.frombuffer(b, dtype=np.uint8)]


def _read_csv(path):
    import gzip
    with (gzip.open(path, "rt") if str(path).endswith(".gz") else open(path)) as f:
        return np.loadtxt(f, delimiter=",", dtype=np.int64, ndmin=2)


def parse_seed_pairs(path):
    """utils.hpp parse_seed_pairs: one `target,query` pair per line (plain or gzipped) -> SEED_PAIR_DTYPE array."""
    a = _read_csv(path)
    out = np.zeros(len(a), dtype=SEED_PAIR_DTYPE)
    if len(a):
        out["target_position_in_read"] = a[:, 0]
        out["query_position_in_read"] = a[:, 1]
    return out


def parse_scored_segment_pairs(path):
    """utils.hpp parse_scored_segment_pairs: `target,query,length,score` lines (plain or gzipped) -> SCORED_SEGMENT_PAIR_DTYPE array."""
    a = _read_csv(path)
    out = np.zeros(len(a), dtype=SCORED_SEGMENT_PAIR_DTYPE)
    for i, name in enumerate(("target_position_in_read", "query_position_in_read", "length", "score")):
        out[name] = a[:, i] if len(a) else 0
    return out


def _as_seeds(seeds):
    s = np.asarray(seeds)
    if s.dtype == SEED_PAIR_DTYPE:
        return np.ascontiguousarray(s)
    s = np.ascontiguousarray(s, dtype=np.uint32).reshape(-1, 2)  # rows of {query, target}, the struct's order
    return s.view(SEED_PAIR_DTYPE).reshape(-1)


class DeviceMemoryAllocationError(MemoryError):
    """device_memory_allocation_exception of the reference (the caller's allocator could not serve a call)."""


class Extender:
    """cudaextender::Extender (extender.hpp:62-134) as create_extender builds it (UngappedXDrop)."""

    def __init__(self, score_matrix, xdrop_threshold, no_entropy=False, stream=None, device_id=0, extension_type=ungapped_xdrop,
                 max_device_memory=None):
        self._h = C.c_void_p()
        mat = np.ascontiguousarray(score_matrix, dtype=np.int32).reshape(-1)
        st = None
        if stream is not None:
            st = stream.stream if hasattr(stream, "stream") else stream.cuda_stream
        self.stream = stream
        self._alloc = self._free = None
        self._blocks = {}
        alloc = free = None
        if max_device_memory is not None:
            # a pool of max_device_memory bytes served from torch's caching allocator: what a DefaultDeviceAllocator of that
            # size is to a C++ caller
            self._budget = int(max_device_memory)
            self._used = 0
            self._alloc = alloc = _ALLOC_FN(self._pool_alloc)
            self._free = free = _FREE_FN(self._pool_free)
        self.device_id = device_id
        check(lib().gwb200_extender_create(C.byref(self._h), mat.ctypes.data_as(C.POINTER(C.c_int32)), C.c_int32(len(mat)),
                                           C.c_int32(xdrop_threshold), C.c_int32(1 if no_entropy else 0), C.c_void_p(st),
                                           C.c_int32(device_id), C.c_int32(extension_type),
                                           None if alloc is None else C.cast(alloc, C.c_void_p),
                                           None if free is None else C.cast(free, C.c_void_p), None))

    def _pool_alloc(self, user, nbytes):
        import torch
        if self._used + nbytes > self._budget:
            return None
        t = torch.empty(int(nbytes), dtype=torch.uint8, device="cuda:%d" % self.device_id)
        self._blocks[t.data_ptr()] = t
        self._used += nbytes
        return t.data_ptr()

    def _pool_free(self, user, ptr, nbytes):
        t = self._blocks.pop(ptr, None)
        if t is not None:
            self._used -= nbytes
            import torch
            torch.cuda.synchronize(self.device_id)

    def _status(self, rc):
        if rc == E_BAD_ALLOC:
            raise DeviceMemoryAllocationError(last_error())
        return check(rc)

    def extend_async(self, query, target, score_threshold, seed_pairs):
        """Host pointer API: encoded query / target (int8 arrays or strings, encoded here) and SeedPairs. Returns a StatusType."""
        q = np.ascontiguousarray(encode_sequence(query) if isinstance(query, (str, bytes)) else query, dtype=np.int8)
        t = np.ascontiguousarray(encode_sequence(target) if isinstance(target, (str, bytes)) else target, dtype=np.int8)
        s = _as_seeds(seed_pairs)
        return self._status(lib().gwb200_extender_extend_host(self._h, q.ctypes.data_as(C.POINTER(C.c_int8)), C.c_int32(len(q)),
                                                              t.ctypes.data_as(C.POINTER(C.c_int8)), C.c_int32(len(t)),
                                                              C.c_int32(score_threshold), s.ctypes.data_as(C.c_void_p), C.c_int32(len(s))))

    def extend_async_device(self, d_query, d_target, score_threshold, d_seed_pairs, d_scored_segment_pairs, d_num_scored_segment_pairs):
        """Device pointer API over torch CUDA tensors: d_query / d_target int8 [len], d_seed_pairs int32/uint32 [n, 2] rows of
        {query, target} (or a flat [2n]), d_scored_segment_pairs int32 [n, 4] (or any tensor of 16 n bytes), d_num int32 [1].
        Stream ordered on the extender's stream. Returns a StatusType."""
        def ptr(x):
            return None if x is None else C.c_void_p(x.data_ptr())

        def length(x):
            return 0 if x is None else int(x.numel())
        n = 0 if d_seed_pairs is None else d_seed_pairs.numel() // 2
        return self._status(lib().gwb200_extender_extend_device(self._h, ptr(d_query), C.c_int32(length(d_query)), ptr(d_target),
                                                                C.c_int32(length(d_target)), C.c_int32(score_threshold), ptr(d_seed_pairs),
                                                                C.c_int32(n), ptr(d_scored_segment_pairs), ptr(d_num_scored_segment_pairs)))

    def sync(self):
        """Waits for the last host-API call and fetches its results; invalid_operation without one."""
        return check(lib().gwb200_extender_sync(self._h))

    def get_scored_segment_pairs(self):
        """Results of the last host-API call as a SCORED_SEGMENT_PAIR_DTYPE array; RuntimeError without one."""
        n = check(lib().gwb200_extender_num_results(self._h))
        out = np.zeros(n, dtype=SCORED_SEGMENT_PAIR_DTYPE)
        if n:
            check(lib().gwb200_extender_get_results(self._h, out.ctypes.data_as(C.c_void_p), C.c_int64(n)))
        return out

    def reset(self):
        check(lib().gwb200_extender_reset(self._h))

    def last_kernel_ms(self):
        return float(lib().gwb200_extender_last_kernel_ms(self._h))

    def last_positions(self):
        return int(lib().gwb200_extender_last_positions(self._h))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            lib().gwb200_extender_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def create_extender(score_matrix, xdrop_threshold, no_entropy=False, stream=None, device_id=0, extension_type=ungapped_xdrop,
                    max_device_memory=None):
    """create_extender (extender.hpp:147-154). score_matrix: 64 ints (8 x 8, row = target code). max_device_memory: size of the
    pool the extender's device memory comes from (None: cudaMalloc as needed)."""
    return Extender(score_matrix, xdrop_threshold, no_entropy, stream, device_id, extension_type, max_device_memory)
