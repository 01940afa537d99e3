"""ctypes binding of the C-ABI in include/dist_b200.h (libdist_b200.so).

The library is the only compute path: if it is missing or fails to load, importing this module
raises -- there is no Python / CPU fallback for scoring or sampling.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libdist_b200.so")

DD, DPD, BB, GP, NICH, NIW, BNB = 0, 1, 2, 3, 4, 5, 6
# dist_b200_option
OPT_VALUE_CDF, OPT_ROW_TILE, OPT_HOST_CHUNKS, OPT_NIW_PATH, OPT_TABLE_KERNEL, OPT_SMALL_TILE, OPT_NICH_PACKED, OPT_NIW_DEBUG, OPT_HOST_ZEROCOPY, OPT_EXP_OFFLOAD = range(10)
MODEL_NAMES = {DD: "dd", DPD: "dpd", BB: "bb", GP: "gp", NICH: "nich", NIW: "niw", BNB: "bnb"}
COLUMN_DTYPE = {DD: np.int32, DPD: np.uint32, BB: np.uint8, GP: np.uint32, NICH: np.float32, NIW: np.float32, BNB: np.uint32}

c_f, c_i, c_sz, c_p = ctypes.c_float, ctypes.c_int, ctypes.c_size_t, ctypes.c_void_p

# every symbol include/dist_b200.h declares: (restype, argtypes)
SIGNATURES = {
    "dist_b200_abi_version": (c_i, []),
    "dist_b200_ctx_create": (c_i, [c_i, ctypes.POINTER(c_p)]),
    "dist_b200_ctx_destroy": (None, [c_p]),
    "dist_b200_last_error": (ctypes.c_char_p, [c_p]),
    "dist_b200_sm_count": (c_i, [c_p]),
    "dist_b200_ctx_set_option": (c_i, [c_p, c_i, c_i]),
    "dist_b200_feature_create": (c_i, [c_p, c_i, ctypes.POINTER(c_p)]),
    "dist_b200_feature_destroy": (None, [c_p]),
    "dist_b200_feature_model": (c_i, [c_p]),
    "dist_b200_feature_groups": (c_i, [c_p]),
    "dist_b200_nich_update_all": (c_i, [c_p, c_p, c_i, c_p, c_p, c_p, c_p]),
    "dist_b200_gp_update_all": (c_i, [c_p, c_p, c_i, c_p, c_p, c_p]),
    "dist_b200_bb_update_all": (c_i, [c_p, c_p, c_i, c_p, c_p, c_p]),
    "dist_b200_bnb_update_all": (c_i, [c_p, c_p, ctypes.c_uint32, c_i, c_p, c_p, c_p]),
    "dist_b200_dd_update_all": (c_i, [c_p, c_i, c_p, c_i, c_p, c_p]),
    "dist_b200_dpd_update_all": (c_i, [c_p, c_f, c_f, c_i, c_p, c_p, c_i, c_p, c_p]),
    "dist_b200_niw_update_all": (c_i, [c_p, c_i, c_p, c_f, c_p, c_f, c_i, c_p, c_p, c_p, c_p]),
    "dist_b200_feature_update_group": (c_i, [c_p, c_i, c_p, c_p]),
    "dist_b200_feature_add_group": (c_i, [c_p, c_p]),
    "dist_b200_feature_remove_group": (c_i, [c_p, c_i, c_p]),
    "dist_b200_feature_add_rows": (c_i, [c_p, c_p, c_p, c_sz, c_p]),
    "dist_b200_add_rows_batch": (c_i, [c_p, c_p, c_i, c_p, c_p, c_sz, c_p]),
    "dist_b200_add_rows_batch_host": (c_i, [c_p, c_p, c_i, c_p, c_p, c_sz]),
    "dist_b200_remove_rows_batch": (c_i, [c_p, c_p, c_i, c_p, c_p, c_sz, c_p]),
    "dist_b200_rows_accumulate": (c_i, [c_p, c_p, c_i, c_p, c_p, c_sz, c_p, c_p]),
    "dist_b200_rows_merge": (c_i, [c_p, c_p, c_i, c_p, c_i, c_p]),
    "dist_b200_rows_xchg_doubles": (c_i, [c_p, c_i, c_p]),
    "dist_b200_remove_rows_batch_host": (c_i, [c_p, c_p, c_i, c_p, c_p, c_sz]),
    "dist_b200_sample_values_batch": (c_i, [c_p, c_p, c_i, c_p, c_sz, ctypes.c_uint64, ctypes.c_uint64, c_p, c_p]),
    "dist_b200_sample_values_batch_host": (c_i, [c_p, c_p, c_i, c_p, c_sz, ctypes.c_uint64, ctypes.c_uint64, c_p]),
    "dist_b200_gp_set_log_prod": (c_i, [c_p, c_p, c_p]),
    "dist_b200_score_data_grid": (c_i, [c_p, c_p, c_sz, c_sz, c_p, c_p]),
    "dist_b200_score_data_grid_host": (c_i, [c_p, c_p, c_sz, c_sz, c_p]),
    "dist_b200_update_all_wire": (c_i, [c_p, c_p, c_sz, c_p, c_p, c_i, c_p]),
    "dist_b200_wire_decode": (c_i, [c_p, c_i, c_p, c_sz, c_p, c_p, c_i, c_p, c_sz, c_p, c_sz, c_p, c_sz, c_p]),
    "dist_b200_prior_wire_host": (c_i, [c_p, c_p, c_sz, c_i, c_p, c_p]),
    "dist_b200_update_all_stream": (c_i, [c_p, c_p, c_sz, c_p, c_sz, c_p]),
    "dist_b200_wire_encode_shared": (c_i, [c_p, c_i, c_p, c_sz, c_p, c_sz, c_p, c_sz, c_p]),
    "dist_b200_wire_split_stream": (c_i, [c_p, c_p, c_sz, c_p, c_p, c_sz, c_p]),
    "dist_b200_feature_dump_groups_wire": (c_i, [c_p, c_p, c_sz, c_p, c_p, c_p]),
    "dist_b200_wire_encode_groups": (c_i, [c_p, c_i, c_i, c_i, c_p, c_p, c_sz, c_p, c_sz, c_p, c_p]),
    "dist_b200_feature_download_stats": (c_i, [c_p, c_p, c_sz, ctypes.POINTER(c_sz), c_p]),
    "dist_b200_count_assignments": (c_i, [c_p, c_p, c_sz, c_i, c_p, c_i, c_p]),
    "dist_b200_prior_pitman_yor_dev": (c_i, [c_p, c_f, c_f, c_i, c_p, c_p, c_p]),
    "dist_b200_prior_low_entropy_host": (c_i, [c_p, c_i, c_i, c_p, c_p]),
    "dist_b200_prior_low_entropy_dev": (c_i, [c_p, c_i, c_i, c_p, c_p, c_p]),
    "dist_b200_feature_download_caches": (c_i, [c_p, c_p, c_sz, ctypes.POINTER(c_sz), c_p]),
    "dist_b200_prior_pitman_yor": (c_i, [c_p, c_f, c_f, c_i, c_p, c_p, c_p]),
    "dist_b200_prior_pitman_yor_host": (c_i, [c_p, c_f, c_f, c_i, c_p, c_p]),
    "dist_b200_score_batch": (c_i, [c_p, c_p, c_i, c_p, c_sz, c_p, c_p, c_i, c_p]),
    "dist_b200_score_sample_batch": (c_i, [c_p, c_p, c_i, c_p, c_sz, c_p, c_p, c_p, c_p, c_p]),
    "dist_b200_sample_from_scores": (c_i, [c_p, c_p, c_sz, c_i, c_p, c_p, c_p]),
    "dist_b200_score_logp_batch": (c_i, [c_p, c_p, c_i, c_p, c_sz, c_p, c_p, c_p]),
    "dist_b200_score_logp_batch_host": (c_i, [c_p, c_p, c_i, c_p, c_sz, c_p, c_p]),
    "dist_b200_logp_from_scores": (c_i, [c_p, c_p, c_sz, c_i, c_p, c_p]),
    "dist_b200_peer_alloc": (c_i, [c_p, c_sz, ctypes.POINTER(c_p), c_p]),
    "dist_b200_peer_open": (c_i, [c_p, c_p, ctypes.POINTER(c_p)]),
    "dist_b200_peer_close": (c_i, [c_p, c_p]),
    "dist_b200_peer_free": (c_i, [c_p, c_p]),
    "dist_b200_score_push_batch": (c_i, [c_p, c_p, c_i, c_p, c_sz, c_sz, c_p, c_p, c_i, c_sz, c_p]),
    "dist_b200_peer_signal": (c_i, [c_p, c_p, c_i, c_i, ctypes.c_uint32, c_p]),
    "dist_b200_peer_wait": (c_i, [c_p, c_p, c_i, ctypes.c_uint32, c_p]),
    "dist_b200_sample_from_slots": (c_i, [c_p, c_p, c_i, c_sz, c_sz, c_i, c_p, c_p, c_p]),
    "dist_b200_score_sample_batch_host": (c_i, [c_p, c_p, c_i, c_p, c_sz, c_p, c_p, c_p, c_p]),
    "dist_b200_score_value_host": (c_i, [c_p, c_p, c_p, c_p]),
    "dist_b200_host_register": (c_i, [c_p, c_p, c_sz]),
    "dist_b200_host_unregister": (c_i, [c_p, c_p]),
    "dist_b200_numerics_probe": (c_i, [c_p, c_i, c_sz, c_p, c_p, c_p]),
    "dist_b200_pipe_peak": (c_i, [c_p, c_i, ctypes.POINTER(ctypes.c_double)]),
    "dist_b200_score_batch_masked": (c_i, [c_p, c_p, c_i, c_p, c_sz, c_p, c_p, c_i, c_p, c_p]),
    "dist_b200_score_sample_batch_masked": (c_i, [c_p, c_p, c_i, c_p, c_sz, c_p, c_p, c_p, c_p, c_p, c_p]),
    "dist_b200_score_logp_batch_masked": (c_i, [c_p, c_p, c_i, c_p, c_sz, c_p, c_p, c_p, c_p]),
    "dist_b200_add_rows_batch_masked": (c_i, [c_p, c_p, c_i, c_p, c_p, c_sz, c_p, c_p]),
    "dist_b200_remove_rows_batch_masked": (c_i, [c_p, c_p, c_i, c_p, c_p, c_sz, c_p, c_p]),
    "dist_b200_rows_accumulate_masked": (c_i, [c_p, c_p, c_i, c_p, c_p, c_sz, c_p, c_p, c_p]),
    "dist_b200_sample_values_batch_masked": (c_i, [c_p, c_p, c_i, c_p, c_sz, ctypes.c_uint64, ctypes.c_uint64, c_p, c_p, c_p]),
}


class DistB200Error(RuntimeError):
    pass


def load_library(path=LIB_PATH):
    if not os.path.exists(path):
        raise DistB200Error(
            "%s is missing: build it with `python -m distributions_b200.build` "
            "(there is no CPU fallback for the scoring path)" % path)
    lib = ctypes.CDLL(path)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.restype = restype
        fn.argtypes = argtypes
    return lib


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = load_library()
    return _lib


def _np_ptr(a):
    return a.ctypes.data if a is not None else None


def _dev_ptr(t):
    """device pointer of a torch tensor / raw int / None"""
    if t is None:
        return None
    if isinstance(t, int):
        return t
    return t.data_ptr()


def pack_observed(mask):
    """a bool column (numpy or torch, True = observed) -> the observed-mask words of the *_masked entries:
    ceil(N / 32) uint32, bit n % 32 of word n / 32 = mask[n] (np.packbits little-endian bit order, read as little-endian
    uint32; bits past N are 0).  Returns the type it was given: a numpy array, or a torch tensor on the input's device."""
    torch_in = not isinstance(mask, np.ndarray) and hasattr(mask, "detach")
    m = mask.detach().cpu().numpy() if torch_in else np.asarray(mask)
    m = np.ascontiguousarray(m, dtype=bool).reshape(-1)
    n_words = (m.size + 31) // 32
    b = np.zeros(4 * n_words, dtype=np.uint8)
    b[:(m.size + 7) // 8] = np.packbits(m, bitorder="little")
    words = b.view("<u4").astype(np.uint32)
    if torch_in:
        import torch
        return torch.from_numpy(words.view(np.int32).copy()).to(mask.device)
    return words


def _masks(observed, F):
    """observed: None or one entry per feature (None = fully observed, else a device tensor / pointer of mask words)"""
    if observed is None:
        return None
    assert len(observed) == F, "observed: one entry per feature"
    return (c_p * F)(*[_dev_ptr(o) for o in observed])


def wire_decode(model, shared_msg, group_msgs):
    """decode serialized Shared / Group messages into (shared floats, keys, stats words); needs no device"""
    L = lib()
    G = len(group_msgs)
    bufs = [ctypes.create_string_buffer(m, len(m)) for m in group_msgs]
    ptrs = (c_p * max(G, 1))(*[ctypes.addressof(b) for b in bufs])
    lens = (c_sz * max(G, 1))(*[len(m) for m in group_msgs])
    counts = (c_sz * 3)()
    args = (None, model, shared_msg, len(shared_msg), ptrs, lens, G)
    rc = L.dist_b200_wire_decode(*args, None, 0, None, 0, None, 0, counts)
    if rc not in (0, 1) or (rc == 1 and not any(counts)):
        raise ValueError("wire_decode: status %d" % rc)
    sh = np.empty(counts[0], np.float32)
    keys = np.empty(counts[1], np.uint32)
    st = np.empty(counts[2], np.uint32)
    rc = L.dist_b200_wire_decode(*args, _np_ptr(sh), sh.size, _np_ptr(keys), keys.size, _np_ptr(st), st.size, counts)
    if rc != 0:
        raise ValueError("wire_decode: status %d" % rc)
    return sh, keys, st


def _split(buf, lens):
    offs = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    raw = buf.tobytes()
    return [raw[offs[i]:offs[i + 1]] for i in range(len(lens))]


def wire_encode_shared(model, shared, keys=None):
    """packed Shared values (wire_decode's) -> the serialized Shared message; needs no device"""
    L = lib()
    shared = np.ascontiguousarray(shared, dtype=np.float32)
    keys = np.ascontiguousarray(keys if keys is not None else [], dtype=np.uint32)
    buf = np.empty(16 + 5 * shared.size + 11 * keys.size, np.uint8)
    n = c_sz()
    rc = L.dist_b200_wire_encode_shared(None, model, _np_ptr(shared), shared.size, _np_ptr(keys) if keys.size else None, keys.size,
                                        _np_ptr(buf), buf.size, ctypes.byref(n))
    if rc != 0:
        raise ValueError("wire_encode_shared: status %d" % rc)
    return buf[:n.value].tobytes()


def wire_split_stream(stream_bytes):
    """records of a [uint32 length][message] stream (the reference's protobuf_stream format): list of bytes"""
    L = lib()
    n = c_sz()
    rc = L.dist_b200_wire_split_stream(None, stream_bytes, len(stream_bytes), None, None, 0, ctypes.byref(n))
    if rc not in (0, 1) or (rc == 1 and n.value == 0):
        raise ValueError("wire_split_stream: status %d" % rc)
    offs, lens = (c_sz * max(n.value, 1))(), (c_sz * max(n.value, 1))()
    rc = L.dist_b200_wire_split_stream(None, stream_bytes, len(stream_bytes), offs, lens, n.value, ctypes.byref(n))
    if rc != 0:
        raise ValueError("wire_split_stream: status %d" % rc)
    return [stream_bytes[offs[i]:offs[i] + lens[i]] for i in range(n.value)]


def wire_encode_groups(model, G, dim, keys, stats):
    """SoA statistics (the arrays wire_decode returns) -> list of serialized Group messages; needs no device"""
    L = lib()
    stats = np.ascontiguousarray(stats, dtype=np.uint32)
    keys = np.ascontiguousarray(keys, dtype=np.uint32) if keys is not None else np.zeros(0, np.uint32)
    n = c_sz()
    lens = (c_sz * max(G, 1))()
    rc = L.dist_b200_wire_encode_groups(None, model, G, dim, _np_ptr(keys) if keys.size else None, _np_ptr(stats), stats.size,
                                        None, 0, lens, ctypes.byref(n))
    if rc != 1 and not (rc == 0 and n.value == 0):
        raise ValueError("wire_encode_groups: status %d" % rc)
    buf = np.empty(n.value, np.uint8)
    rc = L.dist_b200_wire_encode_groups(None, model, G, dim, _np_ptr(keys) if keys.size else None, _np_ptr(stats), stats.size,
                                        _np_ptr(buf), buf.size, lens, ctypes.byref(n))
    if rc != 0:
        raise ValueError("wire_encode_groups: status %d" % rc)
    return _split(buf, [lens[i] for i in range(G)])


class Context:
    def __init__(self, device=0):
        self.L = lib()
        h = c_p()
        rc = self.L.dist_b200_ctx_create(device, ctypes.byref(h))
        if rc != 0:
            raise DistB200Error("dist_b200_ctx_create(device=%d) failed with status %d (no usable CUDA device?)" % (device, rc))
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.dist_b200_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc, what):
        if rc != 0:
            msg = self.L.dist_b200_last_error(self.h)
            raise DistB200Error("%s failed: status %d: %s" % (what, rc, msg.decode() if msg else ""))

    def set_option(self, option, value):
        """measurement knob (dist_b200_option); 0 restores the default"""
        self.check(self.L.dist_b200_ctx_set_option(self.h, int(option), int(value)), "set_option")

    @property
    def sm_count(self):
        return self.L.dist_b200_sm_count(self.h)

    def feature(self, model):
        return Feature(self, model)

    # -- prior ----------------------------------------------------------------------------------
    def prior_pitman_yor(self, alpha, d, group_sizes, prior_dev, stream=None):
        sizes = np.ascontiguousarray(group_sizes, dtype=np.int32)
        self.check(self.L.dist_b200_prior_pitman_yor(self.h, alpha, d, sizes.size, _np_ptr(sizes), _dev_ptr(prior_dev),
                                                     stream), "prior_pitman_yor")

    def prior_pitman_yor_host(self, alpha, d, group_sizes):
        sizes = np.ascontiguousarray(group_sizes, dtype=np.int32)
        out = np.empty(sizes.size, dtype=np.float32)
        self.check(self.L.dist_b200_prior_pitman_yor_host(self.h, alpha, d, sizes.size, _np_ptr(sizes), _np_ptr(out)), "prior_pitman_yor_host")
        return out

    def add_rows_batch(self, features, columns, assign_dev, n_rows, stream=None, observed=None):
        """batched Group::add_value for all features of one kind; nothing is drained, later calls order behind it.
        observed: None, or per feature None / pack_observed words on the device (a missing cell is not added)"""
        F, fa, ca = self._lists(features, columns)
        if observed is not None:
            self.check(self.L.dist_b200_add_rows_batch_masked(self.h, fa, F, ca, _dev_ptr(assign_dev), n_rows, _masks(observed, F),
                                                              stream), "add_rows_batch_masked")
            return
        self.check(self.L.dist_b200_add_rows_batch(self.h, fa, F, ca, _dev_ptr(assign_dev), n_rows, stream), "add_rows_batch")

    def rows_xchg_doubles(self, features):
        """size (float64 elements) of the row-shard exchange buffer: [4][G] per pooled feature, then [G][dim] per dd / dpd table"""
        F = len(features)
        fa = (c_p * F)(*[f.h for f in features])
        n = ctypes.c_size_t(0)
        self.check(self.L.dist_b200_rows_xchg_doubles(fa, F, ctypes.byref(n)), "rows_xchg_doubles")
        return int(n.value)

    def rows_accumulate(self, features, columns, assign_dev, n_rows, xchg_dev, stream=None, observed=None):
        """row shards: this rank's accumulators into xchg_dev (rows_xchg_doubles float64; then all-reduce, then rows_merge)"""
        F, fa, ca = self._lists(features, columns)
        if observed is not None:
            self.check(self.L.dist_b200_rows_accumulate_masked(self.h, fa, F, ca, _dev_ptr(assign_dev), n_rows, _dev_ptr(xchg_dev),
                                                               _masks(observed, F), stream), "rows_accumulate_masked")
            return
        self.check(self.L.dist_b200_rows_accumulate(self.h, fa, F, ca, _dev_ptr(assign_dev), n_rows, _dev_ptr(xchg_dev), stream),
                   "rows_accumulate")

    def rows_merge(self, features, xchg_dev, sign=+1, stream=None):
        F = len(features)
        fa = (c_p * F)(*[f.h for f in features])
        self.check(self.L.dist_b200_rows_merge(self.h, fa, F, _dev_ptr(xchg_dev), sign, stream), "rows_merge")

    def remove_rows_batch(self, features, columns, assign_dev, n_rows, stream=None, observed=None):
        """batched Group::remove_value: the rows leave the groups assign_dev names (observed: as in add_rows_batch)"""
        F, fa, ca = self._lists(features, columns)
        if observed is not None:
            self.check(self.L.dist_b200_remove_rows_batch_masked(self.h, fa, F, ca, _dev_ptr(assign_dev), n_rows,
                                                                 _masks(observed, F), stream), "remove_rows_batch_masked")
            return
        self.check(self.L.dist_b200_remove_rows_batch(self.h, fa, F, ca, _dev_ptr(assign_dev), n_rows, stream), "remove_rows_batch")

    def remove_rows_batch_host(self, features, columns, assign):
        F = len(features)
        cols = [np.ascontiguousarray(c, dtype=COLUMN_DTYPE[f.model]) for f, c in zip(features, columns)]
        assign = np.ascontiguousarray(assign, dtype=np.int32)
        fa = (c_p * F)(*[f.h for f in features])
        ca = (c_p * F)(*[_np_ptr(c) for c in cols])
        self.check(self.L.dist_b200_remove_rows_batch_host(self.h, fa, F, ca, _np_ptr(assign), assign.size), "remove_rows_batch_host")

    def add_rows_batch_host(self, features, columns, assign):
        """host arrays: columns[i] numpy array of COLUMN_DTYPE[model], assign int32"""
        F = len(features)
        cols = [np.ascontiguousarray(c, dtype=COLUMN_DTYPE[f.model]) for f, c in zip(features, columns)]
        assign = np.ascontiguousarray(assign, dtype=np.int32)
        fa = (c_p * F)(*[f.h for f in features])
        ca = (c_p * F)(*[_np_ptr(c) for c in cols])
        self.check(self.L.dist_b200_add_rows_batch_host(self.h, fa, F, ca, _np_ptr(assign), assign.size), "add_rows_batch_host")

    def sample_values_batch(self, features, assign_dev, n_rows, columns_out, seed=0, row0=0, stream=None, observed=None):
        """batched Group::sample_value: columns_out[i][n] (device) <- a posterior-predictive draw of group assign_dev[n]
        of features[i]; rows with an id outside [0, G) keep their values.  Draws depend on (seed, row0 + n, i) only.
        observed (imputation): per feature None / mask words; only MISSING cells are drawn (None: nothing is drawn)."""
        F, fa, ca = self._lists(features, columns_out)
        if observed is not None:
            self.check(self.L.dist_b200_sample_values_batch_masked(self.h, fa, F, _dev_ptr(assign_dev), n_rows, int(seed), int(row0),
                                                                   ca, _masks(observed, F), stream), "sample_values_batch_masked")
            return
        self.check(self.L.dist_b200_sample_values_batch(self.h, fa, F, _dev_ptr(assign_dev), n_rows, int(seed), int(row0), ca, stream),
                   "sample_values_batch")

    def sample_values_batch_host(self, features, assign, seed=0, row0=0, out=None):
        """host form: a list of one array per feature (COLUMN_DTYPE; niw [n][d]).  `out` (optional) supplies the arrays,
        whose rows with an id outside [0, G) are left as they are; fresh arrays are zero-filled."""
        F = len(features)
        assign = np.ascontiguousarray(assign, dtype=np.int32)
        n = assign.size
        if out is None:
            assert all(f.model != NIW or f.dim for f in features), "niw feature of unknown d: pass `out`"
            out = [np.zeros((n, f.dim) if f.model == NIW else n, dtype=COLUMN_DTYPE[f.model]) for f in features]
        for f, o in zip(features, out):
            assert o.dtype == COLUMN_DTYPE[f.model] and o.flags.c_contiguous and o.shape[0] == n, "bad output array"
        fa = (c_p * F)(*[f.h for f in features])
        ca = (c_p * F)(*[_np_ptr(o) for o in out])
        self.check(self.L.dist_b200_sample_values_batch_host(self.h, fa, F, _np_ptr(assign), n, int(seed), int(row0), ca),
                   "sample_values_batch_host")
        return out

    def count_assignments(self, assign_dev, n_rows, G, counts_dev, accumulate=False, stream=None):
        self.check(self.L.dist_b200_count_assignments(self.h, _dev_ptr(assign_dev), n_rows, G, _dev_ptr(counts_dev),
                                                      1 if accumulate else 0, stream), "count_assignments")

    def prior_wire_host(self, clustering_msg, sizes):
        sizes = np.ascontiguousarray(sizes, dtype=np.int32)
        out = np.empty(sizes.size, dtype=np.float32)
        self.check(self.L.dist_b200_prior_wire_host(self.h, clustering_msg, len(clustering_msg), sizes.size, _np_ptr(sizes), _np_ptr(out)),
                   "prior_wire")
        return out

    def prior_low_entropy_host(self, dataset_size, sizes):
        sizes = np.ascontiguousarray(sizes, dtype=np.int32)
        out = np.empty(sizes.size, dtype=np.float32)
        self.check(self.L.dist_b200_prior_low_entropy_host(self.h, int(dataset_size), sizes.size, _np_ptr(sizes), _np_ptr(out)),
                   "prior_low_entropy")
        return out

    def prior_low_entropy_dev(self, dataset_size, G, sizes_dev, prior_dev, stream=None):
        self.check(self.L.dist_b200_prior_low_entropy_dev(self.h, int(dataset_size), G, _dev_ptr(sizes_dev), _dev_ptr(prior_dev), stream),
                   "prior_low_entropy_dev")

    def prior_pitman_yor_dev(self, alpha, d, G, sizes_dev, prior_dev, stream=None):
        self.check(self.L.dist_b200_prior_pitman_yor_dev(self.h, alpha, d, G, _dev_ptr(sizes_dev), _dev_ptr(prior_dev), stream),
                   "prior_pitman_yor_dev")

    # -- hot path (device pointers) --------------------------------------------------------------
    def _lists(self, features, columns):
        F = len(features)
        fa = (c_p * F)(*[f.h for f in features])
        ca = (c_p * F)(*[_dev_ptr(c) for c in columns])
        return F, fa, ca

    def score_batch(self, features, columns, n_rows, prior, scores, accumulate=False, stream=None, observed=None):
        F, fa, ca = self._lists(features, columns)
        if observed is not None:
            self.check(self.L.dist_b200_score_batch_masked(self.h, fa, F, ca, n_rows, _dev_ptr(prior), _dev_ptr(scores),
                                                           1 if accumulate else 0, _masks(observed, F), stream), "score_batch_masked")
            return
        self.check(self.L.dist_b200_score_batch(self.h, fa, F, ca, n_rows, _dev_ptr(prior), _dev_ptr(scores),
                                                1 if accumulate else 0, stream), "score_batch")

    def score_sample_batch(self, features, columns, n_rows, prior, u, assign, scores=None, stream=None, observed=None):
        """observed: None, or per feature None (fully observed) / pack_observed words on the device; a missing cell
        contributes 0 to every group's score"""
        F, fa, ca = self._lists(features, columns)
        if observed is not None:
            self.check(self.L.dist_b200_score_sample_batch_masked(self.h, fa, F, ca, n_rows, _dev_ptr(prior), _dev_ptr(u),
                                                                  _dev_ptr(assign), _dev_ptr(scores), _masks(observed, F), stream),
                       "score_sample_batch_masked")
            return
        self.check(self.L.dist_b200_score_sample_batch(self.h, fa, F, ca, n_rows, _dev_ptr(prior), _dev_ptr(u),
                                                       _dev_ptr(assign), _dev_ptr(scores), stream), "score_sample_batch")

    def sample_from_scores(self, scores, n_rows, G, u, assign, stream=None):
        self.check(self.L.dist_b200_sample_from_scores(self.h, _dev_ptr(scores), n_rows, G, _dev_ptr(u), _dev_ptr(assign),
                                                       stream), "sample_from_scores")

    def score_logp_batch(self, features, columns, n_rows, prior, logp, stream=None, observed=None):
        """logp[n] (device, float32) <- log sum_g exp(prior[g] + sum_f score_f(columns[f][n]; g)); prior may be None.
        observed: as in score_sample_batch (a missing cell's term is left out of the sum)"""
        F, fa, ca = self._lists(features, columns)
        if observed is not None:
            self.check(self.L.dist_b200_score_logp_batch_masked(self.h, fa, F, ca, n_rows, _dev_ptr(prior), _dev_ptr(logp),
                                                                _masks(observed, F), stream), "score_logp_batch_masked")
            return
        self.check(self.L.dist_b200_score_logp_batch(self.h, fa, F, ca, n_rows, _dev_ptr(prior), _dev_ptr(logp), stream),
                   "score_logp_batch")

    def logp_from_scores(self, scores, n_rows, G, logp, stream=None):
        """logp[n] <- log sum_g exp(scores[n][g]) over materialised [n_rows][G] scores (device)"""
        self.check(self.L.dist_b200_logp_from_scores(self.h, _dev_ptr(scores), n_rows, G, _dev_ptr(logp), stream), "logp_from_scores")

    # -- feature shards over peer memory ---------------------------------------------------------
    def peer_alloc(self, nbytes):
        """cudaMalloc a buffer and return (device pointer, 64-byte IPC handle)"""
        ptr = c_p()
        handle = (ctypes.c_ubyte * 64)()
        self.check(self.L.dist_b200_peer_alloc(self.h, nbytes, ctypes.byref(ptr), handle), "peer_alloc")
        return ptr.value, bytes(handle)

    def peer_open(self, handle):
        ptr = c_p()
        buf = (ctypes.c_ubyte * 64).from_buffer_copy(handle)
        self.check(self.L.dist_b200_peer_open(self.h, buf, ctypes.byref(ptr)), "peer_open")
        return ptr.value

    def peer_close(self, ptr):
        self.check(self.L.dist_b200_peer_close(self.h, ptr), "peer_close")

    def peer_free(self, ptr):
        self.check(self.L.dist_b200_peer_free(self.h, ptr), "peer_free")

    def score_push_batch(self, features, columns, n_rows, row0, prior, slot_ptrs, block_rows, stream=None):
        F, fa, ca = self._lists(features, columns)
        sp = (c_p * len(slot_ptrs))(*slot_ptrs)
        self.check(self.L.dist_b200_score_push_batch(self.h, fa, F, ca, n_rows, row0, _dev_ptr(prior), sp, len(slot_ptrs),
                                                     block_rows, stream), "score_push_batch")

    def peer_signal(self, flag_ptrs, my_index, epoch, stream=None):
        fp = (c_p * len(flag_ptrs))(*flag_ptrs)
        self.check(self.L.dist_b200_peer_signal(self.h, fp, len(flag_ptrs), my_index, epoch, stream), "peer_signal")

    def peer_wait(self, flags, n_peers, epoch, stream=None):
        self.check(self.L.dist_b200_peer_wait(self.h, _dev_ptr(flags), n_peers, epoch, stream), "peer_wait")

    def sample_from_slots(self, slots, n_slots, slot_stride, n_rows, G, u, assign, stream=None):
        self.check(self.L.dist_b200_sample_from_slots(self.h, _dev_ptr(slots), n_slots, slot_stride, n_rows, G, _dev_ptr(u),
                                                      _dev_ptr(assign), stream), "sample_from_slots")

    # -- host-buffer forms -----------------------------------------------------------------------
    def score_sample_batch_host(self, features, columns, prior, u, want_scores=False, assign_out=None):
        """Host-buffer entry.  Arrays that are already page-locked (e.g. numpy views of
        torch.Tensor.pin_memory()) are copied from directly; pageable ones are staged by the library."""
        F = len(features)
        cols = [np.ascontiguousarray(c, dtype=COLUMN_DTYPE[f.model]) for f, c in zip(features, columns)]
        n = u.shape[0]
        G = features[0].groups
        for f, c in zip(features, cols):
            assert c.size == n or (f.model == NIW and c.size % n == 0), "column length != len(u)"
        fa = (c_p * F)(*[f.h for f in features])
        ca = (c_p * F)(*[c.ctypes.data for c in cols])
        prior = None if prior is None else np.ascontiguousarray(prior, dtype=np.float32)
        u = np.ascontiguousarray(u, dtype=np.float32)
        assign = assign_out if assign_out is not None else np.empty(n, dtype=np.int32)
        assert assign.dtype == np.int32 and assign.size == n and assign.flags.c_contiguous
        scores = np.empty((n, G), dtype=np.float32) if want_scores else None
        self.check(self.L.dist_b200_score_sample_batch_host(self.h, fa, F, ca, n, _np_ptr(prior), _np_ptr(u), _np_ptr(assign),
                                                            _np_ptr(scores)), "score_sample_batch_host")
        return assign, scores

    def score_logp_batch_host(self, features, columns, prior=None, logp_out=None):
        """Host-buffer form of score_logp_batch: returns the float32 logp of every row.  Page-locked arrays (and a
        page-locked `logp_out`) take the zero-copy route, as in score_sample_batch_host."""
        F = len(features)
        cols = [np.ascontiguousarray(c, dtype=COLUMN_DTYPE[f.model]) for f, c in zip(features, columns)]
        f0 = features[0]
        n = cols[0].shape[0] if f0.model == NIW and cols[0].ndim == 2 else cols[0].size // (f0.dim if f0.model == NIW else 1)
        for f, c in zip(features, cols):
            assert c.size == n * (f.dim if f.model == NIW else 1), "columns of different lengths"
        fa = (c_p * F)(*[f.h for f in features])
        ca = (c_p * F)(*[c.ctypes.data for c in cols])
        prior = None if prior is None else np.ascontiguousarray(prior, dtype=np.float32)
        logp = logp_out if logp_out is not None else np.empty(n, dtype=np.float32)
        assert logp.dtype == np.float32 and logp.size == n and logp.flags.c_contiguous
        self.check(self.L.dist_b200_score_logp_batch_host(self.h, fa, F, ca, n, _np_ptr(prior), _np_ptr(logp)),
                   "score_logp_batch_host")
        return logp

    def host_register(self, array):
        """page-lock a numpy array in place (once): later host-entry calls on it are zero-copy"""
        assert array.flags.c_contiguous
        self.check(self.L.dist_b200_host_register(self.h, array.ctypes.data, array.nbytes), "host_register")
        return array

    def host_unregister(self, array):
        self.check(self.L.dist_b200_host_unregister(self.h, array.ctypes.data), "host_unregister")

    def score_value_host(self, feature, value, scores_accum):
        v = np.ascontiguousarray(value, dtype=COLUMN_DTYPE[feature.model])
        assert scores_accum.dtype == np.float32 and scores_accum.flags.c_contiguous
        self.check(self.L.dist_b200_score_value_host(self.h, feature.h, _np_ptr(v), _np_ptr(scores_accum)), "score_value_host")
        return scores_accum

    def pipe_peak(self, which):
        """lane-ops/s of the MUFU (0) or FP32-FMA (1) pipe (register-only kernels); 2: L2 gather bytes/s"""
        out = ctypes.c_double()
        self.check(self.L.dist_b200_pipe_peak(self.h, which, ctypes.byref(out)), "pipe_peak")
        return out.value

    def numerics_probe(self, fn, x_dev, out_dev, n, stream=None):
        self.check(self.L.dist_b200_numerics_probe(self.h, fn, n, _dev_ptr(x_dev), _dev_ptr(out_dev), stream), "numerics_probe")


class Feature:
    """Device-side MixtureValueScorer of one Model::Mixture."""

    def __init__(self, ctx, model):
        self.ctx = ctx
        self.model = model
        h = c_p()
        ctx.check(ctx.L.dist_b200_feature_create(ctx.h, model, ctypes.byref(h)), "feature_create")
        self.h = h
        self.dim = None  # niw: d of the last update_all (the row length of its columns)

    def close(self):
        if getattr(self, "h", None) and getattr(self.ctx, "h", None):
            self.ctx.L.dist_b200_feature_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def groups(self):
        return self.ctx.L.dist_b200_feature_groups(self.h)

    def update_all(self, w, stream=None):
        """w: a dict of group statistics in the layout of distributions_b200.synth workloads."""
        L, c = self.ctx.L, self.ctx
        f32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)  # noqa: E731
        i32 = lambda a: np.ascontiguousarray(a, dtype=np.int32)  # noqa: E731
        u32 = lambda a: np.ascontiguousarray(a, dtype=np.uint32)  # noqa: E731
        m = self.model
        if m == NICH:
            sh, cnt, mean, ctv = f32(w["shared"]), i32(w["count"]), f32(w["mean"]), f32(w["ctv"])
            c.check(L.dist_b200_nich_update_all(self.h, _np_ptr(sh), cnt.size, _np_ptr(cnt), _np_ptr(mean), _np_ptr(ctv), stream), "nich_update_all")
        elif m == GP:
            sh, cnt, sm = f32(w["shared"]), u32(w["count"]), u32(w["sum"])
            c.check(L.dist_b200_gp_update_all(self.h, _np_ptr(sh), cnt.size, _np_ptr(cnt), _np_ptr(sm), stream), "gp_update_all")
            if w.get("log_prod") is not None and cnt.size:
                self.set_log_prod(w["log_prod"], stream)
        elif m == BNB:
            sh, cnt, sm = f32(w["shared"][:2]), u32(w["count"]), u32(w["sum"])
            c.check(L.dist_b200_bnb_update_all(self.h, _np_ptr(sh), int(w["shared"][2]), cnt.size, _np_ptr(cnt), _np_ptr(sm), stream),
                    "bnb_update_all")
        elif m == BB:
            sh, h, t = f32(w["shared"]), i32(w["heads"]), i32(w["tails"])
            c.check(L.dist_b200_bb_update_all(self.h, _np_ptr(sh), h.size, _np_ptr(h), _np_ptr(t), stream), "bb_update_all")
        elif m == DD:
            al, cnt = f32(w["alphas"]), i32(w["counts"])
            c.check(L.dist_b200_dd_update_all(self.h, al.size, _np_ptr(al), cnt.shape[0], _np_ptr(cnt), stream), "dd_update_all")
        elif m == DPD:
            keys, betas, cnt = u32(w["keys"]), f32(w["betas"]), i32(w["counts"])
            c.check(L.dist_b200_dpd_update_all(self.h, w["alpha"], w["beta0"], keys.size, _np_ptr(keys), _np_ptr(betas),
                                               cnt.shape[0], _np_ptr(cnt), stream), "dpd_update_all")
        elif m == NIW:
            mu, psi, cnt, sx, sxx = f32(w["mu"]), f32(w["psi"]), i32(w["count"]), f32(w["sum_x"]), f32(w["sum_xxT"])
            self.dim = mu.size
            c.check(L.dist_b200_niw_update_all(self.h, mu.size, _np_ptr(mu), w["kappa"], _np_ptr(psi), w["nu"], cnt.size,
                                               _np_ptr(cnt), _np_ptr(sx), _np_ptr(sxx), stream), "niw_update_all")
        else:
            raise ValueError(m)
        return self

    def update_group(self, groupid, stats, stream=None):
        buf = np.ascontiguousarray(stats)
        self.ctx.check(self.ctx.L.dist_b200_feature_update_group(self.h, groupid, _np_ptr(buf), stream), "update_group")

    def add_group(self, stream=None):
        self.ctx.check(self.ctx.L.dist_b200_feature_add_group(self.h, stream), "add_group")

    def remove_group(self, groupid, stream=None):
        self.ctx.check(self.ctx.L.dist_b200_feature_remove_group(self.h, groupid, stream), "remove_group")

    def add_rows(self, column_dev, assign_dev, n_rows, stream=None):
        """batched Group::add_value: fold rows into their assigned groups on the device, rebuild the caches"""
        self.ctx.check(self.ctx.L.dist_b200_feature_add_rows(self.h, _dev_ptr(column_dev), _dev_ptr(assign_dev), n_rows, stream),
                       "add_rows")

    def set_log_prod(self, log_prod, stream=None):
        """gp only: Group::log_prod per group, read by score_data_grid"""
        lp = np.ascontiguousarray(log_prod, dtype=np.float32)
        self.ctx.check(self.ctx.L.dist_b200_gp_set_log_prod(self.h, _np_ptr(lp), stream), "gp_set_log_prod")
        return self

    def score_data_grid(self, shareds):
        """log marginal likelihood of all groups under each packed Shared (host arrays): [n_grid] float32"""
        sh = np.ascontiguousarray(np.atleast_2d(shareds), dtype=np.float32)
        out = np.empty(sh.shape[0], dtype=np.float32)
        self.ctx.check(self.ctx.L.dist_b200_score_data_grid_host(self.h, _np_ptr(sh), sh.shape[0], sh.shape[1], _np_ptr(out)),
                       "score_data_grid")
        return out

    def score_data_grid_dev(self, shareds_dev, n_grid, stride, out_dev, stream=None):
        self.ctx.check(self.ctx.L.dist_b200_score_data_grid(self.h, _dev_ptr(shareds_dev), n_grid, stride, _dev_ptr(out_dev), stream),
                       "score_data_grid")

    def update_all_wire(self, shared_msg, group_msgs, stream=None):
        """Shared + Groups as serialized protobuf messages (bytes) of the reference's schema"""
        G = len(group_msgs)
        bufs = [ctypes.create_string_buffer(m, len(m)) for m in group_msgs]
        ptrs = (c_p * max(G, 1))(*[ctypes.addressof(b) for b in bufs])
        lens = (c_sz * max(G, 1))(*[len(m) for m in group_msgs])
        self.ctx.check(self.ctx.L.dist_b200_update_all_wire(self.h, shared_msg, len(shared_msg), ptrs, lens, G, stream),
                       "update_all_wire")
        return self

    def update_all_stream(self, shared_msg, stream_bytes, stream=None):
        """Groups as one [uint32 length][message] record stream (distributions.io.stream.protobuf_stream_dump)"""
        self.ctx.check(self.ctx.L.dist_b200_update_all_stream(self.h, shared_msg, len(shared_msg), stream_bytes, len(stream_bytes), stream),
                       "update_all_stream")
        return self

    def dump_groups_wire(self, stream=None):
        """the current device-resident statistics as serialized Group messages (list of bytes)"""
        G = self.groups
        n = c_sz()
        lens = (c_sz * max(G, 1))()
        L = self.ctx.L
        rc = L.dist_b200_feature_dump_groups_wire(self.h, None, 0, lens, ctypes.byref(n), stream)
        if rc not in (0, 1):
            self.ctx.check(rc, "dump_groups_wire")
        buf = np.empty(n.value, np.uint8)
        self.ctx.check(L.dist_b200_feature_dump_groups_wire(self.h, _np_ptr(buf), buf.size, lens, ctypes.byref(n), stream), "dump_groups_wire")
        return _split(buf, [lens[i] for i in range(G)])

    def download_stats(self, nbytes, stream=None):
        out = np.empty(nbytes, dtype=np.uint8)
        n = c_sz()
        self.ctx.check(self.ctx.L.dist_b200_feature_download_stats(self.h, _np_ptr(out), out.size, ctypes.byref(n), stream),
                       "download_stats")
        return out[:n.value]

    def download_caches(self, rows, stream=None):
        G = self.groups
        out = np.empty((rows, G), dtype=np.float32)
        n = c_sz()
        self.ctx.check(self.ctx.L.dist_b200_feature_download_caches(self.h, _np_ptr(out), out.size, ctypes.byref(n), stream), "download_caches")
        assert n.value == out.size, (n.value, out.size)
        return out
