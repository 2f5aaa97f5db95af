"""ctypes binding of libb200gbm.so — the Python stand-in for the SWIG `lightgbmlib` class the reference's
Scala code calls (SURVEY.md §8b).  Thin: every method is one C-ABI call plus marshalling, and failures
raise with LGBM_GetLastError() exactly like LightGBMUtils.validate
(lightgbm/src/main/scala/com/microsoft/ml/spark/lightgbm/LightGBMUtils.scala:22-34).

The extension must exist: there is no Python / CPU fallback for any compute entry.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libb200gbm.so")
_LIB = None

DTYPE_FLOAT32, DTYPE_FLOAT64, DTYPE_INT32, DTYPE_INT64 = 0, 1, 2, 3
PREDICT_NORMAL, PREDICT_RAW_SCORE, PREDICT_LEAF_INDEX, PREDICT_CONTRIB = 0, 1, 2, 3


class LightGBMError(Exception):
    pass


def load():
    """Load the C-ABI library (building it is __graft_entry__.build()'s job). Fails loudly if missing."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise LightGBMError(
                "libb200gbm.so is missing (%s). Run `python __graft_entry__.py` to build the CUDA extension; "
                "this package has no CPU fallback." % LIB_PATH)
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        L.LGBM_GetLastError.restype = C.c_char_p
        for name in ("B200GBM_ChunkedArrayGetAddCount", "B200GBM_ChunkedArrayGetChunksCount", "B200GBM_ChunkedArrayGetLastChunkAddCount"):
            getattr(L, name).restype = C.c_int64
            getattr(L, name).argtypes = [C.c_void_p]
        L.B200GBM_ChunkedArrayGetItem.restype = C.c_double
        L.B200GBM_ChunkedArrayGetItem.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_double]
        L.B200GBM_ChunkedArrayAdd.argtypes = [C.c_void_p, C.c_double]
        L.B200GBM_ChunkedArrayAddMany.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.B200GBM_ChunkedArrayCreate.argtypes = [C.c_int, C.c_int64, C.c_void_p]
        L.B200GBM_ChunkedArrayCoalesceTo.argtypes = [C.c_void_p, C.c_void_p]
        for name in ("B200GBM_ChunkedArrayRelease", "B200GBM_ChunkedArrayFree"):
            getattr(L, name).argtypes = [C.c_void_p]
        _LIB = L
    return _LIB


def check(rc):
    if rc != 0:
        raise LightGBMError(load().LGBM_GetLastError().decode())


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _np_dtype_code(a):
    if a.dtype == np.float32:
        return DTYPE_FLOAT32
    if a.dtype == np.float64:
        return DTYPE_FLOAT64
    raise LightGBMError("expected float32/float64 data")


def network_init(machines, local_listen_port, listen_time_out=120, num_machines=1):
    check(load().LGBM_NetworkInit(machines.encode(), C.c_int(local_listen_port), C.c_int(listen_time_out), C.c_int(num_machines)))


def network_free():
    check(load().LGBM_NetworkFree())


def set_device(ordinal):
    check(load().B200GBM_SetDevice(C.c_int(ordinal)))


def sample_indices(n, k, seed=1):
    out = np.zeros(max(min(n, k), 1), dtype=np.int32)
    m = C.c_int(0)
    check(load().B200GBM_SampleIndices(C.c_int(n), C.c_int(k), C.c_int(seed), _ptr(out), C.byref(m)))
    return out[:m.value].copy()


class DeviceBuffer:
    """Raw device allocation on the calling thread's GPU (plumbing for the benchmark's device-resident input)."""

    def __init__(self, nbytes):
        self.ptr = C.c_void_p()
        self.nbytes = nbytes
        check(load().B200GBM_DeviceAlloc(C.c_size_t(nbytes), C.byref(self.ptr)))

    def free(self):
        if self.ptr:
            check(load().B200GBM_DeviceFree(self.ptr))
            self.ptr = C.c_void_p()


class PinnedBuffer:
    def __init__(self, nbytes):
        self.ptr = C.c_void_p()
        self.nbytes = nbytes
        check(load().B200GBM_HostAllocPinned(C.c_size_t(nbytes), C.byref(self.ptr)))

    def as_array(self, dtype, shape):
        n = int(np.prod(shape))
        buf = (C.c_char * (n * np.dtype(dtype).itemsize)).from_address(self.ptr.value)
        return np.frombuffer(buf, dtype=dtype).reshape(shape)

    def free(self):
        if self.ptr:
            check(load().B200GBM_HostFreePinned(self.ptr))
            self.ptr = C.c_void_p()


def _vp(p):
    return p if isinstance(p, C.c_void_p) else C.c_void_p(int(p))


def memcpy(dst_ptr, src_ptr, nbytes):
    check(load().B200GBM_Memcpy(_vp(dst_ptr), _vp(src_ptr), C.c_size_t(nbytes)))


def synthetic_fill(dev_x, dev_label, row_start, nrow, ncol, seed, kind):
    check(load().B200GBM_SyntheticFill(_vp(dev_x), _vp(dev_label) if dev_label is not None else None, C.c_int64(row_start), C.c_int32(nrow), C.c_int32(ncol), C.c_uint64(seed), C.c_int(kind)))


def synthetic_rows(rows, ncol, seed, kind):
    rows = np.ascontiguousarray(rows, dtype=np.int32)
    out = np.zeros((len(rows), ncol), dtype=np.float64)
    lab = np.zeros(len(rows), dtype=np.float32)
    check(load().B200GBM_SyntheticRows(_ptr(rows), C.c_int32(len(rows)), C.c_int32(ncol), C.c_uint64(seed), C.c_int(kind), _ptr(out), _ptr(lab)))
    return out, lab


class Dataset:
    """Mirror of LightGBMDataset (lightgbm/src/main/scala/.../dataset/LightGBMDataset.scala)."""

    def __init__(self, handle, keep=None):
        self.handle = handle
        self._keep = keep

    @classmethod
    def from_mat(cls, X, params="", reference=None, row_major=True):
        X = np.asarray(X)
        if X.dtype not in (np.float32, np.float64):
            X = X.astype(np.float64)
        X = np.ascontiguousarray(X) if row_major else np.asfortranarray(X)
        n, F = X.shape
        h = C.c_void_p()
        check(load().LGBM_DatasetCreateFromMat(_ptr(X), C.c_int(_np_dtype_code(X)), C.c_int32(n), C.c_int32(F), C.c_int(1 if row_major else 0),
                                               params.encode(), reference.handle if reference is not None else None, C.byref(h)))
        return cls(h)

    @classmethod
    def from_device_ptr(cls, ptr, dtype_code, n, F, params="", reference=None):
        h = C.c_void_p()
        check(load().LGBM_DatasetCreateFromMat(_vp(ptr), C.c_int(dtype_code), C.c_int32(n), C.c_int32(F), C.c_int(1), params.encode(),
                                               reference.handle if reference is not None else None, C.byref(h)))
        return cls(h)

    @classmethod
    def from_csr(cls, indptr, indices, data, num_col, params="", reference=None):
        indptr = np.ascontiguousarray(indptr, dtype=np.int32)
        indices = np.ascontiguousarray(indices, dtype=np.int32)
        data = np.ascontiguousarray(data, dtype=np.float64)
        h = C.c_void_p()
        check(load().LGBM_DatasetCreateFromCSR(_ptr(indptr), C.c_int(DTYPE_INT32), _ptr(indices), _ptr(data), C.c_int(DTYPE_FLOAT64),
                                               C.c_int64(len(indptr)), C.c_int64(len(data)), C.c_int64(num_col), params.encode(),
                                               reference.handle if reference is not None else None, C.byref(h)))
        return cls(h)

    @classmethod
    def from_sampled_columns(cls, sample, num_total_row, params=""):
        """sample: [num_sample_row][ncol] float64 (dense sample of rows); zeros are dropped per column as LightGBM expects."""
        sample = np.ascontiguousarray(sample, dtype=np.float64)
        ns, F = sample.shape
        cols, idxs, cnts = [], [], np.zeros(F, dtype=np.int32)
        for f in range(F):
            v = sample[:, f]
            m = (np.abs(v) > 1e-35) | np.isnan(v)
            cols.append(np.ascontiguousarray(v[m]))
            idxs.append(np.ascontiguousarray(np.nonzero(m)[0].astype(np.int32)))
            cnts[f] = int(m.sum())
        pd = (C.POINTER(C.c_double) * F)(*[c.ctypes.data_as(C.POINTER(C.c_double)) for c in cols])
        pi = (C.POINTER(C.c_int) * F)(*[c.ctypes.data_as(C.POINTER(C.c_int)) for c in idxs])
        h = C.c_void_p()
        check(load().LGBM_DatasetCreateFromSampledColumn(pd, pi, C.c_int32(F), _ptr(cnts), C.c_int32(ns), C.c_int32(num_total_row), params.encode(), C.byref(h)))
        return cls(h)

    def push_rows(self, data, start_row, nrow=None, ncol=None, dtype_code=None):
        if isinstance(data, np.ndarray):
            data = np.ascontiguousarray(data)
            nrow, ncol = data.shape
            check(load().LGBM_DatasetPushRows(self.handle, _ptr(data), C.c_int(_np_dtype_code(data)), C.c_int32(nrow), C.c_int32(ncol), C.c_int32(start_row)))
        else:
            check(load().LGBM_DatasetPushRows(self.handle, _vp(data), C.c_int(dtype_code), C.c_int32(nrow), C.c_int32(ncol), C.c_int32(start_row)))

    def set_field(self, name, arr):
        if name in ("label", "weight"):
            a = np.ascontiguousarray(arr, dtype=np.float32); t = DTYPE_FLOAT32
        elif name == "init_score":
            a = np.ascontiguousarray(arr, dtype=np.float64); t = DTYPE_FLOAT64
        elif name == "group":
            a = np.ascontiguousarray(arr, dtype=np.int32); t = DTYPE_INT32
        else:
            raise LightGBMError("Unknown field name: " + name)
        check(load().LGBM_DatasetSetField(self.handle, name.encode(), _ptr(a), C.c_int(len(a)), C.c_int(t)))
        return self

    def get_field(self, name):
        n = C.c_int(0); p = C.c_void_p(); t = C.c_int(0)
        check(load().LGBM_DatasetGetField(self.handle, name.encode(), C.byref(n), C.byref(p), C.byref(t)))
        dt = {0: np.float32, 1: np.float64, 2: np.int32}[t.value]
        buf = (C.c_char * (n.value * np.dtype(dt).itemsize)).from_address(p.value)
        return np.frombuffer(buf, dtype=dt).copy()

    def set_feature_names(self, names):
        arr = (C.c_char_p * len(names))(*[s.encode() for s in names])
        check(load().LGBM_DatasetSetFeatureNames(self.handle, arr, C.c_int(len(names))))

    def num_data(self):
        v = C.c_int(0); check(load().LGBM_DatasetGetNumData(self.handle, C.byref(v))); return v.value

    def num_feature(self):
        v = C.c_int(0); check(load().LGBM_DatasetGetNumFeature(self.handle, C.byref(v))); return v.value

    # --- engine extensions
    def get_bins(self):
        out = np.zeros((self.num_data(), self.num_feature()), dtype=np.uint8)
        check(load().B200GBM_DatasetGetBins(self.handle, _ptr(out)))
        return out

    def get_bins16(self):
        out = np.zeros((self.num_data(), self.num_feature()), dtype=np.uint16)
        check(load().B200GBM_DatasetGetBins16(self.handle, _ptr(out)))
        return out

    def bin_to_cat(self, f):
        out = np.zeros(65536, dtype=np.int32); k = C.c_int(0)
        check(load().B200GBM_DatasetGetBinToCat(self.handle, C.c_int(f), _ptr(out), C.byref(k)))
        return out[:k.value].copy()

    def get_bins_rows(self, rows):
        """bins of the selected rows only (device gather): [len(rows)][num_feature] uint16"""
        rows = np.ascontiguousarray(rows, dtype=np.int32)
        out = np.zeros((len(rows), self.num_feature()), dtype=np.uint16)
        check(load().B200GBM_DatasetGetBinsRows(self.handle, _ptr(rows), C.c_int32(len(rows)), _ptr(out)))
        return out

    def feature_range(self, f):
        out = np.zeros(2, dtype=np.float64)
        check(load().B200GBM_DatasetGetFeatureRange(self.handle, C.c_int(f), _ptr(out)))
        return float(out[0]), float(out[1])

    def feature_info(self, f):
        info = np.zeros(5, dtype=np.int32)
        check(load().B200GBM_DatasetGetFeatureInfo(self.handle, C.c_int(f), _ptr(info)))
        return dict(num_bin=int(info[0]), missing_type=int(info[1]), default_bin=int(info[2]), most_freq_bin=int(info[3]), is_trivial=bool(info[4]))

    def upper_bounds(self, f):
        out = np.zeros(32768, dtype=np.float64); k = C.c_int(0)
        check(load().B200GBM_DatasetGetUpperBounds(self.handle, C.c_int(f), _ptr(out), C.byref(k)))
        return out[:k.value].copy()

    def ingest_ms(self):
        v = C.c_double(0); check(load().B200GBM_DatasetGetIngestMs(self.handle, C.byref(v))); return v.value

    def histogram(self, grad, hess, idx=None):
        g = np.ascontiguousarray(grad, dtype=np.float32); h = np.ascontiguousarray(hess, dtype=np.float32)
        cnt = self.num_data()
        ip = None
        if idx is not None:
            idx = np.ascontiguousarray(idx, dtype=np.int32); cnt = len(idx); ip = _ptr(idx)
        out = np.zeros((self.num_feature(), 256, 2), dtype=np.float64)
        check(load().B200GBM_DatasetHistogram(self.handle, _ptr(g), _ptr(h), ip, C.c_int32(cnt), _ptr(out)))
        return out

    def free(self):
        if self.handle:
            check(load().LGBM_DatasetFree(self.handle))
            self.handle = None


class Booster:
    """Mirror of LightGBMBooster (lightgbm/src/main/scala/.../booster/LightGBMBooster.scala)."""

    def __init__(self, train_set=None, params="", model_str=None):
        self.handle = C.c_void_p()
        self.train_set = train_set
        if model_str is not None:
            it = C.c_int(0)
            check(load().LGBM_BoosterLoadModelFromString(model_str.encode(), C.byref(it), C.byref(self.handle)))
        else:
            check(load().LGBM_BoosterCreate(train_set.handle, params.encode(), C.byref(self.handle)))

    def update_one_iter(self):
        fin = C.c_int(0)
        check(load().LGBM_BoosterUpdateOneIter(self.handle, C.byref(fin)))
        return fin.value == 1

    def update_one_iter_custom(self, grad, hess):
        g = np.ascontiguousarray(grad, dtype=np.float32); h = np.ascontiguousarray(hess, dtype=np.float32)
        fin = C.c_int(0)
        check(load().LGBM_BoosterUpdateOneIterCustom(self.handle, _ptr(g), _ptr(h), C.byref(fin)))
        return fin.value == 1

    def reset_parameter(self, params):
        check(load().LGBM_BoosterResetParameter(self.handle, params.encode()))

    def add_valid(self, ds):
        check(load().LGBM_BoosterAddValidData(self.handle, ds.handle))

    def merge(self, other):
        check(load().LGBM_BoosterMerge(self.handle, other.handle))

    def eval_names(self):
        n = C.c_int(0)
        check(load().LGBM_BoosterGetEvalCounts(self.handle, C.byref(n)))
        bufs = [C.create_string_buffer(128) for _ in range(n.value)]
        arr = (C.c_char_p * max(n.value, 1))(*[C.cast(b, C.c_char_p) for b in bufs])
        out_n = C.c_int(0); need = C.c_size_t(0)
        check(load().LGBM_BoosterGetEvalNames(self.handle, C.c_int(n.value), C.byref(out_n), C.c_size_t(128), C.byref(need), arr))
        return [bufs[i].value.decode() for i in range(out_n.value)]

    def get_eval(self, data_idx):
        cnt = C.c_int(0)
        check(load().LGBM_BoosterGetEvalCounts(self.handle, C.byref(cnt)))
        out = np.zeros(max(cnt.value, 1), dtype=np.float64); n = C.c_int(0)
        check(load().LGBM_BoosterGetEval(self.handle, C.c_int(data_idx), C.byref(n), _ptr(out)))
        return out[:n.value].copy()

    def get_predict(self, data_idx):
        n = C.c_int64(0)
        check(load().LGBM_BoosterGetNumPredict(self.handle, C.c_int(data_idx), C.byref(n)))
        out = np.zeros(n.value, dtype=np.float64)
        check(load().LGBM_BoosterGetPredict(self.handle, C.c_int(data_idx), C.byref(n), _ptr(out)))
        return out

    def _int_getter(self, fn):
        v = C.c_int(0); check(getattr(load(), fn)(self.handle, C.byref(v))); return v.value

    def num_classes(self): return self._int_getter("LGBM_BoosterGetNumClasses")
    def num_model_per_iteration(self): return self._int_getter("LGBM_BoosterNumModelPerIteration")
    def num_total_model(self): return self._int_getter("LGBM_BoosterNumberOfTotalModel")
    def num_feature(self): return self._int_getter("LGBM_BoosterGetNumFeature")
    def current_iteration(self): return self._int_getter("LGBM_BoosterGetCurrentIteration")

    def feature_importance(self, importance_type="split", num_iteration=-1):
        out = np.zeros(self.num_feature(), dtype=np.float64)
        check(load().LGBM_BoosterFeatureImportance(self.handle, C.c_int(num_iteration), C.c_int(0 if importance_type == "split" else 1), _ptr(out)))
        return out

    def _string_call(self, fn, start_iteration, num_iteration, buffer_len):
        # same retry protocol as the SWIG helper: first try a small buffer, then the reported length
        buf = C.create_string_buffer(buffer_len); n = C.c_int64(0)
        check(getattr(load(), fn)(self.handle, C.c_int(start_iteration), C.c_int(num_iteration), C.c_int(0), C.c_int64(buffer_len), C.byref(n), buf))
        if n.value > buffer_len:
            buf = C.create_string_buffer(n.value)
            check(getattr(load(), fn)(self.handle, C.c_int(start_iteration), C.c_int(num_iteration), C.c_int(0), C.c_int64(n.value), C.byref(n), buf))
        return buf.value.decode()

    def save_model_to_string(self, start_iteration=0, num_iteration=-1, buffer_len=10000):
        return self._string_call("LGBM_BoosterSaveModelToString", start_iteration, num_iteration, buffer_len)

    def dump_model(self, start_iteration=0, num_iteration=-1):
        return self._string_call("LGBM_BoosterDumpModel", start_iteration, num_iteration, 10000)

    def predict_for_mat_single(self, row, predict_type=PREDICT_NORMAL, start_iteration=0, num_iteration=-1):
        row = np.ascontiguousarray(row, dtype=np.float64)
        n = C.c_int64(0)
        check(load().LGBM_BoosterCalcNumPredict(self.handle, C.c_int(1), C.c_int(predict_type), C.c_int(start_iteration), C.c_int(num_iteration), C.byref(n)))
        out = np.zeros(max(n.value, 1), dtype=np.float64)
        check(load().LGBM_BoosterPredictForMatSingle(self.handle, _ptr(row), C.c_int(DTYPE_FLOAT64), C.c_int(len(row)), C.c_int(1), C.c_int(predict_type),
                                                     C.c_int(start_iteration), C.c_int(num_iteration), b"max_bin=255", C.byref(n), _ptr(out)))
        return out[:n.value].copy()

    def predict_for_csr_single(self, indices, values, num_col, predict_type=PREDICT_NORMAL, start_iteration=0, num_iteration=-1):
        indices = np.ascontiguousarray(indices, dtype=np.int32); values = np.ascontiguousarray(values, dtype=np.float64)
        indptr = np.array([0, len(values)], dtype=np.int32)
        n = C.c_int64(0)
        check(load().LGBM_BoosterCalcNumPredict(self.handle, C.c_int(1), C.c_int(predict_type), C.c_int(start_iteration), C.c_int(num_iteration), C.byref(n)))
        out = np.zeros(max(n.value, 1), dtype=np.float64)
        check(load().LGBM_BoosterPredictForCSRSingle(self.handle, _ptr(indptr), C.c_int(DTYPE_INT32), _ptr(indices), _ptr(values), C.c_int(DTYPE_FLOAT64),
                                                     C.c_int64(2), C.c_int64(len(values)), C.c_int64(num_col), C.c_int(predict_type), C.c_int(start_iteration),
                                                     C.c_int(num_iteration), b"max_bin=255", C.byref(n), _ptr(out)))
        return out[:n.value].copy()

    def predict_for_mat(self, X, predict_type=PREDICT_NORMAL, start_iteration=0, num_iteration=-1):
        X = np.ascontiguousarray(X, dtype=np.float64)
        nrow, ncol = X.shape
        n = C.c_int64(0)
        check(load().LGBM_BoosterCalcNumPredict(self.handle, C.c_int(nrow), C.c_int(predict_type), C.c_int(start_iteration), C.c_int(num_iteration), C.byref(n)))
        out = np.zeros(max(n.value, 1), dtype=np.float64)
        check(load().LGBM_BoosterPredictForMat(self.handle, _ptr(X), C.c_int(DTYPE_FLOAT64), C.c_int32(nrow), C.c_int32(ncol), C.c_int(1), C.c_int(predict_type),
                                               C.c_int(start_iteration), C.c_int(num_iteration), b"", C.byref(n), _ptr(out)))
        return out[:n.value].reshape(nrow, -1)

    # --- engine extensions
    def predict_device(self, X, predict_type=PREDICT_NORMAL, start_iteration=0, num_iteration=-1, return_ms=False):
        """Batched GPU prediction (B200GBM_BoosterPredictForMatDevice); X: float32/float64 [nrow, ncol] host array."""
        X = np.ascontiguousarray(X)
        if X.dtype not in (np.float32, np.float64):
            X = X.astype(np.float64)
        nrow, ncol = X.shape
        n = C.c_int64(0)
        check(load().LGBM_BoosterCalcNumPredict(self.handle, C.c_int(nrow), C.c_int(predict_type), C.c_int(start_iteration), C.c_int(num_iteration), C.byref(n)))
        out = np.zeros(max(n.value, 1), dtype=np.float64)
        ms = C.c_double(0)
        check(load().B200GBM_BoosterPredictForMatDevice(self.handle, _ptr(X), C.c_int(_np_dtype_code(X)), C.c_int64(nrow), C.c_int32(ncol), C.c_int(predict_type),
                                                        C.c_int(start_iteration), C.c_int(num_iteration), C.byref(n), _ptr(out), C.byref(ms)))
        res = out[:n.value].reshape(nrow, -1)
        return (res, ms.value) if return_ms else res

    def set_profile(self, on=True):
        check(load().B200GBM_BoosterSetProfile(self.handle, C.c_int(1 if on else 0)))

    def get_timing(self, reset=False):
        out = np.zeros(6, dtype=np.float64)
        check(load().B200GBM_BoosterGetTiming(self.handle, _ptr(out), C.c_int(1 if reset else 0)))
        return dict(hist_ms=out[0], total_ms=out[1], hist_rows=int(out[2]), hist_launches=int(out[3]), launches=int(out[4]), iterations=int(out[5]))

    def get_info(self):
        out = np.zeros(4, dtype=np.int32)
        check(load().B200GBM_BoosterGetInfo(self.handle, _ptr(out)))
        return dict(num_machines=int(out[0]), rank=int(out[1]), fused_peer_reduce=int(out[2]) == 1, reduce_mode=int(out[2]), constant_hessian=bool(out[3]))

    def get_memory_info(self):
        out = np.zeros(2, dtype=np.int64)
        check(load().B200GBM_BoosterGetMemoryInfo(self.handle, _ptr(out)))
        return dict(partition_column_copy_bytes=int(out[0]), device_free_bytes=int(out[1]))

    def get_scores(self, data_idx=0):
        n = C.c_int64(0)
        check(load().LGBM_BoosterGetNumPredict(self.handle, C.c_int(data_idx), C.byref(n)))
        out = np.zeros(n.value, dtype=np.float64)
        check(load().B200GBM_BoosterGetScores(self.handle, C.c_int(data_idx), _ptr(out)))
        return out

    def get_gradients(self):
        """For tests: (grad, hess), float32 arrays of K * num_data (class-major), the objective's gradients at the current training
        scores, which before the first iteration are the training set's init_score.  Classes the objective does not train read 0.
        Training is not affected: the model and the scores stay as they are."""
        n = C.c_int64(0)
        check(load().LGBM_BoosterGetNumPredict(self.handle, C.c_int(0), C.byref(n)))
        g = np.zeros(n.value, dtype=np.float32)
        h = np.zeros(n.value, dtype=np.float32)
        check(load().B200GBM_BoosterGetGradients(self.handle, _ptr(g), _ptr(h)))
        return g, h

    def free(self):
        if self.handle:
            check(load().LGBM_BoosterFree(self.handle))
            self.handle = None


class ChunkedArray:
    """Mirror of the SWIG floatChunkedArray/doubleChunkedArray/int32ChunkedArray
    (lightgbm/src/main/scala/.../swig/SwigUtils.scala:22-90)."""

    def __init__(self, dtype_code, chunk_size):
        self.h = C.c_void_p()
        self.dtype_code = dtype_code
        check(load().B200GBM_ChunkedArrayCreate(C.c_int(dtype_code), C.c_int64(chunk_size), C.byref(self.h)))

    def add(self, v): check(load().B200GBM_ChunkedArrayAdd(self.h, C.c_double(v)))

    def add_many(self, arr):
        dt = {0: np.float32, 1: np.float64, 2: np.int32}[self.dtype_code]
        a = np.ascontiguousarray(arr, dtype=dt)
        check(load().B200GBM_ChunkedArrayAddMany(self.h, _ptr(a), C.c_int64(len(a))))

    def get_add_count(self): return load().B200GBM_ChunkedArrayGetAddCount(self.h)
    def get_chunks_count(self): return load().B200GBM_ChunkedArrayGetChunksCount(self.h)
    def get_last_chunk_add_count(self): return load().B200GBM_ChunkedArrayGetLastChunkAddCount(self.h)
    def getitem(self, chunk, idx, default): return load().B200GBM_ChunkedArrayGetItem(self.h, chunk, idx, default)

    def coalesce(self):
        dt = {0: np.float32, 1: np.float64, 2: np.int32}[self.dtype_code]
        out = np.zeros(self.get_add_count(), dtype=dt)
        check(load().B200GBM_ChunkedArrayCoalesceTo(self.h, _ptr(out)))
        return out

    def release(self): check(load().B200GBM_ChunkedArrayRelease(self.h))

    def free(self):
        if self.h:
            check(load().B200GBM_ChunkedArrayFree(self.h)); self.h = None
