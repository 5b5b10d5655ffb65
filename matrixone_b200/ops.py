"""Reference-facing operator calls over the C-ABI (what the Go side would do through cgo, written in Python).

Each function only marshals arguments into mo_xcall_args_t blocks (Vector.FillRawPtrLen layout) and calls XCall /
the mo.h entry points of libmo_b200.so.  Inputs may be numpy arrays (host path: the library stages them) or
DeviceBuffer objects (resident path).  Names follow the reference:

  q6_filter_sum / q1_group_agg     the fused TableScan->Filter->Projection->Group pipelines of TPC-H Q6 / Q1
  agg_sum / agg_count / agg_min / agg_max / agg_avg      aggexec sumAvgExec / countColumnExec / minMaxExecFixed (H0)
  BruteForceIndex                  brute_force.NewBruteForceIndex / .Search / .Destroy (brute_force.go:65-84,248-341)
  IvfflatSearchIndex               ivfflat.IvfflatSearchIndex.Search (ivfflat/search.go:509-630)
  topk_merge                       MergeTop / hnsw sub-index merge
"""
import ctypes as C

import numpy as np

from . import capi
from .vector import DeviceBuffer, Vector, xcall


def _vec(x, length=None, itemsize=None):
    """numpy array / DeviceBuffer / (DeviceBuffer, nbytes) -> Vector"""
    if isinstance(x, Vector):
        return x
    if isinstance(x, DeviceBuffer):
        return Vector(data_ptr=x.ptr, data_nbytes=x.nbytes, length=length)
    a = np.ascontiguousarray(x)
    return Vector(data=a, length=length if length is not None else a.shape[0])


def _params_vec(struct):
    buf = np.frombuffer(bytes(struct), dtype=np.uint8).copy()
    return Vector(data=buf, length=1, const=True)


# ------------------------------------------------------------------------------------------------ aggregates
def _agg(op, T, col, nulls=None, length=None):
    n = length if length is not None else (col.nbytes // np.dtype(capi.NP_OF_T[T]).itemsize if isinstance(col, DeviceBuffer) else len(col))
    res = np.zeros(1, dtype=np.uint64)
    rn = np.zeros(1, dtype=np.uint64)
    rv = Vector(data=res, nulls=rn, length=1)
    cv = _vec(col, n)
    if nulls is not None:
        if isinstance(nulls, DeviceBuffer):
            cv.nulls_ptr = nulls.ptr
        else:
            cv.nulls = np.ascontiguousarray(nulls, dtype=np.uint64)
    cv.length = n
    rc, msg = xcall(capi.XCALL_AGG(op, T), [rv, cv], n, raise_on_error=False)
    if rc not in (0, capi.RC_OUT_OF_RANGE):
        raise capi.MoError(rc, msg)
    return rc, res, bool(rv.nulls[0] & np.uint64(1))


def agg_sum(T, col, nulls=None, length=None):
    """SUM(col): returns (rc, value, is_null); value int64 / uint64 / float64 per SumReturnType (sumavg2.go:69-87)."""
    rc, res, isnull = _agg(capi.AGG_SUM, T, col, nulls, length)
    if T in (capi.T_FLOAT32, capi.T_FLOAT64):
        v = res.view(np.float64)[0]
    elif capi.T_UINT8 <= T <= capi.T_UINT64:
        v = int(res[0])
    else:
        v = int(res.view(np.int64)[0])
    return rc, v, isnull


def agg_avg(T, col, nulls=None, length=None):
    rc, res, isnull = _agg(capi.AGG_AVG, T, col, nulls, length)
    return rc, float(res.view(np.float64)[0]), isnull


def agg_count(T, col, nulls=None, length=None):
    rc, res, _ = _agg(capi.AGG_COUNT, T, col, nulls, length)
    return int(res.view(np.int64)[0])


def _minmax(op, T, col, nulls, length):
    rc, res, isnull = _agg(op, T, col, nulls, length)
    dt = np.dtype(capi.NP_OF_T[T])
    return res.view(np.uint8)[:dt.itemsize].view(dt)[0], isnull


def agg_min(T, col, nulls=None, length=None):
    return _minmax(capi.AGG_MIN, T, col, nulls, length)


def agg_max(T, col, nulls=None, length=None):
    return _minmax(capi.AGG_MAX, T, col, nulls, length)


# ------------------------------------------------------------------------------------------------ TPC-H shapes
def q6_filter_sum(shipdate, discount, quantity, extendedprice, n, date_lo, date_hi, disc_lo, disc_hi, qty_hi):
    """SUM(l_extendedprice*l_discount) WHERE ... (q6.sql).  Returns (sum, qualifying_rows, is_null)."""
    res = np.zeros(2, dtype=np.float64)
    rn = np.zeros(1, dtype=np.uint64)
    rv = Vector(data=res, nulls=rn, length=1)
    p = capi.Q6Params(date_lo, date_hi, disc_lo, disc_hi, qty_hi)
    xcall(capi.XCALL_Q6_FILTER_SUM, [rv, _vec(shipdate, n), _vec(discount, n), _vec(quantity, n), _vec(extendedprice, n), _params_vec(p)], n)
    return float(res[0]), int(res.view(np.int64)[1]), bool(rv.nulls[0] & np.uint64(1))


Q6_RESULT_BYTES = 16
Q1_RESULT_BYTES = C.sizeof(capi.Q1Result)


def q6_filter_sum_device(shipdate, discount, quantity, extendedprice, n, date_lo, date_hi, disc_lo, disc_hi, qty_hi, out_ptr, out_nulls_ptr=None):
    """asynchronous form: resident columns, result {f64 sum, i64 rows} written to caller-owned DEVICE memory at out_ptr, nothing is
    read back and the calling thread's stream is not synchronised (the partial Group of a multi-GPU scan)"""
    rv = Vector(data_ptr=out_ptr, data_nbytes=Q6_RESULT_BYTES, nulls_ptr=out_nulls_ptr, length=1)
    p = capi.Q6Params(date_lo, date_hi, disc_lo, disc_hi, qty_hi)
    xcall(capi.XCALL_Q6_FILTER_SUM, [rv, _vec(shipdate, n), _vec(discount, n), _vec(quantity, n), _vec(extendedprice, n), _params_vec(p)], n)


def q6_merge_device(parts_ptr, nparts, out_ptr, out_nulls_ptr=None):
    """MergeGroup on the device: nparts x {f64 sum, i64 rows} -> one, in order"""
    xcall(capi.XCALL_Q6_MERGE, [Vector(data_ptr=out_ptr, data_nbytes=Q6_RESULT_BYTES, nulls_ptr=out_nulls_ptr, length=1),
                                Vector(data_ptr=parts_ptr, data_nbytes=Q6_RESULT_BYTES * nparts, length=nparts)], nparts)


def q6_merge(parts):
    """host form of the same merge: parts = [(sum, rows), ...] -> (sum, rows, is_null)"""
    buf = np.zeros(2 * len(parts), dtype=np.float64)
    for i, (s_, c_) in enumerate(parts):
        buf[2 * i] = s_
        buf.view(np.int64)[2 * i + 1] = c_
    res = np.zeros(2, dtype=np.float64)
    rn = np.zeros(1, dtype=np.uint64)
    xcall(capi.XCALL_Q6_MERGE, [Vector(data=res, nulls=rn, length=1), Vector(data=buf, length=len(parts))], len(parts))
    return float(res[0]), int(res.view(np.int64)[1]), bool(rn[0] & np.uint64(1))


def _q1_groups(r):
    out = []
    for g in range(r.ngroups):
        s = r.groups[g]
        out.append({k: getattr(s, k) for k in ("returnflag", "linestatus", "first_row", "sum_qty", "sum_base_price", "sum_disc_price",
                                               "sum_charge", "avg_qty", "avg_price", "avg_disc", "sum_disc", "count_order")})
    return out


def q1_result_from_bytes(raw):
    """mo_q1_result_t bytes -> list of group dicts (ngroups = -1: too many distinct keys)"""
    r = capi.Q1Result.from_buffer_copy(bytes(raw))
    if r.ngroups < 0:
        raise capi.MoError(capi.RC_INVALID_ARGUMENT, "q1: more than %d distinct group keys" % capi.Q1_MAX_GROUPS)
    return _q1_groups(r)


def q1_group_agg_device(shipdate, quantity, extendedprice, discount, tax, returnflag, linestatus, n, cutoff, out_ptr, row_base=0):
    """asynchronous form of q1_group_agg: mo_q1_result_t written to DEVICE memory at out_ptr; first_row values are offset by row_base"""
    rv = Vector(data_ptr=out_ptr, data_nbytes=Q1_RESULT_BYTES, length=1)
    xcall(capi.XCALL_Q1_GROUP_AGG, [rv, _vec(shipdate, n), _vec(quantity, n), _vec(extendedprice, n), _vec(discount, n), _vec(tax, n),
                                     _vec(returnflag, n), _vec(linestatus, n), _params_vec(capi.Q1Params(cutoff, 0, row_base))], n)


def q1_merge_device(parts_ptr, nparts, out_ptr):
    xcall(capi.XCALL_Q1_MERGE, [Vector(data_ptr=out_ptr, data_nbytes=Q1_RESULT_BYTES, length=1),
                                Vector(data_ptr=parts_ptr, data_nbytes=Q1_RESULT_BYTES * nparts, length=nparts)], nparts)


def q1_merge(parts_bytes, nparts):
    """host form: nparts concatenated mo_q1_result_t -> merged list of group dicts"""
    buf = np.frombuffer(bytes(parts_bytes), dtype=np.uint8).copy()
    res = np.zeros(Q1_RESULT_BYTES, dtype=np.uint8)
    xcall(capi.XCALL_Q1_MERGE, [Vector(data=res, length=1), Vector(data=buf, length=nparts)], nparts)
    return q1_result_from_bytes(res.tobytes())


def agg_state_device(op, T, col, nulls, n, out_ptr, out_nulls_ptr=None):
    """asynchronous MO_XCALL_AGG: mo_agg_state_t (24 bytes) written to DEVICE memory"""
    cv = _vec(col, n)
    if nulls is not None:
        cv.nulls_ptr = nulls.ptr
    cv.length = n
    xcall(capi.XCALL_AGG(op, T), [Vector(data_ptr=out_ptr, data_nbytes=capi.AGG_STATE_BYTES, nulls_ptr=out_nulls_ptr, length=1), cv], n)


def agg_merge_device(op, T, parts_ptr, nparts, out_ptr, out_bytes=capi.AGG_STATE_BYTES, out_nulls_ptr=None):
    xcall(capi.XCALL_AGG_MERGE(op, T), [Vector(data_ptr=out_ptr, data_nbytes=out_bytes, nulls_ptr=out_nulls_ptr, length=1),
                                        Vector(data_ptr=parts_ptr, data_nbytes=capi.AGG_STATE_BYTES * nparts, length=nparts)], nparts)


def agg_state(op, T, col, nulls=None, length=None):
    """synchronous partial state (bits, count, rc) of one column"""
    n = length if length is not None else (col.nbytes // np.dtype(capi.NP_OF_T[T]).itemsize if isinstance(col, DeviceBuffer) else len(col))
    res = np.zeros(3, dtype=np.uint64)
    rn = np.zeros(1, dtype=np.uint64)
    cv = _vec(col, n)
    if nulls is not None:
        if isinstance(nulls, DeviceBuffer):
            cv.nulls_ptr = nulls.ptr
        else:
            cv.nulls = np.ascontiguousarray(nulls, dtype=np.uint64)
    cv.length = n
    rc, msg = xcall(capi.XCALL_AGG(op, T), [Vector(data=res, nulls=rn, length=1), cv], n, raise_on_error=False)
    if rc not in (0, capi.RC_OUT_OF_RANGE):
        raise capi.MoError(rc, msg)
    return res


def agg_merge(op, T, states, final=True):
    """MergeGroup of partial states (array [n, 3] uint64).  final=True: (rc, value bits as uint64, count, is_null); else the merged state"""
    st = np.ascontiguousarray(states, dtype=np.uint64).reshape(-1, 3)
    res = np.zeros(3 if not final else 2, dtype=np.uint64)
    rn = np.zeros(1, dtype=np.uint64)
    rc, msg = xcall(capi.XCALL_AGG_MERGE(op, T), [Vector(data=res, nulls=rn, length=1), Vector(data=st.reshape(-1), length=st.shape[0])], st.shape[0],
                    raise_on_error=False)
    if rc not in (0, capi.RC_OUT_OF_RANGE):
        raise capi.MoError(rc, msg)
    if not final:
        return res
    return rc, res[0], int(res[1]), bool(rn[0] & np.uint64(1))


def q1_group_agg(shipdate, quantity, extendedprice, discount, tax, returnflag, linestatus, n, cutoff, row_base=0):
    """TPC-H Q1 grouped aggregates (q1.sql).  returnflag/linestatus: packed uint8 columns or varlena cell buffers.
    Returns a list of dicts in first-seen group order."""
    res = np.zeros(C.sizeof(capi.Q1Result), dtype=np.uint8)
    rv = Vector(data=res, length=1)
    cut = _params_vec(capi.Q1Params(cutoff, 0, row_base))
    xcall(capi.XCALL_Q1_GROUP_AGG, [rv, _vec(shipdate, n), _vec(quantity, n), _vec(extendedprice, n), _vec(discount, n), _vec(tax, n),
                                     _vec(returnflag, n), _vec(linestatus, n), cut], n)
    r = capi.Q1Result.from_buffer_copy(res.tobytes())
    out = []
    for g in range(r.ngroups):
        s = r.groups[g]
        out.append({k: getattr(s, k) for k in ("returnflag", "linestatus", "first_row", "sum_qty", "sum_base_price", "sum_disc_price",
                                               "sum_charge", "avg_qty", "avg_price", "avg_disc", "sum_disc", "count_order")})
    return out


# ------------------------------------------------------------------------------------------------ vector search
def _search_params(n, dim, nq, k, metric, nprobe=0, sqrt_out=0, nlist=0, key_base=0):
    return capi.SearchParams(n, dim, nq, k, metric, nprobe, sqrt_out, nlist, key_base)


class BruteForceIndex:
    """brute_force.GoBruteForceIndex: NewBruteForceIndex(dataset, dim, metric) keeps the dataset RESIDENT in HBM
    (the reference keeps it in C-malloc memory, brute_force.go:104-123); Search returns (keys int64[nq*limit],
    distances float64[nq*limit]) row-major, ascending, keys = row ordinals (+ key_base)."""

    def __init__(self, dataset, dim, metric=capi.METRIC_L2, key_base=0, lib=None):
        self.lib = lib or capi.load_library()
        self.dim, self.metric, self.key_base = int(dim), int(metric), int(key_base)
        if isinstance(dataset, DeviceBuffer):
            self.buf, self.owned = dataset, False
            self.n = dataset.nbytes // (4 * self.dim)
        else:
            ds = np.ascontiguousarray(dataset, dtype=np.float32)
            self.n = ds.shape[0]
            self.buf, self.owned = DeviceBuffer.from_numpy(ds, self.lib), True
        self._prepare()

    def _prepare(self):
        # Load: split the resident rows into the tensor-core operand once (L2 metrics; a no-op where it does not apply)
        self.prepared = self.metric in (capi.METRIC_L2, capi.METRIC_L2SQ, capi.METRIC_IP, capi.METRIC_COS) and self.n > 0
        if self.prepared:
            capi.check(self.lib.MoB200_SearchPrepareMetric(self.buf.ptr, self.n, self.dim, self.metric), self.lib)

    def search(self, queries, limit, out_device=False, out=None):
        """out = (keys_device_ptr, distances_device_ptr): results stay in caller-owned device memory (int64 / float64, nq*limit
        each) and nothing is returned -- the form a multi-GPU caller hands straight to NCCL"""
        if isinstance(queries, DeviceBuffer):
            nq = queries.nbytes // (4 * self.dim)
            qv = Vector(data_ptr=queries.ptr, data_nbytes=queries.nbytes, length=nq)
        else:
            q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
            nq = q.shape[0]
            qv = Vector(data=q.reshape(-1), length=nq)
        if limit == 0 or nq == 0:
            return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.float64)
        p = _search_params(self.n, self.dim, nq, limit, self.metric, key_base=self.key_base)
        dv = Vector(data_ptr=self.buf.ptr, data_nbytes=self.n * self.dim * 4, length=self.n)
        if out is not None:
            kv = Vector(data_ptr=out[0], data_nbytes=nq * limit * 8, length=nq)
            dvv = Vector(data_ptr=out[1], data_nbytes=nq * limit * 8, length=nq)
            xcall(capi.XCALL_BRUTEFORCE_TOPK_F32, [kv, dvv, dv, qv, _params_vec(p)], nq)
            return None
        keys = np.zeros(nq * limit, dtype=np.int64)
        dists = np.zeros(nq * limit, dtype=np.float64)
        xcall(capi.XCALL_BRUTEFORCE_TOPK_F32, [Vector(data=keys, length=nq), Vector(data=dists, length=nq), dv, qv, _params_vec(p)], nq)
        return keys, dists

    def destroy(self):
        if self.buf is not None and getattr(self, "prepared", False):
            self.lib.MoB200_SearchRelease(self.buf.ptr)
        if self.owned and self.buf is not None:
            self.buf.free()
        self.buf = None


class IvfflatSearchIndex:
    """ivfflat.IvfflatSearchIndex: centroids + list-ordered entries resident in HBM.  build() takes the entry matrix
    and its list assignment (what the index tables hold) and lays the lists out contiguously."""

    def __init__(self, data, assign, centroids, metric=capi.METRIC_L2, lib=None):
        self.lib = lib or capi.load_library()
        centroids = np.ascontiguousarray(centroids, dtype=np.float32)
        self.nlist, self.dim = centroids.shape
        self.metric = int(metric)
        assign = np.asarray(assign)
        order = np.argsort(assign, kind="stable")   # stable: rows of a list stay in table order
        counts = np.bincount(assign, minlength=self.nlist)
        self.offsets = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
        self.row_ids = order.astype(np.int64)
        self.n = len(order)
        self.d_ids = DeviceBuffer.from_numpy(self.row_ids, self.lib)
        if isinstance(data, DeviceBuffer):          # resident entries: lay them out list by list on the device
            self.d_data = DeviceBuffer(4 * self.n * self.dim, self.lib)
            capi.check(self.lib.MoB200_GatherRowsF32(self.d_data.ptr, data.ptr, self.d_ids.ptr, self.n, self.dim), self.lib)
        else:
            data = np.ascontiguousarray(data, dtype=np.float32)
            self.d_data = DeviceBuffer.from_numpy(data[order], self.lib)
        self.d_cent = DeviceBuffer.from_numpy(centroids, self.lib)
        self.d_off = DeviceBuffer.from_numpy(self.offsets, self.lib)
        self.prepared = self.metric in (capi.METRIC_L2, capi.METRIC_L2SQ) and self.n > 0
        if self.prepared:   # LoadIndex: the list-ordered entries are split (as residuals against their centroid) once
            capi.check(self.lib.MoB200_SearchPrepareIvf(self.d_data.ptr, self.n, self.dim, self.d_cent.ptr, self.nlist, self.d_off.ptr), self.lib)

    @classmethod
    def build(cls, data_dev, n, centroids, metric=capi.METRIC_L2, lib=None, chunk=500_000):
        """index build on resident entries: centroid assignment = Productl2 (brute-force Search(limit=1) against the
        centroids, pkg/sql/colexec/productl2/product_l2.go:317-407) run chunk by chunk, then the list-ordered layout"""
        lib = lib or capi.load_library()
        centroids = np.ascontiguousarray(centroids, dtype=np.float32)
        dim = centroids.shape[1]
        cidx = BruteForceIndex(centroids, dim, metric, lib=lib)
        assign = np.empty(n, dtype=np.int32)
        for r0 in range(0, n, chunk):
            m = min(chunk, n - r0)
            view = DeviceBuffer.__new__(DeviceBuffer)
            view.lib, view.nbytes, view.ptr = lib, 4 * m * dim, data_dev.ptr + 4 * r0 * dim
            keys, _ = cidx.search(view, 1)
            view.ptr = None
            assign[r0:r0 + m] = keys
        cidx.destroy()
        return cls(data_dev, assign, centroids, metric, lib)

    @classmethod
    def build_list_shard(cls, gen_rows, n_total, centroids, rank, world, metric=capi.METRIC_L2, lib=None, chunk=500_000):
        """index build for ONE shard of a list-sharded index (BASELINE config 5: "lists sharded 8 x B200"): every row of the table is assigned to
        its nearest centroid (Productl2, product_l2.go:317-407) and this shard keeps the WHOLE lists l with l % world == rank; the centroid table is
        replicated, the other lists are empty here.  gen_rows(row0, m, device_ptr) materialises table rows [row0, row0 + m) in device memory.
        Row ids are the table's row numbers (primary keys)."""
        lib = lib or capi.load_library()
        centroids = np.ascontiguousarray(centroids, dtype=np.float32)
        dim = centroids.shape[1]
        cidx = BruteForceIndex(centroids, dim, metric, lib=lib)
        cap = n_total if world == 1 else int(n_total / world * 1.1) + chunk
        tmp = DeviceBuffer(4 * cap * dim, lib)
        scratch = DeviceBuffer(4 * min(chunk, n_total) * dim, lib)
        ids, lists, filled = [], [], 0
        for r0 in range(0, n_total, chunk):
            m = min(chunk, n_total - r0)
            gen_rows(r0, m, scratch.ptr)
            keys, _ = cidx.search(scratch.view(4 * m * dim), 1)
            mine = np.flatnonzero(keys % world == rank).astype(np.int64)
            if filled + mine.shape[0] > cap:
                raise capi.MoError(capi.RC_INTERNAL_ERROR, "list shard larger than expected")
            if mine.shape[0]:
                didx = DeviceBuffer.from_numpy(mine, lib)
                capi.check(lib.MoB200_GatherRowsF32(tmp.ptr + 4 * filled * dim, scratch.ptr, didx.ptr, mine.shape[0], dim), lib)
                didx.free()
            ids.append(mine + r0); lists.append(keys[mine].astype(np.int32)); filled += mine.shape[0]
        cidx.destroy(); scratch.free()
        gids = np.concatenate(ids) if ids else np.zeros(0, dtype=np.int64)
        ix = cls(tmp.view(4 * filled * dim), np.concatenate(lists) if lists else np.zeros(0, dtype=np.int32), centroids, metric, lib)
        tmp.free()
        ix.row_ids = gids[ix.row_ids]                  # list-ordered position -> table row number
        ix.d_ids.free(); ix.d_ids = DeviceBuffer.from_numpy(ix.row_ids, lib)
        return ix

    def search(self, queries, limit, nprobe, sqrt_out=False, out=None):
        if isinstance(queries, DeviceBuffer):
            nq = queries.nbytes // (4 * self.dim)
            qvec = Vector(data_ptr=queries.ptr, data_nbytes=queries.nbytes, length=nq)
        else:
            q = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
            nq = q.shape[0]
            qvec = Vector(data=q.reshape(-1), length=nq)
        if out is not None:     # results stay in caller-owned device memory (see BruteForceIndex.search)
            keys = dists = None
            kv = Vector(data_ptr=out[0], data_nbytes=nq * limit * 8, length=nq)
            dvv = Vector(data_ptr=out[1], data_nbytes=nq * limit * 8, length=nq)
        else:
            keys = np.zeros(nq * limit, dtype=np.int64)
            dists = np.zeros(nq * limit, dtype=np.float64)
            kv, dvv = Vector(data=keys, length=nq), Vector(data=dists, length=nq)
        p = _search_params(self.n, self.dim, nq, limit, self.metric, nprobe=nprobe, sqrt_out=int(sqrt_out), nlist=self.nlist)
        xcall(capi.XCALL_IVF_TOPK_F32, [
            kv, dvv,
            Vector(data_ptr=self.d_data.ptr, data_nbytes=self.d_data.nbytes, length=self.n),
            qvec, _params_vec(p),
            Vector(data_ptr=self.d_cent.ptr, data_nbytes=self.d_cent.nbytes, length=self.nlist),
            Vector(data_ptr=self.d_off.ptr, data_nbytes=self.d_off.nbytes, length=self.nlist + 1),
            Vector(data_ptr=self.d_ids.ptr, data_nbytes=self.d_ids.nbytes, length=self.n)], nq)
        return keys, dists

    def destroy(self):
        if self.prepared:
            self.lib.MoB200_SearchRelease(self.d_data.ptr)
        for b in (self.d_data, self.d_cent, self.d_off, self.d_ids):
            b.free()


def topk_merge_device(keys_ptr, dists_ptr, nshards, nq, k, out_keys_ptr, out_dists_ptr):
    """topk_merge on device-resident [nshards, nq, k] results (e.g. straight out of an NCCL all_gather); outputs stay on the device"""
    p = _search_params(nshards, 0, nq, k, 0)
    xcall(capi.XCALL_TOPK_MERGE, [Vector(data_ptr=out_keys_ptr, data_nbytes=nq * k * 8, length=nq), Vector(data_ptr=out_dists_ptr, data_nbytes=nq * k * 8, length=nq),
                                  Vector(data_ptr=keys_ptr, data_nbytes=nshards * nq * k * 8, length=nq),
                                  Vector(data_ptr=dists_ptr, data_nbytes=nshards * nq * k * 8, length=nq), _params_vec(p)], nq)


def topk_merge(keys_shards, dists_shards, nq, k):
    """merge [nshards, nq, k] per-shard results (final keys, float64 distances) into the global top-k."""
    ks = np.ascontiguousarray(keys_shards, dtype=np.int64).reshape(-1)
    ds = np.ascontiguousarray(dists_shards, dtype=np.float64).reshape(-1)
    nsh = ks.shape[0] // (nq * k)
    keys = np.zeros(nq * k, dtype=np.int64)
    dists = np.zeros(nq * k, dtype=np.float64)
    p = _search_params(nsh, 0, nq, k, 0)
    xcall(capi.XCALL_TOPK_MERGE, [Vector(data=keys, length=nq), Vector(data=dists, length=nq), Vector(data=ks, length=nq),
                                  Vector(data=ds, length=nq), _params_vec(p)], nq)
    return keys, dists


# ------------------------------------------------------------------------------------------------ column operators (csrc/colops.cu)
def _with_nulls(x, nulls, length):
    v = _vec(x, length)
    if nulls is not None:
        if isinstance(nulls, DeviceBuffer):
            v.nulls_ptr = nulls.ptr
        else:
            v.nulls = np.ascontiguousarray(nulls, dtype=np.uint64)
    v.length = length
    return v


def filter_sels(bools, nulls=None, length=None):
    """Filter.Call inner loop (filter.go:116-152): ascending row numbers with (!null && true).  Host arrays in, numpy sels out."""
    b = np.ascontiguousarray(bools, dtype=np.uint8)
    n = length if length is not None else b.shape[0]
    sels = np.zeros(max(n, 1), dtype=np.int64)
    cnt = np.zeros(1, dtype=np.int64)
    xcall(capi.XCALL_FILTER_SELS, [Vector(data=sels, length=n), Vector(data=cnt, length=1), _with_nulls(b, nulls, n)], n)
    return sels[:int(cnt[0])]


def filter_sels_device(bools_dev, nulls_dev, n, sels_ptr, count_ptr):
    """asynchronous form on resident vectors: sels (int64[n] capacity) and the count stay on the device"""
    bv = Vector(data_ptr=bools_dev.ptr, data_nbytes=n, nulls_ptr=nulls_dev.ptr if nulls_dev is not None else None, length=n)
    xcall(capi.XCALL_FILTER_SELS, [Vector(data_ptr=sels_ptr, data_nbytes=8 * n, length=n), Vector(data_ptr=count_ptr, data_nbytes=8, length=1), bv], n)


def shuffle(src, sels, src_nulls=None, want_nulls=False):
    """Vector.Shrink / Union (shuffle.FixedLengthShuffle + nulls.Filter): returns dst (and dst nulls words when want_nulls)"""
    a = np.ascontiguousarray(src)
    s = np.ascontiguousarray(sels, dtype=np.int64)
    m = s.shape[0]
    dst = np.zeros(m, dtype=a.dtype)
    dn = np.zeros((m + 63) // 64, dtype=np.uint64) if want_nulls else None
    sv = Vector(data=a.view(np.uint8).reshape(-1), nulls=src_nulls, length=a.shape[0])
    xcall(capi.XCALL_SHUFFLE(a.dtype.itemsize), [Vector(data=dst.view(np.uint8).reshape(-1), nulls=dn, length=m), sv, Vector(data=s, length=m)], m)
    return (dst, dn) if want_nulls else dst


def pack_keys(cols, nulls=None, has_null=True, length=None):
    """fillKeys (inthashmap.go:92-183): <= 8 key bytes per row.  cols: list of fixed-width numpy columns (a 1-element array = const vector).
    Returns (keys uint64[n], skip bitmap words or None)"""
    n = length if length is not None else max(len(c) for c in cols)
    keys = np.zeros(n, dtype=np.uint64)
    skip = None if has_null else np.zeros((n + 63) // 64, dtype=np.uint64)
    prm = np.asarray([len(cols), 1 if has_null else 0], dtype=np.int32)
    vecs = [Vector(data=keys, nulls=skip, length=n), Vector(data=prm.view(np.uint8), length=1, const=True)]
    for i, c in enumerate(cols):
        c = np.ascontiguousarray(c)
        vecs.append(Vector(data=c.view(np.uint8).reshape(-1), nulls=None if nulls is None else nulls[i], length=n))
    xcall(capi.XCALL_PACK_KEYS, vecs, n)
    return keys, skip


class GroupTable:
    """IntHashMap as the group operator sees it: insert(keys) -> 1-based group ids in first-seen order; the table persists across batches"""

    def __init__(self, capacity):
        self.keys = np.zeros(capacity, dtype=np.uint64)
        self.ngroups = np.zeros(1, dtype=np.int64)

    def insert(self, keys, skip=None):
        k = np.ascontiguousarray(keys, dtype=np.uint64)
        n = k.shape[0]
        groups = np.zeros(n, dtype=np.uint64)
        xcall(capi.XCALL_GROUP_IDS, [Vector(data=groups, length=n), Vector(data=self.ngroups, length=1), Vector(data=self.keys, length=self.keys.shape[0]),
                                     Vector(data=k, nulls=skip, length=n)], n)
        return groups

    def insert_device(self, keys_dev, n, groups_dev, d_ngroups, d_table_keys, capacity):
        """all vectors resident (DeviceBuffer); the group count is read back by the call (it sizes the next operator's state)"""
        xcall(capi.XCALL_GROUP_IDS, [Vector(data_ptr=groups_dev.ptr, data_nbytes=8 * n, length=n), Vector(data_ptr=d_ngroups.ptr, data_nbytes=8, length=1),
                                     Vector(data_ptr=d_table_keys.ptr, data_nbytes=8 * capacity, length=capacity),
                                     Vector(data_ptr=keys_dev.ptr, data_nbytes=8 * n, length=n)], n)


def group_agg(op, T, state, state_nulls, counts, groups, col, col_nulls=None, length=None):
    """BatchFill of one aggregate into caller-owned state arrays (numpy, modified in place): state uint64/int64/float64[ngroups] (8-byte slots),
    state_nulls bitmap words (group is NULL), counts int64[ngroups] or None.  Returns rc (0 or RC_OUT_OF_RANGE)."""
    g = np.ascontiguousarray(groups, dtype=np.uint64)
    n = length if length is not None else g.shape[0]
    sv = Vector(data=state.view(np.uint8).reshape(-1), nulls=state_nulls, length=state.shape[0])
    cv = Vector(data=counts, length=state.shape[0]) if counts is not None else Vector(length=0)
    colv = _with_nulls(np.ascontiguousarray(col).view(np.uint8).reshape(-1), col_nulls, n) if col is not None else _with_nulls(np.zeros(0, dtype=np.uint8), col_nulls, n)
    rc, msg = xcall(capi.XCALL_GROUP_AGG(op, T), [sv, cv, Vector(data=g, length=n), colv], n, raise_on_error=False)
    if rc not in (0, capi.RC_OUT_OF_RANGE):
        raise capi.MoError(rc, msg)
    return rc


# ------------------------------------------------------------------------------------------------ the generic fused operator (csrc/plan.cu)
class FusedPlan:
    """Builder for mo_plan_t: table_scan -> filter -> projection -> group in one kernel.

        p = FusedPlan([capi.T_DATE, capi.T_FLOAT64, capi.T_FLOAT64, capi.T_FLOAT64])          # column types
        p.where(0, ">=", lo).where(0, "<", hi).where(1, "between", a, b).where(2, "<", 24.0)
        revenue = p.mul(p.col(3), p.col(1))                                                 # value slots
        p.agg(capi.AGG_SUM, revenue)
        groups = p.run([shipdate, discount, quantity, price], n)
    """

    def __init__(self, col_types, has_null_keys=False, row_base=0):
        self.P = capi.Plan()
        self.P.ncols = len(col_types)
        for i, t in enumerate(col_types):
            self.P.col_type[i] = t
        self.P.has_null_keys = 1 if has_null_keys else 0
        self.P.row_base = row_base

    def where(self, col, op, lo, hi=0.0):
        q = self.P.pred[self.P.npreds]
        q.col, q.op, q.lo, q.hi = col, capi.PLAN_CMP[op], float(lo), float(hi)
        self.P.npreds += 1
        return self

    def _emit(self, op, a=0, b=0, imm=0.0):
        i = self.P.ninstr
        ins = self.P.instr[i]
        ins.op, ins.a, ins.b, ins.imm = op, a, b, float(imm)
        self.P.ninstr += 1
        return self.P.ncols + i

    def col(self, c):
        return c                      # a column IS value slot c

    def const(self, x):
        return self._emit(capi.PLAN_OP_CONST, imm=x)

    def add(self, a, b):
        return self._emit(capi.PLAN_OP_ADD, a, b)

    def sub(self, a, b):
        return self._emit(capi.PLAN_OP_SUB, a, b)

    def mul(self, a, b):
        return self._emit(capi.PLAN_OP_MUL, a, b)

    def div(self, a, b):
        return self._emit(capi.PLAN_OP_DIV, a, b)

    def group_by(self, *cols):
        for c in cols:
            self.P.key_col[self.P.nkeys] = c
            self.P.nkeys += 1
        return self

    def agg(self, kind, value=-1):
        a = self.P.agg[self.P.naggs]
        a.kind, a.value = kind, value
        self.P.naggs += 1
        return self

    def result_bytes(self, max_groups):
        return C.sizeof(capi.PlanHeader) + max_groups * (24 + 16 * self.P.naggs)

    def run(self, cols, n, nulls=None, max_groups=64, out_ptr=None):
        """cols: numpy arrays or DeviceBuffers (one per declared column); nulls: optional list of bitmap words (numpy / DeviceBuffer / None).
        out_ptr: device result buffer of result_bytes(max_groups) -> asynchronous form, returns None.  Else a list of group dicts
        {key, first_row, rows, aggs: [(value, count), ...]} in first-seen order."""
        vecs = []
        for i, c in enumerate(cols):
            nb = None if nulls is None else nulls[i]
            vecs.append(_with_nulls(c if isinstance(c, DeviceBuffer) else np.ascontiguousarray(c).view(np.uint8).reshape(-1), nb, n))
        nbytes = self.result_bytes(max_groups)
        if out_ptr is not None:
            xcall(capi.XCALL_PLAN, [Vector(data_ptr=out_ptr, data_nbytes=nbytes, length=1), _params_vec(self.P)] + vecs, n)
            return None
        res = np.zeros(nbytes, dtype=np.uint8)
        xcall(capi.XCALL_PLAN, [Vector(data=res, length=1), _params_vec(self.P)] + vecs, n)
        return self.parse(res.tobytes())

    def parse(self, raw):
        h = capi.PlanHeader.from_buffer_copy(raw[:C.sizeof(capi.PlanHeader)])
        if h.overflow:
            raise capi.MoError(capi.RC_INVALID_ARGUMENT, "plan: more groups than the result buffer holds")
        rec = 24 + 16 * self.P.naggs
        out = []
        for g in range(h.ngroups):
            b = raw[C.sizeof(capi.PlanHeader) + g * rec: C.sizeof(capi.PlanHeader) + (g + 1) * rec]
            key, first_row, rows = np.frombuffer(b[:8], dtype=np.uint64)[0], np.frombuffer(b[8:16], dtype=np.int64)[0], np.frombuffer(b[16:24], dtype=np.int64)[0]
            aggs = []
            for a in range(self.P.naggs):
                v = np.frombuffer(b[24 + 16 * a: 32 + 16 * a], dtype=np.float64)[0]
                c = np.frombuffer(b[32 + 16 * a: 40 + 16 * a], dtype=np.int64)[0]
                aggs.append((float(v), int(c)))
            out.append({"key": int(key), "first_row": int(first_row), "rows": int(rows), "aggs": aggs})
        if not h.sorted:
            out.sort(key=lambda g: g["first_row"])
        return out


def q6_plan():
    """TPC-H Q6 (q6.sql) as a FusedPlan over columns [shipdate DATE, discount f64, quantity f64, extendedprice f64]"""
    from . import datagen
    lo, hi, dlo, dhi, qhi = datagen.q6_params()
    p = FusedPlan([capi.T_DATE, capi.T_FLOAT64, capi.T_FLOAT64, capi.T_FLOAT64])
    p.where(0, ">=", lo).where(0, "<", hi).where(1, "between", dlo, dhi).where(2, "<", qhi)
    p.agg(capi.AGG_SUM, p.mul(p.col(3), p.col(1)))
    return p


def q1_plan(cutoff, row_base=0):
    """TPC-H Q1 (q1.sql) as a FusedPlan over columns [shipdate, quantity, extendedprice, discount, tax, returnflag u8, linestatus u8]"""
    p = FusedPlan([capi.T_DATE, capi.T_FLOAT64, capi.T_FLOAT64, capi.T_FLOAT64, capi.T_FLOAT64, capi.T_UINT8, capi.T_UINT8], row_base=row_base)
    p.where(0, "<=", cutoff)
    one = p.const(1.0)
    disc_price = p.mul(p.col(2), p.sub(one, p.col(3)))
    charge = p.mul(disc_price, p.add(one, p.col(4)))
    p.group_by(5, 6)
    for kind, v in ((capi.AGG_SUM, 1), (capi.AGG_SUM, 2), (capi.AGG_SUM, disc_price), (capi.AGG_SUM, charge), (capi.AGG_AVG, 1), (capi.AGG_AVG, 2), (capi.AGG_AVG, 3)):
        p.agg(kind, v)
    p.agg(capi.AGG_COUNT, -1)
    return p


# ------------------------------------------------------------------------------------------------ decimals (csrc/decimal.cu)
def dec_arith(op, width, a, b, scale1, scale2, n, n1=None, n2=None, rnulls=None):
    """d64/d128 Add (op 0) / Sub (1) / Mul (2).  a, b: int64 arrays (width 64) or uint64[n, 2] {lo, hi} arrays (width 128); a 1-row operand is a
    const vector.  Returns (rc, result, result nulls words, err_row); result is int64[n] (64-bit + -) or uint64[n, 2]."""
    out128 = op == 2 or width == 128
    r = np.zeros((n, 2), dtype=np.uint64) if out128 else np.zeros(n, dtype=np.int64)
    rn = np.zeros((n + 63) // 64, dtype=np.uint64) if rnulls is None else np.ascontiguousarray(rnulls, dtype=np.uint64).copy()
    prm = np.frombuffer(bytes(capi.DecParams(scale1, scale2, -1)), dtype=np.uint8).copy()
    av = Vector(data=np.ascontiguousarray(a).view(np.uint8).reshape(-1), nulls=n1, length=n)
    bv = Vector(data=np.ascontiguousarray(b).view(np.uint8).reshape(-1), nulls=n2, length=n)
    rc, msg = xcall(capi.XCALL_DEC_ARITH(op, width), [Vector(data=r.view(np.uint8).reshape(-1), nulls=rn, length=n), av, bv, Vector(data=prm, length=1, const=True)], n,
                    raise_on_error=False)
    if rc not in (0, capi.RC_INVALID_ARGUMENT):
        raise capi.MoError(rc, msg)
    return rc, r, rn, int(prm.view(np.int64)[1])


def dec_sum(width, col, sums, counts, groups=None, nulls=None, n=None):
    """SUM/AVG accumulation into sums uint64[ngroups, 2] (Decimal128) and counts int64[ngroups], in place"""
    c = np.ascontiguousarray(col)
    n = n if n is not None else (c.shape[0])
    gv = Vector(data=np.ascontiguousarray(groups, dtype=np.uint64), length=n) if groups is not None else Vector(length=0)
    xcall(capi.XCALL_DEC_SUM(width), [Vector(data=sums.view(np.uint8).reshape(-1), length=sums.shape[0]), Vector(data=counts, length=counts.shape[0]), gv,
                                      _with_nulls(c.view(np.uint8).reshape(-1), nulls, n)], n)


# ---------------------------------------------------------------------------------------------- normalize_l2 (vector-valued)
def normalize_l2(cells, area, length, dtype=np.float32, nulls=None):
    """normalize_l2(v) over a varlena vector column (moarray.NormalizeL2, pkg/vectorize/moarray/external.go:262-285).  Returns
    (result cells uint8[24 * length], result area uint8[len(area)]): the result mirrors the argument's layout."""
    cells = np.ascontiguousarray(cells, dtype=np.uint8)
    area = np.ascontiguousarray(area, dtype=np.uint8)
    ocells = np.zeros(24 * length, dtype=np.uint8)
    oarea = np.zeros(max(area.nbytes, 1), dtype=np.uint8)
    res = Vector(data=ocells, area=oarea, nulls=None if nulls is None else np.array(nulls, dtype=np.uint64, copy=True), length=length)
    fid = capi.XCALL_GO_NORMALIZE_L2_F32 if np.dtype(dtype) == np.float32 else capi.XCALL_GO_NORMALIZE_L2_F64
    xcall(fid, [res, Vector(data=cells, area=area, length=length)], length)
    return ocells, oarea[:area.nbytes]


# ---------------------------------------------------------------------------------------------- hash join (csrc/join.cu)
def _group_sels(groups, nbuild, ngroups):
    """GroupSels.Insert + Finalize over the build side's group ids (JOIN_SELS): (offsets, sels), or (None, None) when every build row has its own
    group or none has one -- Finalize keeps no sels then (joinMapMsg.go:83-89)"""
    if ngroups == nbuild:
        return None, None
    offsets = np.zeros(ngroups + 2, dtype=np.int32)
    sels = np.zeros(max(nbuild, 1), dtype=np.int32)
    cnt = np.zeros(1, dtype=np.int64)
    xcall(capi.XCALL_JOIN_SELS, [Vector(data=offsets, length=ngroups + 2), Vector(data=sels, length=nbuild), Vector(data=cnt, length=1),
                                 Vector(data=groups, length=nbuild)], nbuild)
    if int(cnt[0]) == 0:
        return None, None
    return offsets, sels[:int(cnt[0])]


class JoinMap:
    """message.JoinMap for equality joins over <= 8-byte packed keys (pkg/vm/message/joinMapMsg.go:127-210): the build side's IntHashMap
    (GroupTable: first-seen group ids + key table) and its GroupSels.  HashOnUnique (every build row its own group) keeps no sels."""

    def __init__(self, build_keys, skip=None, prepare=True):
        k = np.ascontiguousarray(build_keys, dtype=np.uint64)
        self.nbuild = k.shape[0]
        tab = GroupTable(max(self.nbuild, 1))
        groups = tab.insert(k, skip)                                   # HashmapBuilder.BuildHashmap: itr.Insert (hashmap.go:340-360)
        self.ngroups = int(tab.ngroups[0])
        self.table_keys = np.ascontiguousarray(tab.keys[:max(self.ngroups, 1)])[:self.ngroups].copy() if self.ngroups else np.zeros(0, np.uint64)
        self.offsets, self.sels = _group_sels(groups, self.nbuild, self.ngroups)
        self.prepared = False
        if prepare and self.ngroups:
            lib = capi.load_library()
            capi.check(lib.MoB200_JoinMapPrepare(self.table_keys.ctypes.data, self.ngroups), lib)
            self.prepared = True

    def hash_on_unique(self):
        return self.offsets is None

    def find(self, keys, nulls=None):
        """intHashMapIterator.Find: 1-based group id per probe key, 0 = no match"""
        k = np.ascontiguousarray(keys, dtype=np.uint64)
        n = k.shape[0]
        vals = np.zeros(n, dtype=np.uint64)
        xcall(capi.XCALL_JOIN_FIND, [Vector(data=vals, length=n), Vector(data=self.table_keys, length=self.ngroups), Vector(data=k, nulls=nulls, length=n)], n)
        return vals

    def probe(self, keys, join_type=capi.JOIN_INNER, nulls=None, capacity=None):
        """(probe rows, build rows) of the join result in the reference's emission order; build row -1 = no build side (left outer / semi / anti)"""
        k = np.ascontiguousarray(keys, dtype=np.uint64)
        n = k.shape[0]
        cap = capacity if capacity is not None else max(2 * n, 1024)
        prm = np.array([join_type, 0], dtype=np.int32)
        while True:
            op, ob, cnt = np.zeros(cap, np.int64), np.zeros(cap, np.int64), np.zeros(1, np.int64)
            vecs = [Vector(data=op, length=cap), Vector(data=ob, length=cap), Vector(data=cnt, length=1), Vector(data=prm.view(np.uint8), length=1),
                    Vector(data=self.table_keys, length=self.ngroups),
                    Vector(data=self.offsets, length=self.ngroups + 2) if self.offsets is not None else Vector(length=0),
                    Vector(data=self.sels, length=len(self.sels)) if self.sels is not None else Vector(length=0),
                    Vector(data=k, nulls=nulls, length=n)]
            rc, msg = xcall(capi.XCALL_JOIN_PROBE, vecs, n, raise_on_error=False)
            if rc == capi.RC_OUT_OF_RANGE and capacity is None:       # the count was reported: size the buffers and ask again
                cap = int(cnt[0])
                continue
            if rc:
                raise capi.MoError(rc, msg)
            return op[:int(cnt[0])], ob[:int(cnt[0])]

    def release(self):
        if self.prepared:
            lib = capi.load_library()
            lib.MoB200_JoinMapRelease(self.table_keys.ctypes.data)
            self.prepared = False


# ---------------------------------------------------------------------------------------------- keys wider than 8 bytes (csrc/strhash.cu)
def pack_str_keys(cols, kinds, nulls=None, has_null=True, const=None, length=None, capacity=None):
    """strHashmapIterator.encodeHashKeys (strhashmap.go:92-385): the exact StrHashMap key bytes of every row.
    cols[k]: a fixed-width numpy column (kinds[k] = element bytes, any width >= 1) or a varlena (cells uint8[24 * n], area) pair (kinds[k] = 0);
    nulls[k]: bitmap words or None; const[k]: column k holds one element that every row repeats (a const NULL: nulls[k] with bit 0 set).
    Returns (offsets int64[n + 1], key bytes uint8[offsets[n]], skip bitmap words -- has_null=False only -- or None)."""
    ncols = len(cols)
    const = const or [False] * ncols
    raw = []
    n = length
    for k, c in enumerate(cols):
        w = int(kinds[k])
        if w:
            data, area = np.ascontiguousarray(c).view(np.uint8).reshape(-1), None
        else:
            data, area = np.ascontiguousarray(c[0], dtype=np.uint8).reshape(-1), np.ascontiguousarray(c[1], dtype=np.uint8).reshape(-1)
        if n is None and not const[k]:
            n = data.nbytes // (w or 24)
        raw.append((data, area))
    n = n if n is not None else 1
    vecs = [Vector(data=d, area=a, nulls=None if nulls is None else nulls[k], length=1 if const[k] else n) for k, (d, a) in enumerate(raw)]
    prm = capi.StrKeyParams(ncols, 1 if has_null else 0)
    for k, w in enumerate(kinds):
        prm.width[k] = int(w)
    offsets = np.zeros(n + 1, dtype=np.int64)
    skip = None if has_null else np.zeros((n + 63) // 64, dtype=np.uint64)
    cap = capacity if capacity is not None else 24 * n + 64
    while True:
        kb = np.zeros(max(cap, 1), dtype=np.uint8)
        rc, msg = xcall(capi.XCALL_PACK_STR_KEYS, [Vector(data=offsets, nulls=skip, length=n), Vector(data=kb, length=cap), _params_vec(prm)] + vecs, n,
                        raise_on_error=False)
        if rc == capi.RC_OUT_OF_RANGE and capacity is None:          # offsets[n] holds the bytes needed: size the buffer and ask again
            cap = int(offsets[n])
            continue
        if rc:
            raise capi.MoError(rc, msg)
        return offsets, kb[:int(offsets[n])], skip


class StrGroupTable:
    """StrHashMap as the group operator sees it: insert(packed keys) -> 1-based group ids in first-seen order.  The key table (offsets + bytes,
    key of group g at bytes[offsets[g - 1] : offsets[g]]) persists across batches and grows when a batch does not fit."""

    def __init__(self, capacity=1024, byte_capacity=None):
        capacity = max(int(capacity), 1)
        self.offsets = np.zeros(capacity + 1, dtype=np.int64)
        self.bytes = np.zeros(max(int(byte_capacity if byte_capacity is not None else 32 * capacity), 16), dtype=np.uint8)
        self.state = np.zeros(4, dtype=np.int64)      # {ngroups, key bytes used, groups needed, bytes needed}

    @property
    def ngroups(self):
        return int(self.state[0])

    def _grow(self, groups, nbytes):
        ng, used = self.ngroups, int(self.state[1])
        if groups > self.offsets.shape[0] - 1:
            off = np.zeros(max(groups, 2 * (self.offsets.shape[0] - 1)) + 1, dtype=np.int64)
            off[:ng + 1] = self.offsets[:ng + 1]
            self.offsets = off
        if nbytes > self.bytes.shape[0]:
            b = np.zeros(max(nbytes, 2 * self.bytes.shape[0]), dtype=np.uint8)
            b[:used] = self.bytes[:used]
            self.bytes = b

    def insert(self, offsets, key_bytes, skip=None):
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        kb = np.ascontiguousarray(key_bytes, dtype=np.uint8)
        n = off.shape[0] - 1
        groups = np.zeros(n, dtype=np.uint64)
        while True:
            rc, msg = xcall(capi.XCALL_STR_GROUP_IDS, [Vector(data=groups, length=n), Vector(data=self.state, length=4),
                                                       Vector(data=self.offsets, length=self.offsets.shape[0]), Vector(data=self.bytes, length=self.bytes.shape[0]),
                                                       Vector(data=off, nulls=skip, length=n), Vector(data=kb, length=kb.shape[0])], n, raise_on_error=False)
            if rc == capi.RC_OUT_OF_RANGE:                            # the table is unchanged and the sizes are reported: grow and repeat
                self._grow(int(self.state[2]), int(self.state[3]))
                continue
            if rc:
                raise capi.MoError(rc, msg)
            return groups

    def table(self):
        """(offsets int64[ngroups + 1], bytes) of the groups so far, copies"""
        ng = self.ngroups
        return self.offsets[:ng + 1].copy(), self.bytes[:int(self.state[1])].copy()

    def key(self, g):
        return self.bytes[self.offsets[g - 1]:self.offsets[g]].tobytes()


class StrJoinMap:
    """message.JoinMap for equality joins over StrHashMap keys (the build side's packed keys): first-seen group ids + key table (StrGroupTable)
    and the GroupSels of JOIN_SELS.  find / probe take the probe side's packed keys (pack_str_keys)."""

    def __init__(self, build_offsets, build_bytes, skip=None, prepare=True):
        off = np.ascontiguousarray(build_offsets, dtype=np.int64)
        self.nbuild = off.shape[0] - 1
        tab = StrGroupTable(max(self.nbuild, 1), max(int(off[-1]), 16))
        groups = tab.insert(off, build_bytes, skip)                    # HashmapBuilder.BuildHashmap: itr.Insert (hashmap.go:340-360)
        self.ngroups = tab.ngroups
        self.key_offsets, self.key_bytes = tab.table()
        self.offsets, self.sels = _group_sels(groups, self.nbuild, self.ngroups)
        self.prepared = False
        if prepare and self.ngroups:
            lib = capi.load_library()
            capi.check(lib.MoB200_StrJoinMapPrepare(self.key_offsets.ctypes.data, self.key_bytes.ctypes.data, self.ngroups), lib)
            self.prepared = True

    def hash_on_unique(self):
        return self.offsets is None

    def _table(self):
        return [Vector(data=self.key_offsets, length=self.ngroups + 1), Vector(data=self.key_bytes, length=self.key_bytes.shape[0])]

    def find(self, offsets, key_bytes, skip=None):
        """strHashmapIterator.Find: 1-based group id per probe key, 0 = no match (or a skipped row)"""
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        n = off.shape[0] - 1
        vals = np.zeros(n, dtype=np.uint64)
        xcall(capi.XCALL_STR_JOIN_FIND, [Vector(data=vals, length=n)] + self._table() +
              [Vector(data=off, nulls=skip, length=n), Vector(data=np.ascontiguousarray(key_bytes, dtype=np.uint8))], n)
        return vals

    def probe(self, offsets, key_bytes, join_type=capi.JOIN_INNER, skip=None, capacity=None):
        """(probe rows, build rows) of the join result in the reference's emission order, as JoinMap.probe"""
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        kb = np.ascontiguousarray(key_bytes, dtype=np.uint8)
        n = off.shape[0] - 1
        cap = capacity if capacity is not None else max(2 * n, 1024)
        prm = np.array([join_type, 0], dtype=np.int32)
        while True:
            op, ob, cnt = np.zeros(cap, np.int64), np.zeros(cap, np.int64), np.zeros(1, np.int64)
            vecs = [Vector(data=op, length=cap), Vector(data=ob, length=cap), Vector(data=cnt, length=1), Vector(data=prm.view(np.uint8), length=1)] + self._table() + [
                Vector(data=self.offsets, length=self.ngroups + 2) if self.offsets is not None else Vector(length=0),
                Vector(data=self.sels, length=len(self.sels)) if self.sels is not None else Vector(length=0),
                Vector(data=off, nulls=skip, length=n), Vector(data=kb, length=kb.shape[0])]
            rc, msg = xcall(capi.XCALL_STR_JOIN_PROBE, vecs, n, raise_on_error=False)
            if rc == capi.RC_OUT_OF_RANGE and capacity is None:
                cap = int(cnt[0])
                continue
            if rc:
                raise capi.MoError(rc, msg)
            return op[:int(cnt[0])], ob[:int(cnt[0])]

    def release(self):
        if self.prepared:
            lib = capi.load_library()
            lib.MoB200_StrJoinMapRelease(self.key_offsets.ctypes.data)
            self.prepared = False


# ---------------------------------------------------------------------------------------------- Elkan k-means (csrc/kmeans.cu)
def kmeans_elkan(vectors, init_centroids, max_iter=500, rnd=None):
    """ElkanClusterer.Cluster (pkg/vectorindex/ivfflat/kmeans/elkans/clusterer.go:330-392), dense variant.  init_centroids: an array [k, dim],
    or an int k = kmeans.Random initialisation (Random.InitCentroids with Go's PCG, gorand.py) and the matching empty-cluster stream.
    Returns (centroids [k, dim], assignments int64[n], iterations)."""
    v = np.ascontiguousarray(vectors)
    assert v.dtype in (np.float32, np.float64)
    n, dim = v.shape
    if isinstance(init_centroids, (int, np.integer)):
        from . import gorand
        k = int(init_centroids)
        if n == k:                                    # Cluster(): vectorCnt == clusterCnt returns the vectors themselves (clusterer.go:337-339)
            return v.copy(), np.arange(n, dtype=np.int64), 0
        init_centroids = v[gorand.random_init_rows(n, k)]
        if rnd is None:
            rnd = np.array(gorand.empty_cluster_stream(min(dim * k * 4, 1 << 20)), dtype=np.float32)
    cent = np.ascontiguousarray(init_centroids, dtype=v.dtype).copy()
    k = cent.shape[0]
    assign = np.zeros(n, dtype=np.int64); iters = np.zeros(1, dtype=np.int64)
    prm = np.array([n, dim, k, max_iter], dtype=np.int64)
    vecs = [Vector(data=cent.reshape(-1), length=k * dim), Vector(data=assign, length=n), Vector(data=iters, length=1), Vector(data=prm.view(np.uint8), length=1),
            Vector(data=v.reshape(-1), length=n * dim),
            Vector(data=np.ascontiguousarray(rnd, dtype=np.float32), length=len(rnd)) if rnd is not None and len(rnd) else Vector(length=0)]
    xcall(capi.XCALL_KMEANS_ELKAN_F32 if v.dtype == np.float32 else capi.XCALL_KMEANS_ELKAN_F64, vecs, n)
    return cent, assign, int(iters[0])


# ---------------------------------------------------------------------------------------------- LZ4 block decode (csrc/lz4.cu)
def lz4_decode_blocks(blocks, sizes):
    """compress.Decompress over many column blocks in one call: blocks = list of compressed byte strings, sizes = their decoded sizes.
    Returns the list of decoded byte strings."""
    src = np.frombuffer(b"".join(blocks), dtype=np.uint8) if blocks else np.zeros(0, np.uint8)
    n = len(blocks)
    desc = np.zeros((n, 4), dtype=np.int64)
    so = do = 0
    for i, (b, s) in enumerate(zip(blocks, sizes)):
        desc[i] = (so, len(b), do, s)
        so += len(b); do += s
    dst = np.zeros(max(do, 1), dtype=np.uint8)
    xcall(capi.XCALL_LZ4_DECODE, [Vector(data=dst, length=do), Vector(data=src if src.size else np.zeros(1, np.uint8), length=so), Vector(data=desc.reshape(-1), length=4 * n)], n)
    return [dst[desc[i, 2]:desc[i, 2] + desc[i, 3]].tobytes() for i in range(n)]


# ---------------------------------------------------------------------------------------------- marshalled vector -> resident vector (csrc/vecdecode.cu)
class VectorView(C.Structure):
    _fields_ = [("vclass", C.c_int32), ("oid", C.c_int32), ("size", C.c_int32), ("width", C.c_int32), ("scale", C.c_int32), ("length", C.c_uint32),
                ("data_len", C.c_uint64), ("area_len", C.c_uint64), ("null_count", C.c_int64), ("nulls_words", C.c_uint64), ("sorted", C.c_int32), ("bad", C.c_int32)]


def vector_unmarshal_device(src_dev, nbytes, data_dev, area_dev, nulls_dev):
    """Vector.UnmarshalBinary on the device: src_dev holds the marshalled bytes (e.g. straight out of lz4 decode), the sections are copied to the
    aligned DeviceBuffers given.  Returns the VectorView."""
    view = np.zeros(C.sizeof(VectorView), dtype=np.uint8)
    vecs = [Vector(data=view, length=1), Vector(data_ptr=data_dev.ptr, data_nbytes=data_dev.nbytes, length=1),
            Vector(data_ptr=area_dev.ptr, data_nbytes=area_dev.nbytes, length=1) if area_dev is not None else Vector(length=0),
            Vector(data_ptr=nulls_dev.ptr, data_nbytes=nulls_dev.nbytes, length=1) if nulls_dev is not None else Vector(length=0),
            Vector(data_ptr=src_dev.ptr, data_nbytes=nbytes, length=1)]
    xcall(capi.XCALL_VECTOR_UNMARSHAL, vecs, 1)
    return VectorView.from_buffer_copy(view.tobytes())
