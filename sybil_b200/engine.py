"""Host-side mirror of sybil's query interface over the C ABI of libsybilgpu.so.

Names, argument meaning and results follow the reference so that the parity tests
read like src/lib/*_test.go:

    Table.LoadAndQueryRecords(loadSpec, querySpec)   src/lib/table_query.go:18
    Table.IntFilter / StrFilter                      src/lib/filter.go:287-310
    Table.Grouping / Aggregation                     src/lib/query_spec.go:195-235
    QuerySpec / QueryParams / Result                 src/lib/query_spec.go:11-105
    Histogram interface                              src/lib/hist.go:9-25
    FLAGS.OP / LOG_HIST / HIST_BUCKET / TIME_*       src/lib/config.go:30-100

In production this layer is Go (see go/sybilgpu and INTEGRATION.md); the Go
toolchain is not in the build image, so the mirror is Python over ctypes.  All
compute goes through the CUDA library: there is no CPU path here.
"""
import ctypes as C
import re

import numpy as np

from . import _ffi as F


class _Flags:
    """The globals of config.go the hot path reads (config.go:123-176 defaults)."""

    def __init__(self):
        self.reset()

    def reset(self):
        self.OP = "avg"
        self.LOG_HIST = False
        self.HIST_BUCKET = 0
        self.TIME_COL = ""
        self.TIME_BUCKET = 0
        self.LIMIT = 100
        self.WEIGHT_COL = ""  # config.go:81; OPTS.WEIGHT_COL / WEIGHT_COL_ID follow from it (cmd_query.go:317-320)


FLAGS = _Flags()


class SybilGpuError(RuntimeError):
    def __init__(self, status, msg):
        super().__init__("libsybilgpu status %d: %s" % (status, msg))
        self.status = status


_CTX = {}


class Context:
    """sg_ctx: one per process and GPU."""

    def __init__(self, device=0):
        self.lib = F.lib()
        st = C.c_int(0)
        self.h = self.lib.sg_create(device, C.byref(st))
        if st.value != F.SG_OK:
            msg = self.lib.sg_last_error(self.h).decode()
            self.lib.sg_destroy(self.h)
            self.h = None
            raise SybilGpuError(st.value, msg)
        self.device = device

    def err(self):
        return self.lib.sg_last_error(self.h).decode()

    def check(self, rc):
        if rc < 0:
            raise SybilGpuError(rc, self.err())
        return rc

    def sm_count(self):
        return self.lib.sg_device_sm_count(self.h)

    def comm_unique_id(self):
        buf = C.create_string_buffer(128)
        self.check(self.lib.sg_comm_unique_id(self.h, buf))
        return buf.raw

    def comm_init(self, uid, rank, nranks):
        self.check(self.lib.sg_comm_init(self.h, uid, rank, nranks))


def get_context(device=0):
    if device not in _CTX:
        _CTX[device] = Context(device)
    return _CTX[device]


# ---- filters / groupings / aggregations -------------------------------------------
class IntFilter:  # filter.go:143-150
    def __init__(self, Field, FieldId, Op, Value):
        self.Field, self.FieldId, self.Op, self.Value = Field, FieldId, Op, int(Value)


class StrFilter:  # filter.go:152-160
    def __init__(self, Field, FieldId, Op, Value):
        self.Field, self.FieldId, self.Op, self.Value = Field, FieldId, Op, Value
        self.regex = re.compile(Value) if Op in ("re", "nre") else None


class SetFilter:  # filter.go:162-169
    def __init__(self, Field, FieldId, Op, Value):
        self.Field, self.FieldId, self.Op, self.Value = Field, FieldId, Op, Value


class StrReplace:  # config.go:102-105; FLAGS.STR_REPLACE "col:pattern:replacement" (table_query.go:34-50)
    def __init__(self, Pattern, Replace):
        self.Pattern, self.Replace = Pattern, Replace
        self.regex = re.compile(Pattern)
        # Go's Expand template ($1, ${1}, ${name}) as Python's (\g<1>); a literal backslash stays one
        t = Replace.replace("\\", "\\\\")
        t = re.sub(r"\$\{(\w+)\}", r"\\g<\1>", t)
        t = re.sub(r"\$(\d+)", r"\\g<\1>", t)
        self._template = t

    def apply(self, s):  # regexp.ReplaceAllString (column_store_io.go:531)
        return self.regex.sub(self._template, s)


class Grouping:  # query_spec.go:73-76
    def __init__(self, Name, name_id):
        self.Name, self.name_id = Name, name_id


class Aggregation:  # query_spec.go:78-83
    def __init__(self, Name, name_id, Op):
        self.Name, self.name_id, self.Op = Name, name_id, Op
        self.HistType = ""
        if Op == "hist":
            self.HistType = "multi" if FLAGS.LOG_HIST else "basic"


class LoadSpec:  # table_load_spec.go:5-72
    def __init__(self, table):
        self.table = table
        self.columns = {}
        self.files = {}

    def Int(self, name):
        self.columns[name] = True
        self.files["int_" + name + ".db"] = True

    def Str(self, name):
        self.columns[name] = True
        self.files["str_" + name + ".db"] = True

    def Set(self, name):
        self.columns[name] = True
        self.files["set_" + name + ".db"] = True


class Hist:
    """Histogram interface (hist.go:9-25) over the merged counters of one (group, aggregation)."""

    def __init__(self, res, gi, ai):
        self._r, self._gi, self._ai = res, gi, ai
        v = F.sg_hist_view()
        rc = res.lib.sg_result_hist(res.h, gi, ai, C.byref(v))
        if rc != 1:
            raise KeyError("no histogram")
        self.Count, self.ExactSum = v.count, v.sum
        self._min, self._max, self.Avg = v.min, v.max, v.avg
        self.NumBuckets, self.BucketSize = v.num_buckets, v.bucket_size
        self.nsubhists = v.nsubhists
        self.Values = np.ctypeslib.as_array(v.values, (v.nvalues,)).copy() if v.values else np.zeros(0, np.int64)
        # the sg_result is freed when LoadAndQueryRecords returns: derive everything now
        lib, h = res.lib, res.h
        out = (C.c_int64 * 100)()
        n = lib.sg_result_percentiles(h, gi, ai, out)
        self._percentiles = [out[i] for i in range(max(n, 0))]
        self._stddev = lib.sg_result_stddev(h, gi, ai)
        n = lib.sg_result_sparse_buckets(h, gi, ai, None, None, 0)
        e, c = (C.c_int64 * max(n, 1))(), (C.c_int64 * max(n, 1))()
        lib.sg_result_sparse_buckets(h, gi, ai, e, c, n)
        self._buckets = {e[i]: c[i] for i in range(max(n, 0))}
        self._r = None

    def Mean(self):
        return self.Avg

    def TotalCount(self):
        return self.Count

    def Min(self):
        return self._min

    def Max(self):
        return self._max

    def Sum(self):  # exact int64 (the reference's Sum() is int64(Avg*Count), hist_basic.go:97-99)
        return self.ExactSum

    def GetPercentiles(self):
        return list(self._percentiles)

    def StdDev(self):
        return self._stddev

    def GetIntBuckets(self):
        return dict(self._buckets)


class Result:  # query_spec.go:85-93
    def __init__(self):
        self.Hists = {}
        self.GroupByKey = ""
        self.BinaryByKey = ()
        self.Count = 0
        self.Samples = 0


def toResultJSON(r, querySpec):
    """Result.toResultJSON (printer.go:109-152): the dict the reference's -json output holds for one group."""
    res = {}
    for agg in querySpec.Aggregations:
        h = r.Hists.get(agg.Name)
        if FLAGS.OP == "hist":
            inner = {}
            res[agg.Name] = inner
            if h is not None:
                inner["percentiles"] = h.GetPercentiles()
                inner["buckets"] = {str(k): v for k, v in h.GetIntBuckets().items() if v > 0}
                inner["stddev"] = h.StdDev()
                inner["avg"] = h.Mean()
                inner["sum"] = h.Mean() * float(h.TotalCount())
                inner["samples"] = h.TotalCount()
        if FLAGS.OP == "avg":
            res[agg.Name] = h.Mean() if h is not None else None
    group_key = r.GroupByKey.split("\t")
    for i, g in enumerate(querySpec.Groups):
        res[g.Name] = group_key[i]
    res["Count"] = r.Count
    res["Samples"] = r.Samples
    return res


class _ResultHandle:
    def __init__(self, lib, h, owner=None):
        self.lib, self.h, self.owner = lib, h, owner

    def groups(self, aggs, with_total):
        out = []
        n = self.lib.sg_result_num_groups(self.h)
        idx = ([-1] if with_total else []) + list(range(n))
        for gi in idx:
            r = Result()
            kb, kl = C.c_void_p(), C.c_int64()
            self.lib.sg_result_group_key(self.h, gi, C.byref(kb), C.byref(kl))
            r.GroupByKey = C.string_at(kb, kl.value).decode("utf-8", "replace")
            cnt, smp = C.c_int64(), C.c_int64()
            key = (C.c_uint64 * F.SG_MAX_GROUPS)()
            self.lib.sg_result_group(self.h, gi, key, C.byref(cnt), C.byref(smp))
            r.Count, r.Samples = cnt.value, smp.value
            r.BinaryByKey = tuple(key[i] for i in range(F.SG_MAX_GROUPS))
            for ai, a in enumerate(aggs):
                try:
                    r.Hists[a.Name] = Hist(self, gi, ai)
                except KeyError:
                    pass
            out.append(r)
        return out


class QueryParams:  # query_spec.go:25-41
    def __init__(self, Filters=None, Groups=None, Aggregations=None, TimeBucket=0, OrderBy="$COUNT", OrderAsc=False, Limit=0,
                 StrReplace=None):
        self.StrReplace = StrReplace or {}  # column name -> StrReplace (query_spec.go:30)
        self.Filters = Filters or []
        self.Groups = Groups or []
        self.Aggregations = Aggregations or []
        self.TimeBucket = TimeBucket
        self.OrderBy = OrderBy    # "$COUNT" (SORT_COUNT), an aggregation's name, or "" (no sort)
        self.OrderAsc = OrderAsc  # query_spec.go:33
        self.Limit = Limit        # FLAGS.LIMIT (the CLI's default is 100); 0 = every group is materialised


class QuerySpec:  # query_spec.go:60-67
    def __init__(self, params=None, **kw):
        self.QueryParams = params or QueryParams(**kw)
        for k in ("Filters", "Groups", "Aggregations", "TimeBucket", "OrderBy", "OrderAsc", "Limit", "StrReplace"):
            setattr(self, k, getattr(self.QueryParams, k))
        self.Results = {}
        self.TimeResults = {}
        self.Cumulative = None
        self.MatchedCount = 0
        self.Sorted = []
        self.BrokenBlocks = 0
        self.SkippedBlocks = 0
        self.stats = None



def make_query_desc(KeyTable, KeyTypes, IntInfo, qs):
    """sg_query_desc for a QuerySpec + the FLAGS globals (usable without a GPU context)."""
    nf, ng, na = len(qs.Filters), len(qs.Groups), len(qs.Aggregations)
    fl = (F.sg_filter_desc * max(nf, 1))()
    keep = []
    for i, f in enumerate(qs.Filters):
        fl[i].col_slot = f.FieldId
        fl[i].op = F.OPS[f.Op]
        if isinstance(f, IntFilter):
            fl[i].col_type = F.SG_COL_INT
            fl[i].int_value = f.Value
        else:
            fl[i].col_type = F.SG_COL_SET if isinstance(f, SetFilter) else F.SG_COL_STR
            b = f.Value if isinstance(f.Value, bytes) else f.Value.encode()
            keep.append(b)
            fl[i].str_value = b
            fl[i].str_len = len(b)
    gr = (F.sg_group_desc * max(ng, 1))()
    for i, g in enumerate(qs.Groups):
        gr[i].col_slot = g.name_id
        gr[i].col_type = KeyTypes[g.name_id]
    ag = (F.sg_agg_desc * max(na, 1))()
    for i, a in enumerate(qs.Aggregations):
        ag[i].col_slot = a.name_id
        mn, mx = IntInfo.get(a.Name, (0, 0))
        ag[i].info_min, ag[i].info_max = mn, mx
    d = F.sg_query_desc()
    d.abi_version = F.SG_ABI_VERSION
    d.op_mode = F.SG_MODE_HIST if FLAGS.OP == "hist" else F.SG_MODE_AVG
    d.hist_kind = F.SG_HIST_MULTI if FLAGS.LOG_HIST else F.SG_HIST_BASIC
    d.hist_bucket = FLAGS.HIST_BUCKET
    d.nfilters, d.ngroups, d.naggs = nf, ng, na
    d.filters = C.cast(fl, C.POINTER(F.sg_filter_desc))
    d.groups = C.cast(gr, C.POINTER(F.sg_group_desc))
    d.aggs = C.cast(ag, C.POINTER(F.sg_agg_desc))
    d.weight_col_slot = KeyTable[FLAGS.WEIGHT_COL] if FLAGS.WEIGHT_COL else -1
    # SortResults(OrderBy, OrderAsc) (aggregate.go:497-525)
    order = getattr(qs, "OrderBy", "$COUNT")
    if order == "$COUNT":
        d.order_by_agg = F.SG_ORDER_COUNT
    elif not order:
        d.order_by_agg = F.SG_ORDER_NONE
    else:
        names = [a.Name for a in qs.Aggregations]
        if order not in names:
            raise ValueError("OrderBy %r is not one of the query's aggregations" % order)
        d.order_by_agg = names.index(order)
    d.order_asc = 1 if getattr(qs, "OrderAsc", False) else 0
    d.limit = int(getattr(qs, "Limit", 0) or 0)
    d.time_col_slot = -1
    if qs.TimeBucket and FLAGS.TIME_COL:
        d.time_col_slot = KeyTable[FLAGS.TIME_COL]
        d.time_bucket = qs.TimeBucket
        mn, mx = IntInfo.get(FLAGS.TIME_COL, (0, 0))
        d.time_min, d.time_max = mn, mx
    return d, (fl, gr, ag, keep)


class Table:
    """sybil.Table as far as the query path needs it: KeyTable, KeyTypes, IntInfo and the blocks.

    Blocks arrive through add_block() (in sybil they are block directories on disk,
    gob-decoded by the Go host); they are staged once into HBM and stay resident.
    """

    def __init__(self, name, key_table, ctx=None):
        self.Name = name
        self.ctx = ctx or get_context()
        self.lib = self.ctx.lib
        self.KeyTable = {}  # name -> column slot (table.go:10-41)
        self.KeyTypes = {}  # slot -> INT_VAL / STR_VAL
        for slot, (n, typ) in enumerate(key_table):
            self.KeyTable[n] = slot
            self.KeyTypes[slot] = typ
        self.IntInfo = {}  # name -> (Min, Max): table info.db (table_column_info.go:18-24)
        types = (C.c_int32 * len(key_table))(*[t for _, t in key_table])
        self.h = self.lib.sg_table_create(self.ctx.h, len(key_table), types)
        if not self.h:
            raise SybilGpuError(F.SG_ERR_CUDA, self.ctx.err())

    def close(self):
        if self.h:
            self.lib.sg_table_free(self.h)
            self.h = None

    def get_key_id(self, name):
        return self.KeyTable[name]

    def add_block(self, blk):
        d = blk.desc() if hasattr(blk, "desc") else blk
        self.ctx.check(self.lib.sg_table_add_block(self.h, C.byref(d) if not isinstance(d, C._Pointer) else d))

    def LoadBlockFromDir(self, dirname, loadSpec=None):
        """Table.LoadBlockFromDir (table_block_io.go:225-310) for a sybil block directory on disk: gob-decode
        `info.db` and the `int_*.db` / `str_*.db` files the LoadSpec names (all, when None) and stage the
        still-encoded arrays (sybil_b200/blockdir.py; no Go involved).  Returns the SavedBlock."""
        from . import blockdir
        cols = set(loadSpec.columns) if loadSpec is not None else None
        key_table = [(n, self.KeyTypes[s]) for n, s in sorted(self.KeyTable.items(), key=lambda kv: kv[1])]
        blk = blockdir.read_block_dir(dirname, key_table, cols, block_index=int(self.lib.sg_table_num_blocks(self.h)))
        self.add_block(blk)
        return blk

    def add_block_desc_ptr(self, p):
        self.ctx.check(self.lib.sg_table_add_block(self.h, p))

    def add_blocks(self, ptr_array, n):
        """sg_table_add_blocks: ptr_array is a ctypes array of sg_block_desc pointers."""
        self.ctx.check(self.lib.sg_table_add_blocks(self.h, ptr_array, n))

    def sync(self):
        self.ctx.check(self.lib.sg_table_sync(self.h))

    def NumRows(self):
        return self.lib.sg_table_num_rows(self.h)

    def dict_strings(self, name):
        slot = self.KeyTable[name]
        n = self.lib.sg_table_dict_size(self.h, slot)
        out = []
        for i in range(n):
            b, l = C.c_void_p(), C.c_int64()
            self.lib.sg_table_dict_get(self.h, slot, i, C.byref(b), C.byref(l))
            out.append(C.string_at(b, l.value))
        return out

    # filter.go:287-310, query_spec.go:195-235, table_load_spec.go:59-72
    def IntFilter(self, name, op, value):
        return IntFilter(name, self.get_key_id(name), op, value)

    def StrFilter(self, name, op, value):
        return StrFilter(name, self.get_key_id(name), op, value)

    def SetFilter(self, name, op, value):
        return SetFilter(name, self.get_key_id(name), op, value)

    def Grouping(self, name):
        return Grouping(name, self.get_key_id(name))

    def Aggregation(self, name, op):
        return Aggregation(name, self.get_key_id(name), op)

    def NewLoadSpec(self):
        return LoadSpec(self)

    def _desc(self, qs):
        return make_query_desc(self.KeyTable, self.KeyTypes, self.IntInfo, qs)

    def LoadAndQueryRecords(self, loadSpec, querySpec, allreduce=False):
        """Table.LoadAndQueryRecords (table_query.go:18-422).  Returns the matched row count and
        fills querySpec.{Results, TimeResults, Cumulative, MatchedCount, Sorted}."""
        pq = self.Prepare(loadSpec, querySpec)
        try:
            return pq.Run(querySpec, allreduce=allreduce)
        finally:
            pq.Close()

    def Prepare(self, loadSpec, querySpec):
        """The same query as a prepared handle (sg_query_begin once, sg_query_run per Run()): a host that
        repeats a query over an unchanged table keeps the block list, the plan and the uploaded work items."""
        return PreparedQuery(self, loadSpec, querySpec)

    def _fill(self, qs, rp):
        lib = self.lib
        rh = _ResultHandle(lib, rp)
        qs.MatchedCount = lib.sg_result_matched_count(rp)
        qs.BrokenBlocks = lib.sg_result_num_broken(rp)
        qs.SkippedBlocks = lib.sg_result_num_skipped(rp)
        qs.NumGroups = lib.sg_result_num_groups_total(rp)
        if not getattr(qs, "materialize", True):
            # counts only: the full result exists in the library (sg_result); building one
            # Python object per group is harness work the caller asked to skip
            qs.Cumulative, qs.Sorted, qs.Results, qs.TimeResults = None, [], {}, {}
            return
        allg = rh.groups(qs.Aggregations, True)
        qs.Cumulative = allg[0]
        qs.Sorted = allg[1:]
        qs.Results = {r.GroupByKey: r for r in qs.Sorted}
        qs.TimeResults = {}
        for b in range(lib.sg_result_num_time_buckets(rp)):
            tb = lib.sg_result_time_bucket(rp, b)
            sl = _ResultHandle(lib, lib.sg_result_time_slice(rp, b))
            qs.TimeResults[tb] = {r.GroupByKey: r for r in sl.groups(qs.Aggregations, False)}


class PreparedQuery:
    """sg_query handle kept across runs (see Table.Prepare)."""

    def __init__(self, table, loadSpec, qs):
        self.table = table
        lib, ctx = table.lib, table.ctx
        if loadSpec is not None:
            for what, name in ([("filter", f.Field) for f in qs.Filters] + [("group", g.Name) for g in qs.Groups] +
                               [("aggregation", a.Name) for a in qs.Aggregations]):
                if name not in loadSpec.columns:
                    raise ValueError("%s column %r is not in the LoadSpec: sybil would not load it" % (what, name))
        d, self._keep = table._desc(qs)
        # StrReplace (table_query.go:34-50, column_store_io.go:515-549): the strings of a rewritten column are
        # rewritten on the host, once per distinct string; its filters travel as RE / NRE bitsets evaluated on
        # the rewritten strings (sybilgpu.h, sg_query_set_str_replace)
        repl = {name: sr for name, sr in (getattr(qs, "StrReplace", None) or {}).items()
                if name in table.KeyTable and table.KeyTypes[table.KeyTable[name]] == F.SG_COL_STR}
        rewritten = {}
        for name, sr in repl.items():
            rewritten[name] = [sr.apply(s.decode("utf-8", "surrogateescape")).encode("utf-8", "surrogateescape")
                               for s in table.dict_strings(name)]
        fl = self._keep[0]
        for i, f in enumerate(qs.Filters):
            if isinstance(f, StrFilter) and f.Field in repl and f.Op in ("eq", "neq"):
                fl[i].op = F.SG_OP_RE if f.Op == "eq" else F.SG_OP_NRE
        self.q = lib.sg_query_begin(ctx.h, table.h, C.byref(d))
        if not self.q:
            raise SybilGpuError(F.SG_ERR_INVALID, ctx.err())
        try:
            for name, strs in rewritten.items():
                blob = b"".join(strs)
                offs = np.zeros(len(strs) + 1, np.uint32)
                if strs:
                    offs[1:] = np.cumsum([len(x) for x in strs])
                buf = np.frombuffer(blob if blob else b"\0", dtype=np.uint8).copy()
                ctx.check(lib.sg_query_set_str_replace(self.q, table.KeyTable[name], buf.ctypes.data, offs.ctypes.data, len(strs)))
            for i, f in enumerate(qs.Filters):
                if isinstance(f, StrFilter) and (f.regex is not None or f.Field in repl):
                    # the host evaluates the regexp once per distinct string (filter.go:215-237)
                    strs = rewritten[f.Field] if f.Field in repl else table.dict_strings(f.Field)
                    bits = np.zeros((len(strs) + 31) // 32 + 1, np.uint32)
                    lit = f.Value if isinstance(f.Value, bytes) else f.Value.encode()
                    for gid, s in enumerate(strs):
                        hit = f.regex.search(s.decode("utf-8", "replace")) if f.regex is not None else s == lit
                        if hit:
                            bits[gid >> 5] |= np.uint32(1 << (gid & 31))
                    ctx.check(lib.sg_query_set_str_lut(self.q, i, bits.ctypes.data, len(strs)))
        except Exception:
            self.Close()
            raise

    def Run(self, qs, allreduce=False, keep_result=False):
        """One pass of the hot path; fills qs like LoadAndQueryRecords.  The result object is freed before
        the call returns (the Python mirror copies what it exposes), unless keep_result: then it stays alive
        as qs.result (Table._fill materialises it later) and the caller frees it with sg_result_free."""
        t = self.table
        lib, ctx = t.lib, t.ctx
        ctx.check(lib.sg_query_run(self.q))
        if allreduce:
            ctx.check(lib.sg_query_allreduce(self.q))
        rp = C.c_void_p()
        ctx.check(lib.sg_query_finish(self.q, C.byref(rp)))
        st = F.sg_stats()
        lib.sg_query_stats(self.q, C.byref(st))
        qs.stats = st
        try:
            t._fill(qs, rp)
        except BaseException:
            lib.sg_result_free(rp)
            raise
        if keep_result:
            qs.result = rp
        else:
            lib.sg_result_free(rp)
        return qs.MatchedCount

    def Close(self):
        if self.q:
            self.table.lib.sg_query_free(self.q)
            self.q = None
