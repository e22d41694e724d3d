"""Host-side mirror of the reference's public API over the infidex_b200 C-ABI.

Mirrors (names, argument meaning, error behaviour) of /root/reference/src/Infidex:
  SearchEngine.CreateDefault / IndexDocuments / Search      SearchEngine.cs:78-92, 96-106, 256-319
  Query (Text, MaxNumberOfRecordsToReturn, EnableCoverage, EnableFacets, CoverageDepth, Filter)   Api/Query.cs
  Result (Records, Facets, TotalCandidates), ScoreEntry (Score, DocumentId, Tiebreaker)            Api/Result.cs, Core/ScoreEntry.cs
  Document / DocumentFields / Field / Weight                                                       Core/Document.cs, Api/*
  Filter.Parse(...) -> INFISCRIPT-V1 bytecode (Filtering/FilterCompiler.cs, BytecodeSerializer.cs) see filter.py

The search itself runs only in libinfidex_gpu.so (CUDA, sm_100a). There is no CPU fallback: constructing an engine
without the library or without a GPU raises. (`_gpu_lib` is a test hook used by the CPU test-suite to load the
kernel *emulation* build; the package never selects it on its own.)
"""
import ctypes as C
import os

import numpy as np

from . import _build
from .filter import Filter

PKG = os.path.dirname(os.path.abspath(__file__))


class Weight:
    High, Med, Low = 0, 1, 2


class Field:
    def __init__(self, name, value=None, weight=Weight.Med, indexable=True, filterable=False, facetable=False):
        self.Name, self.Value, self.Weight = name, value, weight
        self.Indexable, self.Filterable, self.Facetable = indexable, filterable, facetable


class DocumentFields:
    def __init__(self):
        self._fields = {}

    def AddField(self, name, value=None, weight=Weight.Med, indexable=True, filterable=False, facetable=False):
        f = name if isinstance(name, Field) else Field(name, value, weight, indexable, filterable, facetable)
        self._fields[f.Name] = f
        return self

    def GetFieldList(self):
        return list(self._fields.values())


class Document:
    def __init__(self, documentKey, text_or_fields):
        self.DocumentKey = int(documentKey)
        if isinstance(text_or_fields, DocumentFields):
            self.Fields = text_or_fields
        else:
            self.Fields = DocumentFields().AddField("content", text_or_fields)


class Query:
    def __init__(self, text="", maxNumberOfRecordsToReturn=10):
        self.Text = text
        self.MaxNumberOfRecordsToReturn = maxNumberOfRecordsToReturn
        self.EnableCoverage = True
        self.EnableFacets = False
        self.CoverageDepth = 500
        self.Filter = None


class ScoreEntry:
    __slots__ = ("Score", "DocumentId", "Tiebreaker")

    def __init__(self, score, key, tie):
        self.Score, self.DocumentId, self.Tiebreaker = float(score), int(key), int(tie)

    def __repr__(self):
        return "ScoreEntry(Score=%r, DocumentId=%d, Tiebreaker=%d)" % (self.Score, self.DocumentId, self.Tiebreaker)


class Result:
    def __init__(self, records, facets, total, status=0):
        self.Records, self.Facets, self.TotalCandidates, self.Status = records, facets, total, status


# ---- ctypes structures (include/infidex_gpu.h) ----------------------------------------------------------------------
class _Strings(C.Structure):
    _fields_ = [("chars", C.c_void_p), ("off", C.c_void_p), ("n", C.c_int32)]


class _Query(C.Structure):
    _fields_ = [("text", C.c_void_p), ("len", C.c_int32), ("max_results", C.c_int32), ("coverage_depth", C.c_int32),
                ("enable_coverage", C.c_int32), ("filter_id", C.c_int32), ("enable_facets", C.c_int32)]


class _BatchResult(C.Structure):
    _fields_ = [("cap", C.c_int32), ("facet_cap", C.c_int32), ("doc_key", C.c_void_p), ("score", C.c_void_p), ("tie", C.c_void_p),
                ("n", C.c_void_p), ("total_candidates", C.c_void_p), ("status", C.c_void_p), ("facet_column", C.c_void_p),
                ("facet_value", C.c_void_p), ("facet_count", C.c_void_p), ("n_facets", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("ms_total", C.c_float), ("ms_prepare", C.c_float), ("ms_expand", C.c_float), ("ms_stage1", C.c_float),
                ("ms_wordmatch", C.c_float), ("ms_stage2", C.c_float), ("ms_final", C.c_float), ("algo_bytes_stage1", C.c_int64),
                ("kernel_launches", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64), ("s1_query_ms_max", C.c_float), ("s1_query_ms_sum", C.c_float),
                ("ms_s1_select", C.c_float), ("ms_s1_score_warp", C.c_float), ("ms_s1_score_cta", C.c_float), ("ms_s1_finish", C.c_float),
                ("s1_light", C.c_int32), ("s1_heavy", C.c_int32), ("s1_waves", C.c_int32), ("s1_mid", C.c_int32), ("s1_pool_bytes", C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class _Params(C.Structure):
    _fields_ = [("stop_term_limit", C.c_int32), ("device", C.c_int32), ("max_batch", C.c_int32), ("reserved", C.c_int32)]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def pack_strings(strs):
    enc = [s.encode("utf-16-le", "surrogatepass") for s in strs]
    offs = np.zeros(len(enc) + 1, np.int64)
    if enc:
        np.cumsum([len(e) // 2 for e in enc], out=offs[1:])
    blob = np.frombuffer(b"".join(enc), dtype=np.uint16).copy() if offs[-1] else np.zeros(1, np.uint16)
    return blob, offs


class NativeError(RuntimeError):
    pass


def _load_host():
    lib = C.CDLL(_build.build_host())
    lib.ifx_builder_create.restype = C.c_void_p
    lib.ifx_builder_image.restype = C.c_void_p
    return lib


def _load_gpu(path=None):
    path = path or _build.GPU_LIB
    if not os.path.exists(path):
        raise NativeError("libinfidex_gpu.so is not built (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                          "infidex_b200 has no CPU fallback")
    lib = C.CDLL(path)
    lib.ifx_last_error.restype = C.c_char_p
    return lib


class SearchEngine:
    """Drop-in for the reference's SearchEngine (config 400 = CreateDefault)."""

    def __init__(self, device=0, _gpu_lib=None):
        self._host = _load_host()
        self._gpu = _load_gpu(_gpu_lib)
        self._device = device
        self._builder = None
        self._index = C.c_void_p()
        self._schema = None
        self._filters = {}
        self._columns = []      # (name, dict strings) of filter / facet columns, image order
        self._is_indexed = False

    @staticmethod
    def CreateDefault(device=0, _gpu_lib=None):
        return SearchEngine(device, _gpu_lib)

    def __del__(self):
        try:
            self.Dispose()
        except Exception:
            pass

    def Dispose(self):
        if self._index:
            self._gpu.ifx_index_destroy(self._index); self._index = C.c_void_p()
        if self._builder:
            self._host.ifx_builder_destroy(C.c_void_p(self._builder)); self._builder = None

    def _check(self, rc, what):
        if rc != 0:
            raise NativeError("%s failed (%d): %s" % (what, rc, (self._gpu.ifx_last_error() or b"").decode()))

    # ---- indexing ---------------------------------------------------------------------------------------------------
    def IndexDocuments(self, documents):
        docs = list(documents)
        if not docs:
            return
        fields = docs[0].Fields.GetFieldList()      # schema = DocumentFields of the first document (SearchEngine.cs:139-140)
        names = [f.Name for f in fields]
        cols = []
        for f in fields:
            vals = [d.Fields._fields[f.Name].Value if f.Name in d.Fields._fields else None for d in docs]
            if all(isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in vals):
                cols.append(np.array(vals, np.int64))
            elif all(isinstance(v, (float, np.floating)) for v in vals):
                cols.append(np.array(vals, np.float64))
            else:
                cols.append(["" if v is None else str(v) for v in vals])
        self.IndexColumns(np.array([d.DocumentKey for d in docs], np.int64), fields, cols)

    def IndexColumns(self, keys, schema, columns, threads=None, upload=True):
        """Bulk form of IndexDocuments: schema = list[Field] (values ignored), columns[f] = list[str] | int64[] | float64[].
        upload=False stops after the host builder (image_ptr() is valid, no device is touched)."""
        self.Dispose()
        n = len(keys)
        keys = np.ascontiguousarray(keys, np.int64)
        nb, no = pack_strings([f.Name for f in schema])
        w = np.array([f.Weight for f in schema], np.int32)
        fl = np.array([(1 if f.Indexable else 0) | (2 if f.Filterable else 0) | (4 if f.Facetable else 0) for f in schema], np.int32)
        self._builder = self._host.ifx_builder_create(len(schema), _p(nb), _p(no.astype(np.int32)), _p(w), _p(fl))
        self._add_columns(keys, columns)
        self._finish(schema, threads, upload)

    def _add_columns(self, keys, columns):
        n = len(keys)
        kinds = np.zeros(len(columns), np.int32)
        keep, cptr, optr = [], (C.c_void_p * len(columns))(), (C.c_void_p * len(columns))()
        for i, col in enumerate(columns):
            if isinstance(col, np.ndarray) and col.dtype.kind in "iu":
                a = np.ascontiguousarray(col, np.int64); kinds[i] = 2; cptr[i] = a.ctypes.data; keep.append(a)
            elif isinstance(col, np.ndarray) and col.dtype.kind == "f":
                a = np.ascontiguousarray(col, np.float64); kinds[i] = 3; cptr[i] = a.ctypes.data; keep.append(a)
            elif isinstance(col, tuple):          # pre-packed (uint16 blob, int64 offsets)
                blob, o = col; kinds[i] = 1; cptr[i] = blob.ctypes.data; optr[i] = o.ctypes.data; keep += [blob, o]
            else:
                blob, o = pack_strings(col); kinds[i] = 1; cptr[i] = blob.ctypes.data; optr[i] = o.ctypes.data; keep += [blob, o]
        rc = self._host.ifx_builder_add_docs(C.c_void_p(self._builder), n, _p(keys), _p(kinds), cptr, optr)
        if rc:
            raise NativeError("ifx_builder_add_docs failed")

    def _finish(self, schema, threads=None, upload=True):
        self._host.ifx_builder_finish(C.c_void_p(self._builder), threads or max(1, min(len(os.sched_getaffinity(0)), 64)))
        img = self._host.ifx_builder_image(C.c_void_p(self._builder))
        self._schema = list(schema)
        self._columns = []
        buf = np.zeros(4096, np.uint16); b = C.c_void_p(self._builder)
        for c in range(self._host.ifx_builder_num_columns(b)):
            n = self._host.ifx_builder_column_name(b, c, _p(buf), len(buf)); self._columns.append(buf[:n].tobytes().decode("utf-16-le"))
        if upload:
            self._upload(img)

    def IndexChunks(self, schema, chunks, threads=None):
        """Streaming form of IndexColumns for corpora that do not fit one numpy batch: `chunks` yields (keys, columns)."""
        self.Dispose()
        nb, no = pack_strings([f.Name for f in schema])
        w = np.array([f.Weight for f in schema], np.int32)
        fl = np.array([(1 if f.Indexable else 0) | (2 if f.Filterable else 0) | (4 if f.Facetable else 0) for f in schema], np.int32)
        self._builder = self._host.ifx_builder_create(len(schema), _p(nb), _p(no.astype(np.int32)), _p(w), _p(fl))
        for keys, columns in chunks:
            self._add_columns(np.ascontiguousarray(keys, np.int64), columns)
        self._finish(schema, threads)

    def image_ptr(self):
        return self._host.ifx_builder_image(C.c_void_p(self._builder))

    def _upload(self, img_ptr):
        params = _Params(); self._gpu.ifx_params_default(C.byref(params)); params.device = self._device
        idx = C.c_void_p()
        self._check(self._gpu.ifx_index_create(C.c_void_p(img_ptr), C.byref(params), C.byref(idx)), "ifx_index_create")
        self._index = idx
        self._is_indexed = True
        self._filters = {}

    # ---- searching --------------------------------------------------------------------------------------------------
    def _prep_text(self, text):
        a = np.frombuffer(text.encode("utf-16-le", "surrogatepass"), np.uint16) if text else np.zeros(0, np.uint16)
        out = np.zeros(max(len(a), 1), np.uint16)
        n = self._host.ifx_host_prepare_query(_p(np.ascontiguousarray(a)), len(a), _p(out), len(out))
        return out[:n]

    def _filter_id(self, flt):
        if flt is None:
            return -1
        code = flt.bytecode() if isinstance(flt, Filter) else bytes(flt)
        if code not in self._filters:
            if isinstance(flt, Filter):
                # The reference's VM reads any field of the document (FilterVM.cs:160-165); the device only holds columns for fields
                # flagged Filterable or Facetable. A filter on another schema field must fail loudly, not evaluate to "no match".
                have = {c.lower() for c in self._columns}
                missing = sorted(f for f in flt.fields() if f.lower() not in have and any(f.lower() == x.Name.lower() for x in self._schema))
                if missing:
                    raise ValueError("filter uses field(s) %s that are neither Filterable nor Facetable in the schema: no device column exists for them" % missing)
            fid = C.c_int(-1); buf = np.frombuffer(code, np.uint8).copy()
            self._check(self._gpu.ifx_filter_register(self._index, _p(buf), C.c_size_t(len(buf)), C.byref(fid)), "ifx_filter_register")
            self._filters[code] = fid.value
        return self._filters[code]

    def _pack_queries(self, queries):
        texts = [self._prep_text(q.Text) for q in queries]
        arr = (_Query * len(queries))()
        for i, q in enumerate(queries):
            arr[i].text = texts[i].ctypes.data if len(texts[i]) else None
            arr[i].len = len(texts[i]); arr[i].max_results = q.MaxNumberOfRecordsToReturn; arr[i].coverage_depth = q.CoverageDepth
            arr[i].enable_coverage = int(q.EnableCoverage); arr[i].filter_id = self._filter_id(q.Filter); arr[i].enable_facets = int(q.EnableFacets)
        return arr, texts

    def PackBatch(self, queries, facet_cap=0):
        """Host-side marshalling of a batch (what the C# shim does with `fixed` pointers): returns a reusable call object."""
        nq = len(queries)
        arr, keep = self._pack_queries(queries)
        cap = max(1, max(q.MaxNumberOfRecordsToReturn for q in queries))
        fc = facet_cap or (256 if any(q.EnableFacets for q in queries) else 0)
        out = _BatchResult(); out.cap = cap; out.facet_cap = fc
        bufs = dict(keys=np.zeros((nq, cap), np.int64), scores=np.zeros((nq, cap), np.float32), ties=np.zeros((nq, cap), np.uint8),
                    n=np.zeros(nq, np.int32), total=np.zeros(nq, np.int32), status=np.zeros(nq, np.int32),
                    fcol=np.zeros((nq, max(fc, 1)), np.int32), fval=np.zeros((nq, max(fc, 1)), np.int32), fcnt=np.zeros((nq, max(fc, 1)), np.int32), nf=np.zeros(nq, np.int32))
        out.doc_key, out.score, out.tie, out.n, out.total_candidates, out.status = _p(bufs["keys"]), _p(bufs["scores"]), _p(bufs["ties"]), _p(bufs["n"]), _p(bufs["total"]), _p(bufs["status"])
        out.facet_column, out.facet_value, out.facet_count, out.n_facets = _p(bufs["fcol"]), _p(bufs["fval"]), _p(bufs["fcnt"]), _p(bufs["nf"])
        return {"arr": arr, "keep": keep, "nq": nq, "out": out, "bufs": bufs}

    def SearchPacked(self, packed, stats=None):
        """The bare C-ABI call ifx_search_batch on pre-marshalled host buffers (host -> device -> host)."""
        st = stats if stats is not None else Stats()
        self._check(self._gpu.ifx_search_batch(self._index, packed["arr"], packed["nq"], C.byref(packed["out"]), C.byref(st)), "ifx_search_batch")
        return st

    def SearchBatch(self, queries, stats=None, facet_cap=0):
        """Batch form of Search: one C-ABI call for all queries (host buffers in, host buffers out)."""
        if not self._is_indexed:
            return [Result([], None, 0) for _ in queries]
        nq = len(queries)
        arr, keep = self._pack_queries(queries)
        cap = max(1, max(q.MaxNumberOfRecordsToReturn for q in queries))
        fc = facet_cap or (256 if any(q.EnableFacets for q in queries) else 0)
        out = _BatchResult(); out.cap = cap; out.facet_cap = fc
        keys = np.zeros((nq, cap), np.int64); scores = np.zeros((nq, cap), np.float32); ties = np.zeros((nq, cap), np.uint8)
        n = np.zeros(nq, np.int32); total = np.zeros(nq, np.int32); status = np.zeros(nq, np.int32)
        fcol = np.zeros((nq, max(fc, 1)), np.int32); fval = np.zeros((nq, max(fc, 1)), np.int32); fcnt = np.zeros((nq, max(fc, 1)), np.int32); nf = np.zeros(nq, np.int32)
        out.doc_key, out.score, out.tie, out.n, out.total_candidates, out.status = _p(keys), _p(scores), _p(ties), _p(n), _p(total), _p(status)
        out.facet_column, out.facet_value, out.facet_count, out.n_facets = _p(fcol), _p(fval), _p(fcnt), _p(nf)
        st = stats if stats is not None else Stats()
        self._check(self._gpu.ifx_search_batch(self._index, arr, nq, C.byref(out), C.byref(st)), "ifx_search_batch")
        self.last_raw = (keys, scores, ties, n, total, status)
        res = []
        for i in range(nq):
            recs = [ScoreEntry(scores[i, k], keys[i, k], ties[i, k]) for k in range(n[i])]
            facets = None
            if queries[i].EnableFacets:
                facets = {}
                for k in range(nf[i]):
                    facets.setdefault(self._columns[int(fcol[i, k])], []).append((self._facet_value(int(fcol[i, k]), int(fval[i, k])), int(fcnt[i, k])))
            res.append(Result(recs, facets, int(total[i]), int(status[i])))
        return res

    def _facet_value(self, col, vid):
        buf = np.zeros(1024, np.uint16)
        n = self._host.ifx_builder_column_value(C.c_void_p(self._builder), col, vid, _p(buf), len(buf))
        return buf[:n].tobytes().decode("utf-16-le", "surrogatepass")

    def Search(self, query):
        if isinstance(query, str):
            query = Query(query)
        return self.SearchBatch([query])[0]

    # ---- device-resident batches (bench `value`: inputs already in HBM when the timed region starts) -----------------
    def UploadBatch(self, queries):
        arr, keep = self._pack_queries(queries)
        h = C.c_void_p()
        self._check(self._gpu.ifx_batch_upload(self._index, arr, len(queries), C.byref(h)), "ifx_batch_upload")
        return h

    def RunBatch(self, handle, stats=None):
        st = stats if stats is not None else Stats()
        self._check(self._gpu.ifx_batch_run(handle, C.byref(st)), "ifx_batch_run")
        return st

    def DownloadBatch(self, handle, nq, cap):
        """Records of the last RunBatch on `handle` (ifx_batch_download): doc_key / score / tie [nq, cap], n / total_candidates / status [nq].
        `cap` >= the batch's largest MaxNumberOfRecordsToReturn. Row q holds n[q] records; the slots after them are undefined. An uploaded
        batch has no facet capacity, so there are no facet tables to read back."""
        out = _BatchResult(); out.cap = cap; out.facet_cap = 0
        bufs = dict(doc_key=np.zeros((nq, cap), np.int64), score=np.zeros((nq, cap), np.float32), tie=np.zeros((nq, cap), np.uint8),
                    n=np.zeros(nq, np.int32), total_candidates=np.zeros(nq, np.int32), status=np.zeros(nq, np.int32))
        out.doc_key, out.score, out.tie = _p(bufs["doc_key"]), _p(bufs["score"]), _p(bufs["tie"])
        out.n, out.total_candidates, out.status = _p(bufs["n"]), _p(bufs["total_candidates"]), _p(bufs["status"])
        self._check(self._gpu.ifx_batch_download(handle, C.byref(out)), "ifx_batch_download")
        return bufs

    def FreeBatch(self, handle):
        self._gpu.ifx_batch_free(handle)

    def FlushL2(self):
        self._check(self._gpu.ifx_flush_l2(self._index), "ifx_flush_l2")

    def Stage1Batch(self, texts, depth=500, stats=None):
        """Stage-1 (BM25 backbone) lists for a batch: (keys[nq,depth], scores[nq,depth], n[nq], status[nq])."""
        queries = [Query(t) for t in texts]
        arr, keep = self._pack_queries(queries)
        nq = len(queries)
        keys = np.zeros((nq, depth), np.int64); scores = np.zeros((nq, depth), np.float32); n = np.zeros(nq, np.int32); status = np.zeros(nq, np.int32)
        st = stats if stats is not None else Stats()
        self._check(self._gpu.ifx_stage1_batch(self._index, arr, nq, depth, _p(keys), _p(scores), _p(n), _p(status), C.byref(st)), "ifx_stage1_batch")
        return keys, scores, n, status
