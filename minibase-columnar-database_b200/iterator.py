"""Mirror of the reference's ``iterator`` package for the columnar scan path: the CondExpr/FldSpec
predicate and projection structures and the ColumnarFileScan operator, same names and argument meaning
as minijava/src/iterator/*.java.  The operator's work (TupleScan -> PredEval -> Projection per row in the
reference) is one fused GPU scan through the C ABI; ``get_next()`` then slices the result.
"""
from __future__ import annotations

from typing import Optional, Sequence

import numpy as np

from . import _native as N
from .engine import Term
from .global_ import AttrOperator, AttrType, IndexType, SystemDefs, TID
from .heap import Tuple


# ---- exceptions (chainexception/ChainException.java: every checked exception carries `prev`) ----------
class ChainException(Exception):
    def __init__(self, prev: Optional[BaseException] = None, msg: str = ""):
        super().__init__(msg)
        self.prev = prev


class FileScanException(ChainException):
    pass


class TupleUtilsException(ChainException):
    pass


class InvalidRelation(ChainException):
    def __init__(self, msg: str = ""):
        super().__init__(None, msg)


class PredEvalException(ChainException):
    pass


class UnknowAttrType(ChainException):
    pass


class WrongPermat(ChainException):
    def __init__(self, msg: str = ""):
        super().__init__(None, msg)


class IndexException(ChainException):
    pass


class NestedLoopException(ChainException):
    pass


# ---- predicate / projection structures -----------------------------------------------------------------
class RelSpec:
    """iterator/RelSpec.java:3-16"""
    outer, innerRel = 0, 1

    def __init__(self, key: int):
        self.key = key


class FldSpec:
    """iterator/FldSpec.java:4-17: (relation, 1-based field offset)"""

    def __init__(self, relation: RelSpec, offset: int):
        self.relation = relation
        self.offset = offset


class Operand:
    """iterator/Operand.java:5-10"""

    def __init__(self):
        self.symbol: Optional[FldSpec] = None
        self.string: Optional[str] = None
        self.integer: int = 0
        self.real: float = 0.0


class CondExpr:
    """iterator/CondExpr.java:12-57.  A CondExpr[] is a CNF: the array (None-terminated) is AND, the
    ``next`` chain of one element is OR (iterator/PredEval.java:51-54,164-176)."""

    def __init__(self):
        self.op = AttrOperator(AttrOperator.aopNOP)
        self.type1: Optional[AttrType] = None
        self.type2: Optional[AttrType] = None
        self.operand1 = Operand()
        self.operand2 = Operand()
        self.next: Optional["CondExpr"] = None
        self.indexType = IndexType(IndexType.None_)


def _operand_spec(t: AttrType, o: Operand) -> tuple:
    if t.attrType == AttrType.attrSymbol:
        kind = "col" if o.symbol.relation.key == RelSpec.outer else "icol"
        return (kind, o.symbol.offset - 1)                     # symbol.offset is 1-based (PredEval.java:79-91)
    if t.attrType == AttrType.attrInteger:
        return ("int", o.integer)
    if t.attrType == AttrType.attrReal:
        return ("real", o.real)
    if t.attrType == AttrType.attrString:
        return ("str", o.string)
    raise UnknowAttrType(None, "Don't know how to handle attrSymbol, attrNull")


def flatten_condexpr(p: Optional[Sequence[Optional[CondExpr]]]) -> list[Term]:
    """CondExpr[] -> flat term list for the C ABI (conjunct id = array index)."""
    terms: list[Term] = []
    if p is None:
        return terms                                            # p == null: every row qualifies (PredEval.java:46-49)
    for i, head in enumerate(p):
        if head is None:
            break                                               # the array is None-terminated
        cur = head
        while cur is not None:
            terms.append(Term(cur.op.attrOperator, _operand_spec(cur.type1, cur.operand1),
                              _operand_spec(cur.type2, cur.operand2), i))
            cur = cur.next
    return terms


def setup_op_tuple(Jtuple: Tuple, res_attrs: list, in1: Sequence[AttrType], len_in1: int, t1_str_sizes: Sequence[int],
                   proj_list: Sequence[FldSpec], nOutFlds: int) -> list[int]:
    """iterator/TupleUtils.java:295-341: output tuple header of a single-relation projection."""
    sizes = [0] * len_in1
    c = 0
    for i in range(len_in1):
        if in1[i].attrType == AttrType.attrString:
            sizes[i] = t1_str_sizes[c]
            c += 1
    for i in range(nOutFlds):
        if proj_list[i].relation.key != RelSpec.outer:
            raise InvalidRelation("Invalid relation -innerRel")
        res_attrs[i] = AttrType(in1[proj_list[i].offset - 1].attrType)
    res_str_sizes = [sizes[proj_list[i].offset - 1] for i in range(nOutFlds)
                     if in1[proj_list[i].offset - 1].attrType == AttrType.attrString]
    try:
        Jtuple.setHdr(nOutFlds, res_attrs, res_str_sizes)
    except Exception as e:
        raise TupleUtilsException(e, "setHdr() failed")
    return res_str_sizes


class Iterator:
    """iterator/Iterator.java:12-61"""

    def __init__(self):
        self.closeFlag = False

    def get_next(self):
        raise NotImplementedError

    def close(self):
        raise NotImplementedError


class _ResultCursor:
    """Slices an engine Result into reference Tuples, reusing ONE Jtuple like the Java iterators do."""

    def __init__(self, result, out_types: Sequence[AttrType], jtuple: Tuple, whole_fields: bool = False, str_sizes=()):
        self.result = result
        self.jtuple = jtuple
        self.whole_fields = whole_fields        # Tuple.setFld of the stored record: the whole slot is rewritten
        self.str_sizes = list(str_sizes)        # declared width of every output field (0 for numbers)
        self.types = [t.attrType for t in out_types]
        self.positions = result.positions()
        self.cols = [result.column(i) for i in range(len(self.types))]
        self.i = 0

    def next_tuple(self) -> Optional[Tuple]:
        if self.i >= len(self.positions):
            return None
        k = self.i
        self.i += 1
        if self.whole_fields:
            import struct
            for f, t in enumerate(self.types):                 # Jtuple.setFld(j, record bytes) (ColumnarColumnScan.java:167)
                if t == AttrType.attrInteger:
                    self.jtuple.setFld(f + 1, struct.pack(">i", int(self.cols[f][k])))
                elif t == AttrType.attrReal:
                    self.jtuple.setFld(f + 1, struct.pack(">f", float(self.cols[f][k])))
                else:
                    b = bytes(self.cols[f][k]).rstrip(b"\0")
                    self.jtuple.setFld(f + 1, struct.pack(">H", len(b)) + b.ljust(self.str_sizes[f], b"\0"))
            return self.jtuple
        for f, t in enumerate(self.types):                     # Projection.Project (:103-144)
            if t == AttrType.attrInteger:
                self.jtuple.setIntFld(f + 1, int(self.cols[f][k]))
            elif t == AttrType.attrReal:
                self.jtuple.setFloFld(f + 1, float(self.cols[f][k]))
            else:
                self.jtuple.setStrFld(f + 1, bytes(self.cols[f][k]).rstrip(b"\0").decode("utf-8"))
        return self.jtuple

    def next_position(self) -> Optional[int]:
        if self.i >= len(self.positions):
            return None
        self.i += 1
        return int(self.positions[self.i - 1])


class ColumnarFileScan(Iterator):
    """iterator/ColumnarFileScan.java:19-219.

    ColumnarFileScan(file_name, in1, s1_sizes, len_in1, n_out_flds, proj_list, outFilter)   (:51)
    ColumnarFileScan(file_name, in1, s1_sizes, len_in1, outFilter)                          (:102, tid-only / delete query)

    The scan runs on the GPU when the first row is asked for; rows come back in ascending position order
    exactly as TupleScan produces them, deleted rows skipped (columnar/TupleScan.java:85)."""

    def __init__(self, file_name: str, in1: Sequence[AttrType], s1_sizes: Sequence[int], len_in1: int, *rest):
        super().__init__()
        from .columnar import Columnarfile
        if len(rest) == 3:
            n_out_flds, proj_list, outFilter = rest
            self.deleteQuery = False
        elif len(rest) == 1:
            (outFilter,) = rest
            n_out_flds, proj_list = 0, []
            self.deleteQuery = True
        else:
            raise TypeError("ColumnarFileScan(file_name, in1, s1_sizes, len_in1, [n_out_flds, proj_list,] outFilter)")
        self._in1, self.in1_len, self.s_sizes = list(in1), len_in1, list(s1_sizes)
        self.OutputFilter = outFilter
        self.perm_mat = list(proj_list)
        self.nOutFlds = n_out_flds
        self.Jtuple = Tuple()
        self._out_types: list = [None] * n_out_flds
        if not self.deleteQuery:
            setup_op_tuple(self.Jtuple, self._out_types, self._in1, len_in1, self.s_sizes, self.perm_mat, n_out_flds)
        try:
            self.f = Columnarfile(file_name)                    # ColumnarFileScan.java:84-91
        except Exception as e:
            raise FileScanException(e, "Create new heapfile failed")
        if self.f.numColumns != len_in1 or any(a.attrType != b.attrType for a, b in zip(self.f.attrTypes, self._in1)):
            raise FileScanException(None, "openTupleScan() failed")
        self._cursor: Optional[_ResultCursor] = None
        self._result = None

    def show(self):
        return self.perm_mat

    def _open(self) -> _ResultCursor:
        if self._cursor is None:
            try:
                terms = flatten_condexpr(self.OutputFilter)
                proj = [fs.offset - 1 for fs in self.perm_mat]
                self._result = self.f.table.scan(terms, proj=proj, want=N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_HOST)
            except N.MbcError as e:
                raise PredEvalException(e, "TupleUtilsException is caught by PredEval.java")
            self._cursor = _ResultCursor(self._result, self._out_types, self.Jtuple)
        return self._cursor

    def get_next(self) -> Optional[Tuple]:
        return self._open().next_tuple()

    def get_next_tid(self) -> Optional[TID]:
        pos = self._open().next_position()
        return None if pos is None else TID(self.in1_len, pos)

    # what ColumnarNestedLoopJoins needs from an input iterator: its predicate over TABLE columns and the table column
    # behind every field of its output tuple
    def _table_terms(self) -> list:
        return flatten_condexpr(self.OutputFilter)

    def _tuple_columns(self) -> list:
        return [fs.offset - 1 for fs in self.perm_mat]

    def close(self) -> None:
        if not self.closeFlag:
            if self._result is not None:
                self._result.close()
            self._cursor = self._result = None
            self.closeFlag = True

    def restart(self) -> None:
        if self._result is not None:
            self._result.close()
        self._cursor = self._result = None

    def getTupleSize(self) -> int:
        return self.Jtuple.size()

    # ---- extensions the reference does not have (SURVEY.md F5): aggregates over the qualifying set ----
    def aggregate(self, specs: Sequence[tuple]) -> list:
        """specs = [(kind, col)], kind in {COUNT 0, SUM 1, MIN 2, MAX 3}, col 0-based.  Returns (value, valid)."""
        res = self.f.table.scan(flatten_condexpr(self.OutputFilter), want=N.WANT_AGG, aggs=specs)
        out = []
        for a, (kind, col) in enumerate(specs):
            i, f, v = res.agg(a)
            integral = kind == N.AGG_COUNT or self.f.attrTypes[col].attrType == AttrType.attrInteger
            out.append((i if integral else f, v))
        res.close()
        return out

    def group_aggregate(self, key_fields: Sequence[int], specs: Sequence[tuple]) -> list:
        """GROUP BY the 0-based columns key_fields over the rows OutputFilter selects; specs as in aggregate().  Returns
        one (key values..., aggregate values...) tuple per group, groups in ascending key order: ints and COUNT / integer
        aggregates as int, reals as float, strings as str."""
        res = self.f.table.group_aggregate(flatten_condexpr(self.OutputFilter), list(key_fields), aggs=specs)
        try:
            keys = []
            for k, col in enumerate(key_fields):
                vals = res.column(k)
                if self.f.attrTypes[col].attrType == AttrType.attrString:
                    keys.append([bytes(r).split(b"\0", 1)[0].decode("utf-8") for r in vals])
                else:
                    keys.append(vals.tolist())
            aggs = []
            for a, (kind, col) in enumerate(specs):
                i, f = res.group_agg(a)
                integral = kind == N.AGG_COUNT or self.f.attrTypes[col].attrType == AttrType.attrInteger
                aggs.append(i.tolist() if integral else f.tolist())
            return [tuple(k[g] for k in keys) + tuple(a[g] for a in aggs) for g in range(res.count)]
        finally:
            res.close()

    def top_k(self, key_fields: Sequence[int], k: int, descending: bool = False) -> list:
        """ORDER BY the 0-based columns key_fields LIMIT k over the rows OutputFilter selects: one (position, (projected
        field values...)) pair per row in key order, ties by ascending position; the fields are those of perm_mat, ints
        as int, reals as float, strings as str."""
        cols = [fs.offset - 1 for fs in self.perm_mat]
        res = self.f.table.top_k(flatten_condexpr(self.OutputFilter), list(key_fields), k, descending, proj=cols)
        try:
            fields = []
            for i, col in enumerate(cols):
                vals = res.column(i)
                if self.f.attrTypes[col].attrType == AttrType.attrString:
                    fields.append([bytes(r).split(b"\0", 1)[0].decode("utf-8") for r in vals])
                else:
                    fields.append(vals.tolist())
            return [(int(p), tuple(f[g] for f in fields)) for g, p in enumerate(res.positions().tolist())]
        finally:
            res.close()


class _ColumnsScan(Iterator):
    """Shared body of ColumnarColumnScan / ColumnarColumnsScan (SURVEY.md 8f rank 1): the predicate is evaluated over a
    tuple of the scanned columns only (CondExpr field k = the k-th scanned column), the output fields are fetched by
    position from the columns `out_indexes`; deleted rows are skipped (columnar/ColumnScan.java getNext).  Same GPU
    scan as ColumnarFileScan: the filter pass reads only the compared columns, the write pass gathers the rest."""

    def __init__(self, columnarfile, colNos: Sequence[int], rest: tuple, usage: str):
        super().__init__()
        if len(rest) == 4:
            n_out_flds, out_indexes, proj_list, outFilter = rest
            self.deleteQuery = False
        elif len(rest) == 1:                                    # "Only use for delete query": positions only
            (outFilter,) = rest
            n_out_flds, out_indexes, proj_list = 0, [], []
            self.deleteQuery = True
        else:
            raise TypeError(usage)
        self.f = columnarfile
        self.colNos = [int(c) for c in colNos]
        self._in1 = columnarfile.getAttributeTypes()
        self.in1_len = columnarfile.getFieldCount()
        self.s_sizes = columnarfile.getStringSizes()
        if any(c < 0 or c >= self.in1_len for c in self.colNos):
            raise FileScanException(None, "openTupleScan() failed")
        self.OutputFilter = outFilter
        self.perm_mat = list(proj_list)
        self.nOutFlds = n_out_flds
        self.outIndexes = [int(i) for i in out_indexes]
        self.Jtuple = Tuple()
        self._out_types: list = [None] * n_out_flds
        if not self.deleteQuery:
            setup_op_tuple(self.Jtuple, self._out_types, self._in1, self.in1_len, self.s_sizes, self.perm_mat, n_out_flds)
        self.destType = [self._in1[c] for c in self.colNos]     # the predicate tuple's field types
        self._cursor: Optional[_ResultCursor] = None
        self._result = None

    def show(self):
        return self.perm_mat

    def _table_terms(self) -> list:
        terms = []
        for t in flatten_condexpr(self.OutputFilter):           # field k of the predicate tuple -> table column colNos[k]
            ops = []
            for kind, val in (t.lhs, t.rhs):
                if kind == "col":
                    if not 0 <= val < len(self.colNos):
                        raise PredEvalException(None, "FieldNumberOutOfBoundException is caught by PredEval.java")
                    val = self.colNos[val]
                ops.append((kind, val))
            terms.append(Term(t.op, ops[0], ops[1], t.conj))
        return terms

    def _tuple_columns(self) -> list:
        return list(self.outIndexes)

    def getTupleSize(self) -> int:
        return self.Jtuple.size()

    def _open(self) -> _ResultCursor:
        if self._cursor is None:
            terms = self._table_terms()
            try:
                self._result = self.f.table.scan(terms, proj=self.outIndexes, want=N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_HOST)
            except N.MbcError as e:
                raise PredEvalException(e, "TupleUtilsException is caught by PredEval.java")
            sizes = self.f.getAttrSizes()
            self._cursor = _ResultCursor(self._result, self._out_types, self.Jtuple, whole_fields=True,
                                         str_sizes=[sizes[i] if self._in1[i].attrType == AttrType.attrString else 0 for i in self.outIndexes])
        return self._cursor

    def get_next(self) -> Optional[Tuple]:
        return self._open().next_tuple()

    def get_next_tid(self) -> Optional[TID]:
        """The position of the next qualifying row.  (The Java looks the last scanned column's RID up in the FIRST
        column's heap file, ColumnarColumnsScan.java:219 vs :191 -- wrong when the two columns' records differ in size;
        the position returned here is the right one.)"""
        pos = self._open().next_position()
        return None if pos is None else TID(self.in1_len, pos)

    def close(self) -> None:
        if not self.closeFlag:
            if self._result is not None:
                self._result.close()
            self._cursor = self._result = None
            self.closeFlag = True


class ColumnarColumnScan(_ColumnsScan):
    """iterator/ColumnarColumnScan.java:39-88,151-196.

    ColumnarColumnScan(columnarfile, colNo, n_out_flds, out_indexes, proj_list, outFilter)
    ColumnarColumnScan(columnarfile, colNo, outFilter)                  (delete query: get_next_tid only)"""

    def __init__(self, columnarfile, colNo: int, *rest):
        super().__init__(columnarfile, [colNo], rest,
                         "ColumnarColumnScan(columnarfile, colNo, [n_out_flds, out_indexes, proj_list,] outFilter)")
        self.colNo = int(colNo)


class ColumnarColumnsScan(_ColumnsScan):
    """iterator/ColumnarColumnsScan.java:39-101,176-224.

    ColumnarColumnsScan(columnarfile, colNos, n_out_flds, out_indexes, proj_list, outFilter)
    ColumnarColumnsScan(columnarfile, colNos, outFilter)                (delete query: get_next_tid only)"""

    def __init__(self, columnarfile, colNos: Sequence[int], *rest):
        super().__init__(columnarfile, colNos, rest,
                         "ColumnarColumnsScan(columnarfile, colNos, [n_out_flds, out_indexes, proj_list,] outFilter)")


class ColumnarNestedLoopJoins(Iterator):
    """iterator/ColumnarNestedLoopJoins.java:45-231 (SURVEY.md 8f rank 3).

    ColumnarNestedLoopJoins(outerColumnarFile, innerColumnarFile, in1, in1_len, t1_str_sizes, in2, in2_len, t2_str_sizes,
                            outerItr, innerItr, outFilter, rightFilter, joinFilter, proj_list, n_out_flds, amt_of_mem)

    in1 / in2 describe the tuples the two input iterators produce; outFilter / rightFilter are evaluated on those tuples
    (outer / inner), joinFilter on the pair (operand1 = outer field, operand2 = innerRel field), proj_list picks the
    output fields from either tuple.  The input iterators must be this package's scans (ColumnarFileScan,
    ColumnarColumnScan, ColumnarColumnsScan): their predicates and the pending filters are folded into one GPU filter
    scan per side, the join runs as K6, and get_next() hands the joined tuples out in the reference's block order --
    outer blocks of (amt_of_mem - 1) * (1024 / outerItr.getTupleSize()) qualifying tuples, for each block every inner
    tuple in order, the block's outer tuples inside (:157-207)."""

    def __init__(self, outerColumnarFile, innerColumnarFile, in1, in1_len, t1_str_sizes, in2, in2_len, t2_str_sizes,
                 outerItr, innerItr, outFilter, rightFilter, joinFilter, proj_list, n_out_flds, amt_of_mem):
        super().__init__()
        for it in (outerItr, innerItr):
            if not hasattr(it, "_table_terms"):
                raise NestedLoopException(None, "input iterators must be ColumnarFileScan / ColumnarColumn(s)Scan of this package")
        self.outerColumnarFile, self.innerColumnarFile = outerColumnarFile, innerColumnarFile
        self.outerItr, self.innerItr = outerItr, innerItr
        self.OuterFilter, self.RightFilter, self.JoinFilter = outFilter, rightFilter, joinFilter
        self._in1, self._in2 = list(in1)[:in1_len], list(in2)[:in2_len]
        self.perm_mat, self.nOutFlds = list(proj_list), n_out_flds
        self.n_buf_pgs = int(amt_of_mem)
        # two-relation setup_op_tuple (iterator/TupleUtils.java:343-409)
        def sizes_of(types, str_sizes):
            out, k = [], 0
            for t in types:
                if t.attrType == AttrType.attrString:
                    out.append(str_sizes[k]); k += 1
                else:
                    out.append(0)
            return out
        s1, s2 = sizes_of(self._in1, t1_str_sizes), sizes_of(self._in2, t2_str_sizes)
        self.Jtypes, jsizes = [], []
        for fs in self.perm_mat[:n_out_flds]:
            types, sizes = (self._in1, s1) if fs.relation.key == RelSpec.outer else (self._in2, s2)
            self.Jtypes.append(AttrType(types[fs.offset - 1].attrType))
            if types[fs.offset - 1].attrType == AttrType.attrString:
                jsizes.append(sizes[fs.offset - 1])
        self.Jtuple = Tuple()
        try:
            self.Jtuple.setHdr(n_out_flds, self.Jtypes, jsizes)
        except Exception as e:
            raise NestedLoopException(e, "TupleUtilsException is caught by ColumnarNestedLoopsJoins.java")
        self._rows = None
        self._i = 0

    @staticmethod
    def _side_terms(it, pending) -> list:
        """The iterator's own predicate AND the pending filter (fields of the iterator's tuple), over table columns."""
        terms = list(it._table_terms())
        base = 1 + max([t.conj for t in terms], default=-1)
        cols = it._tuple_columns()
        for t in flatten_condexpr(pending):
            ops = [((k, cols[v]) if k == "col" else (k, v)) for k, v in (t.lhs, t.rhs)]
            terms.append(Term(t.op, ops[0], ops[1], base + t.conj))
        return terms

    def _run(self) -> None:
        from .engine import bitmap_join
        want = N.WANT_BITMAP | N.WANT_POSITIONS | N.WANT_HOST
        try:
            osel = self.outerColumnarFile.table.scan(self._side_terms(self.outerItr, self.OuterFilter), want=want)
            isel = self.innerColumnarFile.table.scan(self._side_terms(self.innerItr, self.RightFilter), want=want)
            ocols, icols = self.outerItr._tuple_columns(), self.innerItr._tuple_columns()
            jterms = []
            for t in flatten_condexpr(self.JoinFilter):           # operand1: outer tuple field, operand2: innerRel field
                jterms.append(Term(t.op, ("col", ocols[t.lhs[1]]), ("icol", icols[t.rhs[1]]), t.conj))
            proj = [(N.OPERAND_OUTER, ocols[fs.offset - 1]) if fs.relation.key == RelSpec.outer else (N.OPERAND_INNER, icols[fs.offset - 1])
                    for fs in self.perm_mat[:self.nOutFlds]]
            res = bitmap_join(self.outerColumnarFile.table, self.innerColumnarFile.table, jterms, proj,
                              N.WANT_POSITIONS | N.WANT_COLUMNS | N.WANT_HOST, outer_sel=osel, inner_sel=isel)
        except N.MbcError as e:
            raise NestedLoopException(e, "Exceeption is caught by ColumnarNestedLoopsJoins.java")
        block_rows = max(1, (self.n_buf_pgs - 1) * (1024 // max(self.outerItr.getTupleSize(), 1)))
        po, pi = res.positions(), res.positions2()
        rank = np.searchsorted(osel.positions(), po)              # same key as input.nlj_emission_order
        order = np.lexsort((po, pi, rank // block_rows))
        self._cols = [np.asarray(res.column(i))[order] for i in range(self.nOutFlds)]
        self._rows = len(order)
        res.close(); osel.close(); isel.close()

    def get_next(self) -> Optional[Tuple]:
        if self._rows is None:
            self._run()
        if self._i >= self._rows:
            return None
        k = self._i
        self._i += 1
        for f, t in enumerate(self.Jtypes):                     # Projection.Join (:40-101) into the reused Jtuple
            if t.attrType == AttrType.attrInteger:
                self.Jtuple.setIntFld(f + 1, int(self._cols[f][k]))
            elif t.attrType == AttrType.attrReal:
                self.Jtuple.setFloFld(f + 1, float(self._cols[f][k]))
            else:
                self.Jtuple.setStrFld(f + 1, bytes(self._cols[f][k]).rstrip(b"\0").decode("utf-8"))
        return self.Jtuple

    def close(self) -> None:
        if not self.closeFlag:
            self.innerItr.close()
            self.outerItr.close()
            self._cols, self._rows = None, 0
            self.closeFlag = True
