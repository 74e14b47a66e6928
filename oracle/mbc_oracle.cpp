// mbc_oracle.cpp -- CPU restatement of the reference's columnar scan path.
//
// TEST INFRASTRUCTURE ONLY.  Nothing in the product (libmbcol.so, the Python mirror) links, imports
// or calls this file; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
// reference legs do, and only as the checker / the timed CPU arm.
//
// Parity status: PINNED.  The reference is first-party Java with no native parts and cannot be built
// here (no JDK in the image), so this restatement follows the Java sources line by line and is itself
// validated against the golden session transcript the reference ships (phase3_output, fixtures
// extracted into tests/golden/ by tests/golden/make_golden.py).
//
// The restatement is deliberately literal and row-at-a-time:
//   columnar/TupleScan.java:55-89      one Tuple image per row, all columns, skip markedDeleted
//   heap/Tuple.java:369-440            tuple header: fldCnt, fldOffset[0..n]
//   global/Convert.java:18-126,163-275 big-endian int/float, modified-UTF-8 strings with 2-byte length
//   iterator/PredEval.java:25-183      CNF: array = AND, .next chain = OR, compare type = type of lhs
//   iterator/TupleUtils.java:35-87     int / float / String.compareTo comparison
//   iterator/Projection.java:103-144   Project: copy fields into the (reused) Jtuple
//   iterator/Projection.java:28-83     Join: copy fields of two tuples
//   input/BitMapQuery.java:187-305     bitmap equi-join loop (outer ascending x inner ascending)
//   index/ColumnIndexScan.java:656-740 term -> OR of the bitmaps of the satisfying indexed values
//   index/ColumnarIndexScan.java:130-181 CNF over bitsets
// Aggregates do not exist in the reference (SURVEY.md F5); they are defined here: COUNT = |Q|,
// SUM(int) exact int64, SUM(real) = double sum of (double)float32 in ascending position order,
// MIN/MAX exact, empty Q -> MIN/MAX invalid.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <map>
#include <string>
#include <vector>
#include <thread>

namespace {

enum { ATTR_STRING = 0, ATTR_INTEGER = 1, ATTR_REAL = 2, ATTR_SYMBOL = 3 };
enum { OP_EQ = 0, OP_LT, OP_GT, OP_NE, OP_LE, OP_GE, OP_NOT, OP_NOP, OP_RANGE };
enum { AGG_COUNT = 0, AGG_SUM, AGG_MIN, AGG_MAX };

struct OCol {
    int32_t type, width;
    const void* data;          // nrows packed values: int32/float32 LE or width zero-padded bytes
};
struct OOperand {
    int32_t kind;              // 0 literal, 1 outer column, 2 inner column
    int32_t type;              // literal type
    int32_t col;
    int32_t lit_i;
    float lit_f;
    int32_t lit_slen;
    const uint8_t* lit_s;
};
struct OTerm {
    int32_t op, conj_id;
    OOperand lhs, rhs;
};
struct OAgg {
    int32_t kind, col;
};
struct OAggOut {
    int64_t i;
    double f;
    int32_t valid, pad;
};
struct OProj {
    int32_t rel, col;          // 1 outer, 2 inner
};

// ---- global/Convert.java ------------------------------------------------------------------------
inline void put_short(uint8_t* d, int pos, int v) { d[pos] = (uint8_t)(v >> 8); d[pos + 1] = (uint8_t)v; }
inline int get_short(const uint8_t* d, int pos) { return (int16_t)((d[pos] << 8) | d[pos + 1]); }
inline void put_int(uint8_t* d, int pos, uint32_t v) {
    d[pos] = (uint8_t)(v >> 24); d[pos + 1] = (uint8_t)(v >> 16); d[pos + 2] = (uint8_t)(v >> 8); d[pos + 3] = (uint8_t)v;
}
inline uint32_t get_int(const uint8_t* d, int pos) {
    return ((uint32_t)d[pos] << 24) | ((uint32_t)d[pos + 1] << 16) | ((uint32_t)d[pos + 2] << 8) | d[pos + 3];
}
inline float bits_to_float(uint32_t b) { float f; memcpy(&f, &b, 4); return f; }
inline uint32_t float_to_bits(float f) { uint32_t b; memcpy(&b, &f, 4); return b; }

// DataInputStream.readUTF: modified UTF-8 -> UTF-16 code units
inline void read_utf(const uint8_t* d, int pos, std::vector<uint16_t>* out) {
    int len = ((d[pos] << 8) | d[pos + 1]) & 0xFFFF;
    out->clear();
    const uint8_t* p = d + pos + 2;
    int i = 0;
    while (i < len) {
        int c = p[i];
        if (c < 0x80) { out->push_back((uint16_t)c); i += 1; }
        else if ((c >> 5) == 6) { out->push_back((uint16_t)(((c & 0x1F) << 6) | (p[i + 1] & 0x3F))); i += 2; }
        else { out->push_back((uint16_t)(((c & 0x0F) << 12) | ((p[i + 1] & 0x3F) << 6) | (p[i + 2] & 0x3F))); i += 3; }
    }
}
// String.compareTo
inline int compare_utf16(const std::vector<uint16_t>& a, const std::vector<uint16_t>& b) {
    size_t n = std::min(a.size(), b.size());
    for (size_t i = 0; i < n; ++i)
        if (a[i] != b[i]) return (int)a[i] - (int)b[i];
    return (int)a.size() - (int)b.size();
}

// ---- heap/Tuple.java: header + field access over a byte image ------------------------------------
struct TupleDesc {
    int n = 0;
    std::vector<int> type, size;   // size: 4 or strSize
    std::vector<int> off;          // fldOffset[0..n]
    int length() const { return off[n]; }
};

TupleDesc make_desc(const std::vector<int>& types, const std::vector<int>& sizes) {
    TupleDesc d;
    d.n = (int)types.size();
    d.type = types;
    d.size = sizes;
    d.off.resize(d.n + 1);
    d.off[0] = (d.n + 2) * 2;                                   // Tuple.java:380
    for (int i = 0; i < d.n; ++i) d.off[i + 1] = d.off[i] + (types[i] == ATTR_STRING ? sizes[i] + 2 : 4);
    return d;
}

void set_hdr(const TupleDesc& d, uint8_t* t) {                  // Tuple.java:369-440
    put_short(t, 0, d.n);
    for (int i = 0; i <= d.n; ++i) put_short(t, 2 + 2 * i, d.off[i]);
}

// Convert.setStrValue writes [len][bytes] only: the rest of the slot keeps what it held
inline void set_str_fld(uint8_t* t, int off, const uint8_t* s, int len) {
    put_short(t, off, len);
    memcpy(t + off + 2, s, len);
}

inline int fixed_strlen(const uint8_t* s, int width) {
    int len = 0;
    for (int k = 0; k < width; ++k) if (s[k]) len = k + 1;
    return len;
}

// ---- iterator/PredEval.java + TupleUtils.java ------------------------------------------------------
struct LitTuple {                  // the one-field `value` tuple PredEval builds for a literal
    uint8_t bytes[8 + 2 + 1024];
};

struct Evaluator {
    const TupleDesc* d1;
    const TupleDesc* d2;
    std::vector<uint16_t> sa, sb;

    // field bytes of one operand: literal tuples have their single field at offset 6
    const uint8_t* operand(const OOperand& o, const uint8_t* t1, const uint8_t* t2, LitTuple* lit, int* off) {
        if (o.kind == 0) {
            // value.setHdr(1, {type}, {len+1}) then set*Fld(1, literal)   (PredEval.java:60-78)
            memset(lit->bytes, 0, 16);
            if (o.type == ATTR_INTEGER) put_int(lit->bytes, 6, (uint32_t)o.lit_i);
            else if (o.type == ATTR_REAL) put_int(lit->bytes, 6, float_to_bits(o.lit_f));
            else { memset(lit->bytes, 0, 8 + o.lit_slen + 4); set_str_fld(lit->bytes, 6, o.lit_s, o.lit_slen); }
            *off = 6;
            return lit->bytes;
        }
        const TupleDesc* d = o.kind == 1 ? d1 : d2;
        *off = d->off[o.col];
        return o.kind == 1 ? t1 : t2;
    }

    // TupleUtils.CompareTupleWithTuple: sign of compare under `type`
    int compare(int type, const uint8_t* a, int aoff, const uint8_t* b, int boff) {
        if (type == ATTR_INTEGER) {
            int32_t x = (int32_t)get_int(a, aoff), y = (int32_t)get_int(b, boff);
            return x == y ? 0 : (x < y ? -1 : 1);
        }
        if (type == ATTR_REAL) {
            float x = bits_to_float(get_int(a, aoff)), y = bits_to_float(get_int(b, boff));
            if (x == y) return 0;
            if (x < y) return -1;
            if (x > y) return 1;
            return 2;                                           // NaN: the Java falls through; contract excludes it
        }
        read_utf(a, aoff, &sa);
        read_utf(b, boff, &sb);
        int c = compare_utf16(sa, sb);
        return c > 0 ? 1 : (c < 0 ? -1 : 0);
    }

    bool eval(const OTerm* terms, int nterms, const uint8_t* t1, const uint8_t* t2) {
        if (nterms == 0) return true;                            // p == null (PredEval.java:46-49)
        LitTuple l1, l2;
        int k = 0;
        while (k < nterms) {
            bool row_res = false;
            int conj = terms[k].conj_id;
            for (; k < nterms && terms[k].conj_id == conj; ++k) {
                if (row_res) continue;                           // OR satisfied: the Java breaks out
                const OTerm& t = terms[k];
                int cmp_type = t.lhs.kind == 0 ? t.lhs.type : (t.lhs.kind == 1 ? d1 : d2)->type[t.lhs.col];
                int aoff, boff;
                const uint8_t* a = operand(t.lhs, t1, t2, &l1, &aoff);
                const uint8_t* b = operand(t.rhs, t1, t2, &l2, &boff);
                int c = compare(cmp_type, a, aoff, b, boff);
                bool r = false;
                switch (t.op) {                                  // PredEval.java:137-162
                    case OP_EQ: r = c == 0; break;
                    case OP_LT: r = c < 0; break;
                    case OP_GT: r = c > 0 && c != 2; break;
                    case OP_NE: r = c != 0; break;
                    case OP_LE: r = c <= 0; break;
                    case OP_GE: r = c >= 0 && c != 2; break;
                    case OP_NOT: r = c != 0; break;
                    default: r = false;
                }
                row_res = row_res || r;
            }
            if (!row_res) return false;
        }
        return true;
    }
};

// build the TupleScan image of row r (TupleScan.java:55-89): fresh zeroed tuple, every column
inline void build_row_tuple(const TupleDesc& d, const OCol* cols, int64_t r, uint8_t* t) {
    memset(t, 0, d.length());
    set_hdr(d, t);
    for (int c = 0; c < d.n; ++c) {
        if (d.type[c] == ATTR_STRING) {
            const uint8_t* s = (const uint8_t*)cols[c].data + r * cols[c].width;
            set_str_fld(t, d.off[c], s, fixed_strlen(s, cols[c].width));
        } else {
            put_int(t, d.off[c], ((const uint32_t*)cols[c].data)[r]);
        }
    }
}

// Projection.Project / Join: copy field `src_col` of tuple `src` into field `f` of Jtuple
inline void project_field(const TupleDesc& sd, const uint8_t* src, int src_col, const TupleDesc& jd, uint8_t* j, int f) {
    if (sd.type[src_col] == ATTR_STRING) {
        int len = ((src[sd.off[src_col]] << 8) | src[sd.off[src_col] + 1]) & 0xFFFF;
        set_str_fld(j, jd.off[f], src + sd.off[src_col] + 2, len);   // getStrFld + setStrFld
    } else {
        memcpy(j + jd.off[f], src + sd.off[src_col], 4);
    }
}

// as_i64 of a real aggregate: Java's (long) d -- toward zero, saturated to INT64_MIN / INT64_MAX (±inf too), NaN -> 0
inline int64_t real_as_i64(double d) {
    if (d != d) return 0;
    if (d >= 9223372036854775808.0) return INT64_MAX;
    if (d < -9223372036854775808.0) return INT64_MIN;
    return (int64_t)d;
}

struct AggState {
    int kind, type;
    int64_t i = 0;
    double f = 0;
    bool any = false;
    void add(const uint8_t* t, int off) {
        if (kind == AGG_COUNT) { ++i; any = true; return; }
        if (type == ATTR_INTEGER) {
            int64_t v = (int32_t)get_int(t, off);
            if (kind == AGG_SUM) i += v;
            else if (!any) i = v;
            else i = kind == AGG_MIN ? std::min(i, v) : std::max(i, v);
        } else {
            double v = (double)bits_to_float(get_int(t, off));
            if (kind == AGG_SUM) f += v;
            else if (!any) f = v;
            else f = kind == AGG_MIN ? std::min(f, v) : std::max(f, v);
        }
        any = true;
    }
    void merge(const AggState& o) {
        if (!o.any) return;
        if (kind == AGG_COUNT || kind == AGG_SUM) { i += o.i; f += o.f; }
        else if (!any) { i = o.i; f = o.f; }
        else if (kind == AGG_MIN) { i = std::min(i, o.i); f = std::min(f, o.f); }
        else { i = std::max(i, o.i); f = std::max(f, o.f); }
        any = true;
    }
    void out(OAggOut* o) const {
        bool integral = kind == AGG_COUNT || type == ATTR_INTEGER;
        bool valid = kind == AGG_COUNT || kind == AGG_SUM || any;
        o->valid = valid;
        o->i = valid ? (integral ? i : real_as_i64(f)) : 0;
        o->f = valid ? (integral ? (double)i : f) : 0.0;
    }
};

inline bool bit(const uint64_t* w, int64_t p) { return w && ((w[p >> 6] >> (p & 63)) & 1ull); }

}  // namespace

extern "C" {

// Length of the projected tuple (TupleUtils.setup_op_tuple + Tuple.setHdr).
int32_t orc_tuple_len(int32_t ncols, const OCol* cols, const int32_t* proj, int32_t nproj) {
    std::vector<int> t, s;
    for (int i = 0; i < nproj; ++i) { t.push_back(cols[proj[i]].type); s.push_back(cols[proj[i]].width); }
    (void)ncols;
    return make_desc(t, s).length();
}

// ColumnarFileScan over a whole table.  Returns the number of qualifying rows.
//   out_pos     : nullable, capacity nrows
//   out_tuples  : nullable, capacity nrows * orc_tuple_len
//   stale_padding != 0 reproduces the reused-Jtuple behaviour byte for byte (string padding keeps the
//                 bytes of earlier, longer values: Convert.setStrValue writes len+2 bytes only);
//                 0 gives canonical zero-padded slots.  Forces a single thread.
//   nthreads    : 1 = the literal single-threaded loop; >1 = std::thread over row ranges (CPU baseline)
int64_t orc_scan(int32_t ncols, const OCol* cols, int64_t nrows, const uint64_t* deleted,
                 const OTerm* terms, int32_t nterms, const int32_t* proj, int32_t nproj,
                 int64_t* out_pos, uint8_t* out_tuples, int32_t stale_padding,
                 const OAgg* aggs, int32_t nagg, OAggOut* agg_out, int32_t nthreads) {
    std::vector<int> types, sizes, jt, js;
    for (int c = 0; c < ncols; ++c) { types.push_back(cols[c].type); sizes.push_back(cols[c].width); }
    for (int i = 0; i < nproj; ++i) { jt.push_back(cols[proj[i]].type); js.push_back(cols[proj[i]].width); }
    const TupleDesc d = make_desc(types, sizes);
    const TupleDesc jd = make_desc(jt, js);
    const int jlen = jd.length();
    if (stale_padding) nthreads = 1;
    if (nthreads < 1) nthreads = 1;

    std::vector<std::vector<AggState>> tagg(nthreads);
    std::vector<int64_t> tcount(nthreads, 0);
    std::vector<std::vector<int64_t>> tpos(nthreads);
    std::vector<std::vector<uint8_t>> ttup(nthreads);

    auto worker = [&](const int tid) {
        const int64_t lo = nrows * tid / nthreads, hi = nrows * (tid + 1) / nthreads;
        std::vector<uint8_t> tuple1(d.length() + 8), jtuple(jlen + 8, 0);
        set_hdr(jd, jtuple.data());
        Evaluator ev{&d, nullptr, {}, {}};
        std::vector<AggState> as(nagg);
        for (int a = 0; a < nagg; ++a) { as[a].kind = aggs[a].kind; as[a].type = aggs[a].kind == AGG_COUNT ? ATTR_INTEGER : cols[aggs[a].col].type; }
        int64_t cnt = 0;
        const bool direct = nthreads == 1;
        for (int64_t r = lo; r < hi; ++r) {
            build_row_tuple(d, cols, r, tuple1.data());                    // TupleScan.getNext
            if (bit(deleted, r)) continue;                                 // TupleScan.java:85
            if (!ev.eval(terms, nterms, tuple1.data(), nullptr)) continue; // ColumnarFileScan.java:167
            if (!stale_padding) { memset(jtuple.data(), 0, jlen); set_hdr(jd, jtuple.data()); }
            for (int f = 0; f < nproj; ++f) project_field(d, tuple1.data(), proj[f], jd, jtuple.data(), f);
            for (int a = 0; a < nagg; ++a) as[a].add(tuple1.data(), aggs[a].kind == AGG_COUNT ? 0 : d.off[aggs[a].col]);
            if (direct) {
                if (out_pos) out_pos[cnt] = r;
                if (out_tuples) memcpy(out_tuples + cnt * jlen, jtuple.data(), jlen);
            } else {
                if (out_pos) tpos[tid].push_back(r);
                if (out_tuples) ttup[tid].insert(ttup[tid].end(), jtuple.begin(), jtuple.begin() + jlen);
            }
            ++cnt;
        }
        tcount[tid] = cnt;
        tagg[tid] = as;
    };
    if (nthreads == 1) {
        worker(0);
    } else {
        std::vector<std::thread> pool;
        for (int t = 0; t < nthreads; ++t) pool.emplace_back(worker, t);
        for (auto& th : pool) th.join();
    }
    int64_t total = 0;
    for (int t = 0; t < nthreads; ++t) {
        if (nthreads > 1) {
            if (out_pos && !tpos[t].empty()) memcpy(out_pos + total, tpos[t].data(), tpos[t].size() * 8);
            if (out_tuples && !ttup[t].empty()) memcpy(out_tuples + total * jlen, ttup[t].data(), ttup[t].size());
        }
        total += tcount[t];
    }
    for (int a = 0; a < nagg; ++a) {
        AggState s = tagg[0][a];
        for (int t = 1; t < nthreads; ++t) s.merge(tagg[t][a]);
        s.out(&agg_out[a]);
    }
    return total;
}

// BitMapQuery.executeJoin.  join terms: lhs = outer column, rhs = inner column, op as the user wrote it.
// Returns the number of result pairs; pairs/tuples are written when the buffers are non-NULL and
// the count does not exceed `capacity` (call once with capacity 0 to size).
int64_t orc_bitmap_join(int32_t n_ocols, const OCol* ocols, int64_t n_outer, const uint64_t* outer_sel, const uint64_t* outer_deleted,
                        int32_t n_icols, const OCol* icols, int64_t n_inner, const uint64_t* inner_sel, const uint64_t* inner_deleted,
                        const OTerm* join, int32_t njoin, const OProj* proj, int32_t nproj,
                        int64_t capacity, int64_t* out_opos, int64_t* out_ipos, uint8_t* out_tuples,
                        const OAgg* aggs, int32_t nagg, OAggOut* agg_out) {
    std::vector<int> ot, os, it, is, jt, js;
    for (int c = 0; c < n_ocols; ++c) { ot.push_back(ocols[c].type); os.push_back(ocols[c].width); }
    for (int c = 0; c < n_icols; ++c) { it.push_back(icols[c].type); is.push_back(icols[c].width); }
    for (int f = 0; f < nproj; ++f) {
        const OCol& c = proj[f].rel == 1 ? ocols[proj[f].col] : icols[proj[f].col];
        jt.push_back(c.type); js.push_back(c.width);
    }
    const TupleDesc od = make_desc(ot, os), id = make_desc(it, is), jd = make_desc(jt, js);
    const int jlen = jd.length();
    const int64_t iwords = (n_inner + 63) / 64;

    // "bitmap indexes" of the inner join columns: value bytes -> ascending positions, deleted rows
    // skipped at build time (Columnarfile.createBitMapIndex uses ColumnScan)
    struct Index { std::map<std::string, std::vector<int64_t>> by_value; int type, width; };
    std::map<int, Index> index;
    for (int k = 0; k < njoin; ++k) {
        int c = join[k].rhs.col;
        if (index.count(c)) continue;
        Index& ix = index[c];
        ix.type = icols[c].type; ix.width = icols[c].width;
        for (int64_t r = 0; r < n_inner; ++r) {
            if (bit(inner_deleted, r)) continue;
            std::string key;
            if (ix.type == ATTR_STRING) {
                const uint8_t* s = (const uint8_t*)icols[c].data + r * ix.width;
                key.assign((const char*)s, fixed_strlen(s, ix.width));
            } else {
                uint32_t v = ((const uint32_t*)icols[c].data)[r] ^ 0x80000000u;   // order-preserving key
                uint8_t b[4]; put_int(b, 0, v); key.assign((const char*)b, 4);
            }
            ix.by_value[key].push_back(r);
        }
    }
    auto int_of_key = [](const std::string& k) { return (int32_t)(get_int((const uint8_t*)k.data(), 0) ^ 0x80000000u); };

    std::vector<AggState> as(nagg);
    for (int a = 0; a < nagg; ++a) {
        as[a].kind = aggs[a].kind;
        as[a].type = aggs[a].kind == AGG_COUNT ? ATTR_INTEGER : jt[aggs[a].col];
    }
    std::vector<uint8_t> otup(od.length() + 8), itup(id.length() + 8), jtuple(jlen + 8, 0);
    std::vector<uint64_t> join_bits(iwords), conj_bits(iwords);
    std::vector<uint16_t> sa, sb;
    int64_t count = 0;
    for (int64_t o = 0; o < n_outer; ++o) {                          // outerConditionsBitset.nextSetBit ascending
        if (outer_sel && !bit(outer_sel, o)) continue;
        if (bit(outer_deleted, o)) continue;                         // the side filter already dropped deleted rows
        build_row_tuple(od, ocols, o, otup.data());
        // updateConstraint + new ColumnarIndexScan(inner, constraint)   (:244-247)
        std::fill(join_bits.begin(), join_bits.end(), ~0ull);
        int k = 0;
        while (k < njoin) {
            std::fill(conj_bits.begin(), conj_bits.end(), 0ull);
            int conj = join[k].conj_id;
            for (; k < njoin && join[k].conj_id == conj; ++k) {
                const OTerm& t = join[k];
                const Index& ix = index[t.rhs.col];
                // the reference stores `innerCol op' outerValue` with op' = getOppositeOperator(op) (:453);
                // ColumnIndexScan.getBitSet then ORs the bitmaps of the indexed values v with v op' literal,
                // i.e. exactly the inner values with  outerValue op v.
                if (t.op == OP_EQ) {
                    // EQ selects exactly the literal's own bitmap (ColumnIndexScan.java:660-667): look it up
                    std::string key;
                    if (ix.type == ATTR_STRING) {
                        int len = ((otup[od.off[t.lhs.col]] << 8) | otup[od.off[t.lhs.col] + 1]) & 0xFFFF;
                        key.assign((const char*)otup.data() + od.off[t.lhs.col] + 2, len);
                    } else {
                        uint8_t b[4];
                        put_int(b, 0, get_int(otup.data(), od.off[t.lhs.col]) ^ 0x80000000u);
                        key.assign((const char*)b, 4);
                    }
                    auto it = ix.by_value.find(key);
                    if (it != ix.by_value.end())
                        for (int64_t p : it->second)
                            if (!bit(inner_deleted, p)) conj_bits[p >> 6] |= 1ull << (p & 63);
                    continue;
                }
                for (auto& kv : ix.by_value) {
                    int c;                                           // sign of compare(outer value, v)
                    if (ix.type == ATTR_STRING) {
                        std::vector<uint8_t> a(2 + od.size[t.lhs.col]);
                        read_utf(otup.data(), od.off[t.lhs.col], &sa);
                        sb.clear();
                        std::vector<uint8_t> tmp(2 + kv.first.size());
                        put_short(tmp.data(), 0, (int)kv.first.size());
                        memcpy(tmp.data() + 2, kv.first.data(), kv.first.size());
                        read_utf(tmp.data(), 0, &sb);
                        int cc = compare_utf16(sa, sb);
                        c = cc > 0 ? 1 : (cc < 0 ? -1 : 0);
                    } else {
                        int32_t ov = (int32_t)get_int(otup.data(), od.off[t.lhs.col]);
                        int32_t v = int_of_key(kv.first);
                        c = ov == v ? 0 : (ov < v ? -1 : 1);
                    }
                    bool sel;
                    switch (t.op) {
                        case OP_EQ: sel = c == 0; break;
                        case OP_LT: sel = c < 0; break;
                        case OP_GT: sel = c > 0; break;
                        case OP_NE: sel = c != 0; break;
                        case OP_LE: sel = c <= 0; break;
                        case OP_GE: sel = c >= 0; break;
                        default: sel = false;
                    }
                    if (!sel) continue;
                    for (int64_t p : kv.second)
                        if (!bit(inner_deleted, p)) conj_bits[p >> 6] |= 1ull << (p & 63);   // get_bm_next_tid skips deleted
                }
            }
            for (int64_t w = 0; w < iwords; ++w) join_bits[w] &= conj_bits[w];
        }
        if (inner_sel) for (int64_t w = 0; w < iwords; ++w) join_bits[w] &= inner_sel[w];   // :249
        for (int64_t w = 0; w < iwords; ++w) {
            uint64_t word = join_bits[w];
            while (word) {
                int b = __builtin_ctzll(word);
                word &= word - 1;
                int64_t i = w * 64 + b;
                if (i >= n_inner) break;
                build_row_tuple(id, icols, i, itup.data());
                memset(jtuple.data(), 0, jlen);
                set_hdr(jd, jtuple.data());
                for (int f = 0; f < nproj; ++f) {                    // Projection.Join (:279-280)
                    if (proj[f].rel == 1) project_field(od, otup.data(), proj[f].col, jd, jtuple.data(), f);
                    else project_field(id, itup.data(), proj[f].col, jd, jtuple.data(), f);
                }
                for (int a = 0; a < nagg; ++a) as[a].add(jtuple.data(), aggs[a].kind == AGG_COUNT ? 0 : jd.off[aggs[a].col]);
                if (count < capacity) {
                    if (out_opos) out_opos[count] = o;
                    if (out_ipos) out_ipos[count] = i;
                    if (out_tuples) memcpy(out_tuples + count * jlen, jtuple.data(), jlen);
                }
                ++count;
            }
        }
    }
    for (int a = 0; a < nagg; ++a) as[a].out(&agg_out[a]);
    return count;
}

int32_t orc_max_threads(void) {
    unsigned n = std::thread::hardware_concurrency();
    return n ? (int32_t)n : 1;
}

}  // extern "C"
