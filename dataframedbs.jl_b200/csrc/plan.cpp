// plan.cpp -- parses the serialized view plan (SelectionQueue + Projection) and compiles every
// BlockBroadcasting tree into (a) a typed, tag-free VM program for the generic kernels and (b), when
// the tree is a conjunction of `column <cmp> constant` terms, the term list of the fused fast path.
//
// Reference objects this stands in for:
//   SelectionQueue / RangeToProcess      /root/reference/src/tables/selection.jl:4-10,68-75
//   _check_element (Bool-only predicate) /root/reference/src/tables/selection.jl:52-55
//   BlockBroadcasting result typing      /root/reference/src/tables/broadcast.jl:6-17 (Base._return_type)
//   Projection                           /root/reference/src/tables/projection.jl:1-9
// Julia semantics implemented by the typing below: exact mixed integer/float comparisons, wrapping
// integer arithmetic with promote_type widths, `/` always floating, three-valued logic on missing.
#include <algorithm>
#include <cmath>
#include <limits>
#include <memory>

#include "internal.hpp"

namespace dfdb {
namespace {

struct Rdr {
    const uint8_t *p, *end;
    bool bad = false;
    uint8_t u8() { if (p + 1 > end) { bad = true; return 0; } return *p++; }
    uint32_t u32() { uint32_t v = 0; if (p + 4 > end) { bad = true; return 0; } memcpy(&v, p, 4); p += 4; return v; }
    int64_t i64() { int64_t v = 0; if (p + 8 > end) { bad = true; return 0; } memcpy(&v, p, 8); p += 8; return v; }
    double f64() { double v = 0; if (p + 8 > end) { bad = true; return 0; } memcpy(&v, p, 8); p += 8; return v; }
};

// element tags of an INSET collection
enum { T_I64 = 1, T_U64 = 2, T_F64 = 3, T_STR = 4, T_BOOL = 5, T_MISSING = 6 };

struct Node {
    int op = 0;
    int64_t i = 0;
    double f = 0;
    std::string s;                       // W_STR: the constant; W_INSET: the String elements' bytes
    int sem = 0;                         // W_IN / W_INSET: 0 = `==` (Ref(vector)), 1 = `isequal` (Ref(Set))
    std::vector<uint8_t> tags;           // W_IN / W_INSET: one per element
    std::vector<uint64_t> bits;          // payload: integer / double bits, Bool 0/1, String (offset in s) << 32 | length
    std::vector<std::unique_ptr<Node>> kids;
};

// static type of a VM stack entry
struct TVal {
    int cls = VC_NONE;   // VC_INT, VC_UINT, VC_FLT, VC_BOOL, VC_STR
    int bits = 64;
    bool nullable = false;
    bool dated = false;  // a stored Date / DateTime / Time column (VC_INT payload)
};

int arity(int op)
{
    switch (op) {
    case W_COL: case W_I64: case W_F64: case W_STR: case W_BOOL: return 0;
    case W_NOT: case W_NEG: case W_ISMISSING: case W_IN: case W_INSET: return 1;
    case W_EQ: case W_NE: case W_LT: case W_LE: case W_GT: case W_GE:
    case W_AND: case W_OR: case W_XOR:
    case W_ADD: case W_SUB: case W_MUL: case W_DIV: case W_REM:
    case W_COALESCE: case W_STARTSWITH: case W_ENDSWITH: return 2;
    default: return -1;
    }
}

int parse_tree(Rdr &r, std::unique_ptr<Node> *out)
{
    uint32_t nops = r.u32();
    if (r.bad || nops == 0 || nops > 4096) return fail(DFDB_ERR_ARGUMENT, "bad expression");
    std::vector<std::unique_ptr<Node>> st;
    for (uint32_t k = 0; k < nops; k++) {
        auto n = std::make_unique<Node>();
        n->op = r.u8();
        switch (n->op) {
        case W_COL: case W_I64: n->i = r.i64(); break;
        case W_F64: n->f = r.f64(); break;
        case W_BOOL: n->i = r.u8() != 0; break;
        case W_STR: {
            uint32_t len = r.u32();
            if (r.bad || r.p + len > r.end) return fail(DFDB_ERR_ARGUMENT, "truncated expression");
            n->s.assign(reinterpret_cast<const char *>(r.p), len);
            r.p += len;
            break;
        }
        case W_IN: {
            uint32_t cnt = r.u32();
            if (r.bad || r.p + 8ull * cnt > r.end) return fail(DFDB_ERR_ARGUMENT, "truncated expression");
            n->tags.assign(cnt, T_I64);
            n->bits.resize(cnt);
            if (cnt) memcpy(n->bits.data(), r.p, 8ull * cnt);
            r.p += 8ull * cnt;
            break;
        }
        case W_INSET: {
            n->sem = r.u8();
            uint32_t cnt = r.u32();
            if (r.bad) return fail(DFDB_ERR_ARGUMENT, "truncated expression");
            if (n->sem > 1) return fail(DFDB_ERR_ARGUMENT, "bad in() semantics %d", n->sem);
            if ((uint64_t)cnt > (uint64_t)(r.end - r.p)) return fail(DFDB_ERR_ARGUMENT, "truncated expression");   // every element takes a byte at least
            n->tags.resize(cnt);
            n->bits.resize(cnt);
            for (uint32_t k = 0; k < cnt; k++) {
                const int tag = r.u8();
                uint64_t b = 0;
                switch (tag) {
                case T_I64: case T_U64: case T_F64: b = (uint64_t)r.i64(); break;
                case T_BOOL: b = r.u8() != 0; break;
                case T_MISSING: break;
                case T_STR: {
                    uint32_t len = r.u32();
                    if (r.bad || r.p + len > r.end) return fail(DFDB_ERR_ARGUMENT, "truncated expression");
                    b = (uint64_t)n->s.size() << 32 | len;
                    n->s.append(reinterpret_cast<const char *>(r.p), len);
                    r.p += len;
                    break;
                }
                default:
                    if (r.bad) return fail(DFDB_ERR_ARGUMENT, "truncated expression");
                    return fail(DFDB_ERR_ARGUMENT, "unknown in() element tag %d", tag);
                }
                if (r.bad) return fail(DFDB_ERR_ARGUMENT, "truncated expression");
                n->tags[k] = (uint8_t)tag;
                n->bits[k] = b;
            }
            break;
        }
        default: break;
        }
        if (r.bad) return fail(DFDB_ERR_ARGUMENT, "truncated expression");
        int ar = arity(n->op);
        if (ar < 0) return fail(DFDB_ERR_UNSUPPORTED, "unknown opcode 0x%02x", n->op);
        if ((int)st.size() < ar) return fail(DFDB_ERR_ARGUMENT, "malformed expression (stack underflow)");
        n->kids.resize((size_t)ar);
        for (int a = ar - 1; a >= 0; a--) { n->kids[(size_t)a] = std::move(st.back()); st.pop_back(); }
        st.push_back(std::move(n));
    }
    if (st.size() != 1) return fail(DFDB_ERR_ARGUMENT, "malformed expression");
    *out = std::move(st[0]);
    return DFDB_OK;
}

// The key of collection element (tag, bits) in the domain of value class cls, or false when no value of the class is equal
// to it (`==` for sem 0, `isequal` for sem 1).  Numbers compare exactly: an element is kept only when some value of the class
// has exactly its value.  Keys: signed / unsigned integer bits, Bool 0/1, double bits with `==`'s -0.0 as 0.0 and isequal's
// NaNs as one NaN.  A NaN never equals anything under `==`, and isequal(0, -0.0) is false.
constexpr uint64_t CANON_NAN = 0x7ff8000000000000ull;
bool canon_key(int cls, int sem, int tag, uint64_t bits, uint64_t *key)
{
    if (tag == T_STR || tag == T_MISSING) return false;
    if (cls == VC_FLT) {
        double d;
        if (tag == T_F64) memcpy(&d, &bits, 8);
        else if (tag == T_BOOL) d = bits ? 1.0 : 0.0;
        else if (tag == T_I64) {
            d = (double)(int64_t)bits;
            if (d >= 9223372036854775808.0 || (int64_t)d != (int64_t)bits) return false;
        } else {
            d = (double)bits;
            if (d >= 18446744073709551616.0 || (uint64_t)d != bits) return false;
        }
        if (d != d) {
            if (sem == 0) return false;
            *key = CANON_NAN;
            return true;
        }
        if (sem == 0 && d == 0.0) d = 0.0;
        memcpy(key, &d, 8);
        return true;
    }
    // integer classes: the element as an exact integer
    __int128 v;
    if (tag == T_I64) v = (int64_t)bits;
    else if (tag == T_U64) v = (__int128)bits;
    else if (tag == T_BOOL) v = bits;
    else {
        double d;
        memcpy(&d, &bits, 8);
        if (d != d || std::floor(d) != d || d < -9223372036854775808.0 || d >= 18446744073709551616.0) return false;
        if (d == 0.0 && std::signbit(d) && sem == 1) return false;
        v = d < 0 ? (__int128)(int64_t)d : (__int128)(uint64_t)d;
    }
    if (cls == VC_INT) {
        if (v < -((__int128)1 << 63) || v >= ((__int128)1 << 63)) return false;
    } else if (cls == VC_UINT) {
        if (v < 0 || v >= ((__int128)1 << 64)) return false;
    } else if (v != 0 && v != 1) {   // Bool
        return false;
    }
    *key = (uint64_t)v;
    return true;
}

// the canonical set of an IN / INSET node whose left operand has class cls
void canon_set(const Node *n, int cls, InSet *out)
{
    out->cls = cls;
    out->flags = (n->sem ? SET_ISEQUAL : 0) | (n->tags.empty() ? 0 : SET_NONEMPTY);
    for (size_t k = 0; k < n->tags.size(); k++) {
        const int tag = n->tags[k];
        if (tag == T_MISSING) { out->flags |= SET_MISSING; continue; }
        if (cls == VC_STR) {
            if (tag == T_STR) out->strs.emplace_back(n->s, (size_t)(n->bits[k] >> 32), (size_t)(uint32_t)n->bits[k]);
            continue;
        }
        uint64_t key;
        if (canon_key(cls, n->sem, tag, n->bits[k], &key)) out->keys.push_back(key);
    }
    std::sort(out->keys.begin(), out->keys.end());
    out->keys.erase(std::unique(out->keys.begin(), out->keys.end()), out->keys.end());
    std::sort(out->strs.begin(), out->strs.end());
    out->strs.erase(std::unique(out->strs.begin(), out->strs.end()), out->strs.end());
    for (uint64_t k : out->keys) {
        uint64_t lo = k, hi = k;
        if (cls == VC_FLT) {
            double d;
            memcpy(&d, &k, 8);
            if (d != d) { out->has_nan = true; continue; }
            const bool first = !out->has_range;
            double mn, mx;
            memcpy(&mn, &out->kmin, 8);
            memcpy(&mx, &out->kmax, 8);
            if (first || d < mn) lo = k; else lo = out->kmin;
            if (first || d > mx) hi = k; else hi = out->kmax;
        } else if (out->has_range) {
            const bool uns = cls != VC_INT;
            lo = (uns ? k < out->kmin : (int64_t)k < (int64_t)out->kmin) ? k : out->kmin;
            hi = (uns ? k > out->kmax : (int64_t)k > (int64_t)out->kmax) ? k : out->kmax;
        }
        out->kmin = lo;
        out->kmax = hi;
        out->has_range = true;
    }
}

struct Compiler {
    dfdb_table *tbl;
    dfdb_scan *scan;
    Expr *e;
    VmProgram *prog;
    int nconst = 0, npool = 0;
    int depth = 0, maxdepth = 0;

    int slot_of(int64_t id)
    {
        for (size_t i = 0; i < scan->slots.size(); i++) if (scan->slots[i] == id) return (int)i;
        scan->slots.push_back(id);
        return (int)scan->slots.size() - 1;
    }
    int emit(uint8_t op, uint8_t a = 0, uint8_t b = 0, uint8_t c = 0, int32_t imm = 0)
    {
        if (prog->ninstr >= VM_MAX_INSTR) return fail(DFDB_ERR_UNSUPPORTED, "expression too long");
        prog->instr[prog->ninstr++] = VmInstr{op, a, b, c, imm};
        return DFDB_OK;
    }
    int add_const(int64_t bits, int *idx)
    {
        if (nconst >= VM_MAX_CONST) return fail(DFDB_ERR_UNSUPPORTED, "too many constants in expression");
        prog->consts[nconst] = bits;
        *idx = nconst++;
        return DFDB_OK;
    }
    void push() { if (++depth > maxdepth) maxdepth = depth; }

    static int cls_code(const TVal &v) { return v.cls == VC_FLT ? 3 : v.cls == VC_UINT ? 2 : v.cls == VC_BOOL ? 4 : 1; }

    int compile(const Node *n, TVal *out)
    {
        int rc;
        switch (n->op) {
        case W_COL: {
            Column *c = tbl->find(n->i);
            if (!c) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)n->i);
            int cls = value_class(c->type.kind);
            if (cls == VC_NONE) return fail(DFDB_ERR_UNSUPPORTED, "column %s of type %s is not supported in expressions", c->name.c_str(), c->typestr.c_str());
            int slot = slot_of(n->i);
            if (slot >= MAX_SLOTS) return fail(DFDB_ERR_UNSUPPORTED, "too many columns in one scan (max %d)", MAX_SLOTS);
            if (std::find(e->col_ids.begin(), e->col_ids.end(), n->i) == e->col_ids.end()) e->col_ids.push_back(n->i);
            out->cls = cls;
            out->bits = cls == VC_STR ? 0 : c->type.elsize * 8;
            out->nullable = c->type.nullable;
            out->dated = c->type.kind == DFDB_DATE || c->type.kind == DFDB_DATETIME || c->type.kind == DFDB_TIME;
            push();
            return emit(V_LOAD, (uint8_t)slot);
        }
        case W_I64: {
            int idx;
            if ((rc = add_const(n->i, &idx))) return rc;
            *out = TVal{VC_INT, 64, false};
            push();
            return emit(V_CONST, 0, 0, 0, idx);
        }
        case W_F64: {
            int idx;
            int64_t bits;
            memcpy(&bits, &n->f, 8);
            if ((rc = add_const(bits, &idx))) return rc;
            *out = TVal{VC_FLT, 64, false};
            push();
            return emit(V_CONST, 0, 0, 0, idx);
        }
        case W_BOOL: {
            int idx;
            if ((rc = add_const(n->i ? 1 : 0, &idx))) return rc;
            *out = TVal{VC_BOOL, 8, false};
            push();
            return emit(V_CONST, 0, 0, 0, idx);
        }
        case W_STR: {
            if (npool + (int)n->s.size() > VM_STRPOOL || n->s.size() > 0xFFFF) return fail(DFDB_ERR_UNSUPPORTED, "string constants too long");
            int off = npool;
            memcpy(prog->strpool + npool, n->s.data(), n->s.size());
            npool += (int)n->s.size();
            *out = TVal{VC_STR, 0, false};
            push();
            return emit(V_CONSTSTR, (uint8_t)(n->s.size() & 0xFF), (uint8_t)(n->s.size() >> 8), 0, off);
        }
        default: break;
        }
        TVal a, b;
        if ((rc = compile(n->kids[0].get(), &a))) return rc;
        if (n->kids.size() > 1 && (rc = compile(n->kids[1].get(), &b))) return rc;
        bool nullable = a.nullable || (n->kids.size() > 1 && b.nullable);
        switch (n->op) {
        case W_EQ: case W_NE: case W_LT: case W_LE: case W_GT: case W_GE: {
            int code = n->op - W_EQ;
            depth--;
            *out = TVal{VC_BOOL, 8, nullable};
            if (a.cls == VC_STR || b.cls == VC_STR) {
                if (a.cls == b.cls) return emit(V_STRCMP, (uint8_t)code);
                // ==(::String, ::Number) is false in Julia; ordering is a MethodError
                if (code > 1) return fail(DFDB_ERR_UNSUPPORTED, "ordering comparison between String and non-String");
                return emit(V_STRNUM, (uint8_t)code);
            }
            int la = a.cls == VC_FLT ? 2 : a.cls == VC_UINT ? 1 : 0, lb = b.cls == VC_FLT ? 2 : b.cls == VC_UINT ? 1 : 0;
            static const int cp[3][3] = {{CP_II, CP_IU, CP_IF}, {CP_UI, CP_UU, CP_UF}, {CP_FI, CP_FU, CP_FF}};
            return emit(V_CMP, (uint8_t)code, (uint8_t)cp[la][lb]);
        }
        case W_AND: case W_OR: case W_XOR:
            if (a.cls != VC_BOOL || b.cls != VC_BOOL) return fail(DFDB_ERR_UNSUPPORTED, "bitwise logic is supported on Bool operands only");
            depth--;
            *out = TVal{VC_BOOL, 8, nullable};
            return emit(n->op == W_AND ? V_AND : n->op == W_OR ? V_OR : V_XOR);
        case W_NOT:
            if (a.cls != VC_BOOL) return fail(DFDB_ERR_UNSUPPORTED, "! is supported on Bool operands only");
            *out = TVal{VC_BOOL, 8, nullable};
            return emit(V_NOT);
        case W_ADD: case W_SUB: case W_MUL: case W_DIV: case W_REM: case W_NEG: {
            bool unary = n->op == W_NEG;
            if (a.cls == VC_STR || (!unary && b.cls == VC_STR)) return fail(DFDB_ERR_UNSUPPORTED, "arithmetic on String");
            int code = n->op - W_ADD;
            if (!unary) depth--;
            bool af = a.cls == VC_FLT, bf = !unary && b.cls == VC_FLT;
            uint8_t classes = (uint8_t)(cls_code(a) | ((unary ? 0 : cls_code(b)) << 4));
            if (n->op == W_DIV || af || bf) {
                int bits = 64;
                if (!(n->op == W_DIV && !af && !bf)) {
                    int fa = af ? a.bits : 0, fb = bf ? b.bits : 0;
                    bits = (fa == 64 || fb == 64) ? 64 : 32;
                }
                *out = TVal{VC_FLT, bits, nullable};
                return emit(V_ARITH, (uint8_t)code, classes, (uint8_t)(0x40 | (bits / 8)));
            }
            int abits = (a.cls == VC_INT || a.cls == VC_UINT) ? a.bits : 0;
            int bbits = (!unary && (b.cls == VC_INT || b.cls == VC_UINT)) ? b.bits : 0;
            bool auns = a.cls == VC_UINT, buns = !unary && b.cls == VC_UINT;
            int bits;
            bool uns;
            if (unary) { bits = abits ? abits : 64; uns = auns; }
            else if (!abits && !bbits) { bits = 64; uns = false; }
            else if (!abits) { bits = bbits; uns = buns; }
            else if (!bbits) { bits = abits; uns = auns; }
            else if (abits == bbits) { bits = abits; uns = auns || buns; }
            else if (abits > bbits) { bits = abits; uns = auns; }
            else { bits = bbits; uns = buns; }
            *out = TVal{uns ? VC_UINT : VC_INT, bits, nullable};
            return emit(V_ARITH, (uint8_t)code, classes, (uint8_t)((uns ? 0x80 : 0) | (bits / 8)));
        }
        case W_ISMISSING:
            *out = TVal{VC_BOOL, 8, false};
            return emit(V_ISMISSING);
        case W_COALESCE: {
            bool same = (a.cls == b.cls) || ((a.cls == VC_INT || a.cls == VC_UINT) && (b.cls == VC_INT || b.cls == VC_UINT));
            if (!same || n->kids[1]->kids.size() != 0 || n->kids[1]->op == W_COL)
                return fail(DFDB_ERR_UNSUPPORTED, "coalesce default must be a constant of the same kind");
            depth--;
            *out = a;
            out->nullable = false;
            return emit(V_COALESCE);
        }
        case W_STARTSWITH: case W_ENDSWITH:
            if (a.cls != VC_STR || b.cls != VC_STR) return fail(DFDB_ERR_UNSUPPORTED, "startswith/endswith need String operands");
            depth--;
            *out = TVal{VC_BOOL, 8, nullable};
            return emit(n->op == W_STARTSWITH ? V_STARTSWITH : V_ENDSWITH);
        case W_IN: case W_INSET: {
            // Date, DateTime and Time would compare false against every number in Julia: refused rather than all-false
            if (n->op == W_INSET && a.dated) return fail(DFDB_ERR_UNSUPPORTED, "in() with a collection over a Date / DateTime / Time value");
            if (e->sets.size() >= (size_t)VM_MAX_SETS) return fail(DFDB_ERR_UNSUPPORTED, "too many in() collections in one expression (max %d)", VM_MAX_SETS);
            InSet set;
            canon_set(n, a.cls, &set);
            // `==` with missing on either side gives missing unless some element is equal; isequal is always a Bool
            *out = TVal{VC_BOOL, 8, n->sem == 0 && (a.nullable || (set.flags & SET_MISSING))};
            e->sets.push_back((int)scan->sets.size());
            scan->sets.push_back(std::move(set));
            return emit(V_INSET, (uint8_t)(e->sets.size() - 1));
        }
        default:
            return fail(DFDB_ERR_UNSUPPORTED, "unknown opcode 0x%02x", n->op);
        }
    }
};

// ---- fast path matching ------------------------------------------------------------------------

bool is_numeric_const(const Node *n) { return n->op == W_I64 || n->op == W_F64 || n->op == W_BOOL; }

int flip_code(int code)
{
    switch (code) {
    case 2: return 4;   // LT -> GT
    case 3: return 5;   // LE -> GE
    case 4: return 2;
    case 5: return 3;
    default: return code;
    }
}

// result of `x <code> c` when the comparison is decided by c alone (x below / above c)
int const_cmp(int code, int sign)   // sign = sgn(x - c): -1 means every x is < c
{
    switch (code) {
    case 0: return 0;
    case 1: return 1;
    case 2: case 3: return sign < 0;
    default: return sign > 0;
    }
}

bool make_term(dfdb_table *tbl, dfdb_scan *scan, const Node *col, const Node *cst, int code, Term *t)
{
    Column *c = tbl->find(col->i);
    if (!c) return false;
    int cls = value_class(c->type.kind);
    if (cls != VC_INT && cls != VC_UINT && cls != VC_FLT && cls != VC_BOOL) return false;
    int slot = -1;
    for (size_t i = 0; i < scan->slots.size(); i++) if (scan->slots[i] == col->i) slot = (int)i;
    if (slot < 0) return false;
    t->slot = slot;
    t->code = code;
    t->constant_result = -1;
    t->ci = 0;
    t->cf = 0;
    if (cls == VC_BOOL) cls = VC_UINT;
    t->cls = cls;
    bool cf_const = cst->op == W_F64;
    int64_t ci = cst->i;
    double cf = cst->f;
    if (cls == VC_FLT) {
        if (cf_const) { t->cf = cf; return true; }
        double d = (double)ci;
        bool exact = d >= -9223372036854775808.0 && d < 9223372036854775808.0 && (int64_t)d == ci;
        if (exact) { t->cf = d; return true; }
        // ci lies strictly between two adjacent doubles
        bool d_above = d >= 9223372036854775808.0 || (d > -9223372036854775808.0 && (__int128)(int64_t)d > (__int128)ci);
        double lo = d_above ? std::nextafter(d, -INFINITY) : d, hi = d_above ? d : std::nextafter(d, INFINITY);
        switch (code) {
        case 0: t->constant_result = 0; break;
        case 1: t->constant_result = 1; break;   // NaN != c is true as well
        case 2: case 3: t->code = 3; t->cf = lo; break;
        default: t->code = 5; t->cf = hi; break;
        }
        return true;
    }
    if (!cf_const) {
        if (cls == VC_UINT) {
            if (ci < 0) { t->constant_result = const_cmp(code, +1); return true; }
            t->ci = ci;
            return true;
        }
        t->ci = ci;
        return true;
    }
    // integer column against a Float64 constant: fold to an exact integer comparison
    if (cf != cf) { t->constant_result = code == 1; return true; }
    double lo_lim = cls == VC_UINT ? 0.0 : -9223372036854775808.0;
    double hi_lim = cls == VC_UINT ? 18446744073709551616.0 : 9223372036854775808.0;
    if (cf >= hi_lim) { t->constant_result = const_cmp(code, -1); return true; }
    if (cf < lo_lim) { t->constant_result = const_cmp(code, +1); return true; }
    double fl = std::floor(cf);
    int64_t k = cls == VC_UINT ? (int64_t)(uint64_t)fl : (int64_t)fl;
    t->ci = k;
    if (fl == cf) return true;
    switch (code) {
    case 0: t->constant_result = 0; break;
    case 1: t->constant_result = 1; break;
    case 2: case 3: t->code = 3; break;   // x < c  <=>  x <= floor(c)
    default: t->code = 4; break;          // x > c, x >= c  <=>  x > floor(c)
    }
    return true;
}

bool match_simple(dfdb_table *tbl, dfdb_scan *scan, const Node *n, bool in_coalesce, Expr *e)
{
    if (n->op == W_AND) return match_simple(tbl, scan, n->kids[0].get(), in_coalesce, e) && match_simple(tbl, scan, n->kids[1].get(), in_coalesce, e);
    if (n->op == W_COALESCE) {
        const Node *d = n->kids[1].get();
        if (d->op != W_BOOL || d->i != 0) return false;
        return match_simple(tbl, scan, n->kids[0].get(), true, e);
    }
    if (n->op >= W_EQ && n->op <= W_GE) {
        const Node *l = n->kids[0].get(), *r = n->kids[1].get();
        int code = n->op - W_EQ;
        const Node *col, *cst;
        if (l->op == W_COL && is_numeric_const(r)) { col = l; cst = r; }
        else if (r->op == W_COL && is_numeric_const(l)) { col = r; cst = l; code = flip_code(code); }
        else return false;
        Column *c = tbl->find(col->i);
        if (!c || (c->type.nullable && !in_coalesce)) return false;
        if (e->nterms >= MAX_TERMS) return false;
        Node tmp;
        if (cst->op == W_BOOL) { tmp.op = W_I64; tmp.i = cst->i; cst = &tmp; }
        Term *t = &e->terms[e->nterms];
        if (!make_term(tbl, scan, col, cst, code, t)) return false;
        if (t->constant_result == 1 && c->type.nullable) {
            // true for every value, still false for a missing one (coalesce(missing, false)): keep a comparison that every
            // value passes, so that the scans apply the column's missing bits
            t->constant_result = -1;
            if (t->cls == VC_FLT) { t->code = 1; t->cf = std::numeric_limits<double>::quiet_NaN(); }   // x != NaN
            else { t->code = 5; t->ci = t->cls == VC_INT ? INT64_MIN : 0; }                             // x >= typemin
        }
        e->nterms++;
        return true;
    }
    return false;
}

int compile_expr(dfdb_table *tbl, dfdb_scan *scan, Rdr &r, Expr *e, TVal *result)
{
    const uint8_t *start = r.p;
    std::unique_ptr<Node> root;
    int rc = parse_tree(r, &root);
    if (rc) return rc;
    e->wire.assign(start, r.p);
    memset(&e->prog, 0, sizeof e->prog);
    Compiler c{tbl, scan, e, &e->prog};
    rc = c.compile(root.get(), result);
    if (rc) return rc;
    if (c.maxdepth > VM_MAX_STACK) return fail(DFDB_ERR_UNSUPPORTED, "expression too deep");
    e->prog.result_class = result->cls;
    e->prog.result_nullable = result->nullable;
    e->prog.result_bits = result->bits;
    e->prog.result_uns = result->cls == VC_UINT;
    e->nterms = 0;
    e->simple = result->cls == VC_BOOL && !result->nullable && match_simple(tbl, scan, root.get(), false, e);
    if (!e->simple) e->nterms = 0;
    e->inset_slot = -1;
    if ((root->op == W_IN || root->op == W_INSET) && root->kids[0]->op == W_COL && !result->nullable) {
        const int cls = scan->sets[(size_t)e->sets[0]].cls;
        if (cls != VC_STR)
            for (size_t i = 0; i < scan->slots.size(); i++) if (scan->slots[i] == root->kids[0]->i) e->inset_slot = (int)i;
    }
    return DFDB_OK;
}

}  // namespace

int plan_parse(dfdb_table *t, const uint8_t *bytes, int64_t len, dfdb_scan *s)
{
    Rdr r{bytes, bytes + len};
    if (len < 12 || r.u32() != 0x31504644u) return fail(DFDB_ERR_ARGUMENT, "bad plan magic");
    uint32_t nstages = r.u32();
    if (r.bad || nstages > 1024) return fail(DFDB_ERR_ARGUMENT, "bad plan");
    s->stages.resize(nstages);
    for (auto &st : s->stages) {
        st.kind = r.u8();
        if (st.kind == ST_RANGE) {
            st.start = r.i64(); st.step = r.i64(); st.stop = r.i64();
            if (r.bad) return fail(DFDB_ERR_ARGUMENT, "truncated plan");
            if (st.step == 0) return fail(DFDB_ERR_ARGUMENT, "step cannot be zero");
            bool empty = st.step > 0 ? st.start > st.stop : st.start < st.stop;
            // RangeToProcess takes minimum/maximum of the range, which throw on an empty range (selection.jl:73)
            if (empty) return fail(DFDB_ERR_ARGUMENT, "range must be non-empty");
            st.first = std::min(st.start, st.stop);
            st.last = std::max(st.start, st.stop);
        } else if (st.kind == ST_INDEXVEC) {
            uint32_t n = r.u32();
            if (r.bad || r.p + 8ull * n > r.end) return fail(DFDB_ERR_ARGUMENT, "truncated plan");
            if (n == 0) return fail(DFDB_ERR_ARGUMENT, "reducing over an empty collection is not allowed");
            st.idx.resize(n);
            memcpy(st.idx.data(), r.p, 8ull * n);
            r.p += 8ull * n;
            std::sort(st.idx.begin(), st.idx.end());
            st.idx.erase(std::unique(st.idx.begin(), st.idx.end()), st.idx.end());
            st.first = st.idx.front();
            st.last = st.idx.back();
        } else if (st.kind == ST_PRED) {
            TVal res;
            int rc = compile_expr(t, s, r, &st.e, &res);
            if (rc) return rc;
            // _check_element selection.jl:52-55
            if (res.cls != VC_BOOL || res.nullable) return fail(DFDB_ERR_ARGUMENT, "Function for selection must have Bool result type");
        } else {
            return fail(DFDB_ERR_ARGUMENT, "bad stage kind %d", st.kind);
        }
    }
    uint32_t nproj = r.u32();
    if (r.bad || nproj > 4096) return fail(DFDB_ERR_ARGUMENT, "bad plan");
    s->projs.resize(nproj);
    for (auto &p : s->projs) {
        p.kind = r.u8();
        if (p.kind == PJ_COL) {
            p.col = r.i64();
            if (r.bad) return fail(DFDB_ERR_ARGUMENT, "truncated plan");
            Column *c = t->find(p.col);
            if (!c) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)p.col);
            p.type = c->type;
        } else if (p.kind == PJ_EXPR) {
            TVal res;
            int rc = compile_expr(t, s, r, &p.e, &res);
            if (rc) return rc;
            p.type.nullable = res.nullable;
            if (res.cls == VC_INT || res.cls == VC_UINT) {
                static const int sk[] = {DFDB_I8, DFDB_I16, DFDB_I32, DFDB_I64}, uk[] = {DFDB_U8, DFDB_U16, DFDB_U32, DFDB_U64};
                int w = res.bits == 8 ? 0 : res.bits == 16 ? 1 : res.bits == 32 ? 2 : 3;
                p.type.kind = res.cls == VC_UINT ? uk[w] : sk[w];
                p.type.elsize = res.bits / 8;
            } else if (res.cls == VC_FLT) {
                p.type.kind = res.bits == 32 ? DFDB_F32 : DFDB_F64;
                p.type.elsize = res.bits / 8;
            } else if (res.cls == VC_BOOL) {
                p.type.kind = DFDB_BOOL;
                p.type.elsize = 1;
            } else {
                return fail(DFDB_ERR_UNSUPPORTED, "computed String columns are not supported");
            }
        } else {
            return fail(DFDB_ERR_ARGUMENT, "bad projection kind %d", p.kind);
        }
    }
    if (s->slots.size() > (size_t)MAX_SLOTS) return fail(DFDB_ERR_UNSUPPORTED, "too many columns in one scan (max %d)", MAX_SLOTS);
    return DFDB_OK;
}

}  // namespace dfdb
