/* unique_ref.c -- CPU reference for unique(col): Base.unique over a materialized column (the oracle's block iteration with
 * the selection stages applied), restated in C so that it keeps up with columns of hundreds of millions of rows.
 * Base.unique keeps a Set of the values seen so far (isequal) and emits a value the first time it appears; here the set is
 * an open-addressing table of row indices, and the result is the list of first-appearance rows in row order.
 *
 * isequal: missing is one value, every NaN is one value, -0.0 and 0.0 differ, strings compare by bytes ("" is not missing). */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

enum { K_F16 = 11, K_F32 = 12, K_F64 = 13 };

static uint64_t mix(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

static uint64_t key_of(const uint8_t *p, int es, int kind)
{
    uint64_t v = 0;
    memcpy(&v, p, (size_t)es);
    if (kind == K_F16 && (v & 0x7c00u) == 0x7c00u && (v & 0x3ffu)) return 0x7e00u;
    if (kind == K_F32 && (v & 0x7f800000u) == 0x7f800000u && (v & 0x7fffffu)) return 0x7fc00000u;
    if (kind == K_F64 && (v & 0x7ff0000000000000ull) == 0x7ff0000000000000ull && (v & 0xfffffffffffffull)) return 0x7ff8000000000000ull;
    return v;
}

static size_t table_cap(int64_t n)
{
    size_t cap = 1024;
    while (cap < 2 * (size_t)n) cap <<= 1;
    return cap;
}

/* fixed width: vals n * es bytes, miss n bytes (1 = missing) or NULL; out_idx receives the first-appearance rows; returns
 * their number (-1: out of memory) */
int64_t uref_fixed(const uint8_t *vals, const uint8_t *miss, int es, int kind, int64_t n, int64_t *out_idx)
{
    const size_t cap = table_cap(n);
    int64_t *tab = malloc(cap * sizeof *tab);
    if (!tab) return -1;
    memset(tab, 0xff, cap * sizeof *tab);
    int64_t m = 0;
    for (int64_t i = 0; i < n; i++) {
        const int mi = miss && miss[i];
        const uint64_t k = mi ? 0 : key_of(vals + i * es, es, kind);
        size_t s = (size_t)(mi ? mix(0xA5A5A5A5A5A5A5A5ull) : mix(k)) & (cap - 1);
        for (;; s = (s + 1) & (cap - 1)) {
            const int64_t j = tab[s];
            if (j < 0) { tab[s] = i; out_idx[m++] = i; break; }
            const int mj = miss && miss[j];
            if (mi == mj && (mi || key_of(vals + j * es, es, kind) == k)) break;
        }
    }
    free(tab);
    return m;
}

/* strings: sizes n Int32 (-1 = missing), chars the concatenation of the non-missing values */
int64_t uref_strings(const int32_t *sizes, const uint8_t *chars, int64_t n, int64_t *out_idx)
{
    const size_t cap = table_cap(n);
    int64_t *tab = malloc(cap * sizeof *tab), *off = malloc(((size_t)n + 1) * sizeof *off);
    if (!tab || !off) { free(tab); free(off); return -1; }
    memset(tab, 0xff, cap * sizeof *tab);
    off[0] = 0;
    for (int64_t i = 0; i < n; i++) off[i + 1] = off[i] + (sizes[i] > 0 ? sizes[i] : 0);
    int64_t m = 0;
    for (int64_t i = 0; i < n; i++) {
        const int32_t sz = sizes[i];
        const uint8_t *p = chars + off[i];
        uint64_t f = 0xCBF29CE484222325ull;
        for (int32_t k = 0; k < sz; k++) f = (f ^ p[k]) * 0x100000001B3ull;
        size_t s = (size_t)mix(f ^ ((uint64_t)(uint32_t)sz << 32)) & (cap - 1);
        for (;; s = (s + 1) & (cap - 1)) {
            const int64_t j = tab[s];
            if (j < 0) { tab[s] = i; out_idx[m++] = i; break; }
            if (sizes[j] == sz && (sz <= 0 || memcmp(chars + off[j], p, (size_t)sz) == 0)) break;
        }
    }
    free(tab);
    free(off);
    return m;
}

/* chars of rows idx[0..m) of a string column, concatenated (out holds their total size) */
void uref_take_strings(const int32_t *sizes, const uint8_t *chars, int64_t n, const int64_t *idx, int64_t m, uint8_t *out)
{
    int64_t *off = malloc(((size_t)n + 1) * sizeof *off);
    if (!off) abort();
    off[0] = 0;
    for (int64_t i = 0; i < n; i++) off[i + 1] = off[i] + (sizes[i] > 0 ? sizes[i] : 0);
    for (int64_t k = 0; k < m; k++) {
        const int32_t sz = sizes[idx[k]];
        if (sz > 0) { memcpy(out, chars + off[idx[k]], (size_t)sz); out += sz; }
    }
    free(off);
}
