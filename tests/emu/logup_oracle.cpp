// Column-wise restatement of starky's lookup_helper_columns (starky/src/lookup.rs:579-652) and get_helper_cols
// (lookup.rs:746-789), as a checker for the device path (which works row by row). Test infrastructure only: built by
// tests/test_stark_prove.py into its temporary directory. It takes the flat lookup descriptor of include/plonky2_b200.h
// (types only) and shares no code with the product.
#include <cstdint>
#include <vector>
#include "../../include/plonky2_b200.h"

namespace {
typedef unsigned __int128 u128;
const uint64_t P = 0xFFFFFFFF00000001ull;
uint64_t fadd(uint64_t a, uint64_t b) { return (uint64_t)(((u128)a + b) % P); }
uint64_t fsub(uint64_t a, uint64_t b) { return (uint64_t)(((u128)a + P - b % P) % P); }
uint64_t fmul(uint64_t a, uint64_t b) { return (uint64_t)(((u128)a * b) % P); }
uint64_t fexp(uint64_t b, uint64_t e) {
    uint64_t r = 1;
    for (b %= P; e; e >>= 1, b = fmul(b, b))
        if (e & 1) r = fmul(r, b);
    return r;
}
typedef std::vector<uint64_t> Col;

// F::batch_multiplicative_inverse (field/src/types.rs:133-223): panics on zero -> false
bool batch_multiplicative_inverse(Col& x) {
    Col pre(x.size());
    uint64_t run = 1;
    for (size_t i = 0; i < x.size(); i++) {
        if (x[i] % P == 0) return false;
        run = fmul(run, x[i]);
        pre[i] = run;
    }
    uint64_t inv = fexp(run, P - 2);
    for (size_t i = x.size(); i-- > 0;) {
        const uint64_t xi = i ? fmul(inv, pre[i - 1]) : inv;
        inv = fmul(inv, x[i]);
        x[i] = xi;
    }
    return true;
}

struct Oracle {
    const uint64_t* trace;
    size_t stride, n;
    const gl_logup_desc* d;
    // Column::eval_table (lookup.rs:318-329)
    uint64_t column(uint32_t c, size_t row) const {
        const gl_logup_column col = d->columns[c];
        uint64_t acc = 0;
        for (uint32_t t = 0; t < col.n_terms; t++) {  // linear_combination, then next_row_linear_combination
            const gl_logup_term tm = d->terms[col.term_begin + t];
            if (!tm.next) acc = fadd(acc, fmul(trace[tm.col * stride + row] % P, tm.coeff % P));
        }
        for (uint32_t t = 0; t < col.n_terms; t++) {
            const gl_logup_term tm = d->terms[col.term_begin + t];
            if (tm.next) acc = fadd(acc, fmul(trace[tm.col * stride + (row + 1) % n] % P, tm.coeff % P));
        }
        return fadd(acc, col.constant % P);
    }
    // Filter::eval_table (lookup.rs:114-125)
    uint64_t filter(uint32_t c, size_t row) const {
        const gl_logup_filter f = d->filters[c];
        uint64_t prods = 0, sums = 0;
        for (uint32_t j = 0; j < f.n_prods; j++)
            prods = fadd(prods, fmul(column(d->filter_columns[f.prod_begin + 2 * j], row),
                                     column(d->filter_columns[f.prod_begin + 2 * j + 1], row)));
        for (uint32_t j = 0; j < f.n_sums; j++) sums = fadd(sums, column(d->filter_columns[f.sum_begin + j], row));
        return fadd(prods, sums);
    }
    Col eval_all_rows(uint32_t c) const {
        Col v(n);
        for (size_t r = 0; r < n; r++) v[r] = column(c, r);
        return v;
    }
};
}  // namespace

// All helper columns, lookup-major, challenge-minor (prover.rs:159-173). Returns 1 on a zero denominator.
extern "C" int oracle_logup_helper_columns(const uint64_t* trace, size_t col_stride, uint32_t log_n, const gl_logup_desc* desc,
                                           const uint64_t* challenges, uint32_t n_challenges, uint32_t constraint_degree,
                                           uint64_t* out) {
    const size_t n = (size_t)1 << log_n;
    const Oracle o{trace, col_stride, n, desc};
    const uint32_t chunk = constraint_degree >= 1 ? (constraint_degree - 1 ? constraint_degree - 1 : 0) : 1;
    if (chunk == 0) return 2;  // chunks(0) panics in the reference
    size_t col = 0;
    for (uint32_t l = 0; l < desc->n_lookups; l++) {
        const gl_logup_lookup lk = desc->lookups[l];
        for (uint32_t ci = 0; ci < n_challenges; ci++) {
            const uint64_t challenge = challenges[ci] % P;
            // get_helper_cols: per chunk, per column: combine (beta = 1), invert, multiply by the filter, add
            for (uint32_t k0 = 0; k0 < lk.n_looking; k0 += chunk) {
                Col acc;
                for (uint32_t k = k0; k < lk.n_looking && k < k0 + chunk; k++) {
                    Col combined = o.eval_all_rows(lk.looking_begin + k);
                    for (auto& x : combined) x = fadd(x, challenge);  // reduce_with_powers([f], 1) + gamma
                    if (!batch_multiplicative_inverse(combined)) return 1;
                    for (size_t r = 0; r < n; r++) combined[r] = fmul(combined[r], o.filter(lk.looking_begin + k, r));
                    if (acc.empty()) acc = combined;
                    else
                        for (size_t r = 0; r < n; r++) acc[r] = fadd(acc[r], combined[r]);
                }
                for (size_t r = 0; r < n; r++) out[col * n + r] = acc[r];
                col++;
            }
            const size_t nh = col;  // helper columns of this challenge end here
            const size_t h0 = nh - (lk.n_looking + chunk - 1) / chunk;
            Col table = o.eval_all_rows(lk.table);
            for (auto& x : table) x = fadd(challenge, x);
            if (!batch_multiplicative_inverse(table)) return 1;
            const Col freq = o.eval_all_rows(lk.frequencies);
            // Z(0) = 0, Z(i+1) = Z(i) + sum_k h_k(i) - m(i) / (t(i) + gamma)
            uint64_t z = 0;
            out[col * n] = 0;
            for (size_t i = 0; i + 1 < n; i++) {
                uint64_t x = 0;
                for (size_t c = h0; c < nh; c++) x = fadd(x, out[c * n + i]);
                x = fsub(x, fmul(freq[i], table[i]));
                z = fadd(z, x);
                out[col * n + i + 1] = z;
            }
            col++;
        }
    }
    return 0;
}
