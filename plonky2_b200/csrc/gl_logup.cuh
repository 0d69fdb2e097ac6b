// gl_logup.cuh -- one trace row of starky's logUp helper columns (lookup_helper_columns / get_helper_cols,
// starky/src/lookup.rs:579-652,746-789).
//
// The reference builds the helper columns column by column: for every looking column it evaluates f_i + gamma on all
// rows, inverts the whole column with batch_multiplicative_inverse, multiplies by the filter and adds the chunk's columns;
// then it inverts t + gamma the same way and runs the Z recurrence. Inverses are unique, so a row can do the same work for
// itself: evaluate every denominator of the row (each looking column and the table, for every challenge), invert them with
// ONE batch inversion, and write the chunk sums. The Z recurrence Z(i+1) = Z(i) + d(i) is left to an exclusive prefix
// scan over the rows; this row writes its term d(i) = sum_k h_k(i) - m(i) / (t(i) + gamma).
//
// The same source runs on the host in tests/emu/logup_emu.cpp (threads as a loop).
#pragma once
#include "../../include/plonky2_b200.h"
#include "gl_field.cuh"

namespace gl {

struct LogupParams {
    const uint64_t* trace;  // column c at trace + c * col_stride
    size_t col_stride;
    size_t n;               // rows (a power of two)
    gl_logup_desc d;        // pointers valid where the evaluation runs
    const uint64_t* challenges;
    uint32_t n_challenges;
    uint32_t chunk;         // max(1, constraint_degree - 1)
    uint64_t* out;          // helper columns, column j at out + j * n (the Z columns are filled by the scan)
    uint64_t* zterm;        // one column of n terms d(i) per (lookup, challenge), in output order
};

// Column::eval_table (lookup.rs:318-329)
GL_HD uint64_t logup_column(const LogupParams& p, uint32_t c, size_t i) {
    const gl_logup_column col = p.d.columns[c];
    const size_t inext = (i + 1) & (p.n - 1);
    uint64_t acc = col.constant;
    for (uint32_t t = 0; t < col.n_terms; t++) {
        const gl_logup_term tm = p.d.terms[col.term_begin + t];
        acc = add(acc, mul(p.trace[(size_t)tm.col * p.col_stride + (tm.next ? inext : i)], tm.coeff));
    }
    return acc;
}

// Filter::eval_table (lookup.rs:114-125)
GL_HD uint64_t logup_filter(const LogupParams& p, uint32_t c, size_t i) {
    const gl_logup_filter f = p.d.filters[c];
    uint64_t acc = 0;
    for (uint32_t j = 0; j < f.n_prods; j++)
        acc = add(acc, mul(logup_column(p, p.d.filter_columns[f.prod_begin + 2 * j], i),
                           logup_column(p, p.d.filter_columns[f.prod_begin + 2 * j + 1], i)));
    for (uint32_t j = 0; j < f.n_sums; j++) acc = add(acc, logup_column(p, p.d.filter_columns[f.sum_begin + j], i));
    return acc;
}

// Row i of every helper column. den, pre: GL_LOGUP_MAX_DENOMINATORS words of scratch. Returns false if a denominator is
// zero (the outputs of the row are then meaningless).
GL_HD bool logup_eval_row(const LogupParams& p, size_t i, uint64_t* den, uint64_t* pre) {
    const uint32_t nc = p.n_challenges;
    // denominators, lookup-major, then challenge, then (looking columns..., table): den[o + c*(nl+1) + k]
    uint32_t o = 0;
    for (uint32_t l = 0; l < p.d.n_lookups; l++) {
        const gl_logup_lookup lk = p.d.lookups[l];
        const uint32_t w = lk.n_looking + 1;
        for (uint32_t k = 0; k <= lk.n_looking; k++) {
            const uint64_t f = logup_column(p, k < lk.n_looking ? lk.looking_begin + k : lk.table, i);
            for (uint32_t c = 0; c < nc; c++) den[o + c * w + k] = add(f, p.challenges[c]);  // combine with beta = 1
        }
        o += w * nc;
    }
    // Montgomery batch inversion of the row's o denominators (field/src/types.rs:133-223 computes the same inverses)
    uint64_t run = 1;
    bool ok = true;
    for (uint32_t k = 0; k < o; k++) {
        if (canon(den[k]) == 0) ok = false;
        run = mul(run, den[k]);
        pre[k] = run;
    }
    uint64_t inv_run = inv(run);
    for (uint32_t k = o; k-- > 0;) {
        const uint64_t di = k ? mul(inv_run, pre[k - 1]) : inv_run;
        inv_run = mul(inv_run, den[k]);
        den[k] = di;
    }
    // chunk sums and Z terms; pre[] now holds the lookup's filter values
    o = 0;
    uint32_t col = 0, z = 0;
    for (uint32_t l = 0; l < p.d.n_lookups; l++) {
        const gl_logup_lookup lk = p.d.lookups[l];
        const uint32_t w = lk.n_looking + 1;
        for (uint32_t k = 0; k < lk.n_looking; k++) pre[k] = logup_filter(p, lk.looking_begin + k, i);
        const uint64_t m = logup_column(p, lk.frequencies, i);
        for (uint32_t c = 0; c < nc; c++) {
            const uint64_t* dv = den + o + c * w;
            uint64_t sum = 0;
            for (uint32_t k0 = 0; k0 < lk.n_looking; k0 += p.chunk) {
                const uint32_t k1 = k0 + p.chunk < lk.n_looking ? k0 + p.chunk : lk.n_looking;
                uint64_t h = 0;
                for (uint32_t k = k0; k < k1; k++) h = add(h, mul(pre[k], dv[k]));
                p.out[(size_t)col++ * p.n + i] = canon(h);
                sum = add(sum, h);
            }
            p.zterm[(size_t)z++ * p.n + i] = canon(sub(sum, mul(m, dv[lk.n_looking])));
            col++;  // the Z column itself
        }
        o += w * nc;
    }
    return ok;
}

}  // namespace gl
