// Host run of the device evaluation of starky's logUp helper columns (plonky2_b200/csrc/gl_logup.cuh): the same
// logup_eval_row the kernel k_logup_rows calls per thread, with threads as a loop, then the Z recurrence the device runs as
// an exclusive prefix scan. Test infrastructure: built as a shared library by tests/test_stark_prove.py and compared with
// the column-wise restatement in logup_oracle.cpp.
#include <vector>
#include "../../plonky2_b200/csrc/gl_logup.cuh"
using namespace gl;

// out: the helper columns (column j at out + j * n), laid out like gl_stark_lookup_helper_columns. Returns 1 if a
// denominator was zero, 2 if a row has more than GL_LOGUP_MAX_DENOMINATORS denominators.
extern "C" int emu_logup_helper_columns(const uint64_t* trace, size_t col_stride, uint32_t log_n, const gl_logup_desc* desc,
                                        const uint64_t* challenges, uint32_t n_challenges, uint32_t constraint_degree,
                                        uint64_t* out) {
    const size_t n = (size_t)1 << log_n;
    const uint32_t chunk = constraint_degree > 2 ? constraint_degree - 1 : 1;
    std::vector<uint32_t> zcols;
    uint32_t n_out = 0, n_den = 0;
    for (uint32_t l = 0; l < desc->n_lookups; l++) {
        const gl_logup_lookup lk = desc->lookups[l];
        n_den += (lk.n_looking + 1) * n_challenges;
        for (uint32_t c = 0; c < n_challenges; c++) {
            n_out += (lk.n_looking + chunk - 1) / chunk + 1;
            zcols.push_back(n_out - 1);
        }
    }
    if (n_den > GL_LOGUP_MAX_DENOMINATORS) return 2;
    std::vector<uint64_t> zterm(zcols.size() * n);
    LogupParams p;
    p.trace = trace;
    p.col_stride = col_stride;
    p.n = n;
    p.d = *desc;
    p.challenges = challenges;
    p.n_challenges = n_challenges;
    p.chunk = chunk;
    p.out = out;
    p.zterm = zterm.data();
    int bad = 0;
    for (size_t i = 0; i < n; i++) {  // one "thread" per row
        uint64_t den[GL_LOGUP_MAX_DENOMINATORS], pre[GL_LOGUP_MAX_DENOMINATORS];
        if (!logup_eval_row(p, i, den, pre)) bad = 1;
    }
    for (size_t z = 0; z < zcols.size(); z++) {  // exclusive prefix sums (what k_scan3_*<AddOp> computes)
        uint64_t acc = 0;
        for (size_t i = 0; i < n; i++) {
            out[(size_t)zcols[z] * n + i] = canon(acc);
            acc = add(acc, zterm[z * n + i]);
        }
    }
    return bad;
}
