/*
 * plonky2_b200.h -- C ABI of the B200-native plonky2 prover hot path
 * (Goldilocks NTT / coset-LDE / Poseidon Merkle commitment / FRI commit phase, sm_100a CUDA).
 *
 * The reference (0xPolygonZero/plonky2 @ 5d9da5a) is pure Rust with no FFI; the seam this ABI
 * replaces is the trait/struct surface listed in SURVEY.md section 8(b). Each entry point below
 * cites the reference interface it stands in for. A Rust binding (`extern "C"` block + safe
 * wrappers for PolynomialBatch / MerkleTree / fri_proof) is sketched in INTEGRATION.md.
 *
 * Conventions
 *  - Field element = uint64_t, exactly the reference's #[repr(transparent)] GoldilocksField(pub u64)
 *    (field/src/goldilocks_field.rs:23-25). Inputs may be non-canonical (any u64); every output is
 *    CANONICAL (< p = 2^64 - 2^32 + 1), little-endian host.
 *  - F_{p^2} element = 2 consecutive words (c0, c1), X^2 = 7 (field/src/goldilocks_extensions.rs:14-27).
 *  - Hash = 4 words (plonky2/src/hash/hash_types.rs:20-27).
 *  - `mem` arguments: GL_MEM_HOST (pageable or pinned host memory; the call does the copies) or
 *    GL_MEM_DEVICE (device pointers on the context's device; no copies, stream-ordered).
 *  - Every function returns an int status: GL_OK or a GL_ERR_* code; gl_last_error(ctx) gives text.
 *    Nothing unwinds or aborts across the ABI. Shape errors mirror the reference's panics
 *    (field/src/fft.rs:171-177, plonky2/src/hash/merkle_tree.rs:195-200, plonky2/src/fri/oracle.rs:128).
 *  - One gl_ctx per (device, stream). Calls on one context are serialised by the caller; different
 *    contexts are independent (no global mutable state). The library owns all device memory behind
 *    opaque handles; the caller owns every host buffer.
 *  - There is NO CPU fallback: without a CUDA device gl_ctx_create fails with GL_ERR_CUDA.
 */
#ifndef PLONKY2_B200_H
#define PLONKY2_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GL_OK 0
#define GL_ERR_BAD_SHAPE 1   /* not a power of two, inconsistent degrees, cap_height > log2(leaves) ... */
#define GL_ERR_OOM 2
#define GL_ERR_CUDA 3
#define GL_ERR_UNSUPPORTED 4 /* size beyond this build's limits (log_n > 30 per transform) */
#define GL_ERR_BAD_ARG 5
#define GL_ERR_POW_FAILED 6
#define GL_ERR_DIV_ZERO 7    /* "Tried to invert zero" (field/src/types.rs batch_multiplicative_inverse panics) */

#define GL_MEM_HOST 0
#define GL_MEM_DEVICE 1

#define GL_SALT_SIZE 4 /* plonky2/src/fri/oracle.rs:26 */

typedef struct gl_ctx gl_ctx;
typedef struct gl_commit gl_commit; /* a PolynomialBatch on the device */
typedef struct gl_merkle gl_merkle; /* a MerkleTree on the device */
typedef struct gl_fri gl_fri;       /* FRI commit-phase state on the device */

/* ---- context -------------------------------------------------------------------------------- */
/* stream: a cudaStream_t (NULL = a private non-blocking stream is created). */
int gl_ctx_create(int device, void* stream, gl_ctx** out);
void gl_ctx_destroy(gl_ctx* ctx);
const char* gl_last_error(const gl_ctx* ctx); /* ctx may be NULL: last error of the calling thread */
int gl_ctx_synchronize(gl_ctx* ctx);
/* the cudaStream_t every call on this context is ordered on (callers that mix their own stream work with the
 * library's -- torch tensors, NCCL -- must issue it on this stream or order it with events) */
void* gl_ctx_stream(const gl_ctx* ctx);
/* number of kernels this context has launched so far (for bench.py's gpu_launches) */
uint64_t gl_ctx_launch_count(const gl_ctx* ctx);
/* tuning: columns per multi-pass NTT group (scratch = group * n * 8 bytes; default: as many as fit 1 GiB) */
int gl_ctx_set_ntt_group(gl_ctx* ctx, uint32_t columns);
/* Optional CUDA-event phase timing on the context's stream (the analogue of the reference's TimingTree
 * scopes "IFFT" / "FFT + blinding" / "build Merkle tree", plonky2/src/fri/oracle.rs:65-103). */
#define GL_PHASE_INTT 0          /* from_values' iNTT of all columns */
#define GL_PHASE_LDE 1           /* coset LDE into leaf-major rows (passes A + B, all cosets) */
#define GL_PHASE_LEAF_HASH 2     /* the Poseidon leaf-hash kernel */
#define GL_PHASE_MERKLE_LEVELS 3 /* all two_to_one levels up to the cap */
#define GL_NUM_PHASES 4
int gl_ctx_set_profiling(gl_ctx* ctx, int on);
/* accumulated milliseconds and number of scopes of `phase` since the last reset (synchronises) */
int gl_ctx_phase_ms(gl_ctx* ctx, int phase, double* ms, uint64_t* count);
int gl_ctx_reset_phases(gl_ctx* ctx);

/* ---- NTT  (field/src/fft.rs:53-91 fft_with_options / ifft_with_options;
 *            field/src/polynomial/mod.rs:63-73,280-293 coset_ifft / coset_fft_with_options) -------- */
/* In place, natural order in and out, `batch` columns of n = 2^log_n words, column b at
 * data + b*stride.  inverse = 0: out[k] = sum_j in[j] * (shift*w_n^k)^j;  inverse = 1: the inverse map
 * (coefficients of the polynomial whose values on shift*<w_n> are `data`).  coset_shift = 1 for the
 * plain subgroup.  zero_factor_log is the reference's `zero_factor` hint (top 1 - 2^-r of the input is
 * zero); results do not depend on it. */
int gl_ntt(gl_ctx* ctx, uint64_t* data, uint32_t log_n, uint32_t batch, size_t stride, int inverse,
           uint32_t zero_factor_log, uint64_t coset_shift, int mem);

/* Out-of-place, device-resident variant with up to 8 destinations: column b of the result is written to
 * outs[i] + b*out_stride for EVERY i. With outs[] = the same offset inside each peer GPU's (NVLink-mapped) coefficient
 * buffer -- or one multicast address -- the last pass of the column-sharded iNTT IS the all-gather of SURVEY.md
 * section 8(e): no separate collective, the transfer overlaps the butterflies tile by tile. Natural order in and out,
 * no coset shift; replaces `values.into_par_iter().map(|v| v.ifft())` (oracle.rs:65-69) on G GPUs. */
int gl_ntt_bcast(gl_ctx* ctx, const uint64_t* in, size_t in_stride, uint32_t log_n, uint32_t batch, int inverse,
                 uint64_t* const* outs, uint32_t n_outs, size_t out_stride);

/* Device copy of `words` u64 (even, 16-byte aligned) from this GPU's memory to every destination with 128-byte
 * line stores: the transfer half of the coefficient all-gather when the destinations are peer mappings or a multicast
 * address (measured at link speed, unlike the 64-byte segments gl_ntt_bcast's transposing stores produce).
 * max_ctas bounds the grid (0 = 2 per SM) so the copy can share the GPU with a compute stream. */
int gl_bcast(gl_ctx* ctx, const uint64_t* src, size_t words, uint64_t* const* dests, uint32_t n_dests, uint32_t max_ctas);

/* ---- PolynomialBatch  (plonky2/src/fri/oracle.rs:30-37,57-147) -------------------------------- */
/* from_values (is_coeffs = 0) / from_coeffs (is_coeffs = 1): B columns of n = 2^log_n words at
 * cols + b*col_stride.  salt: NULL (blinding = false) or GL_SALT_SIZE columns of N = n << rate_bits
 * words (column s at salt + s*N) appended to every leaf -- the reference draws them from OsRng
 * (oracle.rs:133-137); here the caller supplies them so the result is deterministic.
 * The handle keeps coefficients (B x n), the LDE (W columns of N values in leaf order, leaf j = LDE row bitrev(j)),
 * digests (reference layout, merkle_tree.rs:50-58) and the cap on the device. */
int gl_commit_create(gl_ctx* ctx, const uint64_t* cols, size_t col_stride, uint32_t B, uint32_t log_n,
                     uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt, int is_coeffs,
                     int mem, gl_commit** out);
/* Row-block sharded variant (one shard per GPU; SURVEY.md section 8e): shard g of G = 2^s <= 2^cap_height
 * builds leaf rows [g*N/G, (g+1)*N/G) -- all columns on the coset (g*w_N^{bitrev_s(g)})<w_{N/G}> -- their
 * digests and cap entries [g*C/G, (g+1)*C/G). Concatenating the shards' leaves / digests / caps in shard
 * order gives exactly the single-device commitment; only the C/G cap entries need to be exchanged
 * (one all-gather). Accessors of a sharded handle return the LOCAL rows / digests / cap entries. */
int gl_commit_create_sharded(gl_ctx* ctx, const uint64_t* cols, size_t col_stride, uint32_t B, uint32_t log_n,
                             uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt, int is_coeffs,
                             int mem, uint32_t shard_index, uint32_t num_shards, gl_commit** out);
/* The same commitment built incrementally, for pipelines whose columns become available in groups (chunks of a
 * host trace in flight, coefficient groups arriving from peer GPUs, Z / partial-product columns computed on the device):
 *   gl_commit_begin        allocates the handle's device state. coeff_storage: NULL, or a caller-owned device matrix of
 *                          B x n words (column b at + b*n) that the handle uses as PolynomialBatch.polynomials (it must
 *                          outlive the handle; columns passed from inside it are not copied);
 *   gl_commit_add_columns  columns [first_col, first_col + count), each exactly once, in any order:
 *                          kind GL_COLS_VALUES (iNTT + LDE), GL_COLS_COEFFS (canonicalise + LDE) or
 *                          GL_COLS_COEFFS_CANONICAL (LDE only);
 *   gl_commit_finish       salt columns (iff blinding) and the Merkle tree. Accessors are valid after it. */
#define GL_COLS_VALUES 0
#define GL_COLS_COEFFS 1
#define GL_COLS_COEFFS_CANONICAL 2
int gl_commit_begin(gl_ctx* ctx, uint32_t B, uint32_t log_n, uint32_t rate_bits, uint32_t cap_height, int blinding,
                    uint32_t shard_index, uint32_t num_shards, uint64_t* coeff_storage, gl_commit** out);
int gl_commit_add_columns(gl_commit* c, uint32_t first_col, uint32_t count, const uint64_t* cols, size_t col_stride,
                          int kind, int mem);
int gl_commit_finish(gl_commit* c, const uint64_t* salt, int mem);
int gl_commit_shard(const gl_commit* c, uint32_t* shard_index, uint32_t* num_shards);
void gl_commit_destroy(gl_commit* c);
/* shape queries */
uint32_t gl_commit_num_polys(const gl_commit* c);  /* B */
uint32_t gl_commit_leaf_width(const gl_commit* c); /* W = B + (salt ? 4 : 0) */
uint32_t gl_commit_degree_log(const gl_commit* c);
uint32_t gl_commit_rate_bits(const gl_commit* c);
uint32_t gl_commit_cap_height(const gl_commit* c);
/* PolynomialBatch.merkle_tree.cap: 4 * 2^cap_height words */
int gl_commit_cap(gl_commit* c, uint64_t* out, int mem);
/* PolynomialBatch.polynomials: B x n coefficients, column-major, column b at out + b*n */
int gl_commit_coeffs(gl_commit* c, uint64_t* out, int mem);
/* MerkleTree.leaves[row_begin .. row_begin + row_count): row-major, W words per leaf */
int gl_commit_leaves(gl_commit* c, size_t row_begin, size_t row_count, uint64_t* out, int mem);
/* MerkleTree.digests: 4 * 2 * (N - 2^cap_height) words, reference layout */
int gl_commit_digests(gl_commit* c, uint64_t* out, int mem);
/* get_lde_values(index, step) (oracle.rs:142-147): B words (salt removed) */
int gl_commit_get_lde_values(gl_commit* c, size_t index, size_t step, uint64_t* out);
/* MerkleTree::get + MerkleTree::prove (merkle_tree.rs:226-237) for `count` leaf indices:
 * out_leaves = count x W, out_paths = count x (log N - cap_height) x 4, siblings bottom-up. Host out. */
int gl_commit_open(gl_commit* c, const uint64_t* leaf_indices, size_t count, uint64_t* out_leaves,
                   uint64_t* out_paths);
/* eval_commitment of OpeningSet::new (plonky2/src/plonk/proof.rs:313-351): every polynomial of the batch
 * evaluated at one point z of F_{p^2}: out = B x 2 words (host). First "next" row of SURVEY section 8(f):
 * it keeps the coefficient D2H off the prover's critical path. */
int gl_commit_eval_ext(gl_commit* c, const uint64_t point[2], uint64_t* out);
/* OpeningSet::new (plonky2/src/plonk/proof.rs:313-351) / StarkOpeningSet::new (starky/src/proof.rs:221-260) as ONE call:
 * request i = every polynomial of commits[i] at points[point_index[i]] (F_{p^2}, 2 words each; e.g. zeta and g*zeta);
 * out = the requests' results concatenated in order, B_i x 2 words each; one power table per distinct point, one
 * D2H (mem = GL_MEM_HOST) or none (GL_MEM_DEVICE). Coefficients never leave the device. */
int gl_openings(gl_ctx* ctx, gl_commit* const* commits, const uint32_t* point_index, size_t n_evals,
                const uint64_t* points, size_t n_points, uint64_t* out, int mem);
/* device views (valid until destroy; for device-resident pipelines such as quotient evaluation).
 * The LDE is kept COLUMN-MAJOR on the device: the value of polynomial (or salt column) k at leaf j -- the LDE row
 * reverse_bits(j), oracle.rs:142-147 -- is at lde[k * col_stride + j]; col_stride = number of local leaves. The
 * reference's row-major MerkleTree.leaves is what gl_commit_leaves / gl_commit_open return. */
const uint64_t* gl_commit_dev_lde(const gl_commit* c, size_t* col_stride);
const uint64_t* gl_commit_dev_coeffs(const gl_commit* c);

/* ---- "next" rows (SURVEY.md section 8f) ------------------------------------------------------------------ */
/* wires_permutation_partial_products_and_zs (plonky2/src/plonk/prover.rs:387-449, util/partial_products.rs:13-37):
 * wires, sigmas = num_routed columns of n = 2^log_n values (column-major); k_is = num_routed host words;
 * out = (ceil(num_routed/degree)) columns of n values: the partial products, then Z LAST (the function's
 * return order). Produces the second commitment's input on the device. Fails with GL_ERR_DIV_ZERO
 * ("Tried to invert zero") where the reference's batch_multiplicative_inverse panics. */
int gl_partial_products_and_zs(gl_ctx* ctx, const uint64_t* wires, const uint64_t* sigmas, const uint64_t* k_is,
                               uint32_t log_n, uint32_t num_routed, uint64_t beta, uint64_t gamma, uint32_t degree,
                               uint64_t* out, int mem);

/* compute_lookup_polys (plonky2/src/plonk/prover.rs:458-577) for ONE challenge set deltas = (A, B, alpha, delta): the RE
 * polynomial followed by the num_partial_lookups partial Sum/LDC polynomials, as value columns of n = 2^log_n rows:
 * out = (num_partial_lookups + 1) columns of n words (column-major), num_partial_lookups =
 * ceil((num_routed_wires / 2) / (max_quotient_degree_factor - 1)). wires: the witness matrix, wire w of row i at
 * wires[w*n + i] (LookupGate wires 2s, 2s+1; LookupTableGate wires 3s, 3s+1, 3s+2: gates/lookup.rs:58-70,
 * gates/lookup_table.rs:64-83). lookup_rows: n_lookup_wires triples (last_lu_gate, last_lut_gate, first_lut_gate)
 * (LookupWire, plonk/circuit_builder.rs:75-87), processed in order like the reference. */
int gl_lookup_polys(gl_ctx* ctx, const uint64_t* wires, uint32_t log_n, uint32_t num_routed_wires,
                    uint32_t max_quotient_degree_factor, const uint64_t deltas[4], const uint32_t* lookup_rows,
                    uint32_t n_lookup_wires, uint64_t* out, int mem);

/* compute_quotient_polys of a STARK (starky/src/prover.rs:488-668): for every challenge alpha_j the values
 * (sum_k alpha_j^.. C_k(x)) / Z_H(x) on the coset g<w_size>, size = n << log2_ceil(quotient_degree_factor), read from the
 * trace commitment's LDE IN PLACE on the device (get_lde_values addressing, oracle.rs:142-147), then coset_ifft: n_alphas
 * polynomials of `size` coefficients at out_coeffs + j*size (DEVICE memory). The coefficients beyond
 * n * quotient_degree_factor are checked to vanish ("Quotient has failed ...", prover.rs:396-401 -> GL_ERR_BAD_ARG).
 * The constraints (Stark::eval_packed_generic, starky/src/stark.rs:40-70) are a straight-line program: value k is the
 * result of instruction k; GL_STARK_EMIT feeds a value to the ConstraintConsumer (constraint_consumer.rs:46-84).
 * consts = the public inputs followed by the program's constants. Split the result into degree-n chunks with
 * gl_commit_begin / gl_commit_add_columns(GL_COLS_COEFFS) to obtain the quotient commitment (prover.rs:391-421). */
#define GL_STARK_LOCAL 0 /* a = trace column: local row value */
#define GL_STARK_NEXT 1  /* a = trace column: next row value */
#define GL_STARK_CONST 2 /* a = index into consts */
#define GL_STARK_ADD 3   /* values a + b */
#define GL_STARK_SUB 4
#define GL_STARK_MUL 5
#define GL_STARK_EMIT 6  /* a = value, b = GL_STARK_CONSTRAINT / _TRANSITION / _FIRST_ROW / _LAST_ROW */
#define GL_STARK_AUX_LOCAL 7 /* a = auxiliary polynomial: local row value (gl_stark_quotient_aux only) */
#define GL_STARK_AUX_NEXT 8  /* a = auxiliary polynomial: next row value */
#define GL_STARK_CONSTRAINT 0
#define GL_STARK_TRANSITION 1
#define GL_STARK_FIRST_ROW 2
#define GL_STARK_LAST_ROW 3
#define GL_STARK_MAX_INSTR 256
#define GL_STARK_MAX_ALPHAS 4
#define GL_STARK_MAX_QD 8
typedef struct {
    uint16_t op, a, b, pad_;
} gl_stark_instr;
int gl_stark_quotient(gl_ctx* ctx, gl_commit* trace, const gl_stark_instr* program, uint32_t n_instr,
                      const uint64_t* consts, uint32_t n_consts, const uint64_t* alphas, uint32_t n_alphas,
                      uint32_t quotient_degree_factor, uint64_t* out_coeffs);
/* The same with the auxiliary polynomials (starky/src/prover.rs:488-668 with auxiliary_polys_commitment): GL_STARK_AUX_LOCAL /
 * GL_STARK_AUX_NEXT read aux's LDE in place with the trace's addressing. aux may be NULL (then this is gl_stark_quotient);
 * otherwise it has the trace's degree and rate. The logUp constraints (eval_packed_lookups_generic, lookup.rs:804-863) are
 * ordinary instructions of the program, emitted after the STARK's own; their challenges travel in consts. */
int gl_stark_quotient_aux(gl_ctx* ctx, gl_commit* trace, gl_commit* aux, const gl_stark_instr* program, uint32_t n_instr,
                          const uint64_t* consts, uint32_t n_consts, const uint64_t* alphas, uint32_t n_alphas,
                          uint32_t quotient_degree_factor, uint64_t* out_coeffs);

/* logUp helper columns of a STARK's lookups (lookup_helper_columns / get_helper_cols, starky/src/lookup.rs:579-652,746-789)
 * for every lookup and every challenge gamma, lookup-major and challenge-minor, as value columns of n = 2^log_n rows:
 *   ceil(n_looking / chunk) helper columns h_k = sum_{i in chunk k} filter_i / (f_i + gamma),  chunk = max(1, constraint_degree - 1),
 *   then Z with Z(0) = 0, Z(i+1) = Z(i) + sum_k h_k(i) - m(i) / (t(i) + gamma).
 * Columns and filters are evaluated like eval_table (lookup.rs:318-329): next-row terms read row (i + 1) mod n. The trace is
 * n_cols columns, column c at trace + c * col_stride; out = the helper columns, column j at out + j * n. trace and out are both
 * host (GL_MEM_HOST) or both device (GL_MEM_DEVICE) memory. A zero denominator fails with GL_ERR_DIV_ZERO ("Tried to invert
 * zero"), where batch_multiplicative_inverse panics. At most GL_LOGUP_MAX_DENOMINATORS = sum over lookups of
 * (n_looking + 1) * n_challenges per row. */
typedef struct {
    uint32_t col, next; /* coeff * trace[col][row], or [row + 1 mod n] if next (Column::linear_combination / next_row_...) */
    uint64_t coeff;
} gl_logup_term;
typedef struct {
    uint32_t term_begin, n_terms; /* Column<F> (lookup.rs:137-160): terms[term_begin ..+ n_terms] + constant */
    uint64_t constant;
} gl_logup_column;
typedef struct {
    uint32_t prod_begin, n_prods; /* Filter<F> (lookup.rs:33-45): sum_j col(fc[prod_begin + 2j]) * col(fc[prod_begin + 2j + 1]) */
    uint32_t sum_begin, n_sums;   /*   + sum_j col(fc[sum_begin + j]),  fc = gl_logup_desc.filter_columns */
} gl_logup_filter;
typedef struct {
    uint32_t looking_begin, n_looking; /* Lookup<F> (lookup.rs:403-416): looking column k = columns[looking_begin + k], */
    uint32_t table, frequencies;       /*   its filter = filters[looking_begin + k]; table / frequencies: column indices */
} gl_logup_lookup;
typedef struct {
    const gl_logup_term* terms;
    const gl_logup_column* columns;
    const uint32_t* filter_columns;
    const gl_logup_filter* filters; /* as many as columns (entries of table / frequency columns are unused) */
    const gl_logup_lookup* lookups;
    uint32_t n_terms, n_columns, n_filter_columns, n_lookups;
} gl_logup_desc;
#define GL_LOGUP_MAX_DENOMINATORS 128
int gl_stark_lookup_helper_columns(gl_ctx* ctx, const uint64_t* trace, size_t col_stride, uint32_t n_cols, uint32_t log_n,
                                   const gl_logup_desc* desc, const uint64_t* challenges, uint32_t n_challenges,
                                   uint32_t constraint_degree, uint64_t* out, int mem);

/* compute_quotient_polys of a plonky2 circuit (plonky2/src/plonk/prover.rs:609-815): for every challenge alpha_k the
 * values eval_vanishing_poly_base_batch(x) / Z_H(x) (plonky2/src/plonk/vanishing_poly.rs:167-340) on the coset g<w_size>,
 * size = n << log2_ceil(quotient_degree_factor), then coset_ifft: n_alphas polynomials of `size` coefficients at
 * out_coeffs + k*size (DEVICE memory); coefficients beyond n * quotient_degree_factor are checked to vanish ("Quotient
 * has failed ...", prover.rs:327-331 -> GL_ERR_BAD_ARG). The LDEs of the commitments (constants_sigmas, wires,
 * zs_partial_products[_lookup], ...: all of one degree and rate, whole on this device) are read IN PLACE with
 * get_lde_values addressing (fri/oracle.rs:142-147).
 * The vanishing polynomial -- every gate's eval_unfiltered_base with its selector filter (gates/gate.rs:159-185,326-333),
 * L_0(x)(Z(x) - 1) and check_partial_products (util/partial_products.rs:52-76) -- is a register program: each
 * instruction writes register dst; GL_VP_TERM contributes vanishing term number b, and the result for challenge k is
 * sum_t alpha_k^t term_t (reduce_with_powers_multi, plonk_common.rs:99-116; the order of the sum does not matter).
 * plonky2_b200/plonk.py builds the program from a gate list the way eval_vanishing_poly_base_batch walks it. */
#define GL_VP_LOCAL 0 /* r[dst] = column b of commitment a at this point's row: get_lde_values(i, step) */
#define GL_VP_NEXT 1  /* ... at the row of point i + next_step (the Z(g x) operand) */
#define GL_VP_CONST 2 /* r[dst] = consts[a | b << 16] */
#define GL_VP_X 3     /* r[dst] = x = coset_shift * w_size^i (shifted_x) */
#define GL_VP_L0 4    /* r[dst] = L_0(x) = Z_H(x) / (n (x - 1)) (ZeroPolyOnCoset::eval_l_0) */
#define GL_VP_ADD 5   /* r[dst] = r[a] + r[b] */
#define GL_VP_SUB 6
#define GL_VP_MUL 7
#define GL_VP_TERM 8  /* vanishing term number b = r[a] */
#define GL_VP_ADDC 9  /* r[dst] = r[a] + consts[b] */
#define GL_VP_MULC 10 /* r[dst] = r[a] * consts[b] */
#define GL_VP_MAX_REGS 256
#define GL_VP_MAX_COMMITS 4
#define GL_VP_MAX_ALPHAS 4
#define GL_VP_MAX_QD 8
typedef struct {
    uint16_t op, dst, a, b;
} gl_vp_instr;
int gl_plonk_quotient(gl_ctx* ctx, gl_commit* const* commits, uint32_t n_commits, const gl_vp_instr* program,
                      uint32_t n_instr, const uint64_t* consts, uint32_t n_consts, const uint64_t* alphas,
                      uint32_t n_alphas, uint32_t n_terms, uint32_t quotient_degree_factor, uint64_t* out_coeffs);

/* ---- Hasher / MerkleTree  (plonky2/src/plonk/config.rs:36-77, plonky2/src/hash/merkle_tree.rs:193-237) */
/* PoseidonPermutation::permute on the HOST for the sequential Fiat-Shamir transcript
 * (plonky2/src/iop/challenger.rs:129-144); the same source as the device permutation. */
void gl_poseidon_permute_host(uint64_t state[12]);
/* Batched PoseidonPermutation::permute (plonky2/src/hash/poseidon.rs:766-777, hashing.rs:62-94): n_items states of
 * 12 words, permuted in place on the device; outputs canonical. */
int gl_poseidon_permute_many(gl_ctx* ctx, uint64_t* states, size_t n_items, int mem);
/* Batched PoseidonHash::hash_or_noop: n_items inputs of W words (row-major) -> n_items x 4 words */
int gl_poseidon_hash_many(gl_ctx* ctx, const uint64_t* in, size_t n_items, uint32_t W, uint64_t* out, int mem);
/* Batched PoseidonHash::hash_no_pad (always the sponge, no no-op branch; hashing.rs:118-145) */
int gl_poseidon_hash_no_pad_many(gl_ctx* ctx, const uint64_t* in, size_t n_items, uint32_t W, uint64_t* out, int mem);
/* Batched PoseidonHash::two_to_one: n_items pairs (8 words each) -> n_items x 4 words */
int gl_poseidon_two_to_one_many(gl_ctx* ctx, const uint64_t* in, size_t n_items, uint64_t* out, int mem);
/* MerkleTree::new(leaves, cap_height): leaves N x W row-major. */
int gl_merkle_build(gl_ctx* ctx, const uint64_t* leaves, size_t N, uint32_t W, uint32_t cap_height, int mem,
                    gl_merkle** out);
void gl_merkle_destroy(gl_merkle* m);
int gl_merkle_cap(gl_merkle* m, uint64_t* out, int mem);
int gl_merkle_digests(gl_merkle* m, uint64_t* out, int mem);
int gl_merkle_open(gl_merkle* m, const uint64_t* leaf_indices, size_t count, uint64_t* out_leaves,
                   uint64_t* out_paths);

/* ---- FRI  (plonky2/src/fri/oracle.rs:176-237 prove_openings; plonky2/src/fri/prover.rs:24-258) --- */
/* One opening batch: a point z in F_{p^2} and the polynomials opened there, each named by
 * (oracle index into the `oracles` array, polynomial index inside it)
 * (plonky2/src/fri/structure.rs:14-60 FriInstanceInfo / FriBatchInfo / FriPolynomialInfo). */
typedef struct {
    uint64_t point[2];
    size_t num_polys;
    const uint32_t* oracle_index;
    const uint32_t* poly_index;
} gl_fri_batch;

/* The part of prove_openings before fri_proof (oracle.rs:186-220): with alpha from the caller's
 * transcript, final_poly = sum_b alpha^{k_b} (F_b(X) - F_b(z_b)) / (X - z_b), F_b = sum_j alpha^j f_{b,j},
 * then its rate-2^-rate_bits coset LDE. The handle holds the n F_{p^2} coefficients and the N values in
 * bit-reversed order (the order fri_committed_trees hashes them in). */
int gl_fri_begin(gl_ctx* ctx, gl_commit* const* oracles, size_t n_oracles, const gl_fri_batch* batches,
                 size_t n_batches, const uint64_t alpha[2], uint32_t rate_bits, uint32_t cap_height,
                 gl_fri** out);
/* The same codeword computed in the VALUE domain, straight from the commitments' LDE rows:
 *   value(x) = sum_b alpha^{k_b} (F_b(x) - F_b(z_b)) / (x - z_b),  F_b(x) = sum_j alpha^j f_{b,j}(x)
 * -- exactly the field elements gl_fri_begin's LDE holds (the quotients are exact), with no pass over the coefficients
 * and no LDE. `opened` = the openings f_{b,j}(z_b) in batch order (2 words each; OpeningSet / gl_openings), as the
 * prover has them at this point (oracle.rs:176-184). If the commitments are row-block shards (gl_commit_create_sharded,
 * all with the same shard), the state holds THIS shard's rows only: every later round is rank-local
 * (gl_fri_commit_round returns the shard's 2^cap_height / G cap entries, gl_fri_fold folds the local leaves), the final
 * polynomial is interpolated by the caller from the gathered gl_fri_values_local. rate_bits comes from the commitments. */
int gl_fri_begin_values(gl_ctx* ctx, gl_commit* const* oracles, size_t n_oracles, const gl_fri_batch* batches,
                        size_t n_batches, const uint64_t* opened, const uint64_t alpha[2], uint32_t cap_height,
                        gl_fri** out);
/* the local block of the current codeword between rounds: *len_out F_{p^2} values (2 words each), bit-reversed order */
int gl_fri_values_local(gl_fri* f, uint64_t* out, size_t cap_words, size_t* len_out);
/* Same, from explicit final-polynomial coefficients (n = 2^log_n F_{p^2} elements, 2n words, host). */
int gl_fri_begin_from_coeffs(gl_ctx* ctx, const uint64_t* coeffs_ext, uint32_t log_n, uint32_t rate_bits,
                             uint32_t cap_height, gl_fri** out);
void gl_fri_destroy(gl_fri* f);
/* final_poly coefficients before folding (n x 2 words), for parity checks */
int gl_fri_coeffs(gl_fri* f, uint64_t* out);
/* One round of fri_committed_trees (prover.rs:96-120), split at the transcript:
 *   commit: leaves = arity consecutive (bit-reversed) values flattened; MerkleTree::new; cap -> host. */
int gl_fri_commit_round(gl_fri* f, uint32_t arity_bits, uint64_t* cap_out /* 4 * 2^cap_height */);
/*   the same with the round's Merkle tree row-block sharded over num_shards GPUs (each hashes its own block of leaves and
 *   returns its 2^cap_height / num_shards cap entries; the caller all-gathers them). Values stay replicated. */
int gl_fri_commit_round_sharded(gl_fri* f, uint32_t arity_bits, uint32_t shard_index, uint32_t num_shards,
                                uint64_t* cap_out);
/*   fold:   with beta from the transcript, values' = fold(values, beta) on the coset shift^arity. */
int gl_fri_fold(gl_fri* f, const uint64_t beta[2]);
/* batch-FRI mixing step (plonky2/src/batch_fri/prover.rs:118-132): when `f`'s codeword has been folded down to the
 * length of `other`'s (the next, lower-degree instance from its own gl_fri_begin), values <- values * beta + other's. */
int gl_fri_mix(gl_fri* f, const gl_fri* other, const uint64_t beta[2]);
/* Final polynomial after the last fold, truncated by 2^rate_bits (prover.rs:134-139):
 * *len_out coefficients (2 words each) written to out (capacity `cap_words` words). */
int gl_fri_final_poly(gl_fri* f, uint64_t* out, size_t cap_words, size_t* len_out);
/* Query openings in the committed FRI trees (prover.rs:236-250): for tree `round`, leaves
 * (arity*2 words each) and Merkle paths for `count` leaf indices. */
int gl_fri_open(gl_fri* f, uint32_t round, const uint64_t* leaf_indices, size_t count, uint64_t* out_leaves,
                uint64_t* out_paths);
uint32_t gl_fri_num_rounds(const gl_fri* f);
/* fri_proof_of_work (prover.rs:153-202): the SMALLEST u64 nonce such that, with the duplex state
 * `state` (sponge state already overwritten by the pending inputs) and the nonce written at lane `pos`,
 * lane 7 of the permuted state has >= min_leading_zeros leading zero bits in canonical form.
 * (The reference's rayon find_any returns an arbitrary qualifying nonce; a sequential run returns
 * the smallest -- maybe_rayon/src/lib.rs:254-259.) */
int gl_fri_pow(gl_ctx* ctx, const uint64_t state[12], uint32_t pos, uint32_t min_leading_zeros,
               uint64_t* nonce_out);

#ifdef __cplusplus
}
#endif
#endif
