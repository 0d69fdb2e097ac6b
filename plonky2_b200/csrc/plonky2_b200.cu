// plonky2_b200.cu -- sm_100a kernels + host orchestration + the C ABI of include/plonky2_b200.h.
//
// Hot path implemented here (reference -> this file):
//   PolynomialBatch::from_values/from_coeffs  plonky2/src/fri/oracle.rs:57-139   -> commit_build()
//   MerkleTree::new / prove                   plonky2/src/hash/merkle_tree.rs:86-237 -> tree_build(), tree_open()
//   prove_openings (pre-FRI part)             plonky2/src/fri/oracle.rs:176-220   -> gl_fri_begin()
//   fri_committed_trees / fri_proof_of_work   plonky2/src/fri/prover.rs:84-202    -> gl_fri_commit_round/fold/pow
// There is no CPU fallback anywhere in this file: every compute entry point launches kernels.
#include <cooperative_groups.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <set>
#include <string>
#include <tuple>
#include <vector>

#include "../../include/plonky2_b200.h"
#include "gl_field.cuh"
#include "gl_ntt.cuh"
#include "gl_poseidon.cuh"
#include "gl_vanishing.cuh"
#include "gl_logup.cuh"

using namespace gl;
typedef uint64_t u64;

// =====================================================================================
// errors / context
// =====================================================================================
static thread_local std::string g_last_error;

struct gl_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    u64 launches = 0;
    std::string err;
    std::map<std::tuple<int, u64, u64>, u64*> step_tabs;  // in-pass step tables by (log, scale, base)
    std::map<std::tuple<int, int, u64>, u64*> post_tabs;  // column-pass post tables by (a, b, base)
    size_t table_bytes = 0;
    std::map<int, u64*> fold_tabs;              // FRI fold tables (w_N^-1 powers, hi | lo) by log N
    cudaStream_t copy_stream = nullptr;         // H2D of column chunks, overlapped with the NTTs of earlier chunks
    std::set<const void*> smem_attr_done;       // kernels whose dynamic-smem attributes are set on THIS device
    u64* scratch = nullptr;                     // NTT group scratch (device)
    size_t scratch_words = 0;
    u64* pinned = nullptr;                      // host staging for small D2H / H2D
    size_t pinned_words = 0;
    u64* dstage = nullptr;                      // device staging for openings
    size_t dstage_words = 0;
    uint32_t ntt_group = 0;                     // 0 = auto
    int ntt_variant = 0;                        // 0 = shared-body column pass for even LOG, 1 = two-copy kernels (A/B switch)
    int sm_count = 0;                           // queried once for ctx->device in gl_ctx_create
    int coop_ok = 0;                            // cooperative launch supported on this device
    int coop_blocks_per_sm = 0;                 // resident CTAs/SM of k_merkle_upper on this device
    // optional CUDA-event phase timing (bench.py's roofline numbers come from here)
    bool prof_on = false;
    struct Pending {
        int phase;
        cudaEvent_t a, b;
    };
    std::vector<Pending> prof_pending;
    double prof_ms[GL_NUM_PHASES] = {0};
    u64 prof_count[GL_NUM_PHASES] = {0};
};

struct PhaseScope {
    gl_ctx* ctx;
    cudaEvent_t a = nullptr, b = nullptr;
    int phase;
    PhaseScope(gl_ctx* c, int ph) : ctx(c), phase(ph) {
        if (!ctx->prof_on) return;
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, ctx->stream);
    }
    ~PhaseScope() {
        if (!a) return;
        cudaEventRecord(b, ctx->stream);
        ctx->prof_pending.push_back({phase, a, b});
    }
};

static int set_err(gl_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
    if (ctx) ctx->err = buf;
    return code;
}
#define CK(ctx, call)                                                                          \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return set_err(ctx, e_ == cudaErrorMemoryAllocation ? GL_ERR_OOM : GL_ERR_CUDA,    \
                           "%s failed: %s", #call, cudaGetErrorString(e_));                    \
    } while (0)
#define CKL(ctx)                                                                               \
    do {                                                                                       \
        (ctx)->launches++;                                                                     \
        cudaError_t e_ = cudaGetLastError();                                                   \
        if (e_ != cudaSuccess)                                                                 \
            return set_err(ctx, GL_ERR_CUDA, "kernel launch failed (%s:%d): %s", __FILE__,     \
                           __LINE__, cudaGetErrorString(e_));                                  \
    } while (0)
#define TRY(expr)                  \
    do {                           \
        int rc_ = (expr);          \
        if (rc_ != GL_OK) return rc_; \
    } while (0)

static int dmalloc(gl_ctx* ctx, u64** p, size_t words) {
    *p = nullptr;
    if (words == 0) return GL_OK;
    CK(ctx, cudaMallocAsync((void**)p, words * 8, ctx->stream));
    return GL_OK;
}
static void dfree(gl_ctx* ctx, u64* p) {
    if (p) cudaFreeAsync(p, ctx->stream);
}
static int ensure_scratch(gl_ctx* ctx, size_t words) {
    if (ctx->scratch_words >= words) return GL_OK;
    if (ctx->scratch) dfree(ctx, ctx->scratch);
    ctx->scratch = nullptr;
    ctx->scratch_words = 0;
    TRY(dmalloc(ctx, &ctx->scratch, words));
    ctx->scratch_words = words;
    return GL_OK;
}
static int ensure_pinned(gl_ctx* ctx, size_t words) {
    if (ctx->pinned_words >= words) return GL_OK;
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    ctx->pinned = nullptr;
    ctx->pinned_words = 0;
    size_t w = words < 65536 ? 65536 : words;
    CK(ctx, cudaHostAlloc((void**)&ctx->pinned, w * 8, cudaHostAllocDefault));
    ctx->pinned_words = w;
    return GL_OK;
}
static int ensure_dstage(gl_ctx* ctx, size_t words) {
    if (ctx->dstage_words >= words) return GL_OK;
    if (ctx->dstage) dfree(ctx, ctx->dstage);
    ctx->dstage = nullptr;
    ctx->dstage_words = 0;
    size_t w = words < 65536 ? 65536 : words;
    TRY(dmalloc(ctx, &ctx->dstage, w));
    ctx->dstage_words = w;
    return GL_OK;
}
// device -> host through pinned staging (stream-ordered, then synchronised)
static int d2h(gl_ctx* ctx, u64* host, const u64* dev, size_t words) {
    if (words == 0) return GL_OK;
    CK(ctx, cudaMemcpyAsync(host, dev, words * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return GL_OK;
}
static int h2d(gl_ctx* ctx, u64* dev, const u64* host, size_t words) {
    if (words == 0) return GL_OK;
    CK(ctx, cudaMemcpyAsync(dev, host, words * 8, cudaMemcpyHostToDevice, ctx->stream));
    return GL_OK;
}
static int copy_out(gl_ctx* ctx, u64* out, const u64* dev, size_t words, int mem) {
    if (mem == GL_MEM_DEVICE) {
        CK(ctx, cudaMemcpyAsync(out, dev, words * 8, cudaMemcpyDeviceToDevice, ctx->stream));
        return GL_OK;
    }
    return d2h(ctx, out, dev, words);
}

// =====================================================================================
// TMA bulk copy of the in-tile twiddle table (cp.async.bulk + mbarrier)
// =====================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void tma_table_issue(u64* dst_smem, const u64* src_gmem, uint32_t bytes, u64* mbar) {
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(mbar)), "r"(bytes)
                     : "memory");
        asm volatile(
            "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                smem_u32(dst_smem)),
            "l"(src_gmem), "r"(bytes), "r"(smem_u32(mbar))
            : "memory");
    }
}
// all threads: called after a __syncthreads() that follows tma_table_issue()
__device__ __forceinline__ void tma_table_wait(u64* mbar) {
    uint32_t done = 0;
    const uint32_t addr = smem_u32(mbar);
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr)
            : "memory");
    }
}

// =====================================================================================
// NTT kernels + orchestration
// =====================================================================================
#include "gl_ntt_host.cuh"

// =====================================================================================
// Poseidon / Merkle kernels
// =====================================================================================
struct TreeView {
    const u64* leaves;  // element k of leaf j at leaves[j*ls + k*es]: row-major (ls = W, es = 1) for MerkleTree::new
                        // and the FRI trees, column-major (ls = 1, es = column stride) for PolynomialBatch LDEs
    u64* digests;       // 4 * 2 * (N - C)
    u64* cap;           // 4 * C
    size_t N, ls, es;
    uint32_t W, log_n, cap_height;
};

// position (in hashes) of node q of layer i inside its subtree's digest block (merkle_tree.rs:176-187)
__host__ __device__ __forceinline__ size_t digest_pos(size_t q, uint32_t i) {
    return 2 * (((q >> 1) << (i + 1)) + ((size_t)1 << i) - 1) + (q & 1);
}

constexpr int HASH_CTA = 128;   // CTA size of the barrier-synchronised Poseidon kernels
constexpr int HASH_MINB = 5;    // 5 CTAs/SM => up to 96 registers/thread (best of the microbench sweep: 820 M perm/s)
__global__ void __launch_bounds__(HASH_CTA, HASH_MINB) k_leaf_hash(TreeView t) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = j < t.N;
    if (!live) j = t.N - 1;  // keep the whole CTA in the per-round barriers; the result is discarded
    u64 h[4];
    hash_or_noop_strided<true, true>(t.leaves + j * t.ls, t.es, t.W, h);
    if (!live) return;
    u64* dst;
    const uint32_t sub_log = t.log_n - t.cap_height;  // log2(leaves per cap subtree)
    if (sub_log == 0) {
        dst = t.cap + 4 * j;
    } else {
        const size_t L = (size_t)1 << sub_log;
        const size_t c = j >> sub_log, q = j & (L - 1);
        dst = t.digests + 4 * (c * 2 * (L - 1) + digest_pos(q, 0));
    }
    dst[0] = h[0];
    dst[1] = h[1];
    dst[2] = h[2];
    dst[3] = h[3];
}
// layer i (>= 1) from layer i-1: one thread per node
__global__ void __launch_bounds__(HASH_CTA, HASH_MINB) k_merkle_level(TreeView t, uint32_t i) {
    const uint32_t sub_log = t.log_n - t.cap_height;
    const size_t nodes_per_sub = (size_t)1 << (sub_log - i);
    const size_t total = nodes_per_sub << t.cap_height;
    size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = g < total;
    if (!live) g = total - 1;
    const size_t c = g >> (sub_log - i), q = g & (nodes_per_sub - 1);
    const size_t L = (size_t)1 << sub_log;
    u64* sub = t.digests + 4 * (c * 2 * (L - 1));
    const u64* pair = sub + 4 * digest_pos(2 * q, i - 1);
    u64 l[4] = {pair[0], pair[1], pair[2], pair[3]};
    u64 r[4] = {pair[4], pair[5], pair[6], pair[7]};
    u64 h[4];
    two_to_one<true>(l, r, h);
    if (!live) return;
    u64* dst = (i == sub_log) ? (t.cap + 4 * c) : (sub + 4 * digest_pos(q, i));
    dst[0] = h[0];
    dst[1] = h[1];
    dst[2] = h[2];
    dst[3] = h[3];
}
// Upper levels in ONE persistent cooperative launch: when a level has fewer nodes than the resident thread
// capacity, per-level launches are latency-bound; here the resident CTAs walk the levels i0..sub_log with a
// grid-wide barrier between levels (every level reads what the previous one wrote).
__global__ void __launch_bounds__(HASH_CTA, HASH_MINB) k_merkle_upper(TreeView t, uint32_t i0) {
    cooperative_groups::grid_group grid = cooperative_groups::this_grid();
    const uint32_t sub_log = t.log_n - t.cap_height;
    const size_t L = (size_t)1 << sub_log;
    const size_t nthreads = (size_t)gridDim.x * blockDim.x;
    for (uint32_t i = i0; i <= sub_log; i++) {
        const size_t nodes_per_sub = (size_t)1 << (sub_log - i);
        const size_t total = nodes_per_sub << t.cap_height;
        // uniform trip count per CTA (the permutation contains CTA barriers)
        const size_t first = (size_t)blockIdx.x * blockDim.x;
        for (size_t base = first; base < total; base += nthreads) {
            size_t g = base + threadIdx.x;
            const bool live = g < total;
            if (!live) g = total - 1;
            const size_t c = g >> (sub_log - i), q = g & (nodes_per_sub - 1);
            u64* sub = t.digests + 4 * (c * 2 * (L - 1));
            const u64* pair = sub + 4 * digest_pos(2 * q, i - 1);
            u64 l[4] = {pair[0], pair[1], pair[2], pair[3]};
            u64 r[4] = {pair[4], pair[5], pair[6], pair[7]};
            u64 h[4];
            two_to_one<true>(l, r, h);
            if (live) {
                u64* dst = (i == sub_log) ? (t.cap + 4 * c) : (sub + 4 * digest_pos(q, i));
                dst[0] = h[0];
                dst[1] = h[1];
                dst[2] = h[2];
                dst[3] = h[3];
            }
        }
        grid.sync();
    }
}
template <bool NOOP_SHORT>
__global__ void __launch_bounds__(128) k_hash_many(const u64* in, size_t n_items, uint32_t W, u64* out) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_items) return;
    u64 h[4];
    hash_or_noop_strided<NOOP_SHORT>(in + j * W, 1, W, h);
    for (int k = 0; k < 4; k++) out[4 * j + k] = h[k];
}
// PoseidonPermutation::permute on n_items independent 12-lane states, in place (hashing.rs:62-94 permute)
__global__ void __launch_bounds__(128) k_permute_many(u64* states, size_t n_items) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_items) return;
    u64 s[12];
#pragma unroll
    for (int k = 0; k < 12; k++) s[k] = states[12 * j + k];
    poseidon_permute(s);
#pragma unroll
    for (int k = 0; k < 12; k++) states[12 * j + k] = canon(s[k]);
}
__global__ void __launch_bounds__(128) k_two_to_one_many(const u64* in, size_t n_items, u64* out) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_items) return;
    u64 l[4], r[4], h[4];
    for (int k = 0; k < 4; k++) {
        l[k] = in[8 * j + k];
        r[k] = in[8 * j + 4 + k];
    }
    two_to_one(l, r, h);
    for (int k = 0; k < 4; k++) out[4 * j + k] = h[k];
}
// Openings: one CTA per queried leaf; copies the leaf and its sibling path (merkle_tree.rs:151-190).
__global__ void k_tree_open(TreeView t, const u64* indices, u64* out_leaves, u64* out_paths) {
    const size_t idx = indices[blockIdx.x];
    const uint32_t num_layers = t.log_n - t.cap_height;
    for (uint32_t k = threadIdx.x; k < t.W; k += blockDim.x)
        out_leaves[(size_t)blockIdx.x * t.W + k] = t.leaves[idx * t.ls + (size_t)k * t.es];
    const size_t L = (size_t)1 << num_layers;
    const size_t tree_index = idx >> num_layers;
    const u64* sub = t.digests + 4 * (tree_index * 2 * (L - 1));
    for (uint32_t k = threadIdx.x; k < num_layers * 4; k += blockDim.x) {
        const uint32_t i = k >> 2, w = k & 3;
        const size_t node = (idx & (L - 1)) >> i;  // ancestor at layer i
        const size_t sib = node ^ 1;
        out_paths[(size_t)blockIdx.x * num_layers * 4 + k] = sub[4 * digest_pos(sib, i) + w];
    }
}

struct Tree {
    u64* leaves = nullptr;  // device
    u64* base = nullptr;    // allocation `leaves` points into when the tree covers a row block of a larger buffer
    bool own_leaves = false;
    u64* digests = nullptr;
    u64* cap = nullptr;
    size_t N = 0;
    size_t ls = 0, es = 1;  // leaf / element strides (ls == 0: row-major, ls = W)
    uint32_t W = 0, log_n = 0, cap_height = 0;
    TreeView view() const { return TreeView{leaves, digests, cap, N, ls ? ls : (size_t)W, es, W, log_n, cap_height}; }
    size_t digest_words() const { return 8 * (N - ((size_t)1 << cap_height)); }
    size_t cap_words() const { return (size_t)4 << cap_height; }
};

static int log2_exact(size_t n, uint32_t* out) {
    if (n == 0 || (n & (n - 1))) return 1;
    uint32_t l = 0;
    while (((size_t)1 << l) < n) l++;
    *out = l;
    return 0;
}

// MerkleTree::new over device leaves (merkle_tree.rs:193-224)
static int tree_build(gl_ctx* ctx, Tree& t) {
    if (log2_exact(t.N, &t.log_n)) return set_err(ctx, GL_ERR_BAD_SHAPE, "Not a power of two: %zu", t.N);
    if (t.cap_height > t.log_n)
        return set_err(ctx, GL_ERR_BAD_SHAPE, "cap_height=%u should be at most log2(leaves.len())=%u", t.cap_height,
                       t.log_n);
    TRY(dmalloc(ctx, &t.digests, t.digest_words()));
    TRY(dmalloc(ctx, &t.cap, t.cap_words()));
    TreeView v = t.view();
    {
        PhaseScope ps(ctx, GL_PHASE_LEAF_HASH);
        // big CTAs (barrier-synchronised rounds) for big trees; small CTAs to spread small trees over the SMs
        const int cta = HASH_CTA;
        k_leaf_hash<<<(unsigned)((t.N + cta - 1) / cta), cta, 0, ctx->stream>>>(v);
        CKL(ctx);
    }
    PhaseScope ps2(ctx, GL_PHASE_MERKLE_LEVELS);
    const uint32_t sub_log = t.log_n - t.cap_height;
    // resident capacity of the persistent upper-level kernel (cooperative launch needs co-residency)
    // (per-context, i.e. per-device, values: gl_ctx_create)
    const size_t coop_threads = ctx->coop_ok ? (size_t)ctx->coop_blocks_per_sm * ctx->sm_count * HASH_CTA : 0;
    for (uint32_t i = 1; i <= sub_log; i++) {
        size_t total = (size_t)1 << (t.log_n - i);
        if (coop_threads && total <= coop_threads && i < sub_log) {
            // this and all higher levels fit the resident grid: one persistent launch finishes the tree
            unsigned nb = (unsigned)((total + HASH_CTA - 1) / HASH_CTA);
            uint32_t i0 = i;
            void* args[] = {(void*)&v, (void*)&i0};
            CK(ctx, cudaLaunchCooperativeKernel((void*)k_merkle_upper, dim3(nb), dim3(HASH_CTA), args, 0, ctx->stream));
            ctx->launches++;
            break;
        }
        const int cta = HASH_CTA;
        k_merkle_level<<<(unsigned)((total + cta - 1) / cta), cta, 0, ctx->stream>>>(v, i);
        CKL(ctx);
    }
    return GL_OK;
}
static void tree_free(gl_ctx* ctx, Tree& t) {
    if (t.own_leaves) dfree(ctx, t.base ? t.base : t.leaves);
    dfree(ctx, t.digests);
    dfree(ctx, t.cap);
    t.leaves = t.digests = t.cap = nullptr;
}
static int tree_open(gl_ctx* ctx, const Tree& t, const u64* leaf_indices, size_t count, u64* out_leaves,
                     u64* out_paths) {
    if (count == 0) return GL_OK;
    for (size_t i = 0; i < count; i++)
        if (leaf_indices[i] >= t.N) return set_err(ctx, GL_ERR_BAD_ARG, "leaf index %llu out of range",
                                                   (unsigned long long)leaf_indices[i]);
    const uint32_t layers = t.log_n - t.cap_height;
    const size_t lw = count * t.W, pw = count * layers * 4;
    TRY(ensure_dstage(ctx, count + lw + pw));
    TRY(ensure_pinned(ctx, count + lw + pw));
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    memcpy(ctx->pinned, leaf_indices, count * 8);
    TRY(h2d(ctx, ctx->dstage, ctx->pinned, count));
    k_tree_open<<<(unsigned)count, 128, 0, ctx->stream>>>(t.view(), ctx->dstage, ctx->dstage + count,
                                                         ctx->dstage + count + lw);
    CKL(ctx);
    TRY(d2h(ctx, ctx->pinned, ctx->dstage + count, lw + pw));
    memcpy(out_leaves, ctx->pinned, lw * 8);
    if (pw) memcpy(out_paths, ctx->pinned + lw, pw * 8);
    return GL_OK;
}

// =====================================================================================
// PolynomialBatch
// =====================================================================================
struct gl_commit {
    gl_ctx* ctx;
    uint32_t B, W, degree_log, rate_bits;
    uint32_t shard_index = 0, shard_log = 0;  // this handle holds leaf rows [g*N/G, (g+1)*N/G)
    bool blinding;
    u64* coeffs = nullptr;  // B x n
    bool own_coeffs = true; // false: caller-owned storage handed to gl_commit_begin
    bool finished = false;  // tree built (handles from gl_commit_begin: after gl_commit_finish)
    u64 sg = 0;             // coset shift of this shard's row block
    Tree tree;
};

// lde[B + s][j] = salt[s][bitrev(j)]  (salt columns are LDE columns in natural order, oracle.rs:133-137)
__global__ void k_salt(const u64* salt, size_t N, uint32_t log_N, size_t row0, size_t rows, u64* lde, size_t lde_stride,
                       uint32_t B) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= rows) return;
    size_t i = (size_t)(__brevll(row0 + j) >> (64 - log_N));
    if (log_N == 0) i = 0;
    for (int s = 0; s < GL_SALT_SIZE; s++) lde[(size_t)(B + s) * lde_stride + j] = canon(salt[(size_t)s * N + i]);
}
// row-major view of a block of LDE rows (MerkleTree.leaves as the reference stores them): out[r*W + k] = lde[k][row0 + r],
// through a 32 x 32 shared-memory tile so that both sides are coalesced
__global__ void k_rows_from_columns(const u64* lde, size_t lde_stride, size_t row0, size_t rows, uint32_t W, u64* out) {
    __shared__ u64 tile[32][33];
    const size_t rb = (size_t)blockIdx.x * 32;
    const uint32_t kb = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const size_t r = rb + threadIdx.x;
        const uint32_t k = kb + i;
        if (r < rows && k < W) tile[i][threadIdx.x] = lde[(size_t)k * lde_stride + row0 + r];
    }
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const size_t r = rb + i;
        const uint32_t k = kb + threadIdx.x;
        if (r < rows && k < W) out[r * W + k] = tile[threadIdx.x][i];
    }
}
// Restriction of a degree-<n polynomial to a coset of size M < n (x^M = sM on it):
// a'[k0] = sum_{k1 < n/M} a[k0 + M*k1] * sM^k1     (SURVEY section 8e, "fold coefficients mod X^M - s^M")
__global__ void k_fold_coeffs(const u64* coeffs, size_t stride, size_t n, size_t M, u64 sM, u64* out) {
    size_t k0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k0 >= M) return;
    const u64* col = coeffs + (size_t)blockIdx.y * stride;
    u64 acc = 0;
    for (size_t k1 = n / M; k1-- > 0;) acc = mul_add(acc, sM, col[k0 + M * k1]);
    out[(size_t)blockIdx.y * M + k0] = acc;
}
__global__ void k_canon(u64* data, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) data[i] = canon(data[i]);
}

// Allocate the device state of a commitment: coefficients (or adopt the caller's matrix) and the column-major LDE.
static int commit_alloc(gl_ctx* ctx, gl_commit* c, uint32_t cap_height, u64* ext_coeffs) {
    const size_t n = (size_t)1 << c->degree_log, N = n << c->rate_bits;
    if (ext_coeffs) {
        c->coeffs = ext_coeffs;
        c->own_coeffs = false;
    } else {
        TRY(dmalloc(ctx, &c->coeffs, (size_t)c->B * n));
    }
    // Row-block sharding (SURVEY section 8e): shard g of G = 2^s owns leaves [g*N/G, (g+1)*N/G), i.e. the
    // LDE points i = g' (mod G), g' = bitrev_s(g): the coset (g * w_N^{g'}) <w_{N/G}> in bit-reversed order.
    const uint32_t sl = c->shard_log;
    const size_t Nloc = N >> sl;
    const uint32_t gprime = bitrev32(c->shard_index, sl);
    c->sg = mul(MULTIPLICATIVE_GROUP_GENERATOR, gl::pow(root_of_unity(c->degree_log + c->rate_bits), gprime));
    Tree& t = c->tree;
    t.N = Nloc;
    t.W = c->W;
    t.cap_height = cap_height - sl;
    t.own_leaves = true;
    t.ls = 1;       // column-major LDE: column k at leaves + k*Nloc, leaf order inside
    t.es = Nloc;
    TRY(dmalloc(ctx, &t.leaves, Nloc * (size_t)c->W));
    return GL_OK;
}
// Columns [g0, g0 + gc) sit in c->coeffs as values (kind 0), coefficients (1) or canonical coefficients (2):
// iNTT ("IFFT", oracle.rs:65-69) / canonicalise, then the leaf-major coset LDE ("FFT + blinding" + "transpose LDEs" +
// bit-reversal, fused) into this shard's rows.
static int commit_chunk(gl_ctx* ctx, gl_commit* c, uint32_t g0, uint32_t gc, int kind) {
    const size_t n = (size_t)1 << c->degree_log;
    const uint32_t sl = c->shard_log;
    Tree& t = c->tree;
    const size_t Nloc = t.N;
    u64* cg = c->coeffs + (size_t)g0 * n;
    if (kind == 0) {
        PhaseScope ps(ctx, GL_PHASE_INTT);
        TRY(ntt_natural(ctx, cg, n, cg, n, (int)c->degree_log, gc, true, 1));
    } else if (kind == 1) {
        size_t tot = (size_t)gc * n;
        k_canon<<<(unsigned)((tot + 255) / 256), 256, 0, ctx->stream>>>(cg, tot);
        CKL(ctx);
    }
    PhaseScope ps(ctx, GL_PHASE_LDE);
    if (sl <= c->rate_bits) {
        const uint32_t rloc = c->rate_bits - sl;
        TRY(lde_columns(ctx, cg, n, gc, (int)c->degree_log, (int)rloc, c->sg, t.leaves + (size_t)g0 * Nloc, Nloc));
    } else {
        // fewer than n points per shard: restrict the polynomials to the sub-coset first
        const uint32_t logM = c->degree_log + c->rate_bits - sl;
        const size_t M = (size_t)1 << logM;
        u64* folded;
        TRY(dmalloc(ctx, &folded, (size_t)gc * M));
        k_fold_coeffs<<<dim3((unsigned)((M + 127) / 128), gc), 128, 0, ctx->stream>>>(cg, n, n, M, gl::pow(c->sg, M), folded);
        CKL(ctx);
        const int rc2 = lde_columns(ctx, folded, M, gc, (int)logM, 0, c->sg, t.leaves + (size_t)g0 * Nloc, Nloc);
        dfree(ctx, folded);
        TRY(rc2);
    }
    return GL_OK;
}
// salt columns (blinding) + "build Merkle tree"
static int commit_finish(gl_ctx* ctx, gl_commit* c, const u64* salt, int mem) {
    const size_t n = (size_t)1 << c->degree_log, N = n << c->rate_bits;
    Tree& t = c->tree;
    const size_t Nloc = t.N;
    if (salt) {
        u64* dsalt = nullptr;
        const u64* sp = salt;
        if (mem == GL_MEM_HOST) {
            TRY(dmalloc(ctx, &dsalt, GL_SALT_SIZE * N));
            TRY(h2d(ctx, dsalt, salt, GL_SALT_SIZE * N));
            sp = dsalt;
        }
        k_salt<<<(unsigned)((Nloc + 255) / 256), 256, 0, ctx->stream>>>(sp, N, c->degree_log + c->rate_bits,
                                                                       (size_t)c->shard_index * Nloc, Nloc, t.leaves,
                                                                       Nloc, c->B);
        CKL(ctx);
        if (dsalt) dfree(ctx, dsalt);
    }
    TRY(tree_build(ctx, t));
    c->finished = true;
    return GL_OK;
}

static int commit_build(gl_ctx* ctx, gl_commit* c, const u64* cols, size_t col_stride, const u64* salt, int is_coeffs,
                        int mem, uint32_t cap_height) {
    const size_t n = (size_t)1 << c->degree_log;
    const uint32_t B = c->B;
    TRY(commit_alloc(ctx, c, cap_height, nullptr));
    // Column chunks flow through  H2D copy -> iNTT -> LDE; the copy of chunk k+1 (separate stream) overlaps the
    // transforms of chunk k.
    // 32-column chunks: launches big enough for full waves; the FIRST chunk is 8 columns so that only ~1.2 ms of H2D
    // (n = 2^20) is exposed before the first transform starts instead of ~5 ms.
    const uint32_t CH = 32, CH0 = 8;
    const bool overlap = (mem == GL_MEM_HOST) && B > CH;
    struct EventList {  // destroyed on every exit path
        std::vector<cudaEvent_t> v;
        ~EventList() {
            for (auto e : v) cudaEventDestroy(e);
        }
    } evl;
    std::vector<cudaEvent_t>& evs = evl.v;
    std::vector<std::pair<uint32_t, uint32_t>> chunks;  // (first column, count)
    if (overlap) {
        for (uint32_t g0 = 0; g0 < B;) {
            const uint32_t want = g0 == 0 ? CH0 : CH, gc = (B - g0 < want) ? B - g0 : want;
            chunks.emplace_back(g0, gc);
            g0 += gc;
        }
        if (!ctx->copy_stream) CK(ctx, cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
        cudaEvent_t ready;
        CK(ctx, cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
        CK(ctx, cudaEventRecord(ready, ctx->stream));  // the stream-ordered allocations above
        CK(ctx, cudaStreamWaitEvent(ctx->copy_stream, ready, 0));
        cudaEventDestroy(ready);
        for (auto& ch : chunks) {
            const uint32_t g0 = ch.first, gc = ch.second;
            if (col_stride == n) {
                CK(ctx, cudaMemcpyAsync(c->coeffs + (size_t)g0 * n, cols + (size_t)g0 * n, (size_t)gc * n * 8,
                                        cudaMemcpyHostToDevice, ctx->copy_stream));
            } else {
                CK(ctx, cudaMemcpy2DAsync(c->coeffs + (size_t)g0 * n, n * 8, cols + (size_t)g0 * col_stride,
                                          col_stride * 8, n * 8, gc, cudaMemcpyHostToDevice, ctx->copy_stream));
            }
            cudaEvent_t e;
            CK(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            CK(ctx, cudaEventRecord(e, ctx->copy_stream));
            evs.push_back(e);
        }
    } else {
        chunks.emplace_back(0u, B);
        CK(ctx, cudaMemcpy2DAsync(c->coeffs, n * 8, cols, col_stride * 8, n * 8, B,
                                  mem == GL_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, ctx->stream));
    }
    for (size_t k = 0; k < chunks.size(); k++) {
        if (overlap) CK(ctx, cudaStreamWaitEvent(ctx->stream, evs[k], 0));
        TRY(commit_chunk(ctx, c, chunks[k].first, chunks[k].second, is_coeffs ? 1 : 0));
    }
    return commit_finish(ctx, c, salt, mem);
}

// =====================================================================================
// FRI
// =====================================================================================
struct PolyRef {
    const u64* ptr;
    u64 a0, a1;  // alpha^j
};
// comp[k] = sum_j alpha^j * f_j[k]   (ReducingFactor::reduce_polys_base, reducing.rs:83-95)
__global__ void k_fri_compose(const PolyRef* refs, uint32_t num, size_t n, u64* comp /* n x 2 */) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    Acc160 a0 = {0, 0, 0}, a1 = {0, 0, 0};
    for (uint32_t j = 0; j < num; j++) {
        const u64 c = refs[j].ptr[k];
        acc_mul(a0, c, refs[j].a0);
        acc_mul(a1, c, refs[j].a1);
    }
    comp[2 * k] = acc_reduce(a0);
    comp[2 * k + 1] = acc_reduce(a1);
}
// z^m via factored tables (F_{p^2}): hi[m >> 12] * lo[m & 4095]
__device__ __forceinline__ E2 e2_pow_tab(const u64* hi, const u64* lo, size_t m) {
    const size_t h = m >> 12, l = m & 4095;
    return e2_mul(E2{hi[2 * h], hi[2 * h + 1]}, E2{lo[2 * l], lo[2 * l + 1]});
}
__global__ void k_fill_e2_pows(E2 base, size_t count, u64* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    E2 r = e2_pow(base, i);
    out[2 * i] = r.a;
    out[2 * i + 1] = r.b;
}
// four power tables in one launch: segment t holds base[t]^i, i < count[t]
struct E2Pows4 {
    E2 base[4];
    size_t count[4];
    u64* out[4];
};
__global__ void k_fill_e2_pows4(E2Pows4 p) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
    for (int t = 0; t < 4; t++) {
        if (i < p.count[t]) {
            E2 r = e2_pow(p.base[t], i);
            p.out[t][2 * i] = r.a;
            p.out[t][2 * i + 1] = r.b;
            return;
        }
        i -= p.count[t];
    }
}
// CTA-wide exclusive SUFFIX sum over F_{p^2} (thread t gets the sum of the values of threads > t, plus `carry`);
// log-step Hillis-Steele in shared memory (sh: 2 * blockDim.x words).
__device__ __forceinline__ E2 block_suffix_excl(E2 v, E2 carry, u64* sh) {
    const int t = threadIdx.x, nt = blockDim.x;
    sh[2 * t] = v.a;
    sh[2 * t + 1] = v.b;
    __syncthreads();
    E2 acc = v;
    for (int off = 1; off < nt; off <<= 1) {
        E2 o = {0, 0};
        if (t + off < nt) o = E2{sh[2 * (t + off)], sh[2 * (t + off) + 1]};
        __syncthreads();
        acc = e2_add(acc, o);
        sh[2 * t] = acc.a;
        sh[2 * t + 1] = acc.b;
        __syncthreads();
    }
    // acc = inclusive suffix; exclusive = inclusive of t+1
    E2 ex = carry;
    if (t + 1 < nt) ex = e2_add(carry, E2{sh[2 * (t + 1)], sh[2 * (t + 1) + 1]});
    __syncthreads();
    return ex;
}
// divide_by_linear (division.rs:75-88) as a suffix scan: acc_k = sum_{m>=k} c_m z^{m-k}
//   = z^{-k} * S_k,  S_k = sum_{m>=k} c_m z^m ;  quotient q_k = acc_{k+1}, q_{n-1} = 0.
constexpr int SCAN_THREADS = 256, SCAN_ITEMS = 8, SCAN_CHUNK = SCAN_THREADS * SCAN_ITEMS;
// phase 1: d_m = c_m * z^m (in place) and per-chunk totals
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_phase1(u64* comp, size_t n, const u64* zhi, const u64* zlo,
                                                            u64* chunk_tot) {
    __shared__ u64 sh[2 * SCAN_THREADS];
    const size_t base = (size_t)blockIdx.x * SCAN_CHUNK + (size_t)threadIdx.x * SCAN_ITEMS;
    E2 tot = {0, 0};
    for (int i = 0; i < SCAN_ITEMS; i++) {
        const size_t m = base + i;
        if (m < n) {
            E2 d = e2_mul(E2{comp[2 * m], comp[2 * m + 1]}, e2_pow_tab(zhi, zlo, m));
            comp[2 * m] = d.a;
            comp[2 * m + 1] = d.b;
            tot = e2_add(tot, d);
        }
    }
    sh[2 * threadIdx.x] = tot.a;
    sh[2 * threadIdx.x + 1] = tot.b;
    __syncthreads();
    for (int off = SCAN_THREADS / 2; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) {
            sh[2 * threadIdx.x] = add(sh[2 * threadIdx.x], sh[2 * (threadIdx.x + off)]);
            sh[2 * threadIdx.x + 1] = add(sh[2 * threadIdx.x + 1], sh[2 * (threadIdx.x + off) + 1]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        chunk_tot[2 * blockIdx.x] = sh[0];
        chunk_tot[2 * blockIdx.x + 1] = sh[1];
    }
}
// phase 2: exclusive suffix sums of the chunk totals, one CTA: each thread owns a contiguous run of chunks
__global__ void __launch_bounds__(1024) k_scan_phase2(u64* chunk_tot, size_t nchunks) {
    __shared__ u64 sh[2 * 1024];
    const size_t per = (nchunks + blockDim.x - 1) / blockDim.x;
    const size_t lo = (size_t)threadIdx.x * per < nchunks ? (size_t)threadIdx.x * per : nchunks;
    const size_t hi = lo + per < nchunks ? lo + per : nchunks;
    E2 tot = {0, 0};
    for (size_t i = lo; i < hi; i++) tot = e2_add(tot, E2{chunk_tot[2 * i], chunk_tot[2 * i + 1]});
    E2 run = block_suffix_excl(tot, E2{0, 0}, sh);
    for (size_t i = hi; i-- > lo;) {
        E2 t = {chunk_tot[2 * i], chunk_tot[2 * i + 1]};
        chunk_tot[2 * i] = run.a;
        chunk_tot[2 * i + 1] = run.b;
        run = e2_add(run, t);
    }
}
// phase 3: S_k inside each chunk (+ carry), q_k = z^{-(k+1)} S_{k+1}; final = final*sh + q, written
// de-interleaved as two base-field columns (c0 column | c1 column) for the LDE.
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_phase3(const u64* d, size_t n, const u64* chunk_carry,
                                                            const u64* zihi, const u64* zilo, E2 shiftmul,
                                                            int first_batch, u64* final_cols /* 2 x n */) {
    __shared__ u64 sh[2 * SCAN_THREADS];
    const size_t base = (size_t)blockIdx.x * SCAN_CHUNK + (size_t)threadIdx.x * SCAN_ITEMS;
    // thread-local suffix sums
    E2 loc[SCAN_ITEMS];
    E2 run = {0, 0};
    for (int i = SCAN_ITEMS - 1; i >= 0; i--) {
        const size_t m = base + i;
        if (m < n) run = e2_add(run, E2{d[2 * m], d[2 * m + 1]});
        loc[i] = run;
    }
    // exclusive suffix over the CTA's threads (log-step scan) + the carry of the later chunks
    const E2 carry = block_suffix_excl(run, E2{chunk_carry[2 * blockIdx.x], chunk_carry[2 * blockIdx.x + 1]}, sh);
    // S_m = loc[i] + carry for m = base + i. q_k = z^{-(k+1)} * S_{k+1}.
    // This thread owns S_m for m in [base, base+ITEMS): emits q_{m-1}.
    for (int i = 0; i < SCAN_ITEMS; i++) {
        const size_t m = base + i;
        if (m >= n || m == 0) continue;
        E2 S = e2_add(loc[i], carry);
        E2 q = e2_mul(S, e2_pow_tab(zihi, zilo, m));
        const size_t k = m - 1;
        E2 f = q;
        if (!first_batch) f = e2_add(e2_mul(E2{final_cols[k], final_cols[n + k]}, shiftmul), q);
        final_cols[k] = canon(f.a);
        final_cols[n + k] = canon(f.b);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        // q_{n-1} = 0 (the reference pads the quotient back to a power of two, oracle.rs:210)
        E2 f = {0, 0};
        if (!first_batch) f = e2_mul(E2{final_cols[n - 1], final_cols[2 * n - 1]}, shiftmul);
        final_cols[n - 1] = canon(f.a);
        final_cols[2 * n - 1] = canon(f.b);
    }
}
// z == 0 special case: q_k = c_{k+1}
__global__ void k_div_by_x(const u64* comp, size_t n, E2 shiftmul, int first_batch, u64* final_cols) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    E2 q = {0, 0};
    if (k + 1 < n) q = E2{comp[2 * (k + 1)], comp[2 * (k + 1) + 1]};
    E2 f = q;
    if (!first_batch) f = e2_add(e2_mul(E2{final_cols[k], final_cols[n + k]}, shiftmul), q);
    final_cols[k] = canon(f.a);
    final_cols[n + k] = canon(f.b);
}

// FRI fold, leaf-local in bit-reversed storage (SURVEY appendix A.10; equals the reference's
// coefficient fold + coset_fft, prover.rs:111-119, and the verifier's compute_evaluation,
// verifier.rs:22-47): leaf l holds v_t = f(x0 * w_arity^{bitrev(t)}), x0 = shift * w_N^{bitrev(l)};
// u = iDFT(v) are x0^i P_i(y); result = sum_i u_i (beta/x0)^i.
struct FoldParams {
    const u64* values;   // N_k x 2 (bit-reversed order)
    u64* out;            // N_k/arity x 2
    size_t n_leaves;
    uint32_t log_leaves; // log2(N_k / arity)
    const u64* winv_hi;  // (w_Nk^-1)^(4096*i)
    const u64* winv_lo;  // (w_Nk^-1)^i, i < 4096
    u64 shift_inv;
    u64 beta0, beta1;
    u64 arity_inv;
    u64 root_inv[32];    // w_arity^-j
    size_t leaf0;        // global index of local leaf 0 (row-block sharded codewords)
};
template <int AB>
__global__ void __launch_bounds__(128) k_fri_fold(FoldParams fp) {
    constexpr int A = 1 << AB;
    const size_t l = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= fp.n_leaves) return;
    E2 e[A];
#pragma unroll
    for (int t = 0; t < A; t++) e[t] = E2{fp.values[2 * (l * A + t)], fp.values[2 * (l * A + t) + 1]};
    // DIT inverse DFT: bit-reversed input (storage order) -> natural-order u (unscaled)
#pragma unroll
    for (int s = 1; s <= AB; s++) {
        const int m = 1 << s, half = m >> 1;
#pragma unroll
        for (int k = 0; k < A; k += m) {
#pragma unroll
            for (int j = 0; j < half; j++) {
                const u64 w = fp.root_inv[j * (A / m)];
                E2 tt = (j == 0) ? e[k + j + half] : e2_scale(e[k + j + half], w);
                E2 uu = e[k + j];
                e[k + j] = e2_add(uu, tt);
                e[k + j + half] = e2_sub(uu, tt);
            }
        }
    }
    // gamma = beta / x0 ; x0^-1 = shift^-1 * w_N^{-bitrev(l)}
    const size_t r = fp.log_leaves ? (size_t)(__brevll(l + fp.leaf0) >> (64 - fp.log_leaves)) : 0;
    const u64 x0inv = mul(fp.shift_inv, mul(fp.winv_hi[r >> 12], fp.winv_lo[r & 4095]));
    const E2 gamma = E2{mul(fp.beta0, x0inv), mul(fp.beta1, x0inv)};
    E2 acc = e[A - 1];
#pragma unroll
    for (int i = A - 2; i >= 0; i--) acc = e2_add(e2_mul(acc, gamma), e[i]);
    acc = e2_scale(acc, fp.arity_inv);
    fp.out[2 * l] = canon(acc.a);
    fp.out[2 * l + 1] = canon(acc.b);
}
// values (bit-reversed, interleaved) -> two natural-order base columns
__global__ void k_unbitrev_split(const u64* values, size_t n, uint32_t log_n, u64* cols) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    size_t j = log_n ? (size_t)(__brevll(i) >> (64 - log_n)) : 0;
    cols[i] = values[2 * j];
    cols[n + i] = values[2 * j + 1];
}
__global__ void k_interleave(const u64* cols, size_t n, size_t count, u64* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    out[2 * i] = cols[i];
    out[2 * i + 1] = cols[n + i];
}
// ---- openings at a point (OpeningSet::new's eval_commitment, plonk/proof.rs:313-351; SURVEY 8(f) row 2) ----
// zt[k] = z^k (F_{p^2}) for k < n, from factored tables
__global__ void k_e2_pow_table(const u64* zhi, const u64* zlo, size_t n, u64* zt) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    E2 v = e2_pow_tab(zhi, zlo, k);
    zt[2 * k] = canon(v.a);
    zt[2 * k + 1] = canon(v.b);
}
// out[b] = sum_k coeffs[b][k] * z^k : one CTA per polynomial, 160-bit lazy accumulators, one reduction per thread
__global__ void __launch_bounds__(256) k_eval_ext(const u64* coeffs, size_t stride, size_t n, const u64* zt, u64* out) {
    __shared__ u64 sh[2 * 256];
    const u64* col = coeffs + (size_t)blockIdx.x * stride;
    Acc160 a0 = {0, 0, 0}, a1 = {0, 0, 0};
    for (size_t k = threadIdx.x; k < n; k += blockDim.x) {
        const u64 c = col[k];
        acc_mul(a0, c, zt[2 * k]);
        acc_mul(a1, c, zt[2 * k + 1]);
    }
    sh[2 * threadIdx.x] = acc_reduce(a0);
    sh[2 * threadIdx.x + 1] = acc_reduce(a1);
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) {
            sh[2 * threadIdx.x] = add(sh[2 * threadIdx.x], sh[2 * (threadIdx.x + off)]);
            sh[2 * threadIdx.x + 1] = add(sh[2 * threadIdx.x + 1], sh[2 * (threadIdx.x + off) + 1]);
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        out[2 * blockIdx.x] = canon(sh[0]);
        out[2 * blockIdx.x + 1] = canon(sh[1]);
    }
}

// ---- Z and partial products (wires_permutation_partial_products_and_zs, plonk/prover.rs:387-449;
//      SURVEY 8(f) row 3). Per (row i, chunk m): c = prod_{j in chunk} (w + beta*k_j*x_i + gamma) /
//      (w + beta*sigma + gamma); then ONE running product over the row-major sequence (i, m).
struct PPParams {
    const u64 *wires, *sigmas, *k_is;
    size_t n;
    uint32_t log_n, num_routed, degree, num_chunks;
    u64 beta, gamma;
    const u64 *xhi, *xlo;  // subgroup element of row i: xhi[i >> 12] * xlo[i & 4095] (w_n^(4096*k), w_n^k)
    u64* seq;              // n * num_chunks chunk products, row-major
    unsigned int* flag;    // set when a denominator is zero
};
constexpr int PP_MAX_CHUNKS = 32;
// One thread per row: the num_chunks chunk denominators of the row are inverted TOGETHER (Montgomery's trick, the
// reference's F::batch_multiplicative_inverse per row, field/src/types.rs:133-223 / prover.rs:421): one field inversion
// and 3 multiplies per chunk instead of one 64-squaring inversion per chunk.
__global__ void __launch_bounds__(128) k_pp_chunks(PPParams p) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const u64 bx = mul(p.beta, mul(p.xhi[i >> 12], p.xlo[i & 4095]));
    u64 num[PP_MAX_CHUNKS], den[PP_MAX_CHUNKS], pre[PP_MAX_CHUNKS];  // pre[m] = den_0 * ... * den_m
    u64 run = 1;
    for (uint32_t m = 0; m < p.num_chunks; m++) {
        u64 nm = 1, dn = 1;
        const uint32_t j1 = min((m + 1) * p.degree, p.num_routed);
        for (uint32_t j = m * p.degree; j < j1; j++) {  // consecutive threads -> consecutive rows: coalesced column reads
            const u64 w = p.wires[(size_t)j * p.n + i];
            const u64 wg = add(w, p.gamma);
            nm = mul(nm, add(wg, mul(bx, p.k_is[j])));
            dn = mul(dn, add(wg, mul(p.beta, p.sigmas[(size_t)j * p.n + i])));
        }
        if (canon(dn) == 0) atomicOr(p.flag, 1u);
        num[m] = nm;
        den[m] = dn;
        run = mul(run, dn);
        pre[m] = run;
    }
    u64 inv_run = gl::inv(run);  // 1 / (den_0 ... den_{M-1})
    for (uint32_t m = p.num_chunks; m-- > 0;) {  // 1/den_m = inv_run * pre[m-1], then inv_run *= den_m
        const u64 dinv = m ? mul(inv_run, pre[m - 1]) : inv_run;
        p.seq[i * p.num_chunks + m] = mul(num[m], dinv);
        inv_run = mul(inv_run, den[m]);
    }
}
// inclusive prefix scan under a field operation (MulOp: partial products; AddOp: logUp Z), 3 phases
struct MulOp {
    static __device__ __forceinline__ u64 id() { return 1; }
    static __device__ __forceinline__ u64 op(u64 a, u64 b) { return mul(a, b); }
};
struct AddOp {
    static __device__ __forceinline__ u64 id() { return 0; }
    static __device__ __forceinline__ u64 op(u64 a, u64 b) { return add(a, b); }
};
template <class Op>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan3_phase1(const u64* seq, size_t L, u64* chunk_tot) {
    __shared__ u64 sh[SCAN_THREADS];
    const size_t base = (size_t)blockIdx.x * SCAN_CHUNK + (size_t)threadIdx.x * SCAN_ITEMS;
    u64 t = Op::id();
    for (int k = 0; k < SCAN_ITEMS; k++)
        if (base + k < L) t = Op::op(t, seq[base + k]);
    sh[threadIdx.x] = t;
    __syncthreads();
    for (int off = SCAN_THREADS / 2; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) sh[threadIdx.x] = Op::op(sh[threadIdx.x], sh[threadIdx.x + off]);
        __syncthreads();
    }
    if (threadIdx.x == 0) chunk_tot[blockIdx.x] = sh[0];
}
// exclusive prefix of the chunk totals, one CTA: each thread owns a contiguous run
template <class Op>
__global__ void __launch_bounds__(1024) k_scan3_phase2(u64* chunk_tot, size_t nchunks) {
    __shared__ u64 sh[1024];
    const size_t per = (nchunks + 1023) / 1024;
    const size_t lo = (size_t)threadIdx.x * per, hi = lo + per < nchunks ? lo + per : nchunks;
    u64 t = Op::id();
    for (size_t k = lo; k < hi; k++) t = Op::op(t, chunk_tot[k]);
    sh[threadIdx.x] = t;
    __syncthreads();
    if (threadIdx.x == 0) {  // 1024 sequential steps
        u64 run = Op::id();
        for (int k = 0; k < 1024; k++) {
            u64 v = sh[k];
            sh[k] = run;
            run = Op::op(run, v);
        }
    }
    __syncthreads();
    u64 run = sh[threadIdx.x];
    for (size_t k = lo; k < hi; k++) {
        u64 v = chunk_tot[k];
        chunk_tot[k] = run;
        run = Op::op(run, v);
    }
}
// phase 3: inclusive prefix inside each chunk; scatter to the output columns:
// acc(i, m) -> partial product column m (m < M-1) at row i, or Z at row i+1 (m == M-1); Z(0) = the identity.
// With M = 1 this is the exclusive scan of one column into out (seq and out must not overlap).
template <class Op>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan3_phase3(const u64* seq, size_t L, const u64* chunk_carry, size_t n,
                                                             uint32_t M, u64* out) {
    __shared__ u64 sh[SCAN_THREADS];
    const size_t base = (size_t)blockIdx.x * SCAN_CHUNK + (size_t)threadIdx.x * SCAN_ITEMS;
    u64 loc[SCAN_ITEMS];
    u64 run = Op::id();
    for (int k = 0; k < SCAN_ITEMS; k++) {
        if (base + k < L) run = Op::op(run, seq[base + k]);
        loc[k] = run;
    }
    sh[threadIdx.x] = run;
    __syncthreads();
    if (threadIdx.x == 0) {
        u64 r = chunk_carry[blockIdx.x];
        for (int t = 0; t < SCAN_THREADS; t++) {
            u64 v = sh[t];
            sh[t] = r;
            r = Op::op(r, v);
        }
    }
    __syncthreads();
    const u64 carry = sh[threadIdx.x];
    for (int k = 0; k < SCAN_ITEMS; k++) {
        const size_t t = base + k;
        if (t >= L) break;
        const u64 acc = canon(Op::op(carry, loc[k]));
        const size_t i = t / M, m = t % M;
        if (m + 1 < M) out[m * n + i] = acc;
        else if (i + 1 < n) out[(size_t)(M - 1) * n + i + 1] = acc;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) out[(size_t)(M - 1) * n] = Op::id();
}

// ---- lookup argument helper columns (compute_lookup_polys, plonk/prover.rs:458-577; SURVEY 8(f) row 3) ----
// For one LookupWire the reference walks the rows from first_lut_row down to last_lu_row and fills
//   RE[row]          = RE[row+1] * delta^L + sum_s combo_B(row, s) * delta^(L-1-s)          (LUT rows only, L = num_lut_slots)
//   SLDC[slot][row]  = running sum over (row descending, slot ascending) of
//                        + sum_{s in slot} multiplicity(row, s) / (alpha - combo_A(row, s))    on LookupTableGate rows
//                        - sum_{s in slot} 1 / (alpha - combo_A(row, s))                        on LookupGate rows
// i.e. one affine and one additive scan over a sequence of T rows (x P slots). k_lookup_terms computes the per-row
// terms (one batch inversion per row, field/src/types.rs:133-223), k_affine_scan runs both scans in one CTA.
struct LookupParams {
    const u64* wires;      // column-major, wire w of row i at wires[w*n + i]
    size_t n;
    uint32_t num_lu_slots, num_lut_slots, P, max_lookup_degree, max_lookup_table_degree;
    u64 dA, dB, dAlpha, dDelta;
    uint32_t first_lut, last_lut, last_lu;  // rows (first_lut >= last_lut > last_lu allowed to be equal ranges)
    u64* term;             // T * P additive terms in scan order
    u64* reh;              // rows_lut Horner values H(row)
    unsigned int* flag;
};
constexpr int LOOKUP_MAX_SLOTS = 64;
__global__ void __launch_bounds__(128) k_lookup_terms(LookupParams p) {
    const uint32_t rows_lut = p.first_lut - p.last_lut + 1, rows_lu = p.last_lut - p.last_lu;
    const uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos >= rows_lut + rows_lu) return;
    const bool lut = pos < rows_lut;
    const size_t row = lut ? (size_t)p.first_lut - pos : (size_t)p.last_lut - 1 - (pos - rows_lut);
    const uint32_t ns = lut ? p.num_lut_slots : p.num_lu_slots, wpe = lut ? 3u : 2u;
    u64 pre[LOOKUP_MAX_SLOTS], den[LOOKUP_MAX_SLOTS];
    u64 run = 1, h = 0;
    for (uint32_t s = 0; s < ns; s++) {
        const u64 inp = p.wires[(size_t)(wpe * s) * p.n + row], out = p.wires[(size_t)(wpe * s + 1) * p.n + row];
        const u64 d = sub(p.dAlpha, add(inp, mul(p.dA, out)));  // alpha - (inp + A * out)
        if (canon(d) == 0) atomicOr(p.flag, 1u);
        den[s] = d;
        run = mul(run, d);
        pre[s] = run;
        if (lut) h = add(mul(h, p.dDelta), add(inp, mul(p.dB, out)));  // new_re = new_re * delta + lookup_combo
    }
    if (lut) p.reh[pos] = h;
    u64 inv_run = gl::inv(run);
    for (uint32_t s = ns; s-- > 0;) {  // den[s] <- 1 / den[s]
        const u64 di = s ? mul(inv_run, pre[s - 1]) : inv_run;
        inv_run = mul(inv_run, den[s]);
        den[s] = di;
    }
    const uint32_t per = lut ? p.max_lookup_table_degree : p.max_lookup_degree;
    for (uint32_t slot = 0; slot < p.P; slot++) {
        u64 acc = 0;
        const uint32_t s1 = min((slot + 1) * per, ns);
        for (uint32_t s = slot * per; s < s1; s++)
            acc = lut ? add(acc, mul(p.wires[(size_t)(3 * s + 2) * p.n + row], den[s])) : add(acc, den[s]);
        p.term[(size_t)pos * p.P + slot] = lut ? acc : neg(acc);
    }
}
// y_k = y_{k-1} * a + b_k over `len` items (a constant; a = 1: additive scan), y_{-1} = init; one CTA of 1024 threads.
// out_of(k) maps item k to its output address (two layouts: SLDC and RE), given by (P, rows_lut, ...) in `p`.
__global__ void __launch_bounds__(1024) k_affine_scan(const u64* b, size_t len, u64 a, u64 init, LookupParams p, int re_mode,
                                                      u64* out) {
    __shared__ u64 sa[1024], sb[1024];
    const size_t per = (len + 1023) / 1024;
    const size_t lo = (size_t)threadIdx.x * per, hi = lo + per < len ? lo + per : len;
    u64 ca = 1, cb = 0;  // composition of my run: y -> y * ca + cb
    for (size_t k = lo; k < hi; k++) {
        ca = mul(ca, a);
        cb = add(mul(cb, a), b[k]);
    }
    sa[threadIdx.x] = ca;
    sb[threadIdx.x] = cb;
    __syncthreads();
    if (threadIdx.x == 0) {  // exclusive scan of the 1024 run compositions, applied to init
        u64 y = init;
        for (int t = 0; t < 1024; t++) {
            const u64 na = sa[t], nb = sb[t];
            sb[t] = y;
            y = add(mul(y, na), nb);
        }
    }
    __syncthreads();
    u64 y = sb[threadIdx.x];
    const uint32_t rows_lut = p.first_lut - p.last_lut + 1;
    for (size_t k = lo; k < hi; k++) {
        y = add(mul(y, a), b[k]);
        size_t pos, col;
        if (re_mode) {
            pos = k;
            col = 0;
        } else {
            pos = k / p.P;
            col = 1 + k % p.P;
        }
        const size_t row = pos < rows_lut ? (size_t)p.first_lut - pos : (size_t)p.last_lut - 1 - (pos - rows_lut);
        out[col * p.n + row] = canon(y);
    }
}

// ---- STARK quotient evaluation (compute_quotient_polys, starky/src/prover.rs:488-668; SURVEY 8(f) row 1) ----
// The constraints (Stark::eval_packed_generic, starky/src/stark.rs) arrive as a small straight-line program over the
// local row, the next row and the public inputs; value k = result of instruction k. One thread per point of the
// quotient coset g*<w_size>, size = n << quotient_degree_bits, reading the trace LDE in place (column-major leaves):
//   local = leaf bitrev(i*step), next = leaf bitrev(((i + next_step) % size) * step)      (get_lde_values, oracle.rs:142-147)
struct StarkQuotientParams {
    const u64* lde;        // trace LDE, column k at lde + k*lde_stride, leaf order
    size_t lde_stride;
    const u64* aux;        // auxiliary polynomials' LDE (same degree and rate, same layout), or null
    size_t aux_stride;
    uint32_t log_N;        // log2 of the LDE size
    uint32_t degree_bits, qd_bits;
    const gl_stark_instr* prog;
    uint32_t n_instr;
    const u64* consts;     // public inputs first, then the program's constants
    u64 alphas[GL_STARK_MAX_ALPHAS];
    uint32_t n_alphas;
    const u64 *xhi, *xlo;  // w_size^i = xhi[i >> 12] * xlo[i & 4095]
    u64 shift;             // coset shift g
    u64 last;              // w_n^-1, the last element of the trace subgroup
    u64 n_field;           // n as a field element
    u64 zh[GL_STARK_MAX_QD], zh_inv[GL_STARK_MAX_QD];  // Z_H on the coset: g^n * w_{2^qd}^j - 1 and inverses (ZeroPolyOnCoset)
    u64* out;              // n_alphas columns of `size` values
    unsigned int* flag;
};
__global__ void __launch_bounds__(128) k_stark_quotient(StarkQuotientParams p) {
    const size_t size = (size_t)1 << (p.degree_bits + p.qd_bits);
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= size) return;
    const uint32_t step_log = p.log_N - p.degree_bits - p.qd_bits;   // step = 2^(rate_bits - qd_bits)
    const size_t inext = (i + ((size_t)1 << p.qd_bits)) & (size - 1);
    const size_t jl = (size_t)(__brevll((unsigned long long)(i << step_log)) >> (64 - p.log_N));
    const size_t jn = (size_t)(__brevll((unsigned long long)(inext << step_log)) >> (64 - p.log_N));
    const u64 x = mul(p.shift, mul(p.xhi[i >> 12], p.xlo[i & 4095]));
    const u64 z_last = sub(x, p.last);
    const u64 zh = p.zh[i & (((size_t)1 << p.qd_bits) - 1)];
    // Lagrange selectors on the coset (PolynomialValues::selector(..).lde_onto_coset, prover.rs:527-531) in closed form:
    // L_0(x) = Z_H(x) / (n (x - 1)),  L_{n-1}(x) = Z_H(x) * last / (n (x - last)); one inversion for both
    const u64 xm1 = sub(x, 1);
    const u64 den = mul(p.n_field, mul(xm1, z_last));
    if (canon(den) == 0) atomicOr(p.flag, 1u);
    const u64 t = mul(zh, gl::inv(den));
    const u64 l_first = mul(t, z_last);
    const u64 l_last = mul(mul(t, p.last), xm1);
    u64 acc[GL_STARK_MAX_ALPHAS];
#pragma unroll
    for (int a = 0; a < GL_STARK_MAX_ALPHAS; a++) acc[a] = 0;
    u64 v[GL_STARK_MAX_INSTR];
    for (uint32_t k = 0; k < p.n_instr; k++) {
        const gl_stark_instr in = p.prog[k];
        u64 r = 0;
        switch (in.op) {
            case GL_STARK_LOCAL: r = p.lde[(size_t)in.a * p.lde_stride + jl]; break;
            case GL_STARK_NEXT: r = p.lde[(size_t)in.a * p.lde_stride + jn]; break;
            case GL_STARK_AUX_LOCAL: r = p.aux[(size_t)in.a * p.aux_stride + jl]; break;
            case GL_STARK_AUX_NEXT: r = p.aux[(size_t)in.a * p.aux_stride + jn]; break;
            case GL_STARK_CONST: r = p.consts[in.a]; break;
            case GL_STARK_ADD: r = add(v[in.a], v[in.b]); break;
            case GL_STARK_SUB: r = sub(v[in.a], v[in.b]); break;
            case GL_STARK_MUL: r = mul(v[in.a], v[in.b]); break;
            default: {  // GL_STARK_EMIT: ConstraintConsumer::constraint* (constraint_consumer.rs:60-84)
                u64 c = v[in.a];
                if (in.b == GL_STARK_TRANSITION) c = mul(c, z_last);
                else if (in.b == GL_STARK_FIRST_ROW) c = mul(c, l_first);
                else if (in.b == GL_STARK_LAST_ROW) c = mul(c, l_last);
                for (uint32_t a = 0; a < p.n_alphas; a++) acc[a] = add(mul(acc[a], p.alphas[a]), c);
            }
        }
        v[k] = r;
    }
    const u64 zi = p.zh_inv[i & (((size_t)1 << p.qd_bits) - 1)];
    for (uint32_t a = 0; a < p.n_alphas; a++) p.out[(size_t)a * size + i] = canon(mul(acc[a], zi));
}
// ---- starky logUp helper columns (lookup_helper_columns, starky/src/lookup.rs:579-652): one thread per trace row; the
// row's evaluation is gl_logup.cuh, the Z columns are the exclusive additive scan (k_scan3_*<AddOp>) of its terms
__global__ void __launch_bounds__(128) k_logup_rows(LogupParams p, unsigned int* flag) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    u64 den[GL_LOGUP_MAX_DENOMINATORS], pre[GL_LOGUP_MAX_DENOMINATORS];
    if (!logup_eval_row(p, i, den, pre)) atomicOr(flag, 1u);
}
// any non-zero word in [begin, begin + count) of each of `cols` columns (stride `stride`) -> flag
__global__ void k_any_nonzero(const u64* data, size_t stride, size_t begin, size_t count, unsigned int* flag) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    if (canon(data[(size_t)blockIdx.y * stride + begin + i]) != 0) atomicOr(flag, 2u);
}

// ---- plonky2 quotient evaluation (compute_quotient_polys, plonk/prover.rs:609-815; SURVEY 8(f) row 1) ----
// one thread per point of the quotient coset; the point's evaluation is gl_vanishing.cuh
__global__ void __launch_bounds__(128) k_plonk_quotient(VanishingParams p) {
    const size_t size = (size_t)1 << (p.degree_bits + p.qd_bits);
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= size) return;
    u64 regs[GL_VP_MAX_REGS];
    if (!vp_eval_point(p, i, regs)) atomicOr(p.flag, 1u);
}

// proof-of-work grind (prover.rs:183-194): smallest qualifying nonce via atomicMin
struct PowParams {
    u64 state[12];
    uint32_t pos, min_lz;
    u64 start, count;
};
__global__ void __launch_bounds__(128) k_fri_pow(PowParams pp, unsigned long long* result) {
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < pp.count; i += stride) {
        const u64 cand = pp.start + i;
        u64 s[12];
#pragma unroll
        for (int k = 0; k < 12; k++) s[k] = pp.state[k];
        s[pp.pos] = cand;
        poseidon_permute(s);
        const u64 resp = canon(s[7]);
        const uint32_t lz = resp ? (uint32_t)__clzll((long long)resp) : 64u;
        if (lz >= pp.min_lz) atomicMin(result, (unsigned long long)cand);
    }
}

struct gl_fri {
    gl_ctx* ctx;
    uint32_t log_n, rate_bits, cap_height;
    u64* coeff_cols = nullptr;  // 2 x n (c0 column, c1 column), natural order
    u64* values = nullptr;      // current round values, N_k x 2, bit-reversed order (owned unless moved to a tree)
    uint32_t log_cur = 0;       // log2(N_k)
    u64 shift = 0;              // current coset shift
    uint32_t pending_arity_bits = 0;
    bool committed = false;     // commit_round done, fold pending
    u64* round_values = nullptr;  // the committed round's whole values buffer (owned by its tree) and leaf count
    size_t round_leaves = 0;
    // value-domain, row-block sharded state (gl_fri_begin_values): `values` holds only rows
    // [vshard_index * 2^(log_cur - vshard_log), ...) of the codeword; log_cur stays the GLOBAL length
    uint32_t vshard_index = 0, vshard_log = 0;
    std::vector<Tree> trees;
};

static int fri_finish_begin(gl_ctx* ctx, gl_fri* f) {
    // lde_final_poly / coset_fft (oracle.rs:215-220) on both F_{p^2} components, leaf-major W = 2
    const size_t n = (size_t)1 << f->log_n, N = n << f->rate_bits;
    TRY(dmalloc(ctx, &f->values, 2 * N));
    u64* cols;
    TRY(dmalloc(ctx, &cols, 2 * N));
    int rc = lde_columns(ctx, f->coeff_cols, n, 2, (int)f->log_n, (int)f->rate_bits, MULTIPLICATIVE_GROUP_GENERATOR, cols, N);
    if (rc == GL_OK) {  // (c0 column | c1 column) -> interleaved F_{p^2} values, the FRI leaves' layout
        k_interleave<<<(unsigned)((N + 255) / 256), 256, 0, ctx->stream>>>(cols, N, N, f->values);
        ctx->launches++;
    }
    dfree(ctx, cols);
    TRY(rc);
    f->log_cur = f->log_n + f->rate_bits;
    f->shift = MULTIPLICATIVE_GROUP_GENERATOR;
    return GL_OK;
}

// =====================================================================================
// C ABI
// =====================================================================================
extern "C" {

int gl_ctx_create(int device, void* stream, gl_ctx** out) {
    if (!out) return set_err(nullptr, GL_ERR_BAD_ARG, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return set_err(nullptr, GL_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                       cudaGetErrorString(e));
    if (device < 0 || device >= count) return set_err(nullptr, GL_ERR_BAD_ARG, "device %d out of range", device);
    gl_ctx* ctx = new gl_ctx();
    ctx->device = device;
    auto init = [&]() -> int {
        CK(ctx, cudaSetDevice(device));
        if (stream) {
            ctx->stream = (cudaStream_t)stream;
        } else {
            CK(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
            ctx->own_stream = true;
        }
        CK(ctx, cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device));
        CK(ctx, cudaDeviceGetAttribute(&ctx->coop_ok, cudaDevAttrCooperativeLaunch, device));
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->coop_blocks_per_sm, k_merkle_upper, HASH_CTA, 0) !=
            cudaSuccess)
            ctx->coop_blocks_per_sm = 0;
        const PoseidonTables& t = host_poseidon_tables();
        CK(ctx, cudaMemcpyToSymbol(c_pos, &t, sizeof(PoseidonTables)));
        return GL_OK;
    };
    const int rc_init = init();
    if (rc_init != GL_OK) {  // no half-built context escapes (and none leaks)
        if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
        delete ctx;
        return rc_init;
    }
    // keep freed blocks in the pool: the commit buffers are large and re-allocated every call
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long thr = ~0ULL;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
    }
    *out = ctx;
    return GL_OK;
}
void gl_ctx_destroy(gl_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto& kv : ctx->step_tabs) cudaFreeAsync(kv.second, ctx->stream);
    for (auto& kv : ctx->post_tabs) cudaFreeAsync(kv.second, ctx->stream);
    for (auto& kv : ctx->fold_tabs) cudaFreeAsync(kv.second, ctx->stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->scratch) cudaFreeAsync(ctx->scratch, ctx->stream);
    if (ctx->dstage) cudaFreeAsync(ctx->dstage, ctx->stream);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}
const char* gl_last_error(const gl_ctx* ctx) { return ctx ? ctx->err.c_str() : g_last_error.c_str(); }
int gl_ctx_synchronize(gl_ctx* ctx) {
    CK(ctx, cudaStreamSynchronize(ctx->stream));
    return GL_OK;
}
uint64_t gl_ctx_launch_count(const gl_ctx* ctx) { return ctx->launches; }
int gl_ctx_set_ntt_group(gl_ctx* ctx, uint32_t columns) {
    // bit 31 selects the kernel variant of the column pass (a measurement switch, see gl_ntt_host.cuh)
    ctx->ntt_variant = (columns >> 31) & 1;
    ctx->ntt_group = columns & 0x7FFFFFFFu;
    return GL_OK;
}
int gl_ctx_set_profiling(gl_ctx* ctx, int on) {
    ctx->prof_on = on != 0;
    return GL_OK;
}
int gl_ctx_phase_ms(gl_ctx* ctx, int phase, double* ms, uint64_t* count) {
    if (phase < 0 || phase >= GL_NUM_PHASES) return set_err(ctx, GL_ERR_BAD_ARG, "bad phase");
    if (!ctx->prof_pending.empty()) {
        CK(ctx, cudaStreamSynchronize(ctx->stream));
        for (auto& p : ctx->prof_pending) {
            float t = 0;
            cudaEventElapsedTime(&t, p.a, p.b);
            ctx->prof_ms[p.phase] += t;
            ctx->prof_count[p.phase]++;
            cudaEventDestroy(p.a);
            cudaEventDestroy(p.b);
        }
        ctx->prof_pending.clear();
    }
    if (ms) *ms = ctx->prof_ms[phase];
    if (count) *count = ctx->prof_count[phase];
    return GL_OK;
}
int gl_ctx_reset_phases(gl_ctx* ctx) {
    TRY(gl_ctx_phase_ms(ctx, 0, nullptr, nullptr));
    for (int i = 0; i < GL_NUM_PHASES; i++) {
        ctx->prof_ms[i] = 0;
        ctx->prof_count[i] = 0;
    }
    return GL_OK;
}

int gl_ntt(gl_ctx* ctx, uint64_t* data, uint32_t log_n, uint32_t batch, size_t stride, int inverse,
           uint32_t zero_factor_log, uint64_t coset_shift, int mem) {
    (void)zero_factor_log;
    if (!ctx || !data) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    CK(ctx, cudaSetDevice(ctx->device));
    if (log_n > 3 * NTT_MAX_LOG_PASS) return set_err(ctx, GL_ERR_UNSUPPORTED, "log_n %u > 30", log_n);
    const size_t n = (size_t)1 << log_n;
    if (batch > 1 && stride < n) return set_err(ctx, GL_ERR_BAD_SHAPE, "stride %zu < n %zu", stride, n);
    if (canon(coset_shift) == 0) return set_err(ctx, GL_ERR_BAD_ARG, "coset_shift must be non-zero");
    if (mem == GL_MEM_DEVICE) return ntt_natural(ctx, data, stride, data, stride, (int)log_n, batch, inverse != 0, coset_shift);
    u64* d;
    TRY(dmalloc(ctx, &d, (size_t)batch * n));
    const size_t pitch = (batch > 1 ? stride : n) * 8;  // one strided copy each way
    int rc = GL_OK;
    if (cudaMemcpy2DAsync(d, n * 8, data, pitch, n * 8, batch, cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
        rc = set_err(ctx, GL_ERR_CUDA, "H2D: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc == GL_OK) rc = ntt_natural(ctx, d, n, d, n, (int)log_n, batch, inverse != 0, coset_shift);
    if (rc == GL_OK) {
        cudaError_t e = cudaMemcpy2DAsync(data, pitch, d, n * 8, n * 8, batch, cudaMemcpyDeviceToHost, ctx->stream);
        if (e != cudaSuccess) rc = set_err(ctx, GL_ERR_CUDA, "D2H: %s", cudaGetErrorString(e));
        if (rc == GL_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess)
            rc = set_err(ctx, GL_ERR_CUDA, "sync failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    dfree(ctx, d);
    return rc;
}

void* gl_ctx_stream(const gl_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int gl_ntt_bcast(gl_ctx* ctx, const uint64_t* in, size_t in_stride, uint32_t log_n, uint32_t batch, int inverse,
                 uint64_t* const* outs, uint32_t n_outs, size_t out_stride) {
    if (!ctx || !in || !outs || n_outs == 0 || n_outs > 8) return set_err(ctx, GL_ERR_BAD_ARG, "need 1..8 destinations");
    CK(ctx, cudaSetDevice(ctx->device));
    if (log_n < 1 || log_n > 3 * NTT_MAX_LOG_PASS) return set_err(ctx, GL_ERR_UNSUPPORTED, "log_n %u not in 1..30", log_n);
    const size_t n = (size_t)1 << log_n;
    if (batch > 1 && (in_stride < n || out_stride < n)) return set_err(ctx, GL_ERR_BAD_SHAPE, "stride < n");
    PeerOuts po;
    for (uint32_t i = 0; i < n_outs; i++) {
        if (!outs[i]) return set_err(ctx, GL_ERR_BAD_ARG, "destination %u is NULL", i);
        if (outs[i] == in) return set_err(ctx, GL_ERR_BAD_ARG, "gl_ntt_bcast is out of place");
        if (i) po.p[po.n++] = outs[i];
    }
    return ntt_natural(ctx, in, in_stride, outs[0], out_stride, (int)log_n, batch, inverse != 0, 1, &po);
}

// src (this GPU's memory) -> every destination, 16 bytes per thread per step: full 128-byte lines per warp instruction,
// the granularity NVLink / NVSwitch multicast writes need to run at link speed (the 64-byte segments of the fused
// natural-order stores reach ~120 GB/s; this copy is bound by the link).
struct BcastDests {
    ulonglong2* p[8];
    int n;
};
__global__ void __launch_bounds__(256) k_bcast_copy(const ulonglong2* __restrict__ src, size_t n16, BcastDests d) {
    // 8 independent 16-byte loads per thread before the first store: with few CTAs (the copy shares the GPU with the
    // transforms) the bytes in flight, not the link, bounded the first version at ~120-190 GB/s
    constexpr int U = 8;
    const size_t step = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (U - 1) * step < n16; i += U * step) {
        ulonglong2 v[U];
#pragma unroll
        for (int u = 0; u < U; u++) v[u] = src[i + u * step];
#pragma unroll
        for (int u = 0; u < U; u++)
            for (int k = 0; k < d.n; k++) d.p[k][i + u * step] = v[u];
    }
    for (; i < n16; i += step) {
        const ulonglong2 v = src[i];
        for (int k = 0; k < d.n; k++) d.p[k][i] = v;
    }
}
int gl_bcast(gl_ctx* ctx, const uint64_t* src, size_t words, uint64_t* const* dests, uint32_t n_dests, uint32_t max_ctas) {
    if (!ctx || !src || !dests || n_dests == 0 || n_dests > 8) return set_err(ctx, GL_ERR_BAD_ARG, "need 1..8 destinations");
    if (words == 0) return GL_OK;
    if ((words & 1) || ((uintptr_t)src & 15)) return set_err(ctx, GL_ERR_BAD_ARG, "gl_bcast needs 16-byte aligned, even-length buffers");
    CK(ctx, cudaSetDevice(ctx->device));
    BcastDests d;
    d.n = (int)n_dests;
    for (uint32_t i = 0; i < n_dests; i++) {
        if (!dests[i] || ((uintptr_t)dests[i] & 15)) return set_err(ctx, GL_ERR_BAD_ARG, "destination %u is NULL or misaligned", i);
        d.p[i] = (ulonglong2*)dests[i];
    }
    const size_t n16 = words / 2;
    size_t ctas = (n16 + 255) / 256;
    const size_t cap = max_ctas ? max_ctas : (size_t)ctx->sm_count * 2;
    if (ctas > cap) ctas = cap;
    k_bcast_copy<<<(unsigned)ctas, 256, 0, ctx->stream>>>((const ulonglong2*)src, n16, d);
    CKL(ctx);
    return GL_OK;
}

static int commit_check_shape(gl_ctx* ctx, uint32_t B, uint32_t log_n, uint32_t rate_bits, uint32_t cap_height,
                              uint32_t shard_index, uint32_t num_shards, uint32_t* shard_log) {
    *shard_log = 0;
    if (log2_exact(num_shards, shard_log) || shard_index >= num_shards)
        return set_err(ctx, GL_ERR_BAD_ARG, "bad shard %u of %u (power of two required)", shard_index, num_shards);
    if (*shard_log > cap_height)
        return set_err(ctx, GL_ERR_BAD_SHAPE, "num_shards=%u exceeds the cap size 2^%u: shards must own whole cap subtrees",
                       num_shards, cap_height);
    if (B == 0) return set_err(ctx, GL_ERR_BAD_SHAPE, "empty polynomial batch");
    if (log_n > 3 * NTT_MAX_LOG_PASS) return set_err(ctx, GL_ERR_UNSUPPORTED, "log_n %u > 30", log_n);
    if (log_n + rate_bits > 32) return set_err(ctx, GL_ERR_BAD_SHAPE, "LDE size exceeds the field's 2-adicity");
    if (cap_height > log_n + rate_bits)
        return set_err(ctx, GL_ERR_BAD_SHAPE, "cap_height=%u should be at most log2(leaves.len())=%u", cap_height,
                       log_n + rate_bits);
    return GL_OK;
}

int gl_commit_begin(gl_ctx* ctx, uint32_t B, uint32_t log_n, uint32_t rate_bits, uint32_t cap_height, int blinding,
                    uint32_t shard_index, uint32_t num_shards, uint64_t* coeff_storage, gl_commit** out) {
    if (!ctx || !out) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    *out = nullptr;
    uint32_t shard_log = 0;
    TRY(commit_check_shape(ctx, B, log_n, rate_bits, cap_height, shard_index, num_shards, &shard_log));
    CK(ctx, cudaSetDevice(ctx->device));
    gl_commit* c = new gl_commit();
    c->ctx = ctx;
    c->B = B;
    c->W = B + (blinding ? GL_SALT_SIZE : 0);
    c->degree_log = log_n;
    c->rate_bits = rate_bits;
    c->blinding = blinding != 0;
    c->shard_index = shard_index;
    c->shard_log = shard_log;
    int rc = commit_alloc(ctx, c, cap_height, coeff_storage);
    if (rc != GL_OK) {
        gl_commit_destroy(c);
        return rc;
    }
    *out = c;
    return GL_OK;
}
int gl_commit_add_columns(gl_commit* c, uint32_t first_col, uint32_t count, const uint64_t* cols, size_t col_stride,
                          int kind, int mem) {
    if (!c) return set_err(nullptr, GL_ERR_BAD_ARG, "null handle");
    gl_ctx* ctx = c->ctx;
    if (c->finished) return set_err(ctx, GL_ERR_BAD_ARG, "commitment already finished");
    if (!cols || kind < 0 || kind > 2) return set_err(ctx, GL_ERR_BAD_ARG, "bad argument");
    if (count == 0) return GL_OK;
    if ((size_t)first_col + count > c->B) return set_err(ctx, GL_ERR_BAD_SHAPE, "columns %u..%u outside the batch of %u", first_col, first_col + count, c->B);
    const size_t n = (size_t)1 << c->degree_log;
    if (count > 1 && col_stride < n) return set_err(ctx, GL_ERR_BAD_SHAPE, "Polynomial degrees inconsistent (stride < n)");
    CK(ctx, cudaSetDevice(ctx->device));
    u64* dst = c->coeffs + (size_t)first_col * n;
    if (!(mem == GL_MEM_DEVICE && cols == dst && (col_stride == n || count == 1)))
        CK(ctx, cudaMemcpy2DAsync(dst, n * 8, cols, col_stride * 8, n * 8, count,
                                  mem == GL_MEM_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, ctx->stream));
    return commit_chunk(ctx, c, first_col, count, kind);
}
int gl_commit_finish(gl_commit* c, const uint64_t* salt, int mem) {
    if (!c) return set_err(nullptr, GL_ERR_BAD_ARG, "null handle");
    gl_ctx* ctx = c->ctx;
    if (c->finished) return set_err(ctx, GL_ERR_BAD_ARG, "commitment already finished");
    if (c->blinding != (salt != nullptr)) return set_err(ctx, GL_ERR_BAD_ARG, "salt must be given exactly when blinding was requested");
    CK(ctx, cudaSetDevice(ctx->device));
    return commit_finish(ctx, c, salt, mem);
}

int gl_commit_create(gl_ctx* ctx, const uint64_t* cols, size_t col_stride, uint32_t B, uint32_t log_n,
                     uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt, int is_coeffs, int mem,
                     gl_commit** out) {
    return gl_commit_create_sharded(ctx, cols, col_stride, B, log_n, rate_bits, cap_height, salt, is_coeffs, mem, 0, 1,
                                    out);
}
int gl_commit_create_sharded(gl_ctx* ctx, const uint64_t* cols, size_t col_stride, uint32_t B, uint32_t log_n,
                             uint32_t rate_bits, uint32_t cap_height, const uint64_t* salt, int is_coeffs, int mem,
                             uint32_t shard_index, uint32_t num_shards, gl_commit** out) {
    if (!ctx || !cols || !out) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    *out = nullptr;
    uint32_t shard_log = 0;
    TRY(commit_check_shape(ctx, B, log_n, rate_bits, cap_height, shard_index, num_shards, &shard_log));
    CK(ctx, cudaSetDevice(ctx->device));
    if (B > 1 && col_stride < ((size_t)1 << log_n))
        return set_err(ctx, GL_ERR_BAD_SHAPE, "Polynomial degrees inconsistent (stride < n)");
    gl_commit* c = new gl_commit();
    c->ctx = ctx;
    c->B = B;
    c->W = B + (salt ? GL_SALT_SIZE : 0);
    c->degree_log = log_n;
    c->rate_bits = rate_bits;
    c->blinding = salt != nullptr;
    c->shard_index = shard_index;
    c->shard_log = shard_log;
    int rc = commit_build(ctx, c, cols, col_stride, salt, is_coeffs, mem, cap_height);
    if (rc != GL_OK) {
        gl_commit_destroy(c);
        return rc;
    }
    *out = c;
    return GL_OK;
}
void gl_commit_destroy(gl_commit* c) {
    if (!c) return;
    cudaSetDevice(c->ctx->device);
    if (c->own_coeffs) dfree(c->ctx, c->coeffs);
    tree_free(c->ctx, c->tree);
    delete c;
}
uint32_t gl_commit_num_polys(const gl_commit* c) { return c->B; }
uint32_t gl_commit_leaf_width(const gl_commit* c) { return c->W; }
uint32_t gl_commit_degree_log(const gl_commit* c) { return c->degree_log; }
uint32_t gl_commit_rate_bits(const gl_commit* c) { return c->rate_bits; }
uint32_t gl_commit_cap_height(const gl_commit* c) { return c->tree.cap_height + c->shard_log; }
#define NEED_FINISHED(c)                                                                                     \
    do {                                                                                                     \
        if (!(c)->finished) return set_err((c)->ctx, GL_ERR_BAD_ARG, "gl_commit_finish has not been called"); \
    } while (0)
int gl_commit_cap(gl_commit* c, uint64_t* out, int mem) {
    NEED_FINISHED(c);
    return copy_out(c->ctx, out, c->tree.cap, c->tree.cap_words(), mem);
}
int gl_commit_coeffs(gl_commit* c, uint64_t* out, int mem) {
    return copy_out(c->ctx, out, c->coeffs, (size_t)c->B << c->degree_log, mem);
}
int gl_commit_leaves(gl_commit* c, size_t row_begin, size_t row_count, uint64_t* out, int mem) {
    gl_ctx* ctx = c->ctx;
    if (row_begin + row_count > c->tree.N) return set_err(ctx, GL_ERR_BAD_ARG, "row range out of bounds");
    if (row_count == 0) return GL_OK;
    CK(ctx, cudaSetDevice(ctx->device));
    // the LDE is column-major on the device; the reference's row-major leaves are produced on demand, in slabs
    const size_t slab = ((size_t)1 << 27) / c->W + 1;  // ~1 GiB of staging at most
    u64* stage = nullptr;
    if (mem == GL_MEM_HOST) TRY(dmalloc(ctx, &stage, (row_count < slab ? row_count : slab) * c->W));
    int rc = GL_OK;
    for (size_t r0 = 0; r0 < row_count && rc == GL_OK; r0 += slab) {
        const size_t rows = row_count - r0 < slab ? row_count - r0 : slab;
        u64* dst = mem == GL_MEM_HOST ? stage : out + r0 * c->W;
        k_rows_from_columns<<<dim3((unsigned)((rows + 31) / 32), (c->W + 31) / 32), dim3(32, 8), 0, ctx->stream>>>(
            c->tree.leaves, c->tree.es, row_begin + r0, rows, c->W, dst);
        ctx->launches++;
        if (cudaGetLastError() != cudaSuccess) rc = set_err(ctx, GL_ERR_CUDA, "k_rows_from_columns launch failed");
        if (rc == GL_OK && mem == GL_MEM_HOST) rc = d2h(ctx, out + r0 * c->W, stage, rows * c->W);
    }
    dfree(ctx, stage);
    return rc;
}
int gl_commit_digests(gl_commit* c, uint64_t* out, int mem) {
    NEED_FINISHED(c);
    return copy_out(c->ctx, out, c->tree.digests, c->tree.digest_words(), mem);
}
int gl_commit_get_lde_values(gl_commit* c, size_t index, size_t step, uint64_t* out) {
    const uint32_t bits = c->degree_log + c->rate_bits;
    size_t idx = index * step;
    if (idx >= ((size_t)1 << bits)) return set_err(c->ctx, GL_ERR_BAD_ARG, "index out of range");
    size_t rev = 0;
    for (uint32_t i = 0; i < bits; i++) rev |= ((idx >> i) & 1) << (bits - 1 - i);
    const size_t row0 = (size_t)c->shard_index * c->tree.N;
    if (rev < row0 || rev >= row0 + c->tree.N) return set_err(c->ctx, GL_ERR_BAD_ARG, "LDE row held by another shard");
    CK(c->ctx, cudaMemcpy2DAsync(out, 8, c->tree.leaves + (rev - row0), c->tree.es * 8, 8, c->B, cudaMemcpyDeviceToHost,
                                 c->ctx->stream));
    CK(c->ctx, cudaStreamSynchronize(c->ctx->stream));
    return GL_OK;
}
int gl_commit_shard(const gl_commit* c, uint32_t* shard_index, uint32_t* num_shards) {
    if (shard_index) *shard_index = c->shard_index;
    if (num_shards) *num_shards = 1u << c->shard_log;
    return GL_OK;
}
int gl_commit_open(gl_commit* c, const uint64_t* leaf_indices, size_t count, uint64_t* out_leaves, uint64_t* out_paths) {
    NEED_FINISHED(c);
    return tree_open(c->ctx, c->tree, leaf_indices, count, out_leaves, out_paths);
}
int gl_commit_eval_ext(gl_commit* c, const uint64_t point[2], uint64_t* out) {
    gl_ctx* ctx = c->ctx;
    if (!point || !out) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)1 << c->degree_log;
    const E2 z = {canon(point[0]), canon(point[1])};
    const size_t hi_cnt = (n >> 12) + 1;
    u64 *zhi = nullptr, *zlo = nullptr, *zt = nullptr, *dout = nullptr;
    auto body = [&]() -> int {
        TRY(dmalloc(ctx, &zhi, 2 * hi_cnt));
        TRY(dmalloc(ctx, &zlo, 2 * 4096));
        TRY(dmalloc(ctx, &zt, 2 * n));
        TRY(dmalloc(ctx, &dout, 2 * (size_t)c->B));
        k_fill_e2_pows<<<(unsigned)((hi_cnt + 127) / 128), 128, 0, ctx->stream>>>(e2_pow(z, 4096), hi_cnt, zhi);
        CKL(ctx);
        k_fill_e2_pows<<<32, 128, 0, ctx->stream>>>(z, 4096, zlo);
        CKL(ctx);
        k_e2_pow_table<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(zhi, zlo, n, zt);
        CKL(ctx);
        k_eval_ext<<<c->B, 256, 0, ctx->stream>>>(c->coeffs, n, n, zt, dout);
        CKL(ctx);
        return d2h(ctx, out, dout, 2 * (size_t)c->B);
    };
    int rc = body();
    dfree(ctx, zhi);
    dfree(ctx, zlo);
    dfree(ctx, zt);
    dfree(ctx, dout);
    return rc;
}
// OpeningSet::new / StarkOpeningSet::new (plonk/proof.rs:313-351, starky/src/proof.rs:221-260) in ONE call: every
// polynomial of commits[i] evaluated at points[point_index[i]], results concatenated in request order, one D2H.
int gl_openings(gl_ctx* ctx, gl_commit* const* commits, const uint32_t* point_index, size_t n_evals, const uint64_t* points,
                size_t n_points, uint64_t* out, int mem) {
    if (!ctx || !commits || !point_index || !points || !out) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    if (n_evals == 0) return GL_OK;
    CK(ctx, cudaSetDevice(ctx->device));
    uint32_t max_log = 0;
    size_t total = 0;
    for (size_t i = 0; i < n_evals; i++) {
        if (!commits[i] || commits[i]->ctx->device != ctx->device) return set_err(ctx, GL_ERR_BAD_ARG, "bad commitment %zu", i);
        if (point_index[i] >= n_points) return set_err(ctx, GL_ERR_BAD_ARG, "point index %u out of range", point_index[i]);
        if (commits[i]->degree_log > max_log) max_log = commits[i]->degree_log;
        total += commits[i]->B;
    }
    const size_t n = (size_t)1 << max_log, hi_cnt = (n >> 12) + 1;
    u64 *zhi = nullptr, *zlo = nullptr, *zt = nullptr, *dout = nullptr;
    auto body = [&]() -> int {
        TRY(dmalloc(ctx, &zhi, 2 * hi_cnt));
        TRY(dmalloc(ctx, &zlo, 2 * 4096));
        TRY(dmalloc(ctx, &zt, 2 * n));
        if (mem == GL_MEM_HOST) TRY(dmalloc(ctx, &dout, 2 * total));
        else dout = out;
        for (size_t p = 0; p < n_points; p++) {  // one power table per distinct point, shared by every request at it
            bool used = false;
            for (size_t i = 0; i < n_evals; i++) used |= point_index[i] == p;
            if (!used) continue;
            const E2 z = {canon(points[2 * p]), canon(points[2 * p + 1])};
            k_fill_e2_pows<<<(unsigned)((hi_cnt + 127) / 128), 128, 0, ctx->stream>>>(e2_pow(z, 4096), hi_cnt, zhi);
            CKL(ctx);
            k_fill_e2_pows<<<32, 128, 0, ctx->stream>>>(z, 4096, zlo);
            CKL(ctx);
            k_e2_pow_table<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(zhi, zlo, n, zt);
            CKL(ctx);
            size_t off = 0;
            for (size_t i = 0; i < n_evals; i++) {
                const gl_commit* c = commits[i];
                if (point_index[i] == p) {
                    const size_t nc = (size_t)1 << c->degree_log;
                    k_eval_ext<<<c->B, 256, 0, ctx->stream>>>(c->coeffs, nc, nc, zt, dout + 2 * off);
                    CKL(ctx);
                }
                off += c->B;
            }
        }
        if (mem == GL_MEM_HOST) return d2h(ctx, out, dout, 2 * total);
        return GL_OK;
    };
    int rc = body();
    dfree(ctx, zhi);
    dfree(ctx, zlo);
    dfree(ctx, zt);
    if (mem == GL_MEM_HOST) dfree(ctx, dout);
    return rc;
}
const uint64_t* gl_commit_dev_lde(const gl_commit* c, size_t* col_stride) {
    if (col_stride) *col_stride = c->tree.es;
    return c->tree.leaves;
}
const uint64_t* gl_commit_dev_coeffs(const gl_commit* c) { return c->coeffs; }

int gl_partial_products_and_zs(gl_ctx* ctx, const uint64_t* wires, const uint64_t* sigmas, const uint64_t* k_is,
                               uint32_t log_n, uint32_t num_routed, uint64_t beta, uint64_t gamma, uint32_t degree,
                               uint64_t* out, int mem) {
    if (!ctx || !wires || !sigmas || !k_is || !out) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    if (degree < 2 || num_routed == 0 || log_n > 26) return set_err(ctx, GL_ERR_BAD_SHAPE, "bad partial-product shape");
    if ((num_routed + degree - 1) / degree > (uint32_t)PP_MAX_CHUNKS)
        return set_err(ctx, GL_ERR_UNSUPPORTED, "more than %d partial-product chunks per row", PP_MAX_CHUNKS);
    CK(ctx, cudaSetDevice(ctx->device));
    const size_t n = (size_t)1 << log_n;
    const uint32_t M = (num_routed + degree - 1) / degree;
    const size_t L = n * M, nchunks = (L + SCAN_CHUNK - 1) / SCAN_CHUNK;
    u64 *dw = nullptr, *ds = nullptr, *dk = nullptr, *seq = nullptr, *tot = nullptr, *dout = nullptr, *dflag = nullptr;
    u64* xtab = nullptr;
    auto body = [&]() -> int {
        const u64 *pw = wires, *ps = sigmas;
        if (mem == GL_MEM_HOST) {
            TRY(dmalloc(ctx, &dw, (size_t)num_routed * n));
            TRY(dmalloc(ctx, &ds, (size_t)num_routed * n));
            TRY(h2d(ctx, dw, wires, (size_t)num_routed * n));
            TRY(h2d(ctx, ds, sigmas, (size_t)num_routed * n));
            pw = dw;
            ps = ds;
            TRY(dmalloc(ctx, &dout, (size_t)M * n));
        } else {
            dout = out;
        }
        TRY(dmalloc(ctx, &dk, num_routed));
        TRY(h2d(ctx, dk, k_is, num_routed));  // k_is is a small host array in both modes
        TRY(dmalloc(ctx, &seq, L));
        TRY(dmalloc(ctx, &tot, nchunks));
        TRY(dmalloc(ctx, &dflag, 1));
        CK(ctx, cudaMemsetAsync(dflag, 0, 8, ctx->stream));
        const u64 wn = root_of_unity(log_n);
        const size_t tcnt = 4096 > (n >> 12) + 1 ? 4096 : (n >> 12) + 1;
        TRY(build_pow_tables(ctx, std::vector<u64>{gl::pow(wn, 4096), wn}, tcnt, &xtab));
        PPParams pp{pw, ps, dk, n, log_n, num_routed, degree, M, canon(beta), canon(gamma), xtab, xtab + tcnt, seq,
                    (unsigned int*)dflag};
        k_pp_chunks<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(pp);
        CKL(ctx);
        k_scan3_phase1<MulOp><<<(unsigned)nchunks, SCAN_THREADS, 0, ctx->stream>>>(seq, L, tot);
        CKL(ctx);
        k_scan3_phase2<MulOp><<<1, 1024, 0, ctx->stream>>>(tot, nchunks);
        CKL(ctx);
        k_scan3_phase3<MulOp><<<(unsigned)nchunks, SCAN_THREADS, 0, ctx->stream>>>(seq, L, tot, n, M, dout);
        CKL(ctx);
        u64 flag = 0;
        TRY(d2h(ctx, &flag, dflag, 1));
        if (flag & 0xFFFFFFFFu) return set_err(ctx, GL_ERR_DIV_ZERO, "Tried to invert zero");
        if (mem == GL_MEM_HOST) TRY(d2h(ctx, out, dout, (size_t)M * n));
        return GL_OK;
    };
    int rc = body();
    dfree(ctx, dw);
    dfree(ctx, ds);
    dfree(ctx, dk);
    dfree(ctx, seq);
    dfree(ctx, tot);
    dfree(ctx, dflag);
    dfree(ctx, xtab);
    if (mem == GL_MEM_HOST) dfree(ctx, dout);
    return rc;
}

int gl_lookup_polys(gl_ctx* ctx, const uint64_t* wires, uint32_t log_n, uint32_t num_routed_wires,
                    uint32_t max_quotient_degree_factor, const uint64_t deltas[4], const uint32_t* lookup_rows,
                    uint32_t n_lookup_wires, uint64_t* out, int mem) {
    if (!ctx || !wires || !deltas || !out || (n_lookup_wires && !lookup_rows)) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    if (max_quotient_degree_factor < 2 || log_n > 26) return set_err(ctx, GL_ERR_BAD_SHAPE, "bad lookup shape");
    const uint32_t num_lu_slots = num_routed_wires / 2, num_lut_slots = num_routed_wires / 3;  // lookup.rs:58-61, lookup_table.rs:64-67
    if (num_lu_slots == 0 || num_lut_slots == 0 || num_lu_slots > (uint32_t)LOOKUP_MAX_SLOTS)
        return set_err(ctx, GL_ERR_UNSUPPORTED, "1..%d lookup slots per row", LOOKUP_MAX_SLOTS);
    const uint32_t max_lookup_degree = max_quotient_degree_factor - 1;
    const uint32_t P = (num_lu_slots + max_lookup_degree - 1) / max_lookup_degree;
    const uint32_t max_lookup_table_degree = (num_lut_slots + P - 1) / P;
    const size_t n = (size_t)1 << log_n;
    const uint32_t num_wires_read = 3 * num_lut_slots > 2 * num_lu_slots ? 3 * num_lut_slots : 2 * num_lu_slots;
    for (uint32_t k = 0; k < n_lookup_wires; k++) {
        const uint32_t last_lu = lookup_rows[3 * k], last_lut = lookup_rows[3 * k + 1], first_lut = lookup_rows[3 * k + 2];
        if (!(last_lu <= last_lut && last_lut <= first_lut && (size_t)first_lut + 1 < n))
            return set_err(ctx, GL_ERR_BAD_ARG, "lookup rows %u: need last_lu <= last_lut <= first_lut < n - 1", k);
    }
    CK(ctx, cudaSetDevice(ctx->device));
    u64 *dw = nullptr, *dout = nullptr, *term = nullptr, *reh = nullptr, *dflag = nullptr;
    auto body = [&]() -> int {
        const u64* pw = wires;
        if (mem == GL_MEM_HOST) {
            TRY(dmalloc(ctx, &dw, (size_t)num_wires_read * n));
            TRY(h2d(ctx, dw, wires, (size_t)num_wires_read * n));
            pw = dw;
            TRY(dmalloc(ctx, &dout, (size_t)(P + 1) * n));
        } else {
            dout = out;
        }
        CK(ctx, cudaMemsetAsync(dout, 0, (size_t)(P + 1) * n * 8, ctx->stream));  // vec![F::ZERO; degree]
        TRY(dmalloc(ctx, &dflag, 1));
        CK(ctx, cudaMemsetAsync(dflag, 0, 8, ctx->stream));
        u64 dL = 1;  // delta^num_lut_slots
        for (uint32_t s = 0; s < num_lut_slots; s++) dL = mul(dL, canon(deltas[3]));
        for (uint32_t k = 0; k < n_lookup_wires; k++) {
            LookupParams p;
            p.wires = pw;
            p.n = n;
            p.num_lu_slots = num_lu_slots;
            p.num_lut_slots = num_lut_slots;
            p.P = P;
            p.max_lookup_degree = max_lookup_degree;
            p.max_lookup_table_degree = max_lookup_table_degree;
            p.dA = canon(deltas[0]);
            p.dB = canon(deltas[1]);
            p.dAlpha = canon(deltas[2]);
            p.dDelta = canon(deltas[3]);
            p.last_lu = lookup_rows[3 * k];
            p.last_lut = lookup_rows[3 * k + 1];
            p.first_lut = lookup_rows[3 * k + 2];
            const uint32_t rows_lut = p.first_lut - p.last_lut + 1, T = rows_lut + (p.last_lut - p.last_lu);
            dfree(ctx, term);
            dfree(ctx, reh);
            term = reh = nullptr;
            TRY(dmalloc(ctx, &term, (size_t)T * P));
            TRY(dmalloc(ctx, &reh, rows_lut));
            p.term = term;
            p.reh = reh;
            p.flag = (unsigned int*)dflag;
            k_lookup_terms<<<(T + 127) / 128, 128, 0, ctx->stream>>>(p);
            CKL(ctx);
            // initial values: the arrays' entries at first_lut_row + 1 (zero unless an earlier LookupWire wrote them)
            u64 init[2];
            CK(ctx, cudaMemcpyAsync(&init[0], dout + p.first_lut + 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
            CK(ctx, cudaMemcpyAsync(&init[1], dout + (size_t)P * n + p.first_lut + 1, 8, cudaMemcpyDeviceToHost, ctx->stream));
            CK(ctx, cudaStreamSynchronize(ctx->stream));
            k_affine_scan<<<1, 1024, 0, ctx->stream>>>(reh, rows_lut, dL, init[0], p, 1, dout);
            CKL(ctx);
            k_affine_scan<<<1, 1024, 0, ctx->stream>>>(term, (size_t)T * P, 1, init[1], p, 0, dout);
            CKL(ctx);
        }
        u64 flag = 0;
        TRY(d2h(ctx, &flag, dflag, 1));
        if (flag & 1u) return set_err(ctx, GL_ERR_DIV_ZERO, "Tried to invert zero");
        if (mem == GL_MEM_HOST) TRY(d2h(ctx, out, dout, (size_t)(P + 1) * n));
        return GL_OK;
    };
    int rc = body();
    dfree(ctx, dw);
    dfree(ctx, term);
    dfree(ctx, reh);
    dfree(ctx, dflag);
    if (mem == GL_MEM_HOST) dfree(ctx, dout);
    return rc;
}

int gl_stark_quotient(gl_ctx* ctx, gl_commit* trace, const gl_stark_instr* program, uint32_t n_instr,
                      const uint64_t* consts, uint32_t n_consts, const uint64_t* alphas, uint32_t n_alphas,
                      uint32_t quotient_degree_factor, uint64_t* out_coeffs) {
    return gl_stark_quotient_aux(ctx, trace, nullptr, program, n_instr, consts, n_consts, alphas, n_alphas,
                                 quotient_degree_factor, out_coeffs);
}

int gl_stark_quotient_aux(gl_ctx* ctx, gl_commit* trace, gl_commit* aux, const gl_stark_instr* program, uint32_t n_instr,
                          const uint64_t* consts, uint32_t n_consts, const uint64_t* alphas, uint32_t n_alphas,
                          uint32_t quotient_degree_factor, uint64_t* out_coeffs) {
    if (!ctx || !trace || !program || !alphas || !out_coeffs) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    if (n_instr == 0 || n_instr > GL_STARK_MAX_INSTR) return set_err(ctx, GL_ERR_UNSUPPORTED, "program of %u instructions (max %d)", n_instr, GL_STARK_MAX_INSTR);
    if (n_alphas == 0 || n_alphas > GL_STARK_MAX_ALPHAS) return set_err(ctx, GL_ERR_UNSUPPORTED, "1..%d challenges", GL_STARK_MAX_ALPHAS);
    if (quotient_degree_factor == 0) return set_err(ctx, GL_ERR_BAD_ARG, "quotient_degree_factor is 0: the STARK has no quotient");
    if (trace->shard_log) return set_err(ctx, GL_ERR_UNSUPPORTED, "quotient evaluation needs the whole LDE on this device");
    NEED_FINISHED(trace);
    if (aux) {
        NEED_FINISHED(aux);
        if (aux->shard_log) return set_err(ctx, GL_ERR_UNSUPPORTED, "quotient evaluation needs the whole LDE on this device");
        if (aux->degree_log != trace->degree_log || aux->rate_bits != trace->rate_bits)
            return set_err(ctx, GL_ERR_BAD_SHAPE, "auxiliary polynomials of degree 2^%u rate_bits %u, trace 2^%u rate_bits %u",
                           aux->degree_log, aux->rate_bits, trace->degree_log, trace->rate_bits);
    }
    uint32_t qd_bits = 0;
    while ((1u << qd_bits) < quotient_degree_factor) qd_bits++;  // log2_ceil
    if (qd_bits > trace->rate_bits)
        return set_err(ctx, GL_ERR_UNSUPPORTED, "Having constraints of degree higher than the rate is not supported yet.");
    if ((1u << qd_bits) > GL_STARK_MAX_QD) return set_err(ctx, GL_ERR_UNSUPPORTED, "quotient degree factor too large");
    for (uint32_t k = 0; k < n_instr; k++) {  // validate once on the host: the kernel trusts the program
        const gl_stark_instr in = program[k];
        bool ok = true;
        switch (in.op) {
            case GL_STARK_LOCAL: case GL_STARK_NEXT: ok = in.a < trace->B; break;
            case GL_STARK_AUX_LOCAL: case GL_STARK_AUX_NEXT: ok = aux && in.a < aux->B; break;
            case GL_STARK_CONST: ok = in.a < n_consts; break;
            case GL_STARK_ADD: case GL_STARK_SUB: case GL_STARK_MUL: ok = in.a < k && in.b < k; break;
            case GL_STARK_EMIT: ok = in.a < k && in.b <= GL_STARK_LAST_ROW; break;
            default: ok = false;
        }
        if (!ok) return set_err(ctx, GL_ERR_BAD_ARG, "constraint program: bad instruction %u", k);
    }
    CK(ctx, cudaSetDevice(ctx->device));
    const uint32_t db = trace->degree_log, size_log = db + qd_bits;
    const size_t size = (size_t)1 << size_log;
    u64 *dprog = nullptr, *dconst = nullptr, *xtab = nullptr, *dflag = nullptr;
    auto body = [&]() -> int {
        const size_t prog_words = ((size_t)n_instr * sizeof(gl_stark_instr) + 7) / 8;
        TRY(dmalloc(ctx, &dprog, prog_words));
        CK(ctx, cudaMemcpyAsync(dprog, program, (size_t)n_instr * sizeof(gl_stark_instr), cudaMemcpyHostToDevice, ctx->stream));
        TRY(dmalloc(ctx, &dconst, n_consts ? n_consts : 1));
        if (n_consts) TRY(h2d(ctx, dconst, consts, n_consts));
        TRY(dmalloc(ctx, &dflag, 1));
        CK(ctx, cudaMemsetAsync(dflag, 0, 8, ctx->stream));
        const u64 ws = root_of_unity(size_log);
        const size_t tcnt = 4096 > (size >> 12) + 1 ? 4096 : (size >> 12) + 1;
        TRY(build_pow_tables(ctx, std::vector<u64>{gl::pow(ws, 4096), ws}, tcnt, &xtab));
        StarkQuotientParams p;
        p.lde = trace->tree.leaves;
        p.lde_stride = trace->tree.es;
        p.aux = aux ? aux->tree.leaves : nullptr;
        p.aux_stride = aux ? aux->tree.es : 0;
        p.log_N = db + trace->rate_bits;
        p.degree_bits = db;
        p.qd_bits = qd_bits;
        p.prog = (const gl_stark_instr*)dprog;
        p.n_instr = n_instr;
        p.consts = dconst;
        p.n_alphas = n_alphas;
        for (uint32_t a = 0; a < GL_STARK_MAX_ALPHAS; a++) p.alphas[a] = a < n_alphas ? canon(alphas[a]) : 0;
        p.xhi = xtab;
        p.xlo = xtab + tcnt;
        p.shift = MULTIPLICATIVE_GROUP_GENERATOR;
        p.last = gl::inv(root_of_unity(db));
        p.n_field = canon((u64)1 << db);
        // ZeroPolyOnCoset::new(degree_bits, qd_bits) (field/src/zero_poly_coset.rs:20-34)
        u64 g_pow_n = MULTIPLICATIVE_GROUP_GENERATOR;
        for (uint32_t k = 0; k < db; k++) g_pow_n = sqr(g_pow_n);
        const u64 wq = root_of_unity(qd_bits);
        u64 xq = 1;
        for (uint32_t j = 0; j < (1u << qd_bits); j++, xq = mul(xq, wq)) {
            p.zh[j] = canon(sub(mul(g_pow_n, xq), 1));
            p.zh_inv[j] = canon(gl::inv(p.zh[j]));
        }
        p.out = out_coeffs;
        p.flag = (unsigned int*)dflag;
        k_stark_quotient<<<(unsigned)((size + 127) / 128), 128, 0, ctx->stream>>>(p);
        CKL(ctx);
        // .coset_ifft(F::coset_shift()) of every challenge's values (prover.rs:661-667)
        TRY(ntt_natural(ctx, out_coeffs, size, out_coeffs, size, (int)size_log, n_alphas, true, MULTIPLICATIVE_GROUP_GENERATOR));
        // trim_to_len(degree * quotient_degree_factor) (prover.rs:396-401): the rest must vanish
        const size_t keep = ((size_t)quotient_degree_factor) << db;
        if (keep < size) {
            k_any_nonzero<<<dim3((unsigned)((size - keep + 255) / 256), n_alphas), 256, 0, ctx->stream>>>(out_coeffs, size, keep,
                                                                                                   size - keep, (unsigned int*)dflag);
            CKL(ctx);
        }
        u64 flag = 0;
        TRY(d2h(ctx, &flag, dflag, 1));
        if (flag & 1u) return set_err(ctx, GL_ERR_DIV_ZERO, "Tried to invert zero");
        if (flag & 2u) return set_err(ctx, GL_ERR_BAD_ARG, "Quotient has failed, the vanishing polynomial is not divisible by Z_H");
        return GL_OK;
    };
    int rc = body();
    dfree(ctx, dprog);
    dfree(ctx, dconst);
    dfree(ctx, xtab);
    dfree(ctx, dflag);
    return rc;
}

int gl_stark_lookup_helper_columns(gl_ctx* ctx, const uint64_t* trace, size_t col_stride, uint32_t n_cols, uint32_t log_n,
                                   const gl_logup_desc* desc, const uint64_t* challenges, uint32_t n_challenges,
                                   uint32_t constraint_degree, uint64_t* out, int mem) {
    if (!ctx || !trace || !desc || !out || (n_challenges && !challenges)) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    if (mem != GL_MEM_HOST && mem != GL_MEM_DEVICE) return set_err(ctx, GL_ERR_BAD_ARG, "bad mem %d", mem);
    if (log_n > 30) return set_err(ctx, GL_ERR_UNSUPPORTED, "log_n %u > 30", log_n);
    const size_t n = (size_t)1 << log_n;
    if (col_stride < n) return set_err(ctx, GL_ERR_BAD_SHAPE, "col_stride %zu < n = %zu", col_stride, n);
    const gl_logup_desc& d = *desc;
    if ((d.n_terms && !d.terms) || (d.n_columns && (!d.columns || !d.filters)) || (d.n_filter_columns && !d.filter_columns) ||
        (d.n_lookups && !d.lookups))
        return set_err(ctx, GL_ERR_BAD_ARG, "null descriptor array");
    // validate once on the host: the kernel trusts the descriptors
    for (uint32_t t = 0; t < d.n_terms; t++)
        if (d.terms[t].col >= n_cols || d.terms[t].next > 1) return set_err(ctx, GL_ERR_BAD_ARG, "lookup term %u: bad column", t);
    for (uint32_t c = 0; c < d.n_columns; c++) {
        const gl_logup_filter f = d.filters[c];
        if ((uint64_t)d.columns[c].term_begin + d.columns[c].n_terms > d.n_terms ||
            (uint64_t)f.prod_begin + 2 * (uint64_t)f.n_prods > d.n_filter_columns ||
            (uint64_t)f.sum_begin + f.n_sums > d.n_filter_columns)
            return set_err(ctx, GL_ERR_BAD_ARG, "lookup column %u: range outside the descriptor arrays", c);
    }
    for (uint32_t k = 0; k < d.n_filter_columns; k++)
        if (d.filter_columns[k] >= d.n_columns) return set_err(ctx, GL_ERR_BAD_ARG, "filter column %u: bad index", k);
    const uint32_t chunk = constraint_degree > 2 ? constraint_degree - 1 : 1;  // constraint_degree.checked_sub(1), at least 1
    uint64_t n_den = 0, n_out = 0;
    std::vector<uint32_t> zcols;  // output column of every (lookup, challenge) Z
    for (uint32_t l = 0; l < d.n_lookups; l++) {
        const gl_logup_lookup lk = d.lookups[l];
        if ((uint64_t)lk.looking_begin + lk.n_looking > d.n_columns || lk.table >= d.n_columns || lk.frequencies >= d.n_columns)
            return set_err(ctx, GL_ERR_BAD_ARG, "lookup %u: bad column index", l);
        n_den += (uint64_t)(lk.n_looking + 1) * n_challenges;
        const uint32_t nh = (lk.n_looking + chunk - 1) / chunk + 1;  // Lookup::num_helper_columns
        for (uint32_t c = 0; c < n_challenges; c++) {
            n_out += nh;
            zcols.push_back((uint32_t)n_out - 1);
        }
    }
    if (n_den > GL_LOGUP_MAX_DENOMINATORS)
        return set_err(ctx, GL_ERR_UNSUPPORTED, "%llu denominators per row (max %d)", (unsigned long long)n_den,
                       GL_LOGUP_MAX_DENOMINATORS);
    if (zcols.empty()) return GL_OK;
    CK(ctx, cudaSetDevice(ctx->device));
    u64 *ddesc = nullptr, *dchal = nullptr, *dtrace = nullptr, *dout = nullptr, *zterm = nullptr, *tot = nullptr, *dflag = nullptr;
    auto body = [&]() -> int {
        // the descriptor arrays, packed into one device buffer
        const size_t sz[5] = {d.n_terms * sizeof(gl_logup_term), d.n_columns * sizeof(gl_logup_column),
                              d.n_columns * sizeof(gl_logup_filter), d.n_lookups * sizeof(gl_logup_lookup),
                              d.n_filter_columns * sizeof(uint32_t)};
        const void* src[5] = {d.terms, d.columns, d.filters, d.lookups, d.filter_columns};
        size_t off[5], words = 0;
        for (int k = 0; k < 5; k++) {
            off[k] = words;
            words += (sz[k] + 15) / 16 * 2;
        }
        TRY(dmalloc(ctx, &ddesc, words ? words : 1));
        for (int k = 0; k < 5; k++)
            if (sz[k]) CK(ctx, cudaMemcpyAsync(ddesc + off[k], src[k], sz[k], cudaMemcpyHostToDevice, ctx->stream));
        TRY(dmalloc(ctx, &dchal, n_challenges));
        std::vector<u64> ch(n_challenges);
        for (uint32_t c = 0; c < n_challenges; c++) ch[c] = canon(challenges[c]);
        TRY(h2d(ctx, dchal, ch.data(), n_challenges));
        LogupParams p;
        p.d = d;
        p.d.terms = (const gl_logup_term*)(ddesc + off[0]);
        p.d.columns = (const gl_logup_column*)(ddesc + off[1]);
        p.d.filters = (const gl_logup_filter*)(ddesc + off[2]);
        p.d.lookups = (const gl_logup_lookup*)(ddesc + off[3]);
        p.d.filter_columns = (const uint32_t*)(ddesc + off[4]);
        if (mem == GL_MEM_HOST) {
            TRY(dmalloc(ctx, &dtrace, (size_t)n_cols * n ? (size_t)n_cols * n : 1));
            if (n_cols)
                CK(ctx, cudaMemcpy2DAsync(dtrace, n * 8, trace, col_stride * 8, n * 8, n_cols, cudaMemcpyHostToDevice, ctx->stream));
            p.trace = dtrace;
            p.col_stride = n;
            TRY(dmalloc(ctx, &dout, n_out * n));
        } else {
            p.trace = trace;
            p.col_stride = col_stride;
            dout = out;
        }
        p.n = n;
        p.challenges = dchal;
        p.n_challenges = n_challenges;
        p.chunk = chunk;
        p.out = dout;
        TRY(dmalloc(ctx, &zterm, zcols.size() * n));
        p.zterm = zterm;
        TRY(dmalloc(ctx, &dflag, 1));
        CK(ctx, cudaMemsetAsync(dflag, 0, 8, ctx->stream));
        k_logup_rows<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(p, (unsigned int*)dflag);
        CKL(ctx);
        // Z(0) = 0, Z(i+1) = Z(i) + d(i): exclusive scan of every Z's terms into its column
        const size_t nchunks = (n + SCAN_CHUNK - 1) / SCAN_CHUNK;
        TRY(dmalloc(ctx, &tot, nchunks));
        for (size_t z = 0; z < zcols.size(); z++) {
            const u64* seq = zterm + z * n;
            k_scan3_phase1<AddOp><<<(unsigned)nchunks, SCAN_THREADS, 0, ctx->stream>>>(seq, n, tot);
            CKL(ctx);
            k_scan3_phase2<AddOp><<<1, 1024, 0, ctx->stream>>>(tot, nchunks);
            CKL(ctx);
            k_scan3_phase3<AddOp><<<(unsigned)nchunks, SCAN_THREADS, 0, ctx->stream>>>(seq, n, tot, n, 1, dout + (size_t)zcols[z] * n);
            CKL(ctx);
        }
        u64 flag = 0;
        TRY(d2h(ctx, &flag, dflag, 1));
        if (flag & 1u) return set_err(ctx, GL_ERR_DIV_ZERO, "Tried to invert zero");
        if (mem == GL_MEM_HOST) TRY(d2h(ctx, out, dout, n_out * n));
        return GL_OK;
    };
    int rc = body();
    dfree(ctx, ddesc);
    dfree(ctx, dchal);
    dfree(ctx, dtrace);
    dfree(ctx, zterm);
    dfree(ctx, tot);
    dfree(ctx, dflag);
    if (mem == GL_MEM_HOST) dfree(ctx, dout);
    return rc;
}

int gl_plonk_quotient(gl_ctx* ctx, gl_commit* const* commits, uint32_t n_commits, const gl_vp_instr* program,
                      uint32_t n_instr, const uint64_t* consts, uint32_t n_consts, const uint64_t* alphas,
                      uint32_t n_alphas, uint32_t n_terms, uint32_t quotient_degree_factor, uint64_t* out_coeffs) {
    if (!ctx || !commits || !program || !alphas || !out_coeffs) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    if (n_commits == 0 || n_commits > GL_VP_MAX_COMMITS) return set_err(ctx, GL_ERR_UNSUPPORTED, "1..%d commitments", GL_VP_MAX_COMMITS);
    if (n_instr == 0) return set_err(ctx, GL_ERR_BAD_ARG, "empty program");
    if (n_alphas == 0 || n_alphas > GL_VP_MAX_ALPHAS) return set_err(ctx, GL_ERR_UNSUPPORTED, "1..%d challenges", GL_VP_MAX_ALPHAS);
    if (n_terms == 0 || n_terms > 65536) return set_err(ctx, GL_ERR_BAD_ARG, "1..65536 vanishing terms");
    if (quotient_degree_factor == 0) return set_err(ctx, GL_ERR_BAD_ARG, "quotient_degree_factor is 0");
    for (uint32_t c = 0; c < n_commits; c++) {
        if (!commits[c]) return set_err(ctx, GL_ERR_BAD_ARG, "null commitment");
        if (commits[c]->ctx != ctx) return set_err(ctx, GL_ERR_BAD_ARG, "commitment %u belongs to another context", c);
        if (commits[c]->shard_log) return set_err(ctx, GL_ERR_UNSUPPORTED, "quotient evaluation needs the whole LDE on this device");
        NEED_FINISHED(commits[c]);
        if (commits[c]->degree_log != commits[0]->degree_log || commits[c]->rate_bits != commits[0]->rate_bits)
            return set_err(ctx, GL_ERR_BAD_SHAPE, "commitments of different degree or rate");
    }
    const uint32_t db = commits[0]->degree_log, rate_bits = commits[0]->rate_bits;
    uint32_t qd_bits = 0;
    while ((1u << qd_bits) < quotient_degree_factor) qd_bits++;  // log2_ceil
    if (qd_bits > rate_bits)
        return set_err(ctx, GL_ERR_UNSUPPORTED, "Having constraints of degree higher than the rate is not supported yet.");
    if ((1u << qd_bits) > GL_VP_MAX_QD) return set_err(ctx, GL_ERR_UNSUPPORTED, "quotient degree factor too large");
    {  // validate once on the host: the kernel trusts the program (operands in range, no register read before it is written)
        bool written[GL_VP_MAX_REGS] = {false};
        auto readable = [&](uint16_t r) { return r < GL_VP_MAX_REGS && written[r]; };
        for (uint32_t k = 0; k < n_instr; k++) {
            const gl_vp_instr in = program[k];
            bool ok = in.dst < GL_VP_MAX_REGS;
            switch (in.op) {
                case GL_VP_LOCAL: case GL_VP_NEXT: ok = ok && in.a < n_commits && in.b < commits[in.a]->W; break;
                case GL_VP_CONST: ok = ok && ((uint32_t)in.a | ((uint32_t)in.b << 16)) < n_consts; break;
                case GL_VP_X: case GL_VP_L0: break;
                case GL_VP_ADD: case GL_VP_SUB: case GL_VP_MUL: ok = ok && readable(in.a) && readable(in.b); break;
                case GL_VP_ADDC: case GL_VP_MULC: ok = ok && readable(in.a) && in.b < n_consts; break;
                case GL_VP_TERM: ok = readable(in.a) && in.b < n_terms; break;
                default: ok = false;
            }
            if (!ok) return set_err(ctx, GL_ERR_BAD_ARG, "vanishing program: bad instruction %u", k);
            if (in.op != GL_VP_TERM) written[in.dst] = true;
        }
    }
    CK(ctx, cudaSetDevice(ctx->device));
    const uint32_t size_log = db + qd_bits;
    const size_t size = (size_t)1 << size_log;
    u64 *dprog = nullptr, *dconst = nullptr, *dapow = nullptr, *xtab = nullptr, *dflag = nullptr;
    auto body = [&]() -> int {
        const size_t prog_words = ((size_t)n_instr * sizeof(gl_vp_instr) + 7) / 8;
        TRY(dmalloc(ctx, &dprog, prog_words));
        TRY(h2d(ctx, dprog, (const u64*)program, prog_words));
        TRY(dmalloc(ctx, &dconst, n_consts ? n_consts : 1));
        if (n_consts) TRY(h2d(ctx, dconst, consts, n_consts));
        std::vector<u64> apow((size_t)n_alphas * n_terms);
        for (uint32_t a = 0; a < n_alphas; a++) {
            u64 pw = 1;
            for (uint32_t t = 0; t < n_terms; t++, pw = mul(pw, alphas[a])) apow[(size_t)a * n_terms + t] = canon(pw);
        }
        TRY(dmalloc(ctx, &dapow, apow.size()));
        TRY(h2d(ctx, dapow, apow.data(), apow.size()));
        TRY(dmalloc(ctx, &dflag, 1));
        CK(ctx, cudaMemsetAsync(dflag, 0, 8, ctx->stream));
        const u64 ws = root_of_unity(size_log);
        const size_t tcnt = 4096 > (size >> 12) + 1 ? 4096 : (size >> 12) + 1;
        TRY(build_pow_tables(ctx, std::vector<u64>{gl::pow(ws, 4096), ws}, tcnt, &xtab));
        VanishingParams p;
        for (uint32_t c = 0; c < GL_VP_MAX_COMMITS; c++) {
            p.lde[c] = c < n_commits ? commits[c]->tree.leaves : nullptr;
            p.lde_stride[c] = c < n_commits ? commits[c]->tree.es : 0;
        }
        p.log_N = db + rate_bits;
        p.degree_bits = db;
        p.qd_bits = qd_bits;
        p.prog = (const gl_vp_instr*)dprog;
        p.n_instr = n_instr;
        p.consts = dconst;
        p.apow = dapow;
        p.n_alphas = n_alphas;
        p.n_terms = n_terms;
        p.xhi = xtab;
        p.xlo = xtab + tcnt;
        p.shift = MULTIPLICATIVE_GROUP_GENERATOR;
        p.n_field = canon((u64)1 << db);
        // ZeroPolyOnCoset::new(degree_bits, qd_bits) (field/src/zero_poly_coset.rs:20-34)
        u64 g_pow_n = MULTIPLICATIVE_GROUP_GENERATOR;
        for (uint32_t k = 0; k < db; k++) g_pow_n = sqr(g_pow_n);
        const u64 wq = root_of_unity(qd_bits);
        u64 xq = 1;
        for (uint32_t j = 0; j < GL_VP_MAX_QD; j++) p.zh[j] = p.zh_inv[j] = 0;
        for (uint32_t j = 0; j < (1u << qd_bits); j++, xq = mul(xq, wq)) {
            p.zh[j] = canon(sub(mul(g_pow_n, xq), 1));
            p.zh_inv[j] = canon(gl::inv(p.zh[j]));
        }
        p.out = out_coeffs;
        p.flag = (unsigned int*)dflag;
        k_plonk_quotient<<<(unsigned)((size + 127) / 128), 128, 0, ctx->stream>>>(p);
        CKL(ctx);
        // .coset_ifft(F::coset_shift()) of every challenge's values (prover.rs:811-814)
        TRY(ntt_natural(ctx, out_coeffs, size, out_coeffs, size, (int)size_log, n_alphas, true, MULTIPLICATIVE_GROUP_GENERATOR));
        // trim_to_len(quotient_degree) (prover.rs:327-331): the rest must vanish
        const size_t keep = ((size_t)quotient_degree_factor) << db;
        if (keep < size) {
            k_any_nonzero<<<dim3((unsigned)((size - keep + 255) / 256), n_alphas), 256, 0, ctx->stream>>>(out_coeffs, size, keep,
                                                                                                   size - keep, (unsigned int*)dflag);
            CKL(ctx);
        }
        u64 flag = 0;
        TRY(d2h(ctx, &flag, dflag, 1));  // synchronises: the host tables above outlive the copies
        if (flag & 1u) return set_err(ctx, GL_ERR_DIV_ZERO, "Tried to invert zero");
        if (flag & 2u) return set_err(ctx, GL_ERR_BAD_ARG, "Quotient has failed, the vanishing polynomial is not divisible by Z_H");
        return GL_OK;
    };
    int rc = body();
    dfree(ctx, dprog);
    dfree(ctx, dconst);
    dfree(ctx, dapow);
    dfree(ctx, xtab);
    dfree(ctx, dflag);
    return rc;
}

void gl_poseidon_permute_host(uint64_t state[12]) {
    poseidon_permute(state);
    for (int i = 0; i < 12; i++) state[i] = canon(state[i]);
}

static int hash_many_impl(gl_ctx* ctx, const u64* in, size_t n_items, size_t in_words_per_item, u64* out, int mem,
                          int which, uint32_t W) {
    if (n_items == 0) return GL_OK;
    const u64* din = in;
    u64 *tin = nullptr, *dout = out;
    if (mem == GL_MEM_HOST) {
        TRY(dmalloc(ctx, &tin, n_items * in_words_per_item));
        TRY(h2d(ctx, tin, in, n_items * in_words_per_item));
        din = tin;
        TRY(dmalloc(ctx, &dout, n_items * 4));
    }
    if (which == 0)
        k_hash_many<true><<<(unsigned)((n_items + 127) / 128), 128, 0, ctx->stream>>>(din, n_items, W, dout);
    else if (which == 2)
        k_hash_many<false><<<(unsigned)((n_items + 127) / 128), 128, 0, ctx->stream>>>(din, n_items, W, dout);
    else
        k_two_to_one_many<<<(unsigned)((n_items + 127) / 128), 128, 0, ctx->stream>>>(din, n_items, dout);
    CKL(ctx);
    if (mem == GL_MEM_HOST) {
        int rc = d2h(ctx, out, dout, n_items * 4);
        dfree(ctx, tin);
        dfree(ctx, dout);
        return rc;
    }
    return GL_OK;
}
int gl_poseidon_hash_many(gl_ctx* ctx, const uint64_t* in, size_t n_items, uint32_t W, uint64_t* out, int mem) {
    if (!ctx || !out || (!in && W)) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    CK(ctx, cudaSetDevice(ctx->device));
    return hash_many_impl(ctx, in, n_items, W, out, mem, 0, W);
}
int gl_poseidon_hash_no_pad_many(gl_ctx* ctx, const uint64_t* in, size_t n_items, uint32_t W, uint64_t* out, int mem) {
    if (!ctx || !out || (!in && W)) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    CK(ctx, cudaSetDevice(ctx->device));
    return hash_many_impl(ctx, in, n_items, W, out, mem, 2, W);
}
int gl_poseidon_two_to_one_many(gl_ctx* ctx, const uint64_t* in, size_t n_items, uint64_t* out, int mem) {
    if (!ctx || !out || !in) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    CK(ctx, cudaSetDevice(ctx->device));
    return hash_many_impl(ctx, in, n_items, 8, out, mem, 1, 8);
}

int gl_poseidon_permute_many(gl_ctx* ctx, uint64_t* states, size_t n_items, int mem) {
    if (!ctx || !states) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    CK(ctx, cudaSetDevice(ctx->device));
    if (n_items == 0) return GL_OK;
    u64* d = states;
    if (mem == GL_MEM_HOST) {
        TRY(dmalloc(ctx, &d, n_items * 12));
        int rc = h2d(ctx, d, states, n_items * 12);
        if (rc != GL_OK) {
            dfree(ctx, d);
            return rc;
        }
    }
    k_permute_many<<<(unsigned)((n_items + 127) / 128), 128, 0, ctx->stream>>>(d, n_items);
    ctx->launches++;
    int rc = cudaGetLastError() == cudaSuccess ? GL_OK : set_err(ctx, GL_ERR_CUDA, "k_permute_many launch failed");
    if (mem == GL_MEM_HOST) {
        if (rc == GL_OK) rc = d2h(ctx, states, d, n_items * 12);
        dfree(ctx, d);
    }
    return rc;
}

struct gl_merkle {
    gl_ctx* ctx;
    Tree tree;
};
int gl_merkle_build(gl_ctx* ctx, const uint64_t* leaves, size_t N, uint32_t W, uint32_t cap_height, int mem,
                    gl_merkle** out) {
    if (!ctx || !out || !leaves) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    *out = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    uint32_t lg;
    if (log2_exact(N, &lg)) return set_err(ctx, GL_ERR_BAD_SHAPE, "Not a power of two: %zu", N);
    if (cap_height > lg)
        return set_err(ctx, GL_ERR_BAD_SHAPE, "cap_height=%u should be at most log2(leaves.len())=%u", cap_height, lg);
    gl_merkle* m = new gl_merkle();
    m->ctx = ctx;
    m->tree.N = N;
    m->tree.W = W;
    m->tree.cap_height = cap_height;
    int rc = GL_OK;
    if (mem == GL_MEM_HOST) {
        m->tree.own_leaves = true;
        rc = dmalloc(ctx, &m->tree.leaves, N * (size_t)W);
        if (rc == GL_OK) rc = h2d(ctx, m->tree.leaves, leaves, N * (size_t)W);
    } else {
        m->tree.leaves = const_cast<u64*>(leaves);  // caller keeps the buffer alive
    }
    if (rc == GL_OK) rc = tree_build(ctx, m->tree);
    if (rc != GL_OK) {
        gl_merkle_destroy(m);
        return rc;
    }
    *out = m;
    return GL_OK;
}
void gl_merkle_destroy(gl_merkle* m) {
    if (!m) return;
    cudaSetDevice(m->ctx->device);
    tree_free(m->ctx, m->tree);
    delete m;
}
int gl_merkle_cap(gl_merkle* m, uint64_t* out, int mem) { return copy_out(m->ctx, out, m->tree.cap, m->tree.cap_words(), mem); }
int gl_merkle_digests(gl_merkle* m, uint64_t* out, int mem) {
    return copy_out(m->ctx, out, m->tree.digests, m->tree.digest_words(), mem);
}
int gl_merkle_open(gl_merkle* m, const uint64_t* leaf_indices, size_t count, uint64_t* out_leaves, uint64_t* out_paths) {
    return tree_open(m->ctx, m->tree, leaf_indices, count, out_leaves, out_paths);
}

// ------------------------------------------------------------------------------- FRI
int gl_fri_begin(gl_ctx* ctx, gl_commit* const* oracles, size_t n_oracles, const gl_fri_batch* batches,
                 size_t n_batches, const uint64_t alpha_in[2], uint32_t rate_bits, uint32_t cap_height, gl_fri** out) {
    if (!ctx || !oracles || !batches || !alpha_in || !out || n_oracles == 0 || n_batches == 0)
        return set_err(ctx, GL_ERR_BAD_ARG, "null/empty argument");
    *out = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    const uint32_t log_n = oracles[0]->degree_log;
    const size_t n = (size_t)1 << log_n;
    for (size_t o = 0; o < n_oracles; o++)
        if (oracles[o]->degree_log != log_n) return set_err(ctx, GL_ERR_BAD_SHAPE, "Polynomial degrees inconsistent");
    gl_fri* f = new gl_fri();
    f->ctx = ctx;
    f->log_n = log_n;
    f->rate_bits = rate_bits;
    f->cap_height = cap_height;
    int rc = GL_OK;
    u64 *comp = nullptr, *chunk = nullptr, *drefs = nullptr, *ztab = nullptr;
    const E2 alpha = {canon(alpha_in[0]), canon(alpha_in[1])};
    const size_t nchunks = (n + SCAN_CHUNK - 1) / SCAN_CHUNK;
    const size_t hi_cnt = (n >> 12) + 1;
    auto body = [&]() -> int {
        TRY(dmalloc(ctx, &f->coeff_cols, 2 * n));
        TRY(dmalloc(ctx, &comp, 2 * n));
        TRY(dmalloc(ctx, &chunk, 2 * nchunks));
        // z / z^-1 power tables: [zhi | zlo | zihi | zilo], one allocation reused by every batch (stream-ordered)
        TRY(dmalloc(ctx, &ztab, 2 * (2 * hi_cnt + 2 * 4096)));
        u64 *zhi = ztab, *zlo = zhi + 2 * hi_cnt, *zihi = zlo + 2 * 4096, *zilo = zihi + 2 * hi_cnt;
        // alpha^j per polynomial (ReducingFactor restarts at alpha^0 for every batch): the references of ALL batches
        // go up in one copy (a pageable source is staged by the runtime before cudaMemcpyAsync returns)
        size_t total_polys = 0;
        for (size_t b = 0; b < n_batches; b++) total_polys += batches[b].num_polys;
        std::vector<PolyRef> refs(total_polys);
        std::vector<E2> shiftmuls(n_batches);
        for (size_t b = 0, at = 0; b < n_batches; b++) {
            const gl_fri_batch& batch = batches[b];
            E2 ap = {1, 0};
            for (size_t j = 0; j < batch.num_polys; j++, at++) {
                const uint32_t oi = batch.oracle_index[j], pi = batch.poly_index[j];
                if (oi >= n_oracles || pi >= oracles[oi]->B) return set_err(ctx, GL_ERR_BAD_ARG, "bad polynomial reference");
                refs[at].ptr = oracles[oi]->coeffs + (size_t)pi * n;
                refs[at].a0 = canon(ap.a);
                refs[at].a1 = canon(ap.b);
                ap = e2_mul(ap, alpha);
            }
            shiftmuls[b] = E2{canon(ap.a), canon(ap.b)};  // alpha^count: alpha.shift_poly (reducing.rs:102-106)
        }
        const size_t ref_words = total_polys * sizeof(PolyRef) / 8;
        TRY(dmalloc(ctx, &drefs, ref_words));
        if (ref_words) TRY(h2d(ctx, drefs, (const u64*)refs.data(), ref_words));
        for (size_t b = 0, at = 0; b < n_batches; at += batches[b].num_polys, b++) {
            const gl_fri_batch& batch = batches[b];
            const E2 shiftmul = shiftmuls[b];
            k_fri_compose<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((const PolyRef*)drefs + at,
                                                                              (uint32_t)batch.num_polys, n, comp);
            CKL(ctx);
            const E2 z = {canon(batch.point[0]), canon(batch.point[1])};
            if (z.a == 0 && z.b == 0) {
                k_div_by_x<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(comp, n, shiftmul, b == 0, f->coeff_cols);
                CKL(ctx);
                continue;
            }
            const E2 zi = e2_inv(z);
            E2Pows4 pw{{e2_pow(z, 4096), z, e2_pow(zi, 4096), zi}, {hi_cnt, 4096, hi_cnt, 4096}, {zhi, zlo, zihi, zilo}};
            const size_t fill_total = 2 * hi_cnt + 2 * 4096;
            k_fill_e2_pows4<<<(unsigned)((fill_total + 127) / 128), 128, 0, ctx->stream>>>(pw);
            CKL(ctx);
            k_scan_phase1<<<(unsigned)nchunks, SCAN_THREADS, 0, ctx->stream>>>(comp, n, zhi, zlo, chunk);
            CKL(ctx);
            k_scan_phase2<<<1, 1024, 0, ctx->stream>>>(chunk, nchunks);
            CKL(ctx);
            k_scan_phase3<<<(unsigned)nchunks, SCAN_THREADS, 0, ctx->stream>>>(comp, n, chunk, zihi, zilo, shiftmul,
                                                                              b == 0, f->coeff_cols);
            CKL(ctx);
        }
        TRY(fri_finish_begin(ctx, f));
        return GL_OK;
    };
    rc = body();
    dfree(ctx, comp);
    dfree(ctx, chunk);
    dfree(ctx, drefs);
    dfree(ctx, ztab);
    if (rc != GL_OK) {
        gl_fri_destroy(f);
        return rc;
    }
    *out = f;
    return GL_OK;
}

// ---- value-domain composition (the pre-FRI part of prove_openings, oracle.rs:186-220, evaluated point by point) ----
// final_poly(x) = sum_b alpha^{k_b} (F_b(x) - F_b(z_b)) / (x - z_b) with F_b(x) = sum_j alpha^j f_{b,j}(x): the same field
// elements as the LDE of the coefficient-domain final polynomial (the quotients are exact), but computed from the
// commitments' LDE rows in place -- rank-local when the commitments are row-block sharded.
struct ValRef {
    const u64* col;  // the polynomial's LDE column (leaf order), local rows
};
struct ValBatch {
    uint32_t first, count;  // slice of the ValRef array
    E2 z, y, shiftmul;      // point, F_b(z_b) = sum_j alpha^j y_{b,j}, alpha^count
};
constexpr int FRI_MAX_BATCHES = 8;
struct ComposeValuesParams {
    const ValRef* refs;
    ValBatch batch[FRI_MAX_BATCHES];
    uint32_t n_batches;
    size_t rows, row0;      // local rows, global index of local row 0
    uint32_t log_N;
    const u64 *xhi, *xlo;   // w_N^i = xhi[i >> 12] * xlo[i & 4095]
    u64 shift;
    E2 alpha;
    u64* out;               // rows x 2
    unsigned int* flag;
};
__global__ void __launch_bounds__(128) k_fri_compose_values(ComposeValuesParams p) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p.rows) return;
    const size_t i = (size_t)(__brevll((unsigned long long)(j + p.row0)) >> (64 - p.log_N));  // LDE point of leaf j
    const u64 x = mul(p.shift, mul(p.xhi[i >> 12], p.xlo[i & 4095]));
    E2 acc = {0, 0};
    for (uint32_t b = 0; b < p.n_batches; b++) {
        const ValBatch vb = p.batch[b];
        E2 s = {0, 0};
        for (uint32_t k = vb.count; k-- > 0;) {  // Horner in alpha over the batch's polynomials
            const u64 v = p.refs[vb.first + k].col[j];
            s = e2_mul(s, p.alpha);
            s.a = add(s.a, v);
        }
        const E2 d = {sub(x, vb.z.a), neg(vb.z.b)};  // x - z_b
        if (canon(d.a) == 0 && canon(d.b) == 0) atomicOr(p.flag, 1u);
        const E2 q = e2_mul(e2_sub(s, vb.y), e2_inv(d));
        acc = e2_add(e2_mul(acc, vb.shiftmul), q);  // alpha.shift_poly(&mut final_poly); final_poly += quotient
    }
    p.out[2 * j] = canon(acc.a);
    p.out[2 * j + 1] = canon(acc.b);
}

int gl_fri_begin_values(gl_ctx* ctx, gl_commit* const* oracles, size_t n_oracles, const gl_fri_batch* batches,
                        size_t n_batches, const uint64_t* opened, const uint64_t alpha_in[2], uint32_t cap_height,
                        gl_fri** out) {
    if (!ctx || !oracles || !batches || !opened || !alpha_in || !out || n_oracles == 0 || n_batches == 0)
        return set_err(ctx, GL_ERR_BAD_ARG, "null/empty argument");
    if (n_batches > (size_t)FRI_MAX_BATCHES) return set_err(ctx, GL_ERR_UNSUPPORTED, "more than %d opening batches", FRI_MAX_BATCHES);
    *out = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    const gl_commit* c0 = oracles[0];
    for (size_t o = 0; o < n_oracles; o++) {
        const gl_commit* c = oracles[o];
        if (!c->finished) return set_err(ctx, GL_ERR_BAD_ARG, "gl_commit_finish has not been called");
        if (c->degree_log != c0->degree_log || c->rate_bits != c0->rate_bits)
            return set_err(ctx, GL_ERR_BAD_SHAPE, "Polynomial degrees inconsistent");
        if (c->shard_index != c0->shard_index || c->shard_log != c0->shard_log)
            return set_err(ctx, GL_ERR_BAD_SHAPE, "commitments are sharded differently");
    }
    if (c0->shard_log > cap_height) return set_err(ctx, GL_ERR_BAD_SHAPE, "more shards than cap entries");
    gl_fri* f = new gl_fri();
    f->ctx = ctx;
    f->log_n = c0->degree_log;
    f->rate_bits = c0->rate_bits;
    f->cap_height = cap_height;
    f->vshard_index = c0->shard_index;
    f->vshard_log = c0->shard_log;
    f->log_cur = c0->degree_log + c0->rate_bits;
    f->shift = MULTIPLICATIVE_GROUP_GENERATOR;
    const size_t rows = c0->tree.N;
    const E2 alpha = {canon(alpha_in[0]), canon(alpha_in[1])};
    u64 *drefs = nullptr, *xtab = nullptr, *dflag = nullptr;
    auto body = [&]() -> int {
        size_t total = 0;
        for (size_t b = 0; b < n_batches; b++) total += batches[b].num_polys;
        std::vector<ValRef> refs(total);
        ComposeValuesParams p;
        p.n_batches = (uint32_t)n_batches;
        for (size_t b = 0, at = 0; b < n_batches; b++) {
            const gl_fri_batch& batch = batches[b];
            E2 ap = {1, 0}, y = {0, 0};
            p.batch[b].first = (uint32_t)at;
            p.batch[b].count = (uint32_t)batch.num_polys;
            for (size_t k = 0; k < batch.num_polys; k++, at++) {
                const uint32_t oi = batch.oracle_index[k], pi = batch.poly_index[k];
                if (oi >= n_oracles || pi >= oracles[oi]->B) return set_err(ctx, GL_ERR_BAD_ARG, "bad polynomial reference");
                refs[at].col = oracles[oi]->tree.leaves + (size_t)pi * oracles[oi]->tree.es;
                const E2 yv = {canon(opened[2 * at]), canon(opened[2 * at + 1])};
                y = e2_add(y, e2_mul(ap, yv));
                ap = e2_mul(ap, alpha);
            }
            p.batch[b].z = E2{canon(batch.point[0]), canon(batch.point[1])};
            p.batch[b].y = E2{canon(y.a), canon(y.b)};
            p.batch[b].shiftmul = E2{canon(ap.a), canon(ap.b)};
        }
        const size_t ref_words = total * sizeof(ValRef) / 8;
        TRY(dmalloc(ctx, &drefs, ref_words ? ref_words : 1));
        if (ref_words) TRY(h2d(ctx, drefs, (const u64*)refs.data(), ref_words));
        const uint32_t log_N = f->log_cur;
        const size_t N = (size_t)1 << log_N;
        const u64 wN = root_of_unity(log_N);
        const size_t tcnt = 4096 > (N >> 12) + 1 ? 4096 : (N >> 12) + 1;
        TRY(build_pow_tables(ctx, std::vector<u64>{gl::pow(wN, 4096), wN}, tcnt, &xtab));
        TRY(dmalloc(ctx, &dflag, 1));
        CK(ctx, cudaMemsetAsync(dflag, 0, 8, ctx->stream));
        TRY(dmalloc(ctx, &f->values, 2 * rows));
        p.refs = (const ValRef*)drefs;
        p.rows = rows;
        p.row0 = (size_t)c0->shard_index * rows;
        p.log_N = log_N;
        p.xhi = xtab;
        p.xlo = xtab + tcnt;
        p.shift = MULTIPLICATIVE_GROUP_GENERATOR;
        p.alpha = alpha;
        p.out = f->values;
        p.flag = (unsigned int*)dflag;
        k_fri_compose_values<<<(unsigned)((rows + 127) / 128), 128, 0, ctx->stream>>>(p);
        CKL(ctx);
        u64 flag = 0;
        TRY(d2h(ctx, &flag, dflag, 1));
        if (flag & 1u) return set_err(ctx, GL_ERR_DIV_ZERO, "Opening point is in the LDE domain");
        return GL_OK;
    };
    int rc = body();
    dfree(ctx, drefs);
    dfree(ctx, xtab);
    dfree(ctx, dflag);
    if (rc != GL_OK) {
        gl_fri_destroy(f);
        return rc;
    }
    *out = f;
    return GL_OK;
}
// the local block of the current codeword (between rounds): 2^(log_cur - shard_log) F_{p^2} values, bit-reversed order
int gl_fri_values_local(gl_fri* f, uint64_t* out, size_t cap_words, size_t* len_out) {
    gl_ctx* ctx = f->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (f->committed || !f->values) return set_err(ctx, GL_ERR_BAD_ARG, "fold the last round first");
    const size_t len = (size_t)1 << (f->log_cur - f->vshard_log);
    if (cap_words < 2 * len) return set_err(ctx, GL_ERR_BAD_ARG, "output buffer too small");
    if (len_out) *len_out = len;
    return d2h(ctx, out, f->values, 2 * len);
}

__global__ void k_split_ext(const u64* inter, size_t n, u64* cols) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    cols[i] = canon(inter[2 * i]);
    cols[n + i] = canon(inter[2 * i + 1]);
}
int gl_fri_begin_from_coeffs(gl_ctx* ctx, const uint64_t* coeffs_ext, uint32_t log_n, uint32_t rate_bits,
                             uint32_t cap_height, gl_fri** out) {
    if (!ctx || !coeffs_ext || !out) return set_err(ctx, GL_ERR_BAD_ARG, "null argument");
    *out = nullptr;
    CK(ctx, cudaSetDevice(ctx->device));
    if (log_n > 3 * NTT_MAX_LOG_PASS) return set_err(ctx, GL_ERR_UNSUPPORTED, "log_n %u > 30", log_n);
    const size_t n = (size_t)1 << log_n;
    gl_fri* f = new gl_fri();
    f->ctx = ctx;
    f->log_n = log_n;
    f->rate_bits = rate_bits;
    f->cap_height = cap_height;
    u64* tmp = nullptr;
    auto body = [&]() -> int {
        TRY(dmalloc(ctx, &f->coeff_cols, 2 * n));
        TRY(dmalloc(ctx, &tmp, 2 * n));
        TRY(h2d(ctx, tmp, coeffs_ext, 2 * n));
        k_split_ext<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(tmp, n, f->coeff_cols);
        CKL(ctx);
        TRY(fri_finish_begin(ctx, f));
        return GL_OK;
    };
    int rc = body();
    dfree(ctx, tmp);
    if (rc != GL_OK) {
        gl_fri_destroy(f);
        return rc;
    }
    *out = f;
    return GL_OK;
}
void gl_fri_destroy(gl_fri* f) {
    if (!f) return;
    cudaSetDevice(f->ctx->device);
    dfree(f->ctx, f->coeff_cols);
    dfree(f->ctx, f->values);
    for (auto& t : f->trees) tree_free(f->ctx, t);
    delete f;
}
int gl_fri_coeffs(gl_fri* f, uint64_t* out) {
    gl_ctx* ctx = f->ctx;
    if (!f->coeff_cols) return set_err(ctx, GL_ERR_BAD_ARG, "this FRI state was built in the value domain: no coefficients");
    const size_t n = (size_t)1 << f->log_n;
    u64* tmp;
    TRY(dmalloc(ctx, &tmp, 2 * n));
    k_interleave<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(f->coeff_cols, n, n, tmp);
    CKL(ctx);
    int rc = d2h(ctx, out, tmp, 2 * n);
    dfree(ctx, tmp);
    return rc;
}
uint32_t gl_fri_num_rounds(const gl_fri* f) { return (uint32_t)f->trees.size(); }

// One round's Merkle commitment; with num_shards = G > 1 only the row block [g*L/G, (g+1)*L/G) of the L leaves is hashed
// (FRI leaves are consecutive bit-reversed values, so a row block is a set of whole cap subtrees, like the initial
// commitment): cap_out receives this shard's C/G cap entries, the values stay replicated for the (cheap) fold.
static int fri_commit_round(gl_fri* f, uint32_t arity_bits, uint32_t shard_index, uint32_t num_shards, uint64_t* cap_out) {
    gl_ctx* ctx = f->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (f->committed) return set_err(ctx, GL_ERR_BAD_ARG, "fold the previous round first");
    if (arity_bits < 1 || arity_bits > 5) return set_err(ctx, GL_ERR_UNSUPPORTED, "arity_bits %u not in 1..5", arity_bits);
    if (arity_bits > f->log_cur) return set_err(ctx, GL_ERR_BAD_SHAPE, "arity exceeds the codeword length");
    uint32_t sl = 0;
    if (log2_exact(num_shards, &sl) || shard_index >= num_shards)
        return set_err(ctx, GL_ERR_BAD_ARG, "bad shard %u of %u (power of two required)", shard_index, num_shards);
    if (f->cap_height > f->log_cur - arity_bits)
        return set_err(ctx, GL_ERR_BAD_SHAPE, "cap_height=%u should be at most log2(leaves.len())=%u", f->cap_height,
                       f->log_cur - arity_bits);
    if (sl > f->cap_height)
        return set_err(ctx, GL_ERR_BAD_SHAPE, "num_shards=%u exceeds the cap size 2^%u", num_shards, f->cap_height);
    if (f->vshard_log) {  // the codeword itself is sharded: the local buffer is this shard's block of leaves
        if (num_shards != 1 && (sl != f->vshard_log || shard_index != f->vshard_index))
            return set_err(ctx, GL_ERR_BAD_ARG, "this FRI state is row-block sharded %u of %u", f->vshard_index, 1u << f->vshard_log);
        sl = f->vshard_log;
        shard_index = 0;  // no offset inside the local buffer
        if (f->log_cur < arity_bits + sl || sl > f->cap_height)
            return set_err(ctx, GL_ERR_BAD_SHAPE, "round too small for %u shards", 1u << sl);
    }
    const size_t L = (size_t)1 << (f->log_cur - arity_bits);
    Tree t;
    t.N = L >> sl;
    t.W = 2u << arity_bits;
    t.cap_height = f->cap_height - sl;
    t.base = f->values;
    t.leaves = f->values + (size_t)shard_index * t.N * t.W;  // chunks(arity).map(flatten) of the bit-reversed values == this buffer
    t.own_leaves = false;
    int rc = tree_build(ctx, t);
    if (rc != GL_OK) {
        tree_free(ctx, t);
        return rc;
    }
    t.own_leaves = true;  // ownership of the values buffer moves to the tree
    f->round_values = f->values;
    f->round_leaves = f->vshard_log ? t.N : L;
    f->values = nullptr;
    f->trees.push_back(t);
    f->pending_arity_bits = arity_bits;
    f->committed = true;
    return d2h(ctx, cap_out, t.cap, t.cap_words());
}
int gl_fri_commit_round(gl_fri* f, uint32_t arity_bits, uint64_t* cap_out) { return fri_commit_round(f, arity_bits, 0, 1, cap_out); }
int gl_fri_commit_round_sharded(gl_fri* f, uint32_t arity_bits, uint32_t shard_index, uint32_t num_shards, uint64_t* cap_out) {
    return fri_commit_round(f, arity_bits, shard_index, num_shards, cap_out);
}

int gl_fri_fold(gl_fri* f, const uint64_t beta[2]) {
    gl_ctx* ctx = f->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (!f->committed) return set_err(ctx, GL_ERR_BAD_ARG, "commit the round first");
    const uint32_t ab = f->pending_arity_bits;
    const size_t leaves = f->round_leaves;
    u64* out;
    TRY(dmalloc(ctx, &out, 2 * leaves));
    FoldParams fp{};
    fp.values = f->round_values;
    fp.out = out;
    fp.n_leaves = leaves;
    fp.leaf0 = (size_t)f->vshard_index * leaves;
    fp.log_leaves = f->log_cur - ab;
    const u64 wN = root_of_unity(f->log_cur);
    const u64 winv = gl::inv(wN);
    const size_t hi_cnt = ((size_t)1 << (f->log_cur > 12 ? f->log_cur - 12 : 0)) + 1;  // covers any arity
    const size_t tcnt = hi_cnt > 4096 ? hi_cnt : 4096;
    u64* tabs;
    {
        auto it = ctx->fold_tabs.find((int)f->log_cur);
        if (it == ctx->fold_tabs.end()) {
            TRY(build_pow_tables(ctx, std::vector<u64>{gl::pow(winv, 4096), winv}, tcnt, &tabs));
            ctx->fold_tabs[(int)f->log_cur] = tabs;
        } else {
            tabs = it->second;
        }
    }
    fp.winv_hi = tabs;
    fp.winv_lo = tabs + tcnt;
    fp.shift_inv = gl::inv(f->shift);
    fp.beta0 = canon(beta[0]);
    fp.beta1 = canon(beta[1]);
    fp.arity_inv = inverse_2exp(ab);
    const u64 wa_inv = gl::inv(root_of_unity(ab));
    for (uint32_t j = 0; j < (1u << ab); j++) fp.root_inv[j] = gl::pow(wa_inv, j);
    const unsigned nb = (unsigned)((leaves + 127) / 128);
    switch (ab) {
        case 1: k_fri_fold<1><<<nb, 128, 0, ctx->stream>>>(fp); break;
        case 2: k_fri_fold<2><<<nb, 128, 0, ctx->stream>>>(fp); break;
        case 3: k_fri_fold<3><<<nb, 128, 0, ctx->stream>>>(fp); break;
        case 4: k_fri_fold<4><<<nb, 128, 0, ctx->stream>>>(fp); break;
        case 5: k_fri_fold<5><<<nb, 128, 0, ctx->stream>>>(fp); break;
    }
    CKL(ctx);
    f->values = out;
    f->log_cur -= ab;
    f->shift = gl::pow(f->shift, (u64)1 << ab);  // shift = shift.exp_u64(arity), prover.rs:118
    f->committed = false;
    return GL_OK;
}

// batch-FRI (batch_fri/prover.rs:118-132): after a fold, when the codeword has shrunk to the size of the next (smaller)
// instance's LDE, final_values <- final_values * beta + values[next], element by element in natural order -- which is
// element by element in the shared bit-reversed order too.
__global__ void k_fri_mix(u64* vals, const u64* other, size_t count, E2 beta) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const E2 v = {vals[2 * i], vals[2 * i + 1]}, w = {other[2 * i], other[2 * i + 1]};
    const E2 r = e2_add(e2_mul(v, beta), w);
    vals[2 * i] = canon(r.a);
    vals[2 * i + 1] = canon(r.b);
}
int gl_fri_mix(gl_fri* f, const gl_fri* other, const uint64_t beta[2]) {
    if (!f || !other || !beta) return set_err(f ? f->ctx : nullptr, GL_ERR_BAD_ARG, "null argument");
    gl_ctx* ctx = f->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (f->committed || other->committed || !f->values || !other->values)
        return set_err(ctx, GL_ERR_BAD_ARG, "both codewords must be between rounds (folded, not committed)");
    if (f->log_cur != other->log_cur) return set_err(ctx, GL_ERR_BAD_SHAPE, "codeword lengths differ: 2^%u vs 2^%u", f->log_cur, other->log_cur);
    const size_t count = (size_t)1 << f->log_cur;
    k_fri_mix<<<(unsigned)((count + 255) / 256), 256, 0, ctx->stream>>>(f->values, other->values, count,
                                                                         E2{canon(beta[0]), canon(beta[1])});
    CKL(ctx);
    return GL_OK;
}

int gl_fri_final_poly(gl_fri* f, uint64_t* out, size_t cap_words, size_t* len_out) {
    gl_ctx* ctx = f->ctx;
    CK(ctx, cudaSetDevice(ctx->device));
    if (f->committed) return set_err(ctx, GL_ERR_BAD_ARG, "fold the last round first");
    if (f->vshard_log) return set_err(ctx, GL_ERR_BAD_ARG, "sharded codeword: gather gl_fri_values_local and interpolate");
    const size_t Nf = (size_t)1 << f->log_cur;
    if (f->log_cur < f->rate_bits) return set_err(ctx, GL_ERR_BAD_SHAPE, "codeword shorter than the blowup");
    const size_t len = Nf >> f->rate_bits;
    if (cap_words < 2 * len) return set_err(ctx, GL_ERR_BAD_ARG, "output buffer too small");
    u64 *cols, *inter;
    TRY(dmalloc(ctx, &cols, 2 * Nf));
    TRY(dmalloc(ctx, &inter, 2 * len));
    k_unbitrev_split<<<(unsigned)((Nf + 255) / 256), 256, 0, ctx->stream>>>(f->values, Nf, f->log_cur, cols);
    CKL(ctx);
    // coset_ifft on the current coset (the reference keeps coefficients; we recover them once)
    int rc = ntt_natural(ctx, cols, Nf, cols, Nf, (int)f->log_cur, 2, true, f->shift);
    if (rc == GL_OK) {
        k_interleave<<<(unsigned)((len + 255) / 256), 256, 0, ctx->stream>>>(cols, Nf, len, inter);
        ctx->launches++;
        rc = d2h(ctx, out, inter, 2 * len);
    }
    dfree(ctx, cols);
    dfree(ctx, inter);
    if (rc == GL_OK && len_out) *len_out = len;
    return rc;
}

int gl_fri_open(gl_fri* f, uint32_t round, const uint64_t* leaf_indices, size_t count, uint64_t* out_leaves,
                uint64_t* out_paths) {
    if (round >= f->trees.size()) return set_err(f->ctx, GL_ERR_BAD_ARG, "round %u out of range", round);
    CK(f->ctx, cudaSetDevice(f->ctx->device));
    return tree_open(f->ctx, f->trees[round], leaf_indices, count, out_leaves, out_paths);
}

int gl_fri_pow(gl_ctx* ctx, const uint64_t state[12], uint32_t pos, uint32_t min_leading_zeros, uint64_t* nonce_out) {
    if (!ctx || !state || !nonce_out || pos >= 8) return set_err(ctx, GL_ERR_BAD_ARG, "bad argument");
    CK(ctx, cudaSetDevice(ctx->device));
    unsigned long long* dres;
    TRY(dmalloc(ctx, (u64**)&dres, 1));
    PowParams pp;
    for (int i = 0; i < 12; i++) pp.state[i] = canon(state[i]);
    pp.pos = pos;
    pp.min_lz = min_leading_zeros;
    // batches grow geometrically from ~2x the expected number of tries so that an easy grind costs one
    // small launch; candidates are scanned in increasing order, so the first hit batch holds the minimum.
    u64 batch = (u64)2 << (min_leading_zeros < 24 ? min_leading_zeros : 24);
    if (batch < 4096) batch = 4096;
    int rc = GL_OK;
    u64 found = ~0ULL;
    for (u64 start = 0; start < P; start += batch, batch = batch < ((u64)1 << 24) ? batch * 4 : batch) {
        if (cudaMemsetAsync(dres, 0xFF, 8, ctx->stream) != cudaSuccess) {
            rc = set_err(ctx, GL_ERR_CUDA, "cudaMemsetAsync failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
        pp.start = start;
        pp.count = (P - start < batch) ? P - start : batch;
        const u64 nb_max = (u64)ctx->sm_count * 8;
        const unsigned nb = (unsigned)((pp.count + 127) / 128 < nb_max ? (pp.count + 127) / 128 : nb_max);
        k_fri_pow<<<nb, 128, 0, ctx->stream>>>(pp, dres);
        ctx->launches++;
        if (cudaGetLastError() != cudaSuccess) {
            rc = set_err(ctx, GL_ERR_CUDA, "k_fri_pow launch failed");
            break;
        }
        rc = d2h(ctx, &found, (u64*)dres, 1);
        if (rc != GL_OK || found != ~0ULL) break;
        if (start > ((u64)1 << 40)) {
            rc = set_err(ctx, GL_ERR_POW_FAILED, "Proof of work failed. This is highly unlikely!");
            break;
        }
    }
    dfree(ctx, (u64*)dres);
    if (rc == GL_OK) *nonce_out = found;
    return rc;
}

}  // extern "C"
