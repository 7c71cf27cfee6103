// capi.cu — C ABI (include/winterfell_b200.h): context, device matrices, NTT/LDE planning,
// commitments, FRI prover. Host orchestration only; all arithmetic on field data happens in the
// kernels of ntt.cu / commit.cu / fri.cu / layout.cu. There is no CPU fallback for device work.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>

#include <algorithm>
#include <map>
#include <set>
#include <string>
#include <thread>
#include <vector>

#include "internal.hpp"

void wf_mark(wf_ctx* ctx, const char* name) {
    if (!ctx->profiling) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, ctx->st);
    ctx->marks.push_back({name, e});
}
int wf_fail(wf_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    return code;
}
// The context's device is made current on the calling thread wherever work for it starts (allocation, pass launch, gather,
// stage mark, sync): a process may hold contexts for several GPUs, or call from a thread whose current device is another one.
static inline void wf_use_device(wf_ctx* ctx) {
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != ctx->device) cudaSetDevice(ctx->device);
}
int wf_dev_alloc(wf_ctx* ctx, size_t bytes, void** out) {
    wf_use_device(ctx);
    bytes = (bytes + 255) & ~(size_t)255;
    if (bytes == 0) bytes = 256;
    auto it = ctx->pool.find(bytes);
    if (it != ctx->pool.end()) {
        *out = it->second;
        ctx->pool.erase(it);
        ctx->live[*out] = bytes;
        return WF_OK;
    }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        // release the cache and retry once
        for (auto& kv : ctx->pool) cudaFree(kv.second);
        ctx->pool.clear();
        e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return wf_fail(ctx, WF_ERR_CUDA, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    }
    ctx->live[p] = bytes;
    *out = p;
    return WF_OK;
}
// Buffers return to the pool in stream order: all work is issued on ctx->st, so a later user of the
// same buffer is ordered after the earlier kernels that touched it.
void wf_dev_free(wf_ctx* ctx, void* p) {
    if (!p) return;
    auto it = ctx->live.find(p);
    if (it == ctx->live.end()) return;
    ctx->pool.insert({it->second, p});
    ctx->live.erase(it);
}
int wf_mat_alloc(wf_ctx* ctx, size_t rows, u32 cols, wf_mat** out) { return wf_mat_alloc_w(ctx, rows, cols, seg_width_for(cols), out); }
int wf_mat_alloc_w(wf_ctx* ctx, size_t rows, u32 cols, int W, wf_mat** out) {
    wf_mat* m = new wf_mat();
    m->m.rows = rows;
    m->m.cols = cols;
    m->m.W = W;
    m->m.seg_stride = rows * m->m.W;
    void* p;
    int r = wf_dev_alloc(ctx, m->m.words() * 8, &p);
    if (r != WF_OK) { delete m; return r; }
    m->m.base = (u64*)p;
    *out = m;
    return WF_OK;
}

// -------------------------------------------------------------------------------------------------
// twiddle / scale tables (built once per size, cached in the context)
// -------------------------------------------------------------------------------------------------
__global__ void pow_table_kernel(u64* out, u64 base, u64 scale, size_t count) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = gl_mul(scale, gl_pow(base, i));
}
__global__ void pow_table2_kernel(u64* out, const u64* bases, size_t count, size_t nbases) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count * nbases) out[i] = gl_pow(bases[i / count], i % count);
}

int wf_get_twiddles(wf_ctx* ctx, u32 log_n, const u64** out) {
    auto it = ctx->tw.find(log_n);
    if (it != ctx->tw.end()) { *out = it->second; return WF_OK; }
    if (log_n < 1 || log_n > 32) return wf_fail(ctx, WF_ERR_INVALID, "no 2^%u-th root of unity", log_n);
    size_t half = log_n >= 1 ? ((size_t)1 << (log_n - 1)) : 1;
    void* p;
    // never returned to the pool: cudaMalloc directly
    cudaError_t e = cudaMalloc(&p, std::max(half * 8, (size_t)16));
    if (e != cudaSuccess) return wf_fail(ctx, WF_ERR_CUDA, "cudaMalloc twiddles: %s", cudaGetErrorString(e));
    pow_table_kernel<<<(unsigned)((half + 255) / 256), 256, 0, ctx->st>>>((u64*)p, gl_root_of_unity(log_n), 1, half);
    ctx->launches++;
    CK(cudaGetLastError());
    ctx->tw[log_n] = (u64*)p;
    *out = (u64*)p;
    return WF_OK;
}

// w_(2^log_order)^i for i < 2^log_count (full power table; two of them replace the gather over w_M^i, i < M/2)
static int get_pow_table(wf_ctx* ctx, u32 log_order, u32 log_count, const u64** out) {
    auto key = std::make_pair(log_order, log_count);
    auto it = ctx->pow_tab.find(key);
    if (it != ctx->pow_tab.end()) { *out = it->second; return WF_OK; }
    size_t cnt = (size_t)1 << log_count;
    void* p;
    cudaError_t e = cudaMalloc(&p, std::max(cnt * 8, (size_t)16));
    if (e != cudaSuccess) return wf_fail(ctx, WF_ERR_CUDA, "cudaMalloc power table: %s", cudaGetErrorString(e));
    pow_table_kernel<<<(unsigned)((cnt + 255) / 256), 256, 0, ctx->st>>>((u64*)p, log_order ? gl_root_of_unity(log_order) : 1, 1, cnt);
    ctx->launches++;
    CK(cudaGetLastError());
    ctx->pow_tab[key] = (u64*)p;
    *out = (u64*)p;
    return WF_OK;
}
static int get_round_tw(wf_ctx* ctx, u32 logS, const u64** out) {
    auto it = ctx->round_tw.find(logS);
    if (it != ctx->round_tw.end()) { *out = it->second; return WF_OK; }
    void* p;
    cudaError_t e = cudaMalloc(&p, ntt2_tw_entries((int)logS) * 8);
    if (e != cudaSuccess) return wf_fail(ctx, WF_ERR_CUDA, "cudaMalloc round twiddles: %s", cudaGetErrorString(e));
    CK(ntt2_build_tw((int)logS, (u64*)p, ctx->st));
    ctx->launches++;
    ctx->round_tw[logS] = (u64*)p;
    *out = (u64*)p;
    return WF_OK;
}
// One pass: fills in the twiddle tables the kernel family of this sub-transform size reads, then launches.
// p.logS, p.logM, p.has_post, p.W and the geometry must be set; sub_tw / master / tw_hi / tw_lo are set here.
static int launch_pass(wf_ctx* ctx, int mode, NttPassParams& p, u32 n_segments, u32 n_batch) {
    wf_use_device(ctx);
    if (p.logS >= NTT2_MIN_LOGS) {
        CKI(get_round_tw(ctx, (u32)p.logS, &p.sub_tw));
        if (p.has_post) {
            p.tw_split = p.logM / 2;
            CKI(get_pow_table(ctx, p.logM, p.tw_split, &p.tw_lo));
            CKI(get_pow_table(ctx, p.logM - p.tw_split, p.logM - p.tw_split, &p.tw_hi));
        }
        p.vec_in = p.vec_out = (p.W >= 2 || mode == NTT_STRIDED) ? 1 : 0;
        CK(ntt2_launch_pass(mode, p, n_segments, n_batch, ctx->st));
    } else {
        CKI(wf_get_twiddles(ctx, std::max((u32)p.logS, 1u), &p.sub_tw));
        if (p.has_post) CKI(wf_get_twiddles(ctx, p.logM, &p.master));
        CK(ntt_launch_pass(mode, p, n_segments, n_batch, ctx->st));
    }
    ctx->launches++;
    return WF_OK;
}

// n = R * C split for the two-pass schedule (sub-transforms of at most 2^NTT_MAX_LOGS points)
static void split_log(u32 log_n, u32* logR, u32* logC) {
    if (log_n <= NTT_MAX_LOGS) { *logR = 0; *logC = log_n; return; }
    u32 r = (log_n + 1) / 2;
    if (r > NTT_MAX_LOGS) r = NTT_MAX_LOGS;
    *logR = r;
    *logC = log_n - r;
}

// tables for the first LDE pass of an n = R * C split (logR = 0: single pass over n = C points)
static int get_lde_tables(wf_ctx* ctx, u32 log_n, u32 log_b, u32 logR, LdeTables* out) {
    auto key = std::make_pair(log_n | (logR << 8), log_b);
    auto it = ctx->lde_tabs.find(key);
    if (it != ctx->lde_tabs.end()) { *out = it->second; return WF_OK; }
    const u32 logC = log_n - logR;
    size_t b = (size_t)1 << log_b, R = (size_t)1 << logR, C = (size_t)1 << logC;
    u64 g = gl_root_of_unity(log_n + log_b);
    // s_k = 7 * w_N^k (coset k of the LDE domain; natural row i = b*j + k)
    std::vector<u64> bases(b);
    size_t cnt = logR == 0 ? C : R;
    for (size_t k = 0; k < b; k++) {
        u64 sk = gl_mul(GL_GENERATOR, gl_pow(g, k));
        bases[k] = logR == 0 ? sk : gl_pow(sk, C);
    }
    LdeTables t{nullptr, nullptr};
    void *p, *pb;
    CK(cudaMalloc(&p, b * cnt * 8));
    CK(cudaMalloc(&pb, b * 8));
    CK(cudaMemcpyAsync(pb, bases.data(), b * 8, cudaMemcpyHostToDevice, ctx->st));
    pow_table2_kernel<<<(unsigned)((b * cnt + 255) / 256), 256, 0, ctx->st>>>((u64*)p, (u64*)pb, cnt, b);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->st));  // `bases` is a stack vector
    cudaFree(pb);
    t.pre = (u64*)p;
    if (logR != 0) {
        void* q;
        CK(cudaMalloc(&q, C * 8));
        pow_table_kernel<<<(unsigned)((C + 255) / 256), 256, 0, ctx->st>>>((u64*)q, GL_GENERATOR, 1, C);
        ctx->launches++;
        CK(cudaGetLastError());
        t.pow7 = (u64*)q;
    }
    ctx->lde_tabs[key] = t;
    *out = t;
    return WF_OK;
}

// -------------------------------------------------------------------------------------------------
// NTT / LDE drivers on segment matrices
// -------------------------------------------------------------------------------------------------
static void pass_defaults(NttPassParams& p, const SegMatrix& in, const SegMatrix& out) {
    memset(&p, 0, sizeof(p));
    p.in = in.base;
    p.out = out.base;
    p.in_seg_stride = in.seg_stride;
    p.out_seg_stride = out.seg_stride;
    p.W = in.W;
    p.out_W = (u32)out.W;
    p.out_row_mul = 1;
    p.cconst = 1;
}
// three-pass split for n > 2^22: n = 2^lr * 2^lc with the size-2^lc step itself two-pass (2^lr2 * 2^lc2)
static int split3(wf_ctx* ctx, u32 log_n, u32* lr, u32* lc, u32* lr2, u32* lc2) {
    *lr = (log_n + 2) / 3;
    *lc = log_n - *lr;
    split_log(*lc, lr2, lc2);
    if (*lr2 == 0 || *lc2 > NTT_MAX_LOGS || *lr > NTT_MAX_LOGS)
        return wf_fail(ctx, WF_ERR_UNSUPPORTED, "transform of 2^%u points exceeds the three-pass limit", log_n);
    return WF_OK;
}

// out = DFT (inverse: iDFT with 1/n) of every column of `in`; in/out: n rows. `tmp` (n rows, same
// shape) is needed when log_n > NTT_MAX_LOGS. in == out is allowed.
static int run_ntt(wf_ctx* ctx, const SegMatrix& in, SegMatrix& out, const SegMatrix* tmp, u32 log_n, int inverse) {
    u32 logR, logC;
    split_log(log_n, &logR, &logC);
    u64 inv_n = gl_inv(((u64)1 << log_n) % GL_P);
    NttPassParams p;
    if (logC > NTT_MAX_LOGS) {
        // THREE passes (n > 2^22): pass A is the strided size-R step of the four-step scheme over the whole array; the
        // contiguous size-C step is then a batch of R independent two-pass transforms (batch index = j1) whose last
        // pass writes X[j1 + R * j].
        if (!tmp) return wf_fail(ctx, WF_ERR_STATE, "run_ntt: scratch matrix required");
        u32 lr, lc, lr2, lc2;
        CKI(split3(ctx, log_n, &lr, &lc, &lr2, &lc2));
        pass_defaults(p, in, *tmp);  // pass A
        p.logS = (int)lr; p.logR = lr; p.logC = lc; p.inverse = inverse;
        p.has_post = 1; p.logM = log_n; p.a_mul = 1; p.b_mul = 0; p.cconst = inverse ? inv_n : 1;
        CKI(launch_pass(ctx, NTT_STRIDED, p, in.nseg(), 1));
        pass_defaults(p, *tmp, *tmp);  // pass B: in place, batch = row j1 of the R x C matrix
        p.in_batch_stride = p.out_batch_stride = ((size_t)1 << lc) * in.W;
        p.logS = (int)lr2; p.logR = lr2; p.logC = lc2; p.inverse = inverse;
        p.has_post = 1; p.logM = lc; p.a_mul = 1; p.b_mul = 0;
        CKI(launch_pass(ctx, NTT_STRIDED, p, in.nseg(), 1u << lr));
        pass_defaults(p, *tmp, out);  // pass C: X[j1 + R * (inner index)]
        p.in_batch_stride = ((size_t)1 << lc) * in.W;
        p.logS = (int)lc2; p.logR = lr2; p.logC = lc2; p.inverse = inverse;
        p.out_row_mul = 1u << lr; p.out_row_add = 1;
        CKI(launch_pass(ctx, NTT_CONTIG, p, in.nseg(), 1u << lr));
        return WF_OK;
    }
    if (logR == 0) {
        pass_defaults(p, in, out);
        p.logS = (int)logC; p.logR = 0; p.logC = logC; p.inverse = inverse;
        if (inverse) p.cconst = inv_n;
        return launch_pass(ctx, NTT_CONTIG, p, in.nseg(), 1);
    }
    if (!tmp) return wf_fail(ctx, WF_ERR_STATE, "run_ntt: scratch matrix required");
    // pass 1: strided size-R transforms + twiddle w_n^(+-j1*m2) (and 1/n for the inverse)
    pass_defaults(p, in, *tmp);
    p.logS = (int)logR; p.logR = logR; p.logC = logC; p.inverse = inverse;
    p.has_post = 1; p.logM = log_n; p.a_mul = 1; p.b_mul = 0; p.cconst = inverse ? inv_n : 1;
    CKI(launch_pass(ctx, NTT_STRIDED, p, in.nseg(), 1));
    // pass 2: contiguous size-C transforms, transposed write-back
    pass_defaults(p, *tmp, out);
    p.logS = (int)logC; p.logR = logR; p.logC = logC; p.inverse = inverse;
    return launch_pass(ctx, NTT_CONTIG, p, in.nseg(), 1);
}

// LDE of coefficient columns over 7 * <w_N>: out has n << log_b rows, row b*j + k = P(7 w_N^k w_n^j).
// `out` may be a view of a wider matrix: segment width out.W >= polys.W, the polys' columns landing at
// column offset out_col0 of each out row (column-chunked trace pipeline, wf_trace_lde_from_host).
static int set_scatter(wf_ctx* ctx, NttPassParams& p, const LdeScatter& sc, u32 log_b, u32 coset) {
    if (p.logS < NTT2_MIN_LOGS || p.W < 2) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "scattered LDE output needs sub-transforms of >= 64 points and W >= 2");
    p.sc_on = 1; p.sc_log_nj = sc.log_nj; p.sc_log_b = log_b; p.sc_coset = coset; p.sc_seg0 = sc.seg0; p.sc_seg_stride = sc.seg_stride; p.sc_world = sc.world;
    for (int q = 0; q < 8; q++) p.sc_peer[q] = sc.peer[q];
    return WF_OK;
}
// k0 <= k < k1 (k1 = 0: all cosets) selects the cosets computed; coset k, point j lands in out row j * row_mul + (k - k0) * row_add
// (row_mul = 0: the natural order b*j + k). Coset-major output (row_mul = 1, row_add = n) is what a rank of a sharded proof
// produces for the cosets it owns (prover.cu, composition polynomial).
static int run_lde(wf_ctx* ctx, const SegMatrix& polys, SegMatrix& out, u32 log_n, u32 log_b, u32 out_col0 = 0, u32 k0 = 0, u32 k1 = 0,
                   u32 row_mul = 0, u32 row_add = 1, const LdeScatter* sc = nullptr) {
    u32 logR, logC;
    split_log(log_n, &logR, &logC);
    u32 b = 1u << log_b;
    if (k1 == 0) k1 = b;
    if (row_mul == 0) { row_mul = b; row_add = 1; }
    LdeTables tabs;
    NttPassParams p;
    if (sc && logC > NTT_MAX_LOGS) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "scattered LDE output is limited to two-pass sizes");
    if (logC > NTT_MAX_LOGS) {
        // THREE passes per coset (n > 2^22), same structure as run_ntt: pass A carries the coset scaling
        // and the four-step twiddle, the contiguous size-C step is a batch of R two-pass transforms whose
        // last pass writes row b*(j1 + R*j) + k.
        u32 lr, lc, lr2, lc2;
        CKI(split3(ctx, log_n, &lr, &lc, &lr2, &lc2));
        CKI(get_lde_tables(ctx, log_n, log_b, lr, &tabs));
        SegMatrix y = polys;
        void* yp;
        CKI(wf_dev_alloc(ctx, polys.words() * 8, &yp));
        y.base = (u64*)yp;
        int rc = WF_OK;
        for (u32 k = k0; k < k1 && rc == WF_OK; k++) {
            pass_defaults(p, polys, y);  // pass A
            p.logS = (int)lr; p.logR = lr; p.logC = lc;
            p.pre_tab = tabs.pre + ((size_t)k << lr); p.pre_batch_stride = 0;
            p.has_post = 1; p.logM = log_n + log_b; p.a_mul = b; p.b_mul = 1; p.batch0 = k;
            p.ctab = tabs.pow7;
            rc = launch_pass(ctx, NTT_STRIDED, p, polys.nseg(), 1);
            if (rc != WF_OK) break;
            pass_defaults(p, y, y);  // pass B (in place), batch = j1
            p.in_batch_stride = p.out_batch_stride = ((size_t)1 << lc) * polys.W;
            p.logS = (int)lr2; p.logR = lr2; p.logC = lc2;
            p.has_post = 1; p.logM = lc; p.a_mul = 1; p.b_mul = 0;
            rc = launch_pass(ctx, NTT_STRIDED, p, polys.nseg(), 1u << lr);
            if (rc != WF_OK) break;
            pass_defaults(p, y, out);  // pass C: row b*(j1 + R*j) + k
            p.in_batch_stride = ((size_t)1 << lc) * polys.W;
            p.logS = (int)lc2; p.logR = lr2; p.logC = lc2;
            p.out_row_mul = row_mul << lr; p.out_row_add = row_mul; p.out_col0 = out_col0;
            p.out = out.base + (size_t)(k - k0) * row_add * out.W;
            rc = launch_pass(ctx, NTT_CONTIG, p, polys.nseg(), 1u << lr);
        }
        wf_dev_free(ctx, yp);  // stream-ordered pool: also correct on the error path
        return rc;
    }
    CKI(get_lde_tables(ctx, log_n, log_b, logR, &tabs));
    if (logR == 0) {
        pass_defaults(p, polys, out);
        p.logS = (int)logC; p.logR = 0; p.logC = logC;
        p.pre_tab = tabs.pre + ((size_t)k0 << log_n); p.pre_batch_stride = (size_t)1 << log_n;
        p.out_row_mul = row_mul; p.out_row_add = row_add; p.out_col0 = out_col0;
        if (sc) CKI(set_scatter(ctx, p, *sc, log_b, k0));
        return launch_pass(ctx, NTT_CONTIG, p, polys.nseg(), k1 - k0);
    }
    // Cosets per launch (grid.z = coset). The scratch Y of one coset is as large as the polynomials; while
    // it fits in half of the 126 MB L2 the contiguous pass finds most of it there, so cosets are processed
    // kb at a time with kb chosen to keep kb * |polys| <= 64 MiB (never less than one coset; narrow matrices
    // whose tiles would not fill the SMs take all cosets at once).
    const size_t poly_bytes = polys.words() * 8;
    const size_t tiles_per_coset = (((size_t)1 << logC) * polys.nseg());  // strided-pass blocks (x chunks)
    u32 kb = b;
    while (kb > 1 && poly_bytes * kb > ((size_t)64 << 20) && tiles_per_coset * (kb / 2) >= 4 * 296) kb >>= 1;
    while (kb > 1 && poly_bytes * kb > ((size_t)1 << 30)) kb >>= 1;
    while (kb > k1 - k0 || (k1 - k0) % kb) kb >>= 1;
    SegMatrix y = polys;
    void* yp;
    CKI(wf_dev_alloc(ctx, poly_bytes * kb, &yp));
    y.base = (u64*)yp;
    int rc = WF_OK;
    for (u32 k = k0; k < k1 && rc == WF_OK; k += kb) {
        // pass 1: Y_k[j1][m2] = 7^m2 w_N^((b j1 + k) m2) sum_m1 a[C m1 + m2] (s_k^C)^m1 w_R^(j1 m1)
        pass_defaults(p, polys, y);
        p.logS = (int)logR; p.logR = logR; p.logC = logC;
        p.pre_tab = tabs.pre + ((size_t)k << logR); p.pre_batch_stride = (size_t)1 << logR;
        p.out_batch_stride = polys.words();
        // exponent (b*j1 + k)*m2 = (j1*a_mul + (batch0 + z)*b_mul)*m2
        p.has_post = 1; p.logM = log_n + log_b; p.a_mul = b; p.b_mul = 1; p.batch0 = k;
        p.ctab = tabs.pow7;
        rc = launch_pass(ctx, NTT_STRIDED, p, polys.nseg(), kb);
        if (rc != WF_OK) break;
        // pass 2: X_k[j1 + R j2] = sum_m2 Y_k[j1][m2] w_C^(j2 m2)  -> row b*(j1 + R j2) + k
        pass_defaults(p, y, out);
        p.logS = (int)logC; p.logR = logR; p.logC = logC;
        p.in_batch_stride = polys.words();
        p.out_row_mul = row_mul; p.out_row_add = row_add; p.out_col0 = out_col0;
        p.out = out.base + (size_t)(k - k0) * row_add * out.W;  // first coset of the launch; the launch's coset z adds z * row_add rows
        if (sc) { rc = set_scatter(ctx, p, *sc, log_b, k); if (rc != WF_OK) break; }
        rc = launch_pass(ctx, NTT_CONTIG, p, polys.nseg(), kb);
    }
    wf_dev_free(ctx, yp);
    return rc;
}

// =================================================================================================
// C ABI
// =================================================================================================
template <int K>
__device__ __forceinline__ void field_shift_store(u64 a, u64* out, size_t n, size_t i, int slot) { out[(4 + slot) * n + i] = gl_mul_2exp<K>(a); }
__global__ void field_ops_kernel(const u64* a, const u64* b, size_t n, u64* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u64 x = a[i], y = b[i];
    out[i] = gl_mul(x, y);
    out[n + i] = gl_add(x, y);
    out[2 * n + i] = gl_sub(x, y);
    out[3 * n + i] = x ? gl_inv(x) : 0;
    u64 s = x, d = y;
    gl_butterfly(s, d);
    if (s != out[n + i] || d != out[2 * n + i]) out[n + i] = ~0ULL;  // butterfly must agree with add / sub
    field_shift_store<1>(x, out, n, i, 0);   field_shift_store<3>(x, out, n, i, 1);   field_shift_store<6>(x, out, n, i, 2);
    field_shift_store<12>(x, out, n, i, 3);  field_shift_store<24>(x, out, n, i, 4);  field_shift_store<31>(x, out, n, i, 5);
    field_shift_store<32>(x, out, n, i, 6);  field_shift_store<33>(x, out, n, i, 7);  field_shift_store<48>(x, out, n, i, 8);
    field_shift_store<63>(x, out, n, i, 9);  field_shift_store<64>(x, out, n, i, 10); field_shift_store<65>(x, out, n, i, 11);
    field_shift_store<72>(x, out, n, i, 12); field_shift_store<80>(x, out, n, i, 13); field_shift_store<84>(x, out, n, i, 14);
    field_shift_store<90>(x, out, n, i, 15); field_shift_store<95>(x, out, n, i, 16); field_shift_store<96>(x, out, n, i, 17);
}

// extension-field KAT kernel: out[0] = a * b, out[1] = a^-1, out[2] = frobenius(a), out[3] = a.mul_base(b[0]),
// out[4] = a + b, out[5] = a - b, each [n][D] (ExtensibleField<2>/<3> for BaseElement, math/src/field/f64/mod.rs:401-499)
template <int D>
__global__ void ext_ops_kernel(const u64* a, const u64* b, size_t n, u64* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    GlExt<D> x, y;
#pragma unroll
    for (int q = 0; q < D; q++) { x.v[q] = a[i * D + q]; y.v[q] = b[i * D + q]; }
    const GlExt<D> r[6] = {ext_mul(x, y), ext_inv(x), ext_frobenius(x), ext_mul_base(x, y.v[0]), ext_add(x, y), ext_sub(x, y)};
#pragma unroll
    for (int k = 0; k < 6; k++)
#pragma unroll
        for (int q = 0; q < D; q++) out[((size_t)k * n + i) * D + q] = r[k].v[q];
}

template <int K>
static u64 m2e(u64 x) { return gl_mul_2exp<K>(x); }

extern "C" {

const char* wf_version(void) { return "winterfell_b200 0.1 (sm_100a)"; }

int wf_ctx_create(wf_ctx** out, int device, void* stream) {
    if (!out) return WF_ERR_INVALID;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) return WF_ERR_CUDA;  // no CPU fallback
    if (device < 0 || device >= n) return WF_ERR_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return WF_ERR_CUDA;
    wf_ctx* ctx = new wf_ctx();
    ctx->device = device;
    ctx->st = (cudaStream_t)stream;
    ctx->launches = 0;
    ctx->pinned = nullptr;
    ctx->pinned_bytes = 0;
    ctx->profiling = false;
    *out = ctx;
    return WF_OK;
}
void wf_ctx_destroy(wf_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->st);
    for (auto& kv : ctx->pool) cudaFree(kv.second);
    for (auto& kv : ctx->live) cudaFree(kv.first);
    for (auto& kv : ctx->tw) cudaFree(kv.second);
    for (auto& kv : ctx->lde_tabs) { cudaFree(kv.second.pre); if (kv.second.pow7) cudaFree(kv.second.pow7); }
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    for (auto& kv : ctx->ipc_opened) cudaIpcCloseMemHandle(kv.second);   // other ranks' buffers mapped by sharded proofs
    for (auto& kv : ctx->jit_cache) if (kv.second.first) cudaLibraryUnload((cudaLibrary_t)kv.second.first);
    for (int i = 0; i < 4; i++) if (ctx->push_st[i]) { cudaStreamSynchronize(ctx->push_st[i]); cudaStreamDestroy(ctx->push_st[i]); }
    for (int i = 0; i < 16; i++) if (ctx->push_ev[i]) cudaEventDestroy(ctx->push_ev[i]);
    if (ctx->copy_st) {
        cudaStreamSynchronize(ctx->copy_st);
        for (int i = 0; i < 2; i++) { cudaEventDestroy(ctx->ev_up[i]); cudaEventDestroy(ctx->ev_used[i]); }
        cudaEventDestroy(ctx->ev_start);
        cudaStreamDestroy(ctx->copy_st);
    }
    delete ctx;
}
int wf_ctx_set_profiling(wf_ctx* ctx, int on) {
    if (!ctx) return WF_ERR_INVALID;
    ctx->profiling = on != 0;
    for (auto& m : ctx->marks) cudaEventDestroy(m.second);
    ctx->marks.clear();
    return WF_OK;
}
int wf_ctx_stage_times(wf_ctx* ctx, char* names, size_t names_cap, float* ms, size_t* count) {
    if (!ctx || !names || !ms || !count) return WF_ERR_INVALID;
    CK(cudaStreamSynchronize(ctx->st));
    size_t n = ctx->marks.size() > 0 ? ctx->marks.size() - 1 : 0, used = 0;
    if (n > *count) n = *count;
    names[0] = 0;
    for (size_t i = 0; i < n; i++) {
        CK(cudaEventElapsedTime(&ms[i], ctx->marks[i].second, ctx->marks[i + 1].second));
        const std::string& nm = ctx->marks[i + 1].first;
        if (used + nm.size() + 2 < names_cap) { memcpy(names + used, nm.c_str(), nm.size()); used += nm.size(); names[used++] = ','; names[used] = 0; }
    }
    *count = n;
    for (auto& m : ctx->marks) cudaEventDestroy(m.second);
    ctx->marks.clear();
    return WF_OK;
}
const char* wf_last_error(const wf_ctx* ctx) { return ctx ? ctx->err.c_str() : "no context (is a CUDA device present?)"; }
int wf_ctx_sync(wf_ctx* ctx) { wf_use_device(ctx); CK(cudaStreamSynchronize(ctx->st)); return WF_OK; }
uint64_t wf_ctx_launch_count(const wf_ctx* ctx) { return ctx->launches; }
int wf_ctx_mem_stats(const wf_ctx* ctx, uint64_t* live_buffers, uint64_t* live_bytes, uint64_t* pooled_bytes) {
    if (!ctx) return WF_ERR_INVALID;
    uint64_t lb = 0, pb = 0;
    for (auto& kv : ctx->live) lb += kv.second;
    for (auto& kv : ctx->pool) pb += kv.first;
    if (live_buffers) *live_buffers = ctx->live.size();
    if (live_bytes) *live_bytes = lb;
    if (pooled_bytes) *pooled_bytes = pb;
    return WF_OK;
}

// ---- matrices -----------------------------------------------------------------------------------
int wf_mat_from_device_columns(wf_ctx* ctx, const uint64_t* d_cols, uint32_t ncols, size_t nrows, wf_mat** out) {
    if (!ctx || !d_cols || !out || ncols == 0 || nrows == 0) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    wf_mat* m;
    CKI(wf_mat_alloc(ctx, nrows, ncols, &m));
    CK(layout_cols_to_seg(d_cols, nrows, 1, 0, m->m, ctx->st));
    ctx->launches++;
    *out = m;
    return WF_OK;
}

// `nbase` base columns from host columns of d-component elements: base column q = component (q0 + q) % d of host column
// (q0 + q) / d, so the block may start and end inside an element
static int mat_from_host_elements(wf_ctx* ctx, const uint64_t* const* cols, uint32_t nbase, size_t nrows, int d, u32 q0, int mont,
                                  wf_mat** out) {
    // stage: host column j (nrows * d words, elements interleaved) -> device [ne][nrows*d]
    const size_t col_words = nrows * d;
    const u32 ne = (q0 + nbase - 1) / d + 1;
    void* stage;
    CKI(wf_dev_alloc(ctx, (size_t)ne * col_words * 8, &stage));
    for (uint32_t j = 0; j < ne; j++)
        CK(cudaMemcpyAsync((u64*)stage + (size_t)j * col_words, cols[j], col_words * 8, cudaMemcpyHostToDevice, ctx->st));
    wf_mat* m;
    int r = wf_mat_alloc(ctx, nrows, nbase, &m);
    if (r != WF_OK) { wf_dev_free(ctx, stage); return r; }
    // element (row, q) at stage[((q0+q)/d)*col_words + row*d + (q0+q)%d]
    CK(layout_cols_to_seg((u64*)stage, nrows, d, mont, m->m, ctx->st, (int)q0));
    ctx->launches++;
    wf_dev_free(ctx, stage);
    *out = m;
    return WF_OK;
}
int wf_mat_from_host_columns(wf_ctx* ctx, const uint64_t* const* cols, uint32_t ncols, size_t nrows, int ext_degree,
                             int mont, wf_mat** out) {
    if (!ctx || !cols || !out || ncols == 0 || nrows == 0 || ext_degree < 1 || ext_degree > 3)
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    return mat_from_host_elements(ctx, cols, ncols * ext_degree, nrows, ext_degree, 0, mont, out);
}
// Non-owning handle over caller-allocated device memory already in the segment layout of a rows x cols
// matrix (segment width as for any matrix of `cols` columns: 8 for cols >= 8). wf_mat_free releases the
// handle only. Lets an LDE be written into, or a commitment be taken from, a buffer that a collective
// sends or receives (winterfell_b200/dist.py).
int wf_mat_wrap_device(wf_ctx* ctx, uint64_t* d_segments, size_t rows, uint32_t cols, wf_mat** out) {
    if (!ctx || !d_segments || !out || rows == 0 || cols == 0) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    wf_mat* m = new wf_mat();
    m->m.rows = rows;
    m->m.cols = cols;
    m->m.W = seg_width_for(cols);
    m->m.seg_stride = rows * m->m.W;
    m->m.base = d_segments;  // not in ctx->live: wf_dev_free ignores it
    *out = m;
    return WF_OK;
}
int wf_mat_select_columns(wf_ctx* ctx, const wf_mat* m, uint32_t first, uint32_t count, wf_mat** out) {
    if (!ctx || !m || !out || count == 0 || first + count > m->m.cols) return wf_fail(ctx, WF_ERR_INVALID, "bad column range");
    wf_mat* o;
    CKI(wf_mat_alloc(ctx, m->m.rows, count, &o));
    CK(layout_select_cols(m->m, first, o->m, ctx->st));
    ctx->launches++;
    *out = o;
    return WF_OK;
}
int wf_mat_free(wf_ctx* ctx, wf_mat* m) {
    if (!m) return WF_OK;
    wf_dev_free(ctx, m->m.base);
    delete m;
    return WF_OK;
}
size_t wf_mat_rows(const wf_mat* m) { return m->m.rows; }
uint32_t wf_mat_cols(const wf_mat* m) { return m->m.cols; }

static int mat_export(wf_ctx* ctx, const wf_mat* m, uint64_t* dst, int to_host, int mont, int row_major) {
    if (!ctx || !m || !dst) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    size_t words = m->m.rows * m->m.cols;
    u64* d = dst;
    void* tmp = nullptr;
    if (to_host) { CKI(wf_dev_alloc(ctx, words * 8, &tmp)); d = (u64*)tmp; }
    CK(layout_seg_to_flat(m->m, d, row_major, mont, ctx->st));
    ctx->launches++;
    if (to_host) {
        CK(cudaMemcpyAsync(dst, d, words * 8, cudaMemcpyDeviceToHost, ctx->st));
        CK(cudaStreamSynchronize(ctx->st));
        wf_dev_free(ctx, tmp);
    }
    return WF_OK;
}
int wf_mat_to_columns(wf_ctx* ctx, const wf_mat* m, uint64_t* dst, int to_host, int mont) { return mat_export(ctx, m, dst, to_host, mont, 0); }
int wf_mat_to_rows(wf_ctx* ctx, const wf_mat* m, uint64_t* dst, int to_host, int mont) { return mat_export(ctx, m, dst, to_host, mont, 1); }

int wf_mat_read_rows(wf_ctx* ctx, const wf_mat* m, const uint64_t* positions, size_t k, uint64_t* dst, int mont) {
    if (!ctx || !m || !positions || !dst) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    if (k == 0) return WF_OK;
    for (size_t i = 0; i < k; i++)
        if (positions[i] >= m->m.rows) return wf_fail(ctx, WF_ERR_INVALID, "row %llu out of range", (unsigned long long)positions[i]);
    void *dpos, *dout;
    CKI(wf_dev_alloc(ctx, k * 8, &dpos));
    CKI(wf_dev_alloc(ctx, k * m->m.cols * 8, &dout));
    CK(cudaMemcpyAsync(dpos, positions, k * 8, cudaMemcpyHostToDevice, ctx->st));
    CK(layout_gather_rows(m->m, (const u64*)dpos, k, (u64*)dout, mont, ctx->st));
    ctx->launches++;
    CK(cudaMemcpyAsync(dst, dout, k * m->m.cols * 8, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    wf_dev_free(ctx, dpos);
    wf_dev_free(ctx, dout);
    return WF_OK;
}

static int log2_exact(size_t n, u32* out) {
    if (n == 0 || (n & (n - 1))) return -1;
    u32 l = 0;
    while (((size_t)1 << l) < n) l++;
    *out = l;
    return 0;
}

static int mat_transform(wf_ctx* ctx, const wf_mat* in, int inverse, wf_mat** out) {
    if (!ctx || !in || !out) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    u32 log_n;
    if (log2_exact(in->m.rows, &log_n) || log_n < 1) return wf_fail(ctx, WF_ERR_INVALID, "rows must be a power of two >= 2");
    wf_mat* o;
    CKI(wf_mat_alloc(ctx, in->m.rows, in->m.cols, &o));
    SegMatrix tmp = in->m;
    void* tp = nullptr;
    if (log_n > NTT_MAX_LOGS) {
        int r = wf_dev_alloc(ctx, in->m.words() * 8, &tp);
        if (r != WF_OK) { wf_mat_free(ctx, o); return r; }
        tmp.base = (u64*)tp;
    }
    int r = run_ntt(ctx, in->m, o->m, tp ? &tmp : nullptr, log_n, inverse);
    wf_dev_free(ctx, tp);
    if (r != WF_OK) { wf_mat_free(ctx, o); return r; }
    *out = o;
    return WF_OK;
}
int wf_mat_interpolate(wf_ctx* ctx, const wf_mat* evals, wf_mat** polys) { return mat_transform(ctx, evals, 1, polys); }
int wf_mat_evaluate(wf_ctx* ctx, const wf_mat* polys, wf_mat** evals) { return mat_transform(ctx, polys, 0, evals); }

int wf_mat_lde(wf_ctx* ctx, const wf_mat* polys, uint32_t log_blowup, wf_mat** lde) {
    if (!ctx || !polys || !lde) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    u32 log_n;
    if (log2_exact(polys->m.rows, &log_n) || log_n < 1) return wf_fail(ctx, WF_ERR_INVALID, "rows must be a power of two >= 2");
    if (log_blowup > 7 || log_n + log_blowup > 32) return wf_fail(ctx, WF_ERR_INVALID, "bad blowup");
    wf_mat* o;
    CKI(wf_mat_alloc(ctx, polys->m.rows << log_blowup, polys->m.cols, &o));
    int r = run_lde(ctx, polys->m, o->m, log_n, log_blowup);
    if (r != WF_OK) { wf_mat_free(ctx, o); return r; }
    *lde = o;
    return WF_OK;
}

int wf_mat_lde_into(wf_ctx* ctx, const wf_mat* polys, uint32_t log_blowup, wf_mat* lde) {
    if (!ctx || !polys || !lde) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    u32 log_n;
    if (log2_exact(polys->m.rows, &log_n) || log_n < 1) return wf_fail(ctx, WF_ERR_INVALID, "rows must be a power of two >= 2");
    if (log_blowup > 7 || lde->m.rows != (polys->m.rows << log_blowup) || lde->m.cols != polys->m.cols || lde->m.W != polys->m.W)
        return wf_fail(ctx, WF_ERR_INVALID, "output matrix does not match the LDE shape");
    return run_lde(ctx, polys->m, lde->m, log_n, log_blowup);
}

// Cosets k0 <= k < k1 of the LDE only, coset-major: row (k - k0) * n + j of `lde` = P(7 w_N^k w_n^j). One rank's share of a
// transform whose columns are too few to shard by column (the composition polynomial of a sharded proof).
int wf_mat_lde_cosets(wf_ctx* ctx, const wf_mat* polys, uint32_t log_blowup, uint32_t k0, uint32_t k1, wf_mat* lde) {
    if (!ctx || !polys || !lde) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    u32 log_n;
    if (log2_exact(polys->m.rows, &log_n) || log_n < 1) return wf_fail(ctx, WF_ERR_INVALID, "rows must be a power of two >= 2");
    if (log_blowup > 7 || k0 >= k1 || k1 > (1u << log_blowup) || lde->m.rows != polys->m.rows * (k1 - k0) || lde->m.cols != polys->m.cols ||
        lde->m.W != polys->m.W || ((k1 - k0) & (k1 - k0 - 1)))
        return wf_fail(ctx, WF_ERR_INVALID, "coset range / output matrix do not match");
    return run_lde(ctx, polys->m, lde->m, log_n, log_blowup, 0, k0, k1, 1, (u32)polys->m.rows);
}

// DefaultTraceLde::new up to the commitment (trace_lde/default/mod.rs:63-100, build_trace_commitment
// :245-282) from HOST columns, with the upload pipelined against the transforms: the columns are cut
// into chunks (whole 8-column segments when there are several, else the two halves of the one segment);
// chunk k+1 crosses PCIe on a copy stream while chunk k is laid out, interpolated and extended on the
// compute stream. Columns are independent, so the result equals from_host_columns -> interpolate -> lde.
int wf_trace_lde_from_host(wf_ctx* ctx, const uint64_t* const* cols, uint32_t ncols, size_t nrows, int mont, uint32_t log_blowup,
                           wf_mat** polys_out, wf_mat** lde_out) {
    return wf_trace_lde_cosetwise(ctx, cols, nullptr, ncols, nrows, mont, log_blowup, polys_out, lde_out, false, nullptr, nullptr, 1, 0);
}
// The same pipeline with two knobs for the sharded prover (prover.cu): coset_major = the LDE is written coset-major
// (row k * n + j = P(7 w_N^k w_n^j); *lde_out must then be preallocated, with the natural segment width of `ncols` columns or
// a wider one: a rank of a sharded proof writes its columns at the segment width of the whole trace) and after_coset(k)
// is called once coset k of ALL columns has been enqueued on the ctx stream — the caller starts that coset's exchange there.
// d_cols != NULL: the columns are already on the device (column-major), no upload stage.
// d > 1 (host columns only): cols are columns of d-component elements ([nrows][d] words each, as wf_mat_from_host_columns) and
// the ncols BASE columns transformed are components q0, q0 + 1, ... of them: base column i = component (q0 + i) % d of host
// column (q0 + i) / d (a rank's block of an auxiliary segment, which may start and end inside an element).
int wf_trace_lde_cosetwise(wf_ctx* ctx, const uint64_t* const* cols, const uint64_t* d_cols, uint32_t ncols, size_t nrows, int mont,
                           uint32_t log_blowup, wf_mat** polys_out, wf_mat** lde_out, bool coset_major,
                           const std::function<int(u32)>* after_coset, const LdeScatter* scatter, int d, uint32_t q0) {
    if (!ctx || (!cols && !d_cols) || !polys_out || (!lde_out && !scatter) || ncols == 0 || d < 1 || d > 3 || q0 >= (u32)d ||
        (d_cols && d != 1))
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    u32 log_n;
    if (log2_exact(nrows, &log_n) || log_n < 1) return wf_fail(ctx, WF_ERR_INVALID, "rows must be a power of two >= 2");
    if (log_blowup > 7 || log_n + log_blowup > 32) return wf_fail(ctx, WF_ERR_INVALID, "bad blowup");
    const int Wn = seg_width_for(ncols);
    const bool prealloc = coset_major && !scatter;
    if (prealloc && (!lde_out || !*lde_out || (*lde_out)->m.rows != (nrows << log_blowup) || (*lde_out)->m.W < Wn || (*lde_out)->m.cols != ncols))
        return wf_fail(ctx, WF_ERR_INVALID, "coset-major output must be preallocated");
    const int Wout = prealloc ? (*lde_out)->m.W : Wn;
    const u32 nseg_out = (ncols + Wout - 1) / Wout;
    const u32 nb = 1u << log_blowup;
    // cosets of one column chunk: all at once, or one by one with the callback when this is the last chunk
    auto extend = [&](const SegMatrix& pv, SegMatrix& ov, u32 out_col0, bool last, u32 out_seg) -> int {
        if (scatter) {  // every coset straight into the owners' row shards (natural order there); `ov` is not written
            LdeScatter s2 = *scatter;
            s2.seg0 += out_seg;
            return run_lde(ctx, pv, ov, log_n, log_blowup, out_col0, 0, nb, 0, 1, &s2);
        }
        if (!after_coset || !last) {
            if (!coset_major) return run_lde(ctx, pv, ov, log_n, log_blowup, out_col0);
            return run_lde(ctx, pv, ov, log_n, log_blowup, out_col0, 0, nb, 1, (u32)nrows);
        }
        for (u32 k = 0; k < nb; k++) {   // run_lde places its FIRST coset at the view's origin: shift the view to coset k's rows
            SegMatrix ok = ov;
            ok.base += (coset_major ? (size_t)k * nrows : (size_t)k) * ov.W;
            if (coset_major) CKI(run_lde(ctx, pv, ok, log_n, log_blowup, out_col0, k, k + 1, 1, (u32)nrows));
            else CKI(run_lde(ctx, pv, ok, log_n, log_blowup, out_col0, k, k + 1, nb, 1));
            CKI((*after_coset)(k));
        }
        return WF_OK;
    };
    int Wc = nseg_out >= 2 ? Wout : (Wn >= 4 ? Wn / 2 : 0);
    // (measured on cfg2, 8 columns: halves 7.03 ms e2e, quarters 7.35 — W = 2 tiles cost more than the
    // shorter upload head saves — no pipeline 7.36)
    if (d_cols || Wc == 0 || log_n < 12) {  // resident columns, or too narrow / too small to be worth a pipeline
        wf_mat* tr;
        if (d_cols) CKI(wf_mat_from_device_columns(ctx, d_cols, ncols, nrows, &tr));
        else CKI(mat_from_host_elements(ctx, cols, ncols, nrows, d, q0, mont, &tr));
        int r = wf_mat_interpolate(ctx, tr, polys_out);
        wf_mat_free(ctx, tr);
        if (r != WF_OK) return r;
        if (scatter) { SegMatrix none = (*polys_out)->m; none.W = Wout; return extend((*polys_out)->m, none, 0, true, 0); }
        if (!coset_major && !after_coset) return wf_mat_lde(ctx, *polys_out, log_blowup, lde_out);
        if (!coset_major) CKI(wf_mat_alloc(ctx, nrows << log_blowup, ncols, lde_out));
        return extend((*polys_out)->m, (*lde_out)->m, 0, true, 0);
    }
    if (!ctx->copy_st) {
        CK(cudaStreamCreateWithFlags(&ctx->copy_st, cudaStreamNonBlocking));
        for (int i = 0; i < 2; i++) {
            CK(cudaEventCreateWithFlags(&ctx->ev_up[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->ev_used[i], cudaEventDisableTiming));
        }
        CK(cudaEventCreateWithFlags(&ctx->ev_start, cudaEventDisableTiming));
    }
    const u32 nchunks = (ncols + Wc - 1) / Wc;
    wf_mat *polys = nullptr, *lde = nullptr, *tr = nullptr;
    void* stage[2] = {nullptr, nullptr};
    void* tmp = nullptr;
    auto release = [&](bool results_too) {  // buffers return to the pool in stream order
        wf_mat_free(ctx, tr);
        for (int i = 0; i < 2; i++) wf_dev_free(ctx, stage[i]);
        wf_dev_free(ctx, tmp);
        if (results_too) { wf_mat_free(ctx, polys); if (!coset_major && !scatter) wf_mat_free(ctx, lde); }
    };
    auto body = [&]() -> int {
        CKI(wf_mat_alloc_w(ctx, nrows, ncols, Wc, &polys));
        if (coset_major || scatter) lde = lde_out ? *lde_out : nullptr;
        else CKI(wf_mat_alloc(ctx, nrows << log_blowup, ncols, &lde));
        CKI(wf_mat_alloc_w(ctx, nrows, Wc, Wc, &tr));                       // one chunk of trace values (reused)
        // a chunk of Wc base columns touches at most ne_max host columns of d components: each is uploaded whole
        const size_t ne_max = (size_t)(Wc + d - 2) / d + 1;
        for (int i = 0; i < 2; i++) CKI(wf_dev_alloc(ctx, ne_max * d * nrows * 8, &stage[i]));
        CKI(wf_dev_alloc(ctx, (size_t)Wc * nrows * 8, &tmp));               // two-pass scratch
        if (lde && lde->m.W > (int)ncols) CK(cudaMemsetAsync(lde->m.base, 0, lde->m.words() * 8, ctx->st));  // padding columns
        // the copy stream must not write pool buffers before their previous users on the compute stream are done
        CK(cudaEventRecord(ctx->ev_start, ctx->st));
        CK(cudaStreamWaitEvent(ctx->copy_st, ctx->ev_start, 0));
        for (u32 k = 0; k < nchunks; k++) {
            const u32 c0 = k * Wc, cw = std::min<u32>(Wc, ncols - c0);
            const int sb = k & 1;
            if (k >= 2) CK(cudaStreamWaitEvent(ctx->copy_st, ctx->ev_used[sb], 0));
            const u32 e0 = (q0 + c0) / d, e1 = (q0 + c0 + cw - 1) / d;   // host columns holding base columns [c0, c0 + cw)
            for (u32 e = e0; e <= e1; e++)
                CK(cudaMemcpyAsync((u64*)stage[sb] + (size_t)(e - e0) * d * nrows, cols[e], (size_t)d * nrows * 8, cudaMemcpyHostToDevice,
                                   ctx->copy_st));
            CK(cudaEventRecord(ctx->ev_up[sb], ctx->copy_st));
            CK(cudaStreamWaitEvent(ctx->st, ctx->ev_up[sb], 0));
            SegMatrix trv = tr->m;
            trv.cols = cw;
            CK(layout_cols_to_seg((const u64*)stage[sb], nrows, d, mont, trv, ctx->st, (int)((q0 + c0) % d)));
            CK(cudaEventRecord(ctx->ev_used[sb], ctx->st));
            ctx->launches++;
            SegMatrix pv = polys->m;                                          // segment k of the W = Wc polys matrix
            pv.base = polys->m.base + (size_t)k * polys->m.seg_stride;
            pv.cols = cw;
            SegMatrix tv = trv;
            tv.base = (u64*)tmp;
            CKI(run_ntt(ctx, trv, pv, &tv, log_n, 1));
            SegMatrix ov = pv;                                                // out segment holding columns c0..
            ov.W = Wout;
            if (lde) { ov = lde->m; ov.base = lde->m.base + (size_t)(c0 / Wout) * lde->m.seg_stride; }
            ov.cols = cw;
            CKI(extend(pv, ov, c0 % Wout, k + 1 == nchunks, c0 / Wout));
        }
        return WF_OK;
    };
    int rc = body();
    if (rc != WF_OK) {
        cudaStreamSynchronize(ctx->copy_st);  // no copy may still target a buffer that goes back to the pool
        release(true);
        return rc;
    }
    release(false);
    *polys_out = polys;
    if (lde_out) *lde_out = lde;
    return WF_OK;
}

int wf_mat_interpolate_with_offset(wf_ctx* ctx, const wf_mat* evals, uint64_t domain_offset, wf_mat** polys) {
    // fft/serial.rs:84-101: iNTT, then coefficient i *= offset^-i (the 1/n is already in the iNTT)
    if (domain_offset == 0 || domain_offset >= GL_P) return wf_fail(ctx, WF_ERR_INVALID, "bad domain offset");
    wf_mat* p;
    CKI(mat_transform(ctx, evals, 1, &p));
    CK(layout_scale_rows_by_powers(p->m, gl_inv(domain_offset), ctx->st));
    ctx->launches++;
    *polys = p;
    return WF_OK;
}

// ---- commitments --------------------------------------------------------------------------------
static int tree_alloc(wf_ctx* ctx, int hash_id, size_t nleaves, wf_tree** out) {
    if (nleaves < 2 || (nleaves & (nleaves - 1))) return wf_fail(ctx, WF_ERR_INVALID, "number of leaves must be a power of two >= 2");
    wf_tree* t = new wf_tree();
    t->hash_id = hash_id;
    t->nleaves = nleaves;
    void *a, *b;
    int r = wf_dev_alloc(ctx, nleaves * 32, &a);
    if (r != WF_OK) { delete t; return r; }
    r = wf_dev_alloc(ctx, nleaves * 32, &b);
    if (r != WF_OK) { wf_dev_free(ctx, a); delete t; return r; }
    t->leaves = (u64*)a;
    t->nodes = (u64*)b;
    *out = t;
    return WF_OK;
}
static u32 merkle_launches(size_t nleaves) {
    u32 l = 0;
    size_t m = nleaves / 2;
    while (m > (1u << 13)) { l++; m >>= 1; }
    for (;;) {
        l++;
        if (m <= 256) break;
        m = (m >> 8) >> 1;
        if (m == 0) break;
    }
    return l;
}
int wf_commit_rows_partitioned(wf_ctx* ctx, int hash_id, const wf_mat* m, uint32_t partition_size, wf_tree** out) {
    if (!ctx || !m || !out) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    if (!WF_HASH_IS_KNOWN(hash_id)) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "unknown hash %d", hash_id);
    if (partition_size != 0 && partition_size != m->m.cols && (m->m.cols + partition_size - 1) / partition_size > 16)
        return wf_fail(ctx, WF_ERR_INVALID, "more than 16 partitions");
    wf_tree* t;
    CKI(tree_alloc(ctx, hash_id, m->m.rows, &t));
    CK(commit_hash_rows(hash_id, m->m, t->leaves, ctx->st, partition_size));
    CK(commit_merkle_nodes(hash_id, t->leaves, t->nleaves, t->nodes, ctx->st));
    ctx->launches += 1 + merkle_launches(t->nleaves);
    *out = t;
    return WF_OK;
}
int wf_commit_rows(wf_ctx* ctx, int hash_id, const wf_mat* m, wf_tree** out) {
    if (!ctx || !m || !out) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    if (!WF_HASH_IS_KNOWN(hash_id)) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "unknown hash %d", hash_id);
    wf_tree* t;
    CKI(tree_alloc(ctx, hash_id, m->m.rows, &t));
    CK(commit_hash_rows(hash_id, m->m, t->leaves, ctx->st));
    CK(commit_merkle_nodes(hash_id, t->leaves, t->nleaves, t->nodes, ctx->st));
    ctx->launches += 1 + merkle_launches(t->nleaves);
    *out = t;
    return WF_OK;
}
int wf_tree_from_leaves(wf_ctx* ctx, int hash_id, const uint8_t* leaves, size_t nleaves, int on_device, wf_tree** out) {
    if (!ctx || !leaves || !out) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    wf_tree* t;
    CKI(tree_alloc(ctx, hash_id, nleaves, &t));
    CK(cudaMemcpyAsync(t->leaves, leaves, nleaves * 32, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->st));
    CK(commit_merkle_nodes(hash_id, t->leaves, nleaves, t->nodes, ctx->st));
    ctx->launches += merkle_launches(nleaves);
    if (!on_device) CK(cudaStreamSynchronize(ctx->st));
    *out = t;
    return WF_OK;
}
int wf_tree_free(wf_ctx* ctx, wf_tree* t) {
    if (!t) return WF_OK;
    wf_dev_free(ctx, t->leaves);
    wf_dev_free(ctx, t->nodes);
    delete t;
    return WF_OK;
}
size_t wf_tree_num_leaves(const wf_tree* t) { return t->nleaves; }
int wf_tree_root(wf_ctx* ctx, const wf_tree* t, uint8_t root[32]) {
    if (!ctx || !t || !root) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    CK(cudaMemcpyAsync(root, t->nodes + 4, 32, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    return WF_OK;
}
int wf_tree_to_host(wf_ctx* ctx, const wf_tree* t, uint8_t* leaves, uint8_t* nodes) {
    if (!ctx || !t) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    if (leaves) CK(cudaMemcpyAsync(leaves, t->leaves, t->nleaves * 32, cudaMemcpyDeviceToHost, ctx->st));
    if (nodes) CK(cudaMemcpyAsync(nodes, t->nodes, t->nleaves * 32, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    return WF_OK;
}

// MerkleTree::prove_batch (crypto/src/merkle/mod.rs:217-272) on a device tree: the walk decides
// which digests are needed (host, indices only), one gather kernel fetches them.
}  // extern "C"

// ---- batched openings ------------------------------------------------------------------------------
// MerkleTree::prove_batch (crypto/src/merkle/mod.rs:217-272) split into a host-only PLAN (which
// digests are needed: pure index arithmetic) and a FINISH step (serialisation, proofs.rs:390-401), so
// that all the gathers of a proof (trace rows, constraint rows, every FRI layer) share ONE index
// upload, ONE result download and ONE stream synchronisation (GatherBatch).
int wf_open_plan(wf_ctx* ctx, size_t n, const uint64_t* positions, size_t k, OpenPlan& pl) {
    pl.depth = 0;
    while (((size_t)1 << pl.depth) < n) pl.depth++;
    if (k == 0) return wf_fail(ctx, WF_ERR_INVALID, "no positions");
    std::map<size_t, size_t> index_map;
    for (size_t i = 0; i < k; i++) {
        if (positions[i] >= n) return wf_fail(ctx, WF_ERR_INVALID, "leaf index out of bounds");
        index_map[positions[i]] = i;
    }
    if (index_map.size() != k) return wf_fail(ctx, WF_ERR_INVALID, "duplicate leaf index");
    std::set<size_t> norm;
    for (size_t i = 0; i < k; i++) norm.insert(positions[i] & ~(size_t)1);
    // gather list: entries < n address nodes[], entries >= n address leaves[entry - n]
    pl.want.clear();
    pl.vec_slots.clear();
    pl.leaf_slot.assign(k, 0);
    std::vector<size_t> next;
    for (size_t index : norm) {
        std::vector<size_t> slots;
        for (size_t i = index; i < index + 2; i++) {
            auto it = index_map.find(i);
            pl.want.push_back(n + i);
            if (it != index_map.end()) pl.leaf_slot[it->second] = pl.want.size() - 1;
            else slots.push_back(pl.want.size() - 1);
        }
        pl.vec_slots.push_back(slots);
        next.push_back((index + n) >> 1);
    }
    for (u32 lvl = 1; lvl < pl.depth; lvl++) {
        std::vector<size_t> idx = next;
        next.clear();
        size_t i = 0;
        while (i < idx.size()) {
            size_t sib = idx[i] ^ 1;
            if (i + 1 < idx.size() && idx[i + 1] == sib) i += 1;
            else { pl.want.push_back(sib); pl.vec_slots[i].push_back(pl.want.size() - 1); }
            next.push_back(sib >> 1);
            i += 1;
        }
    }
    return WF_OK;
}
void wf_open_finish(const OpenPlan& pl, const uint8_t* got, uint8_t* leaves_out, ByteVec& proof) {
    if (leaves_out)
        for (size_t i = 0; i < pl.leaf_slot.size(); i++) memcpy(leaves_out + i * 32, got + pl.leaf_slot[i] * 32, 32);
    proof.u8_((u8)pl.depth);  // BatchMerkleProof::write_into (proofs.rs:390-401)
    proof.usize(pl.vec_slots.size());
    for (auto& v : pl.vec_slots) {
        proof.usize(v.size());
        for (size_t s : v) proof.bytes(got + s * 32, pl.digest_bytes);   // 32-byte slots, ByteDigest<N> writes N bytes
    }
}

static int pinned_reserve(wf_ctx* ctx, size_t bytes) {
    if (ctx->pinned_bytes >= bytes) return WF_OK;
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    ctx->pinned = nullptr;
    ctx->pinned_bytes = 0;
    bytes = std::max(bytes * 2, (size_t)1 << 20);
    CK(cudaMallocHost(&ctx->pinned, bytes));
    ctx->pinned_bytes = bytes;
    return WF_OK;
}

size_t GatherBatch::add_rows(const SegMatrix& m, const std::vector<u64>& pos) {
    rows.push_back({m, pos, 0, 0});
    return rows.size() - 1;
}
int GatherBatch::add_opening(wf_ctx* ctx, const wf_tree* t, const std::vector<u64>& pos, size_t* id) {
    digs.emplace_back();
    digs.back().t = t;
    CKI(wf_open_plan(ctx, t->nleaves, pos.data(), pos.size(), digs.back().plan));
    digs.back().plan.digest_bytes = WF_DIGEST_BYTES(t->hash_id);
    digs.back().idx = digs.back().plan.want;
    *id = digs.size() - 1;
    return WF_OK;
}
int GatherBatch::add_opening_sharded(wf_ctx* ctx, const wf_tree* t, size_t n_global, int world, int rank, const std::vector<u64>& pos,
                                     size_t* id, std::vector<std::pair<size_t, u64>>* top_slots) {
    digs.emplace_back();
    DigJob& j = digs.back();
    j.t = t;
    CKI(wf_open_plan(ctx, n_global, pos.data(), pos.size(), j.plan));
    if (t) j.plan.digest_bytes = WF_DIGEST_BYTES(t->hash_id);   // (the host-only planning export passes no tree)
    const size_t n_local = n_global / (size_t)world;
    u32 log_w = 0;
    while ((1 << log_w) < world) log_w++;
    j.idx.assign(j.plan.want.size(), ~(u64)0);
    for (size_t s = 0; s < j.plan.want.size(); s++) {
        const u64 e = j.plan.want[s];
        if (e >= n_global) {  // leaf digest e - n
            const u64 leaf = e - n_global;
            if ((int)(leaf / n_local) == rank) j.idx[s] = n_local + leaf % n_local;
        } else if (e < (u64)world) {  // node of the top log2(world) levels: held on the host by every rank
            if (top_slots) top_slots->push_back({s, e});
        } else {
            u32 depth = 63 - (u32)__builtin_clzll(e);        // node e sits at depth `depth` (root = depth 0)
            const u32 rel = depth - log_w;                     // depth inside its subtree
            const u64 owner = (e >> rel) - (u64)world;
            if ((int)owner == rank) j.idx[s] = ((u64)1 << rel) | (e & (((u64)1 << rel) - 1));
        }
    }
    *id = digs.size() - 1;
    return WF_OK;
}
int GatherBatch::run(wf_ctx* ctx) {
    wf_use_device(ctx);
    size_t idx_words = 0, out_words = 0;
    for (auto& j : rows) { j.idx_off = idx_words; j.out_off = out_words; idx_words += j.pos.size(); out_words += j.pos.size() * j.m.cols; }
    for (auto& j : digs) { j.idx_off = idx_words; j.out_off = out_words; idx_words += j.plan.want.size(); out_words += j.plan.want.size() * 4; }
    if (idx_words == 0) return WF_OK;
    CKI(pinned_reserve(ctx, (idx_words + out_words) * 8));
    u64* h_idx = (u64*)ctx->pinned;
    u64* h_out = h_idx + idx_words;
    for (auto& j : rows) memcpy(h_idx + j.idx_off, j.pos.data(), j.pos.size() * 8);
    for (auto& j : digs) memcpy(h_idx + j.idx_off, j.idx.data(), j.idx.size() * 8);
    void *d_idx, *d_out;
    CKI(wf_dev_alloc(ctx, idx_words * 8, &d_idx));
    CKI(wf_dev_alloc(ctx, out_words * 8, &d_out));
    CK(cudaMemcpyAsync(d_idx, h_idx, idx_words * 8, cudaMemcpyHostToDevice, ctx->st));
    for (auto& j : rows) {
        CK(layout_gather_rows(j.m, (const u64*)d_idx + j.idx_off, j.pos.size(), (u64*)d_out + j.out_off, 0, ctx->st));
        ctx->launches++;
    }
    for (auto& j : digs) {
        CK(layout_gather_digests(j.t->nodes, j.t->leaves, j.t->nleaves, (const u64*)d_idx + j.idx_off, j.plan.want.size(),
                                 (u64*)d_out + j.out_off, ctx->st));
        ctx->launches++;
    }
    if (comm && comm->world > 1 && comm->all_reduce_sum(comm->user, d_out, out_words) != 0)
        return wf_fail(ctx, WF_ERR_STATE, "all_reduce_sum callback failed");
    CK(cudaMemcpyAsync(h_out, d_out, out_words * 8, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    wf_dev_free(ctx, d_idx);
    wf_dev_free(ctx, d_out);
    result = h_out;
    return WF_OK;
}

int wf_tree_open_many_bytes(wf_ctx* ctx, const wf_tree* t, const uint64_t* positions, size_t k, uint8_t* leaves_out,
                            ByteVec& proof) {
    GatherBatch gb;
    size_t id;
    CKI(gb.add_opening(ctx, t, std::vector<u64>(positions, positions + k), &id));
    CKI(gb.run(ctx));
    wf_open_finish(gb.digs[id].plan, gb.digest_result(id), leaves_out, proof);
    return WF_OK;
}
extern "C" {
int wf_tree_open_many(wf_ctx* ctx, const wf_tree* t, const uint64_t* positions, size_t k, uint8_t* leaves_out,
                      uint8_t* proof, size_t* proof_len) {
    if (!ctx || !t || !positions || !leaves_out || !proof || !proof_len) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    ByteVec bv;
    CKI(wf_tree_open_many_bytes(ctx, t, positions, k, leaves_out, bv));
    if (bv.v.size() > *proof_len) return wf_fail(ctx, WF_ERR_INVALID, "proof buffer too small (%zu needed)", bv.v.size());
    memcpy(proof, bv.v.data(), bv.v.size());
    *proof_len = bv.v.size();
    return WF_OK;
}

}  // extern "C"
// leaf digests of one FRI layer + the Merkle tree over them (fri/src/prover/mod.rs:202-222, :321-336); vals: `len`
// evaluations of degree d, ld words apart, natural order
int wf_fri_layer_tree(wf_ctx* ctx, int hash_id, const u64* vals, size_t len, int d, int ld, int nf, wf_tree** out) {
    const size_t m = len / (size_t)nf;
    wf_tree* t;
    CKI(tree_alloc(ctx, hash_id, m, &t));
    CK(fri_hash_layer(hash_id, vals, len, d, ld, nf, t->leaves, ctx->st));
    CK(commit_merkle_nodes(hash_id, t->leaves, m, t->nodes, ctx->st));
    ctx->launches += 1 + merkle_launches(m);
    *out = t;
    return WF_OK;
}
extern "C" {
// ---- FRI ----------------------------------------------------------------------------------------
int wf_fri_free(wf_ctx* ctx, wf_fri* f) {
    if (!f) return WF_OK;
    for (auto& l : f->layers) { wf_dev_free(ctx, l.evals); wf_tree_free(ctx, l.tree); }
    delete f;
    return WF_OK;
}

}  // extern "C"
// What a commit phase under construction owns: the wf_fri with its finished layers, the tree of the layer in flight and the
// scratch buffers — all of it returns to the pool on every early error return.
struct FriBuild {
    wf_ctx* ctx;
    wf_fri* f;
    wf_tree* t = nullptr;
    DevScratch tmp;
    FriBuild(wf_ctx* c, wf_fri* fr) : ctx(c), f(fr), tmp(c) {}
    ~FriBuild() { if (t) wf_tree_free(ctx, t); if (f) wf_fri_free(ctx, f); }
};
extern "C" {
int wf_fri_build_layers(wf_ctx* ctx, int hash_id, const wf_mat* evals, int d, uint32_t folding, uint32_t rem_max_deg,
                        uint32_t blowup, wf_fri_commit_fn commit, wf_fri_draw_fn draw_alpha, void* user, wf_fri** out) {
    if (!ctx || !evals || !commit || !draw_alpha || !out) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    if (d < 1 || d > 3 || (int)evals->m.cols != d) return wf_fail(ctx, WF_ERR_INVALID, "evaluations must have ext_degree base columns");
    if (folding != 2 && folding != 4 && folding != 8 && folding != 16) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "folding factor %u", folding);
    size_t len = evals->m.rows;
    u32 logL;
    if (log2_exact(len, &logL)) return wf_fail(ctx, WF_ERR_INVALID, "domain size must be a power of two");
    wf_fri* f = new wf_fri();
    FriBuild g(ctx, f);
    f->hash_id = hash_id; f->d = d; f->folding = folding; f->blowup = blowup;
    f->ld = evals->m.W;  // d base columns live in one segment of width W >= d
    const int ld = f->ld;
    // layer 0 evaluations: copy of the segment (the prover keeps its own copy, fri/src/prover/mod.rs:217-221)
    void* cur;
    CKI(g.tmp.alloc(len * ld * 8, &cur));
    CK(cudaMemcpyAsync(cur, evals->m.base, len * ld * 8, cudaMemcpyDeviceToDevice, ctx->st));
    size_t max_rem = (size_t)(rem_max_deg + 1) * blowup;  // fri/src/options.rs:85-93
    while (len > max_rem) {
        size_t m = len / folding;
        wf_tree* t;
        CKI(tree_alloc(ctx, hash_id, m, &t));
        g.t = t;
        CK(fri_hash_layer(hash_id, (u64*)cur, len, d, ld, (int)folding, t->leaves, ctx->st));
        CK(commit_merkle_nodes(hash_id, t->leaves, m, t->nodes, ctx->st));
        ctx->launches += 1 + merkle_launches(m);
        uint8_t root[32];
        CK(cudaMemcpyAsync(root, t->nodes + 4, 32, cudaMemcpyDeviceToHost, ctx->st));
        CK(cudaStreamSynchronize(ctx->st));
        commit(user, root);
        u64 alpha[3] = {0, 0, 0};
        draw_alpha(user, alpha);
        const u64* master;
        u32 ll = 0;
        while (((size_t)1 << ll) < len) ll++;
        CKI(wf_get_twiddles(ctx, ll, &master));
        void* nxt;
        CKI(g.tmp.alloc(m * ld * 8, &nxt));
        if (ld > d) CK(cudaMemsetAsync(nxt, 0, m * ld * 8, ctx->st));
        CK(fri_fold_layer((u64*)cur, len, d, ld, (int)folding, alpha, master, (u64*)nxt, ld, ctx->st));
        ctx->launches++;
        f->layers.push_back(FriLayer{(u64*)g.tmp.keep(cur), len, t});   // the wf_fri owns layer and tree from here
        g.t = nullptr;
        cur = nxt;
        len = m;
    }
    // remainder (fri/src/prover/mod.rs:230-239)
    std::vector<u64> raw(len * ld), v(len * d);
    CK(cudaMemcpyAsync(raw.data(), cur, len * ld * 8, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    g.tmp.free(cur);
    for (size_t i = 0; i < len; i++)
        for (int c = 0; c < d; c++) v[i * d + c] = raw[i * ld + c];
    wf_host_dft(v, len, d, true, GL_GENERATOR);
    size_t rsize = len / blowup;
    f->remainder.resize(rsize * d);
    for (size_t i = 0; i < rsize; i++)
        for (int c = 0; c < d; c++) f->remainder[i * d + c] = v[(rsize - 1 - i) * d + c];
    Digest rc = hh_hash_elements(hash_id, f->remainder.data(), f->remainder.size());
    commit(user, rc.b);
    g.f = nullptr;   // the caller's now
    *out = f;
    return WF_OK;
}

}  // extern "C"
// FriProver::build_layers with the transcript replicated on the device: every layer's leaf hashing, tree,
// coin step (fri_coin_step: reseed with the root, draw alpha) and fold are enqueued back to back, and the
// host synchronises ONCE at the end, replays commit_fri_layer / draw_fri_alpha on its own coin and checks
// that it draws the alphas the device used. (The callback form above pays a device-to-host round trip
// per layer: ~20 us x 8 layers on the 2^23-point codeword of cfg2.)
int wf_fri_build_layers_coin(wf_ctx* ctx, int hash_id, const wf_mat* evals, int d, uint32_t folding, uint32_t rem_max_deg,
                             uint32_t blowup, PublicCoin& coin, std::vector<Digest>& commitments, wf_fri** out) {
    if (!ctx || !evals || !out) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    if (d < 1 || d > 3 || (int)evals->m.cols != d) return wf_fail(ctx, WF_ERR_INVALID, "evaluations must have ext_degree base columns");
    if (folding != 2 && folding != 4 && folding != 8 && folding != 16) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "folding factor %u", folding);
    size_t len = evals->m.rows;
    u32 logL;
    if (log2_exact(len, &logL)) return wf_fail(ctx, WF_ERR_INVALID, "domain size must be a power of two");
    wf_fri* f = new wf_fri();
    FriBuild g(ctx, f);
    f->hash_id = hash_id; f->d = d; f->folding = folding; f->blowup = blowup;
    f->ld = evals->m.W;
    const int ld = f->ld;
    const size_t max_rem = (size_t)(rem_max_deg + 1) * blowup;  // fri/src/options.rs:85-93
    size_t nlayers = 0;
    for (size_t l = len; l > max_rem; l /= folding) nlayers++;
    void *cur, *dstate, *dalpha, *dlog;
    CKI(g.tmp.alloc(len * ld * 8, &cur));
    CK(cudaMemcpyAsync(cur, evals->m.base, len * ld * 8, cudaMemcpyDeviceToDevice, ctx->st));
    CKI(g.tmp.alloc(8 * 8, &dstate));
    CKI(g.tmp.alloc(8 * 8, &dalpha));
    CKI(g.tmp.alloc(std::max<size_t>(nlayers, 1) * 8 * 8, &dlog));
    u64 seed_words[4];
    memcpy(seed_words, coin.seed.b, 32);
    CK(cudaMemcpyAsync(dstate, seed_words, 32, cudaMemcpyHostToDevice, ctx->st));
    size_t layer = 0;
    while (len > max_rem) {
        size_t m = len / folding;
        wf_tree* t;
        CKI(tree_alloc(ctx, hash_id, m, &t));
        g.t = t;
        CK(fri_hash_layer(hash_id, (u64*)cur, len, d, ld, (int)folding, t->leaves, ctx->st));
        CK(commit_merkle_nodes(hash_id, t->leaves, m, t->nodes, ctx->st));
        CK(fri_coin_step(hash_id, (u64*)dstate, t->nodes + 4, d, (u64*)dalpha, (u64*)dlog + 8 * layer, ctx->st));
        ctx->launches += 2 + merkle_launches(m);
        const u64* master;
        u32 ll = 0;
        while (((size_t)1 << ll) < len) ll++;
        CKI(wf_get_twiddles(ctx, ll, &master));
        void* nxt;
        CKI(g.tmp.alloc(m * ld * 8, &nxt));
        if (ld > d) CK(cudaMemsetAsync(nxt, 0, m * ld * 8, ctx->st));
        CK(fri_fold_layer((u64*)cur, len, d, ld, (int)folding, nullptr, master, (u64*)nxt, ld, ctx->st, (const u64*)dalpha));
        ctx->launches++;
        f->layers.push_back(FriLayer{(u64*)g.tmp.keep(cur), len, t});   // the wf_fri owns layer and tree from here
        g.t = nullptr;
        cur = nxt;
        len = m;
        layer++;
    }
    std::vector<u64> raw(len * ld), v(len * d), log(std::max<size_t>(nlayers, 1) * 8);
    CK(cudaMemcpyAsync(raw.data(), cur, len * ld * 8, cudaMemcpyDeviceToHost, ctx->st));
    if (nlayers) CK(cudaMemcpyAsync(log.data(), dlog, nlayers * 8 * 8, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    g.tmp.free(cur);
    g.tmp.free(dstate); g.tmp.free(dalpha); g.tmp.free(dlog);
    // replay on the host coin: commit_fri_layer, draw_fri_alpha (prover/src/channel.rs:215-234)
    for (size_t l = 0; l < nlayers; l++) {
        Digest root;
        memcpy(root.b, &log[8 * l], 32);
        commitments.push_back(root);
        coin.reseed(root);
        u64 alpha[3] = {0, 0, 0};
        bool ok = coin.draw(d, alpha) && log[8 * l + 7] == 1;
        for (int k = 0; k < d; k++) ok = ok && alpha[k] == log[8 * l + 4 + k];
        if (!ok) return wf_fail(ctx, WF_ERR_STATE, "device and host FRI transcripts diverged at layer %zu", l);
    }
    // remainder (fri/src/prover/mod.rs:230-239)
    for (size_t i = 0; i < len; i++)
        for (int c = 0; c < d; c++) v[i * d + c] = raw[i * ld + c];
    wf_host_dft(v, len, d, true, GL_GENERATOR);
    size_t rsize = len / blowup;
    f->remainder.resize(rsize * d);
    for (size_t i = 0; i < rsize; i++)
        for (int c = 0; c < d; c++) f->remainder[i * d + c] = v[(rsize - 1 - i) * d + c];
    Digest rc = hh_hash_elements(hash_id, f->remainder.data(), f->remainder.size());
    commitments.push_back(rc);
    coin.reseed(rc);
    g.f = nullptr;   // the caller's now
    *out = f;
    return WF_OK;
}
extern "C" {

struct DefaultChannel {
    PublicCoin coin;
    int d;
    std::vector<Digest> commitments;
};
int wf_fri_build_layers_default_channel(wf_ctx* ctx, int hash_id, const wf_mat* evals, int d, uint32_t folding,
                                        uint32_t rem_max_deg, uint32_t blowup, uint8_t* roots_out, size_t roots_cap,
                                        wf_fri** out) {
    DefaultChannel ch{PublicCoin(hash_id, nullptr, 0), d, {}};
    CKI(wf_fri_build_layers_coin(ctx, hash_id, evals, d, folding, rem_max_deg, blowup, ch.coin, ch.commitments, out));
    if (roots_out) {
        if (roots_cap < ch.commitments.size() * 32) return wf_fail(ctx, WF_ERR_INVALID, "roots buffer too small");
        for (size_t i = 0; i < ch.commitments.size(); i++) memcpy(roots_out + 32 * i, ch.commitments[i].b, 32);
    }
    return WF_OK;
}
uint32_t wf_fri_num_layers(const wf_fri* f) { return (uint32_t)f->layers.size(); }
size_t wf_fri_remainder(const wf_fri* f, uint64_t* coeffs, size_t cap_words) {
    if (coeffs && cap_words >= f->remainder.size()) memcpy(coeffs, f->remainder.data(), f->remainder.size() * 8);
    return f->remainder.size() / f->d;
}

}  // extern "C"
int wf_fri_queue_proof(wf_ctx* ctx, wf_fri* f, const std::vector<u64>& positions, GatherBatch& gb, FriProofPlan& plan) {
    // fri/src/prover/mod.rs:254-319: per layer fold the positions, queue the row values and the opening
    std::vector<u64> pos = positions;
    for (auto& L : f->layers) {
        size_t m = L.len / f->folding;
        std::vector<u64> fp;  // fold_positions (fri/src/folding/mod.rs:159-176)
        for (u64 p : pos) {
            u64 q = p % m;
            if (std::find(fp.begin(), fp.end(), q) == fp.end()) fp.push_back(q);
        }
        pos = fp;
        // queried values: row `position` of the transposed layer = v[pos + j*m], j < folding
        std::vector<u64> gpos(pos.size() * f->folding);
        for (size_t i = 0; i < pos.size(); i++)
            for (u32 j = 0; j < f->folding; j++) gpos[i * f->folding + j] = pos[i] + (u64)j * m;
        SegMatrix lm;
        lm.base = L.evals; lm.rows = L.len; lm.cols = (u32)f->d; lm.W = f->ld; lm.seg_stride = L.len * f->ld;
        plan.row_ids.push_back(gb.add_rows(lm, gpos));
        size_t id;
        CKI(gb.add_opening(ctx, L.tree, pos, &id));
        plan.dig_ids.push_back(id);
        plan.nq.push_back(pos.size());
    }
    return WF_OK;
}
void wf_fri_finish_proof(const wf_fri* f, const GatherBatch& gb, const FriProofPlan& plan, ByteVec& bv) {
    // FriProof / FriProofLayer wire format (fri/src/proof.rs:149-163, 275-285)
    bv.u8_((u8)f->layers.size());
    for (size_t l = 0; l < f->layers.size(); l++) {
        size_t nvals = plan.nq[l] * f->folding * f->d;
        ByteVec paths;
        wf_open_finish(gb.digs[plan.dig_ids[l]].plan, gb.digest_result(plan.dig_ids[l]), nullptr, paths);
        bv.u32_((u32)(nvals * 8));
        bv.bytes(gb.row_result(plan.row_ids[l]), nvals * 8);
        bv.u32_((u32)paths.v.size());
        bv.bytes(paths.v.data(), paths.v.size());
    }
    bv.u16_((uint16_t)(f->remainder.size() * 8));
    bv.bytes(f->remainder.data(), f->remainder.size() * 8);
    bv.u8_(0);  // log2(num_partitions = 1)
}
extern "C" {
int wf_fri_build_proof(wf_ctx* ctx, wf_fri* f, const uint64_t* positions, size_t k, uint8_t* out, size_t* len) {
    if (!ctx || !f || !positions || !out || !len) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    GatherBatch gb;
    FriProofPlan plan;
    CKI(wf_fri_queue_proof(ctx, f, std::vector<u64>(positions, positions + k), gb, plan));
    CKI(gb.run(ctx));
    ByteVec bv;
    wf_fri_finish_proof(f, gb, plan, bv);
    if (bv.v.size() > *len) return wf_fail(ctx, WF_ERR_INVALID, "proof buffer too small (%zu needed)", bv.v.size());
    memcpy(out, bv.v.data(), bv.v.size());
    *len = bv.v.size();
    return WF_OK;
}

// ---- plain kernels on caller-owned device buffers -------------------------------------------------
int wf_ntt_dev(wf_ctx* ctx, uint64_t* d_data, uint32_t log_n, uint32_t cols, int inverse) {
    if (!ctx || !d_data || cols == 0 || log_n < 1) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    wf_mat *m, *o;
    CKI(wf_mat_from_device_columns(ctx, d_data, cols, (size_t)1 << log_n, &m));
    int r = mat_transform(ctx, m, inverse, &o);
    wf_mat_free(ctx, m);
    if (r != WF_OK) return r;
    r = wf_mat_to_columns(ctx, o, d_data, 0, 0);
    wf_mat_free(ctx, o);
    return r;
}
int wf_hash_rows_dev(wf_ctx* ctx, int hash_id, const uint64_t* d_rows, size_t nrows, uint32_t cols, uint8_t* d_digests) {
    if (!ctx || !d_rows || !d_digests || cols == 0) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    // a row-major matrix is a single segment of width `cols`; reuse the generic kernel through a
    // one-segment view when cols is a supported width, else convert
    wf_mat* m;
    CKI(wf_mat_alloc(ctx, nrows, cols, &m));
    CK(layout_rows_to_seg(d_rows, m->m, ctx->st));
    CK(commit_hash_rows(hash_id, m->m, (u64*)d_digests, ctx->st));
    ctx->launches += 2;
    wf_mat_free(ctx, m);
    return WF_OK;
}
int wf_merkle_dev(wf_ctx* ctx, int hash_id, const uint8_t* d_leaves, size_t nleaves, uint8_t* d_nodes) {
    if (!ctx || !d_leaves || !d_nodes) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    if (nleaves < 2 || (nleaves & (nleaves - 1))) return wf_fail(ctx, WF_ERR_INVALID, "number of leaves must be a power of two >= 2");
    CK(commit_merkle_nodes(hash_id, (const u64*)d_leaves, nleaves, (u64*)d_nodes, ctx->st));
    ctx->launches += merkle_launches(nleaves);
    return WF_OK;
}
// field-arithmetic self-test hook: out[0..n) = a*b, out[n..2n) = a+b, out[2n..3n) = a-b,
// out[3n..4n) = 1/a (0 for a = 0), then out[(4+k) n ..) = a * 2^shift[k] for the 18 compile-time shifts
// the mini-DFTs use. Inputs canonical. Exists because uniform random data reaches the reduction's
// canonicalisation branch with probability 2^-32 per operation: tests feed crafted operands.
int wf_field_ops_dev(wf_ctx* ctx, const uint64_t* d_a, const uint64_t* d_b, size_t n, uint64_t* d_out) {
    if (!ctx || !d_a || !d_b || !d_out || n == 0) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    field_ops_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx->st>>>(d_a, d_b, n, d_out);
    ctx->launches++;
    CK(cudaGetLastError());
    return WF_OK;
}
int wf_ext_ops_dev(wf_ctx* ctx, uint32_t ext, const uint64_t* d_a, const uint64_t* d_b, size_t n, uint64_t* d_out) {
    if (!ctx || !d_a || !d_b || !d_out || n == 0 || (ext != 2 && ext != 3)) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    const unsigned blocks = (unsigned)((n + 127) / 128);
    if (ext == 2) ext_ops_kernel<2><<<blocks, 128, 0, ctx->st>>>(d_a, d_b, n, d_out);
    else ext_ops_kernel<3><<<blocks, 128, 0, ctx->st>>>(d_a, d_b, n, d_out);
    ctx->launches++;
    CK(cudaGetLastError());
    return WF_OK;
}
int wf_fri_fold_dev(wf_ctx* ctx, const uint64_t* d_evals, size_t len, int d, uint32_t folding, const uint64_t* alpha,
                    uint64_t* d_next) {
    if (!ctx || !d_evals || !alpha || !d_next || d < 1 || d > 3) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    u32 ll;
    if (log2_exact(len, &ll) || len < folding) return wf_fail(ctx, WF_ERR_INVALID, "bad length");
    const u64* master;
    CKI(wf_get_twiddles(ctx, std::max(ll, 1u), &master));
    CK(fri_fold_layer(d_evals, len, d, d, (int)folding, alpha, master, d_next, d, ctx->st));
    ctx->launches++;
    return WF_OK;
}

// ---- host helpers --------------------------------------------------------------------------------
int wf_host_hash_elements(int hash_id, const uint64_t* elems, size_t n, uint8_t out[32]) {
    Digest d = hh_hash_elements(hash_id, elems, n);
    memcpy(out, d.b, 32);
    return WF_OK;
}
int wf_host_merge(int hash_id, const uint8_t two[64], uint8_t out[32]) {
    Digest a, b;
    memcpy(a.b, two, 32);
    memcpy(b.b, two + 32, 32);
    Digest d = hh_merge(hash_id, a, b);
    memcpy(out, d.b, 32);
    return WF_OK;
}
int wf_host_merge_with_int(int hash_id, const uint8_t seed[32], uint64_t value, uint8_t out[32]) {
    Digest s;
    memcpy(s.b, seed, 32);
    Digest d = hh_merge_with_int(hash_id, s, value);
    memcpy(out, d.b, 32);
    return WF_OK;
}
uint64_t wf_host_mul(uint64_t a, uint64_t b) { return gl_mul(a, b); }
uint64_t wf_host_mul_2exp(uint64_t x, uint32_t k) {
    switch (k) {
        case 0: return m2e<0>(x); case 3: return m2e<3>(x); case 6: return m2e<6>(x); case 12: return m2e<12>(x);
        case 24: return m2e<24>(x); case 36: return m2e<36>(x); case 48: return m2e<48>(x); case 60: return m2e<60>(x);
        case 63: return m2e<63>(x); case 64: return m2e<64>(x); case 65: return m2e<65>(x); case 72: return m2e<72>(x);
        case 84: return m2e<84>(x); case 95: return m2e<95>(x); case 96: return m2e<96>(x);
        default: return gl_mul(x, gl_pow(2, k));
    }
}
uint64_t wf_host_mont_to_canonical(uint64_t m) { return gl_from_mont(m); }
uint64_t wf_host_canonical_to_mont(uint64_t x) { return gl_to_mont(x); }
size_t wf_host_write_usize(uint64_t value, uint8_t out[9]) {  // the serializer's vint64 (byte_writer.rs:77-92)
    ByteVec b;
    b.usize(value);
    memcpy(out, b.v.data(), b.v.size());
    return b.v.size();
}
// FibSmallProver::build_trace (examples/src/fibonacci/fib_small/prover.rs:37-53) for the "FibSmall x k" family:
// pair j starts at (j + 1, j + 1) and steps state[0] += state[1]; state[1] += state[0]. cols: [2k][n] canonical
// words (column-major, the layout wf_prove_fib / wf_prove_fib_dev take); results[j] = last value of column 2j+1.
int wf_host_build_fib_trace(uint32_t k, size_t n, uint64_t* cols, uint64_t* results) {
    if (!cols || !results || k == 0 || n == 0) return WF_ERR_INVALID;
    auto pair = [&](uint32_t j) {
        u64 a = j + 1, b = j + 1;
        u64 *ca = cols + (size_t)(2 * j) * n, *cb = ca + n;
        for (size_t i = 0; i < n; i++) {
            ca[i] = a;
            cb[i] = b;
            a = gl_add_host(a, b);
            b = gl_add_host(b, a);
        }
        results[j] = cb[n - 1];
    };
    const unsigned nt = std::max(1u, std::min(std::min(k, 16u), std::thread::hardware_concurrency()));
    std::vector<std::thread> th;  // pairs are independent
    for (unsigned t = 0; t < nt; t++) th.emplace_back([&, t]() { for (uint32_t j = t; j < k; j += nt) pair(j); });
    for (auto& x : th) x.join();
    return WF_OK;
}
// Index arithmetic of a sharded opening (GatherBatch::add_opening_sharded), exposed for the CPU tests of the multi-rank
// logic: the batch proof of `positions` in a tree of n_global leaves needs the digests want[0..count) (entries < n_global:
// heap nodes, else leaves, as MerkleTree::prove_batch walks them, crypto/src/merkle/mod.rs:217-272); idx[i] = where rank
// `rank` of `world` finds want[i] in ITS subtree (node index < n_local, else n_local + leaf), ~0 if another rank holds it,
// ~0 - 1 if it is one of the top log2(world) levels every rank keeps on the host. Returns count, or -1.
long wf_host_sharded_opening_plan(size_t n_global, int world, int rank, const uint64_t* positions, size_t k, uint64_t* want,
                                  uint64_t* idx, size_t cap) {
    if (!positions || !want || !idx || world < 1 || (world & (world - 1)) || n_global % (size_t)world) return -1;
    GatherBatch gb;
    size_t id;
    std::vector<std::pair<size_t, u64>> top;
    if (gb.add_opening_sharded(nullptr, nullptr, n_global, world, rank, std::vector<u64>(positions, positions + k), &id, &top) != WF_OK) return -1;
    const auto& j = gb.digs[id];
    if (j.idx.size() > cap) return -1;
    for (size_t i = 0; i < j.idx.size(); i++) { want[i] = j.plan.want[i]; idx[i] = j.idx[i]; }
    for (auto& t : top) idx[t.first] = ~(u64)0 - 1;
    return (long)j.idx.size();
}
// DefaultRandomCoin on the host (crypto/src/random/default.rs): seed from elements, optional reseed with a
// digest, then draw `count` elements of extension degree d -> out[count][d]. Returns 0, or -1 if a draw fails.
int wf_host_coin_draw(int hash_id, const uint64_t* seed_elems, size_t n_seed, const uint8_t* reseed32, int d, size_t count,
                      uint64_t* out) {
    if (d < 1 || d > 3 || !out) return -1;
    PublicCoin coin(hash_id, seed_elems, n_seed);
    if (reseed32) { Digest dg; memcpy(dg.b, reseed32, 32); coin.reseed(dg); }
    for (size_t i = 0; i < count; i++) if (!coin.draw(d, out + i * d)) return -1;
    return 0;
}

}  // extern "C"
