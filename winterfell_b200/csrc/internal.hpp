// internal.hpp — shared host-side definitions of the C-ABI implementation (capi.cu, prover.cu).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <map>
#include <set>
#include <string>
#include <functional>
#include <vector>

#include "../../include/winterfell_b200.h"
#include "commit.cuh"
#include "fri.cuh"
#include "host_transcript.hpp"
#include "layout.cuh"
#include "ntt.cuh"

// =================================================================================================
// context
// =================================================================================================
struct LdeTables {
    u64* pre;    // two-pass: [blowup][R] (s_k^C)^m1 ; single pass: [blowup][n] s_k^m
    u64* pow7;   // two-pass: [C] 7^m2 ; single pass: null
};

struct wf_ctx {
    int device;
    cudaStream_t st;
    std::string err;
    uint64_t launches;
    std::multimap<size_t, void*> pool;       // free device buffers by size
    std::map<void*, size_t> live;            // allocated device buffers
    std::map<u32, u64*> tw;                  // log_n -> w_n^i, i < n/2
    std::map<u32, u64*> round_tw;            // logS -> round-twiddle table of the ntt2 plan
    std::map<std::pair<u32, u32>, u64*> pow_tab;  // (log order, log count) -> w_(2^order)^i, i < 2^count
    std::map<std::pair<u32, u32>, LdeTables> lde_tabs;  // (log_n, log_blowup)
    void* pinned;                            // staging buffer (pinned host)
    size_t pinned_bytes;
    cudaStream_t copy_st = nullptr;          // H2D stream of the chunked trace pipeline (created on first use)
    cudaEvent_t ev_up[2], ev_used[2], ev_start;
    // sharded proofs: device memory of the other ranks mapped through CUDA IPC (key = the 64-byte handle), the streams the
    // peer copies are issued on (copy engines: no SM is taken from the kernels they overlap) and one event per coset
    std::map<std::string, void*> ipc_opened;
    cudaStream_t push_st[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t push_ev[16] = {};
    // constraint kernels compiled per AIR (jit.cu): generated source -> (cudaLibrary_t, cudaKernel_t); (null, null) = failed
    std::map<std::string, std::pair<void*, void*>> jit_cache;
    bool jit_enabled = true;
    uint64_t jit_compiled = 0, jit_hits = 0, jit_fallbacks = 0;
    bool profiling;                          // record a CUDA event at every pipeline stage boundary
    std::vector<std::pair<std::string, cudaEvent_t>> marks;
};
// stage marker (tracing spans of the reference: prover/src/lib.rs:312-466 info_span!/instrument)
void wf_mark(wf_ctx* ctx, const char* name);

struct wf_mat {
    SegMatrix m;
};
struct wf_tree {
    int hash_id;
    size_t nleaves;
    u64* leaves;  // nleaves x 4 words
    u64* nodes;   // nleaves x 4 words
};

// Small host-side transforms for transcript-sized data (FRI remainder, periodic column tables):
// plain radix-2 on `n` elements of `d` interleaved components. inverse: a_j = (1/n) sum v_i w^(-ij),
// then coefficient j scaled by offset^-j (fft/serial.rs:84-101 interpolate_poly_with_offset);
// forward: coefficient j scaled by offset^j first, then v_i = sum a_j w^(ij) (evaluation over offset*<w>).
static inline void wf_host_dft(std::vector<u64>& v, size_t n, int d, bool inverse, u64 offset) {
    u32 log_n = 0;
    while (((size_t)1 << log_n) < n) log_n++;
    u64 w0 = n > 1 ? gl_root_of_unity(log_n) : 1;
    if (inverse) w0 = gl_inv(w0);
    if (!inverse && offset != 1) {
        u64 f = 1;
        for (size_t i = 0; i < n; i++) { for (int c = 0; c < d; c++) v[i * d + c] = gl_mul(v[i * d + c], f); f = gl_mul(f, offset); }
    }
    for (size_t i = 0; i < n; i++) {  // bit-reverse, then DIT butterflies
        size_t j = 0;
        for (u32 b = 0; b < log_n; b++) j |= ((i >> b) & 1) << (log_n - 1 - b);
        if (j > i) for (int c = 0; c < d; c++) std::swap(v[i * d + c], v[j * d + c]);
    }
    for (size_t len = 2; len <= n; len <<= 1) {
        u64 wl = gl_pow(w0, n / len);
        for (size_t s = 0; s < n; s += len) {
            u64 w = 1;
            for (size_t i = 0; i < len / 2; i++) {
                for (int c = 0; c < d; c++) {
                    u64 a = v[(s + i) * d + c], b = gl_mul(v[(s + i + len / 2) * d + c], w);
                    v[(s + i) * d + c] = gl_add(a, b);
                    v[(s + i + len / 2) * d + c] = gl_sub(a, b);
                }
                w = gl_mul(w, wl);
            }
        }
    }
    if (inverse) {
        u64 scale = gl_inv((u64)n % GL_P), oinv = gl_inv(offset);
        for (size_t i = 0; i < n; i++) {
            for (int c = 0; c < d; c++) v[i * d + c] = gl_mul(v[i * d + c], scale);
            scale = gl_mul(scale, oinv);
        }
    }
}

int wf_fail(wf_ctx* ctx, int code, const char* fmt, ...);
// jit.cu
std::string wf_jit_source(int D, u32 w, u32 nper, u32 nregs, const std::vector<u32>& prog, const std::vector<u64>& consts, u32 aw, u32 nr,
                          u32 naregs, const std::vector<u32>& aprog);
int wf_jit_compile(const std::string& src, std::vector<char>& cubin, std::string& log);
int wf_jit_get_kernel(wf_ctx* ctx, const std::string& src, cudaKernel_t* kernel);
int wf_dev_alloc(wf_ctx* ctx, size_t bytes, void** out);
void wf_dev_free(wf_ctx* ctx, void* p);
// Scratch buffers of one call: whatever is still registered when the scope ends (every early error return included) goes back
// to the context's pool. free() hands one back early, keep() passes ownership on (the buffer outlives the call).
struct DevScratch {
    wf_ctx* ctx;
    std::vector<void*> bufs;
    explicit DevScratch(wf_ctx* c) : ctx(c) {}
    DevScratch(const DevScratch&) = delete;
    DevScratch& operator=(const DevScratch&) = delete;
    ~DevScratch() { for (void* p : bufs) if (p) wf_dev_free(ctx, p); }
    int alloc(size_t bytes, void** out) {
        int r = wf_dev_alloc(ctx, bytes, out);
        if (r == WF_OK) bufs.push_back(*out);
        return r;
    }
    void forget(void* p) { for (void*& q : bufs) if (q == p) { q = nullptr; return; } }
    void free(void* p) { if (!p) return; forget(p); wf_dev_free(ctx, p); }
    void* keep(void* p) { forget(p); return p; }
};
int wf_mat_alloc(wf_ctx* ctx, size_t rows, u32 cols, wf_mat** out);
int wf_mat_alloc_w(wf_ctx* ctx, size_t rows, u32 cols, int W, wf_mat** out);
// LDE output scattered into the row shards of the ranks of a sharded proof (NttPassParams::sc_*, ntt.cuh)
struct LdeScatter {
    u64* peer[8];        // shard base per rank (peer memory mapped through CUDA IPC; own rank: the local shard)
    size_t seg_stride;   // words between segments of a shard
    u32 seg0;            // global segment the first local segment maps to
    u32 log_nj;          // log2(points of one coset per rank)
    u32 world;           // > 0: also write the halo rows of the previous rank (NttPassParams::sc_world)
};
extern "C" int wf_trace_lde_cosetwise(wf_ctx* ctx, const uint64_t* const* cols, const uint64_t* d_cols, uint32_t ncols, size_t nrows, int mont,
                           uint32_t log_blowup, wf_mat** polys_out, wf_mat** lde_out, bool coset_major,
                           const std::function<int(u32)>* after_coset, const LdeScatter* scatter, int d, uint32_t q0);
extern "C" int wf_mat_lde_cosets(wf_ctx* ctx, const wf_mat* polys, uint32_t log_blowup, uint32_t k0, uint32_t k1, wf_mat* lde);  // internal (not in the public header)
struct PublicCoin;
struct Digest;
struct wf_fri;
int wf_fri_build_layers_coin(wf_ctx* ctx, int hash_id, const wf_mat* evals, int d, uint32_t folding, uint32_t rem_max_deg,
                             uint32_t blowup, PublicCoin& coin, std::vector<Digest>& commitments, wf_fri** out);
int wf_get_twiddles(wf_ctx* ctx, u32 log_n, const u64** out);
struct wf_tree;
int wf_fri_layer_tree(wf_ctx* ctx, int hash_id, const u64* vals, size_t len, int d, int ld, int nf, wf_tree** out);
struct OpenPlan {
    u32 depth;
    u32 digest_bytes = 32;                       // bytes a digest serializes to (24 for Blake3_192), set from the tree's hasher
    std::vector<u64> want;                       // < n: nodes[want]; >= n: leaves[want - n]
    std::vector<std::vector<size_t>> vec_slots;  // per proof vector: slots into `want`
    std::vector<size_t> leaf_slot;               // per queried position: slot of its leaf digest
};
int wf_open_plan(wf_ctx* ctx, size_t n, const uint64_t* positions, size_t k, OpenPlan& pl);
void wf_open_finish(const OpenPlan& pl, const uint8_t* got, uint8_t* leaves_out, ByteVec& proof);
// all row / digest gathers of one proof: one upload, one download, one synchronisation
// Sharded proofs (wf_comm): every rank queues the SAME jobs; a row / digest this rank does not hold is queued with the
// index ~0 (gathered as zero) and the gathered words are summed over the ranks before the download.
struct GatherBatch {
    struct RowJob { SegMatrix m; std::vector<u64> pos; size_t idx_off, out_off; };
    struct DigJob { const wf_tree* t; OpenPlan plan; std::vector<u64> idx; size_t idx_off, out_off; };  // idx: indices into t (or ~0)
    std::vector<RowJob> rows;
    std::vector<DigJob> digs;
    const wf_comm* comm = nullptr;
    u64* result = nullptr;  // pinned host buffer, valid until the next run()
    size_t add_rows(const SegMatrix& m, const std::vector<u64>& pos);
    int add_opening(wf_ctx* ctx, const wf_tree* t, const std::vector<u64>& pos, size_t* id);
    // opening in a tree of n_global leaves stored as `world` local subtrees (this rank: `t`, n_global / world leaves):
    // nodes above the subtree roots are not gathered (the caller patches them in from its host copy, see top_slots)
    int add_opening_sharded(wf_ctx* ctx, const wf_tree* t, size_t n_global, int world, int rank, const std::vector<u64>& pos,
                            size_t* id, std::vector<std::pair<size_t, u64>>* top_slots);
    int run(wf_ctx* ctx);
    const u64* row_result(size_t id) const { return result + rows[id].out_off; }
    const u8* digest_result(size_t id) const { return (const u8*)(result + digs[id].out_off); }
    u64* digest_words(size_t id) { return result + digs[id].out_off; }
};
struct FriLayer {
    u64* evals;   // len x ld words (natural order)
    size_t len;
    wf_tree* tree;
};
struct wf_fri {
    int hash_id, d, ld;
    u32 folding, blowup;
    std::vector<FriLayer> layers;
    std::vector<u64> remainder;  // reversed coefficients, d words each
};

// FriProver::build_proof split the same way: queue the gathers, then serialise
struct FriProofPlan { std::vector<size_t> row_ids, dig_ids; std::vector<size_t> nq; };
int wf_fri_queue_proof(wf_ctx* ctx, wf_fri* f, const std::vector<u64>& positions, GatherBatch& gb, FriProofPlan& plan);
void wf_fri_finish_proof(const wf_fri* f, const GatherBatch& gb, const FriProofPlan& plan, ByteVec& out);
int wf_tree_open_many_bytes(wf_ctx* ctx, const wf_tree* t, const uint64_t* positions, size_t k, uint8_t* leaves_out,
                            ByteVec& proof);

#define CK(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t _e = (call);                                                                          \
        if (_e != cudaSuccess)                                                                            \
            return wf_fail(ctx, WF_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
    } while (0)
#define CKI(call)                   \
    do {                            \
        int _r = (call);            \
        if (_r != WF_OK) return _r; \
    } while (0)
