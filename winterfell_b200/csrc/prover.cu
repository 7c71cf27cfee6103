// prover.cu — the full proving pipeline on device behind one C-ABI call (wf_prove_fib / wf_prove_air /
// wf_prove_air_aux), i.e. the body of winterfell's Prover::generate_proof (prover/src/lib.rs:282-492) with
// every hot loop on the GPU, and the same steps as separate exports (wf_eval_constraints, ...):
//   K1-K4  trace commitment          (ntt.cu, commit.cu)          DefaultTraceLde::new, set_aux_trace
//   K5     constraint evaluation     (fib_ / generic_constraints) DefaultConstraintEvaluator::evaluate
//   K6/K7  composition poly + commit (ntt.cu, commit.cu)          DefaultConstraintCommitment::new
//   K8     out-of-domain frames      (ood_partial_kernel)         TracePolyTable/CompositionPoly::get_ood_frame
//   K9/K10 DEEP composition          (deep_sum/div_kernel)        DeepCompositionPoly::{add_trace_polys, evaluate}
//   K11    FRI commit phase          (fri.cu, device coin)        FriProver::build_layers
//   K13    proof-of-work grinding    (grind_kernel)               ProverChannel::grind_query_seed, smallest nonce
// The Fiat-Shamir transcript (ProverChannel, prover/src/channel.rs) and the proof wire format
// (air/src/proof/*.rs) are host code here, bit-exact with the reference; during the FRI commit phase the
// coin is mirrored on the device and the host replays it afterwards.
//
// The DEEP composition is computed in EVALUATION form over the LDE domain,
//   D(x) = (S(x) - S(z)) / (x - z) + (S(x) - S(zg)) / (x - zg),  S = sum_j cc_j T_j + sum_j cc'_j H_j,
// which is the same polynomial the reference builds in coefficient form by synthetic division
// (composer/mod.rs:67-210) and evaluates by LDE (:171): exact field arithmetic, identical values
// (SURVEY.md A.4), but row-parallel and without the extra LDE.
//
// Constraint evaluation needs the AIR on the device (Air::evaluate_transition is user Rust code,
// air/src/air/mod.rs:210): generic AIRs arrive as a flat description (transition programs for both
// segments, periodic columns, single / periodic / sequence assertions, exemptions; format in
// include/winterfell_b200.h) and run on a bytecode evaluator; the "FibSmall x k" family = k copies of
// examples/src/fibonacci/fib_small/air.rs:16-69 side by side (k = 1 is the reference example, k = 4 / 32
// the 8- / 64-column configurations of BASELINE.json) has a specialised kernel.
#include <algorithm>
#include <chrono>

#include "internal.hpp"
#include "blake3.cuh"
#include "alg_hash.cuh"

// =================================================================================================
// kernels
// =================================================================================================
#include "constraints_generic.cuh"  // ld_ext / seg_at, GenEvalParams, generic_constraints_kernel (also the source NVRTC compiles per AIR)

#ifndef FIB_ROWS_D3
#define FIB_ROWS_D3 2   // CE rows per thread sharing one inversion, cubic extension (register budget)
#endif
struct FibEvalParams {
    SegMatrix lde;      // N x 2k trace LDE
    SegMatrix out;      // ce x D combined constraint evaluations
    u32 k, log_n, log_blowup, log_ce_blowup;
    const u64* coef;    // [k][5][D]: per pair j the coefficients of t0, t1 (transition), of column 2j and 2j+1 in the
                        // step-0 boundary group, and of column 2j+1 in the last-step group
    u64 K0[3], K1[3];   // constants of the two boundary groups: sum_q bcoef0_q * value_q, sum_j bcoef1_j * result_j
    const u64* tw_ce;   // w_ce^i, i < ce/2
    u64 zt[8];          // 1 / (x^n - 1) at CE step i mod ce_blowup
    u64 last;           // g_trace^(n-1): transition exemption point and divisor offset of group 1
    // row-sharded evaluation (multi-GPU): this launch covers CE rows [row0, row0 + ce_rows); `lde` then holds the LDE
    // rows of that range followed by `blowup` halo rows (the first rows of the next shard), so the next-state row is
    // local row + blowup without wrap-around. ce_rows = 0: the whole domain.
    size_t row0, ce_rows;
};

// CE-domain rows, FIB_ROWS per thread sharing one field inversion (evaluator/default.rs:165-214
// evaluate_fragment_main + evaluation_table.rs:317-367 acc_column, fused). The three linear forms of a row
// (transition combination, the two boundary groups) are dot products of base-field frame values with extension
// coefficients: they run on delayed-reduction accumulators (GlAcc), one reduction per row and form instead of one per
// term — the first version spent 22 k instructions per row of the 64-column cubic configuration in gl_mul / gl_add.
template <int D>
__global__ void __launch_bounds__(256) fib_constraints_kernel(FibEvalParams p) {
    extern __shared__ __align__(16) u64 fsm[];
    constexpr int ROWS = D == 3 ? FIB_ROWS_D3 : 4;
    for (u32 i = threadIdx.x; i < p.k * 5 * D; i += blockDim.x) fsm[i] = p.coef[i];
    __syncthreads();
    const size_t ce_all = (size_t)1 << (p.log_n + p.log_ce_blowup);
    const size_t ce = p.ce_rows ? p.ce_rows : ce_all;   // rows of this launch
    const size_t N = (size_t)1 << (p.log_n + p.log_blowup);
    const u32 lde_shift = p.log_blowup - p.log_ce_blowup;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const u32 half = (u32)(ce_all >> 1);
    const int W = p.lde.W;
    GlExt<D> T[ROWS], B0[ROWS], B1[ROWS];
    u64 d0[ROWS], d1[ROWS];
#pragma unroll
    for (int r = 0; r < ROWS; r++) {
        const size_t il = tid + r * stride;   // row of this launch
        const size_t i = il + p.row0;         // row of the CE domain
        T[r] = ext_zero<D>(); B0[r] = ext_zero<D>(); B1[r] = ext_zero<D>();
        d0[r] = 1; d1[r] = 1;
        if (il >= ce) continue;
        const size_t ls = il << lde_shift;
        const size_t nx = p.ce_rows ? ls + ((size_t)1 << p.log_blowup)
                                    : ((ls + ((size_t)1 << p.log_blowup)) & (N - 1));  // trace_lde/default/mod.rs:169-180
        GlAcc aT[D], a0[D], a1[D];
#pragma unroll
        for (int q = 0; q < D; q++) { aT[q] = acc_zero(); a0[q] = acc_zero(); a1[q] = acc_zero(); }
#pragma unroll 2
        for (u32 j = 0; j < p.k; j++) {
            // columns 2j, 2j+1 are adjacent words of one segment row: one 16-byte load per frame row
            const size_t off = (size_t)((2 * j) / W) * p.lde.seg_stride + (2 * j) % W;
            const ulonglong2 cur = __ldg(reinterpret_cast<const ulonglong2*>(p.lde.base + off + ls * W));
            const ulonglong2 nxt = __ldg(reinterpret_cast<const ulonglong2*>(p.lde.base + off + nx * W));
            const u64 t0 = gl_sub(nxt.x, gl_add(cur.x, cur.y));  // fib_small/air.rs:58
            const u64 t1 = gl_sub(nxt.y, gl_add(cur.y, nxt.x));  // :59
            const u64* cf = fsm + (size_t)j * 5 * D;
#pragma unroll
            for (int q = 0; q < D; q++) {
                acc_mad(aT[q], cf[q], t0);
                acc_mad(aT[q], cf[D + q], t1);
                acc_mad(a0[q], cf[2 * D + q], cur.x);
                acc_mad(a0[q], cf[3 * D + q], cur.y);
                acc_mad(a1[q], cf[4 * D + q], cur.y);
            }
        }
#pragma unroll
        for (int q = 0; q < D; q++) {
            T[r].v[q] = acc_reduce(aT[q]);
            B0[r].v[q] = gl_sub(acc_reduce(a0[q]), p.K0[q]);
            B1[r].v[q] = gl_sub(acc_reduce(a1[q]), p.K1[q]);
        }
        u64 w = p.tw_ce[i & (half - 1)];
        if (i & half) w = gl_neg(w);
        u64 x = gl_mul(w, GL_GENERATOR);  // domain.rs:123 get_ce_x_at
        d0[r] = gl_sub(x, 1);             // boundary divisor of the step-0 group
        d1[r] = gl_sub(x, p.last);        // boundary divisor of the last-step group = transition exemption
    }
    // batch inversion of the products d0*d1 (never zero: x lies on the coset 7<w>, 1 and g^(n-1) do not)
    u64 prod[ROWS], pre[ROWS], run = 1;
#pragma unroll
    for (int r = 0; r < ROWS; r++) { prod[r] = gl_mul(d0[r], d1[r]); pre[r] = run; run = gl_mul(run, prod[r]); }
    run = gl_inv(run);
#pragma unroll
    for (int r = ROWS - 1; r >= 0; r--) { u64 inv = gl_mul(run, pre[r]); run = gl_mul(run, prod[r]); prod[r] = inv; }
#pragma unroll
    for (int r = 0; r < ROWS; r++) {
        const size_t il = tid + r * stride, i = il + p.row0;
        if (il >= ce) continue;
        u64 z0 = gl_mul(prod[r], d1[r]), z1 = gl_mul(prod[r], d0[r]);                   // 1/(x - 1), 1/(x - g^(n-1))
        u64 zt = gl_mul(p.zt[i & (((size_t)1 << p.log_ce_blowup) - 1)], d1[r]);         // e(x) / (x^n - 1)
        GlExt<D> acc = ext_add(ext_add(ext_mul_base(T[r], zt), ext_mul_base(B0[r], z0)), ext_mul_base(B1[r], z1));
        u64* o = p.out.base + il * p.out.W;
#pragma unroll
        for (int q = 0; q < D; q++) o[q] = acc.v[q];
    }
}

// composition_poly.rs:128-140 segment(): column j = coefficients [j*n, (j+1)*n) of the interpolated
// CE-domain polynomial; each is an extension column of D base columns.
__global__ void comp_split_kernel(SegMatrix coefs, size_t n, u32 kc, int D, SegMatrix out) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t total = n * kc * D;
    if (idx >= total) return;
    size_t i = idx / (kc * D);
    u32 col = (u32)(idx % (kc * D));
    u32 j = col / D, comp = col % D;
    u64 v = coefs.base[(j * n + i) * coefs.W + comp];
    out.base[(size_t)(col / out.W) * out.seg_stride + i * out.W + (col % out.W)] = v;
}

// Evaluation of every base-coefficient column at TWO extension points (z and z*g), as per-block partial sums
// (polynom::eval, math/src/polynom/mod.rs:55-62; ColMatrix::evaluate_columns_at :245; TracePolyTable::get_ood_frame
// poly_table.rs:68-76). Block = 32 row groups x 8 lanes (lane = column of the segment); a thread owns OOD_RPT
// consecutive coefficients of ONE column and accumulates sum_r a_r z^r for both points on delayed-reduction
// accumulators against a shared table of z^r (one base-by-extension product per coefficient and point, no reduction
// inside the loop); the row-group power (z^OOD_RPT)^rg and the block power z^(first row of the block) — the latter
// from a table filled by ood_pow_kernel, an ext_pow per thread there instead of per coefficient chunk here — are
// applied once per thread / once per block. partial[col][chunk][point] = sum_{m in chunk} a_m z^m.
#define OOD_RPT 64
#define OOD_ROWS_PER_BLOCK (32 * OOD_RPT)
template <int D>
__global__ void ood_pow_kernel(GlExt<D> z0, GlExt<D> z1, u32 chunks, u64* zb /*[2][chunks][D]*/) {
    const u32 idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= 2 * chunks) return;
    const u32 pt = idx / chunks, c = idx % chunks;
    const GlExt<D> v = ext_pow(pt ? z1 : z0, (u64)c * OOD_ROWS_PER_BLOCK);
#pragma unroll
    for (int d = 0; d < D; d++) zb[(size_t)idx * D + d] = v.v[d];
}
template <int D>
__global__ void __launch_bounds__(256) ood_partial_kernel(SegMatrix polys, GlExt<D> z0, GlExt<D> z1, const u64* zb,
                                                          u64* partial /*[cols][chunks][2][D]*/, u32 chunks) {
    const u32 g = blockIdx.y, chunk = blockIdx.x, t = threadIdx.x;
    const int W = polys.W;
    const size_t n = polys.rows;
    const u64* base = polys.base + (size_t)g * polys.seg_stride;
    __shared__ u64 zpow[2][OOD_RPT][D];   // z^r
    __shared__ u64 zrg[2][32][D];         // z^(OOD_RPT * rg)
    __shared__ u64 red[2][32][8][D];
    if (t < 2 * OOD_RPT) {
        const GlExt<D> v = ext_pow(t < OOD_RPT ? z0 : z1, t % OOD_RPT);
#pragma unroll
        for (int d = 0; d < D; d++) zpow[t / OOD_RPT][t % OOD_RPT][d] = v.v[d];
    } else if (t < 2 * OOD_RPT + 64) {
        const u32 u = t - 2 * OOD_RPT, pt = u / 32, rg = u % 32;
        const GlExt<D> v = ext_pow(pt ? z1 : z0, (u64)rg * OOD_RPT);
#pragma unroll
        for (int d = 0; d < D; d++) zrg[pt][rg][d] = v.v[d];
    }
    __syncthreads();
    const u32 rg = t >> 3, lane = t & 7;
    const size_t start = (size_t)chunk * OOD_ROWS_PER_BLOCK + (size_t)rg * OOD_RPT;
    GlAcc acc[2][D];
#pragma unroll
    for (int pt = 0; pt < 2; pt++)
#pragma unroll
        for (int d = 0; d < D; d++) acc[pt][d] = acc_zero();
    if (lane < (u32)W) {
        const u64* src = base + start * W + lane;
#pragma unroll 1
        for (int r0 = 0; r0 < OOD_RPT; r0 += 8) {
            u64 cf[8];
#pragma unroll
            for (int k = 0; k < 8; k++) cf[k] = (start + r0 + k < n) ? __ldg(src + (size_t)(r0 + k) * W) : 0;
#pragma unroll
            for (int k = 0; k < 8; k++) {
#pragma unroll
                for (int d = 0; d < D; d++) {
                    acc_mad(acc[0][d], zpow[0][r0 + k][d], cf[k]);
                    acc_mad(acc[1][d], zpow[1][r0 + k][d], cf[k]);
                }
            }
        }
    }
#pragma unroll
    for (int pt = 0; pt < 2; pt++) {
        GlExt<D> v;
#pragma unroll
        for (int d = 0; d < D; d++) v.v[d] = acc_reduce(acc[pt][d]);
        v = ext_mul(v, ld_ext<D>(&zrg[pt][rg][0]));
#pragma unroll
        for (int d = 0; d < D; d++) red[pt][rg][lane][d] = v.v[d];
    }
    __syncthreads();
    if (t < 16) {
        const u32 pt = t >> 3, q = t & 7, col = g * W + q;
        if (q < (u32)W && col < polys.cols) {
            GlExt<D> sacc = ext_zero<D>();
            for (int k = 0; k < 32; k++) sacc = ext_add(sacc, ld_ext<D>(&red[pt][k][q][0]));
            sacc = ext_mul(sacc, ld_ext<D>(zb + ((size_t)pt * chunks + chunk) * D));
            u64* o = partial + (((size_t)col * chunks + chunk) * 2 + pt) * D;
#pragma unroll
            for (int d = 0; d < D; d++) o[d] = sacc.v[d];
        }
    }
}
// one warp per (column, point): lanes stride over the chunks (2048 of them for a 2^22-row column — a single thread
// walking them serially took 0.5 ms per call), then a shuffle tree over the extension components
template <int D>
__global__ void __launch_bounds__(256) ood_reduce_kernel(const u64* partial, u32 cols, u32 chunks, u64* out /*[cols][2][D]*/) {
    const u32 idx = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (idx >= cols * 2) return;   // warp-uniform
    const u32 col = idx >> 1, pt = idx & 1;
    GlExt<D> s = ext_zero<D>();
    for (u32 c = lane; c < chunks; c += 32) s = ext_add(s, ld_ext<D>(partial + (((size_t)col * chunks + c) * 2 + pt) * D));
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        GlExt<D> o;
#pragma unroll
        for (int c = 0; c < D; c++) o.v[c] = __shfl_down_sync(0xffffffffu, s.v[c], off);
        s = ext_add(s, o);
    }
    if (lane == 0)
        for (int c = 0; c < D; c++) out[(size_t)idx * D + c] = s.v[c];
}

struct DeepParams {
    SegMatrix trace;   // N x c
    SegMatrix cons;    // N x kc*D
    SegMatrix out;     // N x D
    SegMatrix aux;     // N x aw*D (aux segment LDE; aw == 0 when single-segment)
    u32 c, kc, log_N, aw;
    const u64* acc;    // [aw][D] DEEP coefficients for aux columns (composer/mod.rs:100-125)
    const u64* tcc;    // [c][D]  DEEP coefficients for trace columns
    const u64* ccc;    // [kc][D] DEEP coefficients for composition columns
    const u64* tw_N;   // w_N^i, i < N/2
    size_t row0, nrows;  // row-sharded launch: rows [row0, row0 + nrows) of the LDE domain (nrows = 0: all N rows)
};
// DeepCompositionPoly in evaluation form, two kernels:
//   deep_sum_kernel: S(x) = sum_j cc_j T_j(x) + sum_j cc'_j A_j(x) + sum_j cc''_j H_j(x) for every LDE row — the
//     pass that reads the whole LDE; one row per thread, coefficients in shared memory, ~40 registers, so
//     the SMs stay full (the earlier single kernel needed 242 registers per thread with cubic elements:
//     12 % occupancy, 28 % issue utilisation, 2.0 ms for 2^21 rows x 64 columns);
//   deep_div_kernel: D(x) = (S(x) - S(z)) / (x - z) + (S(x) - S(zg)) / (x - zg) in place, DEEP_ROWS rows per
//     thread sharing one batch inversion (math/src/utils/mod.rs:169).
// (Tried and dropped: chains of rows i, i + b, ... that reuse 1 / (x_{i-b} - z) = g / (x_i - z g) to halve
// the inversions — the strided row pattern cost more than the arithmetic saved.)
#ifndef DEEP_SUM_THREADS
#define DEEP_SUM_THREADS 256
#endif
template <int D>
__global__ void __launch_bounds__(DEEP_SUM_THREADS) deep_sum_kernel(DeepParams p) {
    extern __shared__ __align__(16) u64 dsm[];
    u64* s_t = dsm;                                  // [c][D]
    u64* s_a = s_t + (size_t)p.c * D;                // [aw][D]
    u64* s_c = s_a + (size_t)p.aw * D;               // [kc][D]
    for (u32 i = threadIdx.x; i < p.c * D; i += DEEP_SUM_THREADS) s_t[i] = p.tcc[i];
    for (u32 i = threadIdx.x; i < p.aw * D; i += DEEP_SUM_THREADS) s_a[i] = p.acc[i];
    for (u32 i = threadIdx.x; i < p.kc * D; i += DEEP_SUM_THREADS) s_c[i] = p.ccc[i];
    __syncthreads();
    const size_t N = p.nrows ? p.nrows : ((size_t)1 << p.log_N);   // rows of this launch
    const size_t row = (size_t)blockIdx.x * DEEP_SUM_THREADS + threadIdx.x;
    if (row >= N) return;
    // S over the base-field trace columns = D dot products of the row with the coefficient components: delayed-reduction
    // accumulators, one reduction per component per row
    GlAcc acc[D];
#pragma unroll
    for (int d = 0; d < D; d++) acc[d] = acc_zero();
    if (p.trace.W == 8) {
        // one 64-byte segment row = four 16-byte loads; the next segment's row is requested before this one is consumed
        // (the kernel was latency-bound on these loads: 3.2 long-scoreboard stalls per issue, profiles/r2_cubic_stages.txt)
        const u32 nseg = (p.c + 7) / 8;
        ulonglong2 nx[4];
        {
            const ulonglong2* rp = reinterpret_cast<const ulonglong2*>(p.trace.base + row * 8);
#pragma unroll
            for (int k = 0; k < 4; k++) nx[k] = __ldg(rp + k);
        }
        for (u32 g = 0; g < nseg; g++) {
            u64 v[8];
#pragma unroll
            for (int k = 0; k < 4; k++) { v[2 * k] = nx[k].x; v[2 * k + 1] = nx[k].y; }
            if (g + 1 < nseg) {
                const ulonglong2* rp = reinterpret_cast<const ulonglong2*>(p.trace.base + (size_t)(g + 1) * p.trace.seg_stride + row * 8);
#pragma unroll
                for (int k = 0; k < 4; k++) nx[k] = __ldg(rp + k);
            }
#pragma unroll
            for (int q = 0; q < 8; q++) {
                u32 j = g * 8 + q;
                if (j < p.c) {
#pragma unroll
                    for (int d = 0; d < D; d++) acc_mad(acc[d], s_t[(size_t)j * D + d], v[q]);
                }
            }
        }
    } else {
        for (u32 j = 0; j < p.c; j++) {
            const u64 v = seg_at(p.trace, row, j);
#pragma unroll
            for (int d = 0; d < D; d++) acc_mad(acc[d], s_t[(size_t)j * D + d], v);
        }
    }
    GlExt<D> S;
#pragma unroll
    for (int d = 0; d < D; d++) S.v[d] = acc_reduce(acc[d]);
    for (u32 j = 0; j < p.aw; j++) {
        GlExt<D> av;
#pragma unroll
        for (int q = 0; q < D; q++) av.v[q] = seg_at(p.aux, row, j * D + q);
        S = ext_add(S, ext_mul(ld_ext<D>(s_a + (size_t)j * D), av));
    }
    for (u32 j = 0; j < p.kc; j++) {
        GlExt<D> hv;
#pragma unroll
        for (int q = 0; q < D; q++) hv.v[q] = seg_at(p.cons, row, j * D + q);
        S = ext_add(S, ext_mul(ld_ext<D>(s_c + (size_t)j * D), hv));
    }
    u64* o = p.out.base + row * p.out.W;
#pragma unroll
    for (int q = 0; q < D; q++) o[q] = S.v[q];
}

// rows per thread sharing one batch inversion
#ifndef DEEP_ROWS1
#define DEEP_ROWS1 8
#endif
#ifndef DEEP_ROWS2
#define DEEP_ROWS2 8
#endif
#ifndef DEEP_ROWS3
#define DEEP_ROWS3 8
#endif
#ifndef DEEP_DIV_MINB
#define DEEP_DIV_MINB 2
#endif
#define DEEP_ROWS (D == 1 ? DEEP_ROWS1 : (D == 2 ? DEEP_ROWS2 : DEEP_ROWS3))
// 1 / (x - z) for x in the BASE field and z in the extension, without an extension-field inversion: with m_z the minimal
// polynomial of z over the base field (degree D, base-field coefficients) and Q_z(X) = m_z(X) / (X - z) (degree D - 1, extension
// coefficients, monic),   1 / (x - z) = Q_z(x) / m_z(x),   m_z(x) = N(x - z) in the base field.
// So the per-row inversion is a BASE-field one (3 multiplications per denominator in a batch inversion instead of 3
// extension products = 18 for the cubic extension) and Q_z(x) costs D - 1 base-by-extension products. The host supplies
//   D = 3: m = X^3 - t X^2 + s X - n (t = trace, n = norm), Q = X^2 - q1 X + q0, q1 = z' + z'', q0 = z' z'' (Frobenius conjugates)
//   D = 2: m = X^2 - t X + n,                                Q = X - q0,          q0 = z'
//   D = 1: m = X - z,                                        Q = 1.
template <int D>
struct DeepPoint {
    u64 t, s, n;        // base-field coefficients of m_z
    GlExt<D> q1, q0;    // extension coefficients of Q_z
};
template <int D>
__device__ __forceinline__ u64 deep_m(const DeepPoint<D>& pt, u64 x, u64 x2) {
    if (D == 1) return gl_sub(x, pt.n);                                          // x - z
    if (D == 2) return gl_add(gl_sub(x2, gl_mul(pt.t, x)), pt.n);               // x^2 - t x + n
    return gl_sub(gl_add(gl_mul(x2, gl_sub(x, pt.t)), gl_mul(pt.s, x)), pt.n);  // x^2 (x - t) + s x - n
}
template <int D>
__device__ __forceinline__ GlExt<D> deep_q(const DeepPoint<D>& pt, u64 x, u64 x2) {
    GlExt<D> q;
    if (D == 1) { q.v[0] = 1; return q; }
    if (D == 2) { q = ext_sub(ext_from_base<D>(x), pt.q0); return q; }
    q = ext_sub(pt.q0, ext_mul_base(pt.q1, x));
    q.v[0] = gl_add(q.v[0], x2);
    return q;
}
template <int D>
__global__ void __launch_bounds__(256, DEEP_DIV_MINB) deep_div_kernel(DeepParams p, DeepPoint<D> pz, DeepPoint<D> pzg, GlExt<D> Sz, GlExt<D> Szg) {
    const size_t N = p.nrows ? p.nrows : ((size_t)1 << p.log_N);   // rows of this launch
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    constexpr int ROWS = DEEP_ROWS;
    u64 xs[D == 1 ? 1 : ROWS], den[2 * ROWS];   // x is only needed again by Q_z for D > 1
    const u32 half = (u32)(((size_t)1 << p.log_N) >> 1);
#pragma unroll
    for (int r = 0; r < ROWS; r++) {
        size_t row = tid + r * stride;
        if (D > 1) xs[r] = 0;
        den[2 * r] = 1; den[2 * r + 1] = 1;
        if (row >= N) continue;
        const size_t grow = row + p.row0;   // row of the LDE domain
        u64 w = p.tw_N[grow & (half - 1)];
        if (grow & half) w = gl_neg(w);
        const u64 x = gl_mul(w, GL_GENERATOR), x2 = gl_sqr(x);
        if (D > 1) xs[r] = x;
        den[2 * r] = deep_m<D>(pz, x, x2);
        den[2 * r + 1] = deep_m<D>(pzg, x, x2);
    }
    // batch inversion in the base field; the norms are never zero (z is outside the base-field LDE domain with overwhelming
    // probability; a zero would also break the reference's synthetic division)
    u64 pre[2 * ROWS], run = 1;
#pragma unroll
    for (int q = 0; q < 2 * ROWS; q++) { pre[q] = run; run = gl_mul(run, den[q]); }
    run = gl_inv(run);
#pragma unroll
    for (int q = 2 * ROWS - 1; q >= 0; q--) { const u64 inv = gl_mul(run, pre[q]); run = gl_mul(run, den[q]); den[q] = inv; }
#pragma unroll
    for (int r = 0; r < ROWS; r++) {
        size_t row = tid + r * stride;
        if (row >= N) continue;
        u64* o = p.out.base + row * p.out.W;
        const GlExt<D> S = ld_ext<D>(o);
        const u64 x = D > 1 ? xs[r] : 0, x2 = D > 1 ? gl_sqr(x) : 0;
        const GlExt<D> a = ext_mul_base(ext_mul(ext_sub(S, Sz), deep_q<D>(pz, x, x2)), den[2 * r]);
        const GlExt<D> b = ext_mul_base(ext_mul(ext_sub(S, Szg), deep_q<D>(pzg, x, x2)), den[2 * r + 1]);
        const GlExt<D> v = ext_add(a, b);
#pragma unroll
        for (int q = 0; q < D; q++) o[q] = v.v[q];
    }
}
// host side of DeepPoint: the conjugates of z under the Frobenius map (math/src/field/f64/mod.rs:431, :490-498)
template <int D>
static bool deep_point(const GlExt<D>& z, DeepPoint<D>& pt) {
    pt.t = pt.s = pt.n = 0;
    pt.q1 = ext_zero<D>(); pt.q0 = ext_zero<D>();
    if (D == 1) { pt.n = z.v[0]; return true; }
    const GlExt<D> z1 = ext_frobenius(z);
    if (D == 2) {
        const GlExt<D> tr = ext_add(z, z1), nm = ext_mul(z, z1);
        pt.t = tr.v[0]; pt.n = nm.v[0]; pt.q0 = z1;
        return tr.v[1] == 0 && nm.v[1] == 0;
    }
    const GlExt<D> z2 = ext_frobenius(z1);
    const GlExt<D> tr = ext_add(z, ext_add(z1, z2));
    const GlExt<D> z12 = ext_mul(z1, z2);
    const GlExt<D> sm = ext_add(ext_mul(z, ext_add(z1, z2)), z12), nm = ext_mul(z, z12);
    pt.t = tr.v[0]; pt.s = sm.v[0]; pt.n = nm.v[0];
    pt.q1 = ext_add(z1, z2); pt.q0 = z12;
    bool ok = true;
    for (int k = 1; k < D; k++) ok = ok && tr.v[k] == 0 && sm.v[k] == 0 && nm.v[k] == 0;
    return ok;
}

// Proof-of-work grinding (K13; prover/src/channel.rs:169-184, crypto/src/random/default.rs:141-146):
// thread idx tests nonce = start + idx: trailing_zeros(LE u64 of merge_with_int(seed, nonce)[..8]) >=
// grinding. atomicMin keeps the SMALLEST qualifying nonce of the batch, and batches are scanned in
// increasing order, so the result is the serial-semantics nonce (the reference's `concurrent`
// find_any is nondeterministic; byte-identity is defined against the serial branch).
__global__ void __launch_bounds__(256) grind_kernel(int hash_id, const u64* seed /*4 words*/, u64 start, u64 count, u32 grinding,
                                                    unsigned long long* result) {
    u64 idx = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= count) return;
    u64 nonce = start + idx;
    u64 head;
    if (WF_HASH_IS_BLAKE3(hash_id)) {
        u32 ws[8], cv[8];
#pragma unroll
        for (int i = 0; i < 4; i++) { ws[2 * i] = (u32)seed[i]; ws[2 * i + 1] = (u32)(seed[i] >> 32); }
        if (hash_id == WF_HASH_BLAKE3_256) b3_merge_with_int_words<8>(ws, nonce, cv, b3_runtime_one());  // blake/mod.rs:41-46
        else b3_merge_with_int_words<6>(ws, nonce, cv, b3_runtime_one());                                 // :95-102
        head = (u64)cv[0] | ((u64)cv[1] << 32);
    } else {
        u64 sd[4], o[4];
#pragma unroll
        for (int i = 0; i < 4; i++) sd[i] = seed[i];
        if (hash_id == WF_HASH_RP64_256) alg_merge_with_int<WF_HASH_RP64_256>(sd, nonce, o);       // rp64_256/mod.rs:198-218
        else if (hash_id == WF_HASH_SHA3_256) alg_merge_with_int<WF_HASH_SHA3_256>(sd, nonce, o);  // sha/mod.rs:38-43
        else alg_merge_with_int<WF_HASH_RPJIVE64_256>(sd, nonce, o);                                // rp64_256_jive/mod.rs:206-229
        head = o[0];
    }
    u64 mask = grinding >= 64 ? ~0ULL : ((1ULL << grinding) - 1);
    if ((head & mask) == 0) atomicMin(result, (unsigned long long)nonce);
}

// =================================================================================================
// host orchestration
// =================================================================================================
static int grind_on_device(wf_ctx* ctx, int hash_id, const Digest& seed, u32 grinding, u64* nonce_out) {
    if (grinding == 0) { *nonce_out = 1; return WF_OK; }
    void *d_seed, *d_res;
    CKI(wf_dev_alloc(ctx, 32, &d_seed));
    CKI(wf_dev_alloc(ctx, 8, &d_res));
    CK(cudaMemcpyAsync(d_seed, seed.b, 32, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaMemsetAsync(d_res, 0xff, 8, ctx->st));
    const u64 batch = WF_HASH_IS_BLAKE3(hash_id) ? (1ULL << 20) : (1ULL << 16);
    u64 start = 1, found = ~0ULL;
    while (found == ~0ULL) {
        grind_kernel<<<(unsigned)((batch + 255) / 256), 256, 0, ctx->st>>>(hash_id, (const u64*)d_seed, start, batch, grinding,
                                                                         (unsigned long long*)d_res);
        ctx->launches++;
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(&found, d_res, 8, cudaMemcpyDeviceToHost, ctx->st));
        CK(cudaStreamSynchronize(ctx->st));
        start += batch;
    }
    wf_dev_free(ctx, d_seed);
    wf_dev_free(ctx, d_res);
    *nonce_out = found;
    return WF_OK;
}

namespace {

struct Options {
    u32 num_queries, blowup, grinding, ext, folding, rem_max_deg, batch_c, batch_d, num_partitions, hash_rate;
    int hash_id;
    // PartitionOptions::partition_size::<E>(num_columns) (air/src/options.rs:428-438) in BASE columns, for `cols` columns of
    // extension degree `deg`; cols * deg = the row is hashed whole (RowMatrix::commit_to_rows, row_matrix.rs:191-193)
    u32 part_words(u32 cols, u32 deg) const {
        if (num_partitions <= 1) return cols * deg;
        const u32 min_ps = hash_rate / deg, ps = (cols + num_partitions - 1) / num_partitions;
        return (ps > min_ps ? ps : min_ps) * deg;
    }
};

// Host-side AIR description (mirrors oracle/wf_prover.cpp `Air`; flat format documented at
// wf_prove_air in include/winterfell_b200.h)
// stride 0: Assertion::single; one value + stride: ::periodic; n / stride values: ::sequence
// (air/src/air/assertions/mod.rs:62-120). Main values: one word each; aux values: three words each.
struct AirAssertion { u64 column, first_step, stride; std::vector<u64> values; };
typedef AirAssertion AuxAssertion;
struct AirHost {
    u32 w = 0;
    // auxiliary segment (air/src/air/trace_info.rs:24-40): aw columns over E, nr random elements
    u32 aw = 0, nr = 0, aux_num_regs = 0;
    std::vector<std::pair<u32, std::vector<u32>>> aux_degrees;
    std::vector<u32> aux_prog;
    std::vector<AuxAssertion> aux_asserts;
    std::vector<std::pair<u32, std::vector<u32>>> all_degrees() const {  // context.rs:268-271
        auto r = degrees; r.insert(r.end(), aux_degrees.begin(), aux_degrees.end()); return r;
    }
    std::vector<u64> pub_inputs;
    std::vector<std::pair<u32, std::vector<u32>>> degrees;
    std::vector<std::vector<u64>> periodic;
    std::vector<u64> consts;
    std::vector<u32> prog;  // 4 words per instruction
    u32 num_regs = 0;
    std::vector<AirAssertion> asserts;
    u32 exemptions = 1;
    bool is_fib = false;  // FibSmall x k: use the specialised kernel
    u32 fib_k = 0;
    std::vector<u64> fib_results;
    u32 log_ce_blowup() const {  // air/src/air/context.rs:87-100, transition/degree.rs min_blowup_factor
        u32 r = 1;
        for (auto& dg : all_degrees()) {
            u32 bound = dg.first + (u32)dg.second.size() - 1, l = 0;
            while ((1u << l) < bound) l++;
            r = std::max(r, std::max(l, 1u));
        }
        return r;
    }
    u32 num_comp_cols(size_t n) const {  // context.rs:265-285
        size_t hi = 0;
        for (auto& dg : all_degrees()) {
            size_t e = (size_t)dg.first * (n - 1);
            for (u32 cyc : dg.second) e += (n / cyc) * (cyc - 1);
            hi = std::max(hi, e);
        }
        size_t div = n - exemptions;
        return (u32)std::max((hi - div + n - 1) / n, (size_t)1);
    }
    std::vector<AuxAssertion> sorted_aux_assertions() const {
        std::vector<AuxAssertion> a = aux_asserts;
        std::stable_sort(a.begin(), a.end(), [](const AuxAssertion& x, const AuxAssertion& y) {
            if (x.stride != y.stride) return x.stride < y.stride;
            if (x.first_step != y.first_step) return x.first_step < y.first_step;
            return x.column < y.column;
        });
        return a;
    }
    std::vector<AirAssertion> sorted_assertions() const {  // assertions/mod.rs:301-315
        std::vector<AirAssertion> a = asserts;
        std::stable_sort(a.begin(), a.end(), [](const AirAssertion& x, const AirAssertion& y) {
            if (x.stride != y.stride) return x.stride < y.stride;
            if (x.first_step != y.first_step) return x.first_step < y.first_step;
            return x.column < y.column;
        });
        return a;
    }
};
static AirHost fib_air_host(u32 k, size_t n, const u64* results) {
    AirHost a;
    a.w = 2 * k;
    a.pub_inputs.assign(results, results + k);
    a.is_fib = true; a.fib_k = k; a.fib_results.assign(results, results + k);
    for (u32 j = 0; j < k; j++) {
        a.degrees.push_back({1, {}});
        a.degrees.push_back({1, {}});
        a.asserts.push_back({2 * j, 0, 0, {(u64)(j + 1)}});
        a.asserts.push_back({2 * j + 1, 0, 0, {(u64)(j + 1)}});
        a.asserts.push_back({2 * j + 1, n - 1, 0, {results[j]}});
    }
    return a;
}
static bool parse_air_host(const u64* d, size_t len, AirHost& a) {
    size_t p = 0;
    auto rd = [&](u64& v) { if (p >= len) return false; v = d[p++]; return true; };
    u64 v, cnt;
    if (!rd(v) || v == 0 || v > 255) return false;
    a.w = (u32)v;
    if (!rd(cnt) || cnt == 0 || cnt > 4096) return false;
    for (u64 i = 0; i < cnt; i++) {
        u64 base, nc;
        if (!rd(base) || !rd(nc) || base == 0 || nc > 16) return false;
        std::vector<u32> cyc;
        // TransitionConstraintDegree::with_cycles asserts cycle lengths that are powers of two >= 2 (transition/degree.rs:62-79)
        for (u64 j = 0; j < nc; j++) { if (!rd(v) || v < 2 || (v & (v - 1)) || v > (1ull << 32)) return false; cyc.push_back((u32)v); }
        if (base + nc - 1 > 128) return false;  // min_blowup_factor would exceed the largest blowup (options.rs:132-190)
        a.degrees.push_back({(u32)base, cyc});
    }
    if (!rd(cnt) || cnt > 64) return false;
    for (u64 i = 0; i < cnt; i++) {
        u64 ln;
        if (!rd(ln) || ln < 2 || (ln & (ln - 1))) return false;
        std::vector<u64> col;
        for (u64 j = 0; j < ln; j++) { if (!rd(v) || v >= GL_P) return false; col.push_back(v); }
        a.periodic.push_back(col);
    }
    if (!rd(cnt)) return false;
    for (u64 i = 0; i < cnt; i++) { if (!rd(v) || v >= GL_P) return false; a.consts.push_back(v); }
    if (!rd(v) || v > GEN_MAX_REGS || v < 2 * a.w + a.periodic.size()) return false;
    a.num_regs = (u32)v;
    if (!rd(cnt) || cnt > (1u << 20)) return false;
    for (u64 i = 0; i < cnt; i++) {
        u64 op, ds, x, y;
        if (!rd(op) || !rd(ds) || !rd(x) || !rd(y) || op > 4) return false;
        const u64 first_tmp = 2 * a.w + a.periodic.size();  // inputs are read-only: boundary terms re-read them
        if (op == 4) { if (ds >= a.degrees.size() || x >= a.num_regs) return false; }
        else if (op == 3) { if (ds >= a.num_regs || ds < first_tmp || x >= a.consts.size()) return false; }
        else if (ds >= a.num_regs || ds < first_tmp || x >= a.num_regs || y >= a.num_regs) return false;
        a.prog.insert(a.prog.end(), {(u32)op, (u32)ds, (u32)x, (u32)y});
    }
    if (!rd(cnt) || cnt == 0) return false;
    for (u64 i = 0; i < cnt; i++) {
        AirAssertion as;
        u64 nv;
        if (!rd(as.column) || !rd(as.first_step) || !rd(as.stride) || !rd(nv) || as.column >= a.w || nv == 0 || nv > len) return false;
        for (u64 j = 0; j < nv; j++) { if (!rd(v) || v >= GL_P) return false; as.values.push_back(v); }
        a.asserts.push_back(as);
    }
    if (!rd(cnt)) return false;
    for (u64 i = 0; i < cnt; i++) { if (!rd(v) || v >= GL_P) return false; a.pub_inputs.push_back(v); }
    if (!rd(v) || v == 0 || v > 8) return false;
    a.exemptions = (u32)v;
    if (p == len) return true;
    // optional aux section: [aw, nr, nTa, {base, ncyc, cyc...}*, aux_num_regs, nIa, {op,dst,a,b}*,
    //                        nAa, {column, first_step, stride, nvals, {v0, v1, v2} x nvals}*]
    if (!rd(v) || v == 0 || v > 255) return false;
    a.aw = (u32)v;
    if (!rd(v) || v > 255) return false;
    a.nr = (u32)v;
    if (!rd(cnt) || cnt == 0 || cnt > 4096) return false;   // context.rs:104-113
    for (u64 i = 0; i < cnt; i++) {
        u64 base, nc;
        if (!rd(base) || !rd(nc) || base == 0 || nc > 16) return false;
        std::vector<u32> cyc;
        for (u64 j = 0; j < nc; j++) { if (!rd(v) || v < 2 || (v & (v - 1)) || v > (1ull << 32)) return false; cyc.push_back((u32)v); }
        if (base + nc - 1 > 128) return false;
        a.aux_degrees.push_back({(u32)base, cyc});
    }
    const u64 first_tmp = 2 * a.w + 2 * a.aw + a.periodic.size() + a.nr;
    if (!rd(v) || v > AUX_MAX_REGS || v < first_tmp) return false;
    a.aux_num_regs = (u32)v;
    if (!rd(cnt) || cnt > (1u << 20)) return false;
    for (u64 i = 0; i < cnt; i++) {
        u64 op, ds, x, y;
        if (!rd(op) || !rd(ds) || !rd(x) || !rd(y) || op > 4) return false;
        if (op == 4) { if (ds >= a.aux_degrees.size() || x >= a.aux_num_regs) return false; }
        else if (op == 3) { if (ds >= a.aux_num_regs || ds < first_tmp || x >= a.consts.size()) return false; }
        else if (ds >= a.aux_num_regs || ds < first_tmp || x >= a.aux_num_regs || y >= a.aux_num_regs) return false;
        a.aux_prog.insert(a.aux_prog.end(), {(u32)op, (u32)ds, (u32)x, (u32)y});
    }
    if (!rd(cnt) || cnt == 0) return false;
    for (u64 i = 0; i < cnt; i++) {
        AuxAssertion as;
        u64 nv;
        if (!rd(as.column) || !rd(as.first_step) || !rd(as.stride) || !rd(nv) || as.column >= a.aw || nv == 0 || nv > len) return false;
        for (u64 j = 0; j < 3 * nv; j++) { if (!rd(v) || v >= GL_P) return false; as.values.push_back(v); }
        a.aux_asserts.push_back(as);
    }
    return p == len;
}

template <int D>
struct Channel {  // ProverChannel (prover/src/channel.rs)
    PublicCoin coin;
    ByteVec commitments;
    Channel(int h, const std::vector<u64>& seed) : coin(h, seed.data(), seed.size()) {}
    void commit(const u8 root[32]) {  // commit_trace / commit_constraints / commit_fri_layer
        commitments.bytes(root, WF_DIGEST_BYTES(coin.hash_id));   // ByteDigest<N>::write_into: N bytes
        Digest d;
        memcpy(d.b, root, 32);
        coin.reseed(d);
    }
    GlExt<D> draw() {
        GlExt<D> r = ext_zero<D>();
        coin.draw(D, r.v);
        return r;
    }
    // air/src/air/coefficients.rs:201-218: Linear / Algebraic / Horner batching
    std::vector<GlExt<D>> draw_coeffs(u32 method, size_t n) {
        std::vector<GlExt<D>> r;
        if (method == 0) { for (size_t i = 0; i < n; i++) r.push_back(draw()); return r; }
        GlExt<D> a = draw(), x = ext_from_base<D>(1);
        for (size_t i = 0; i < n; i++) { r.push_back(x); x = ext_mul(x, a); }
        if (method == 2) std::reverse(r.begin(), r.end());
        return r;
    }
};

// Channel seed: Context::to_elements || public inputs (prover/src/channel.rs:57-82, air/src/air/context.rs:119-136), with
// TraceInfo::to_elements (air/src/air/trace_info.rs:209-238)
static std::vector<u64> channel_seed(const AirHost& air, size_t n, const Options& o) {
    const u32 c = air.w, aw = air.aw;
    const size_t n_cons = air.degrees.size() + air.aux_degrees.size() + air.asserts.size() + air.aux_asserts.size();
    const u64 ti0 = aw ? ((((((u64)c << 8) | 1) << 8) | aw) << 8) | air.nr : ((u64)c << 8);
    std::vector<u64> seed = {ti0, (u64)n, 1, 0xFFFFFFFFULL, (u64)n_cons,
                             ((u64)o.ext << 24) | ((u64)o.folding << 16) | ((u64)o.rem_max_deg << 8) | o.blowup,
                             o.grinding, o.num_queries};
    for (u64 v : air.pub_inputs) seed.push_back(v);
    return seed;
}
// Head of the proof object (prover/src/lib.rs:464-489; air/src/proof/mod.rs:189-200): the Context (context.rs:142-151:
// TraceInfo, modulus, ProofOptions, number of constraints), the number of query positions and the commitments
static void write_proof_head(ByteVec& w, const AirHost& air, u32 log_n, const Options& o, size_t num_positions, const ByteVec& commitments) {
    const size_t n_cons = air.degrees.size() + air.aux_degrees.size() + air.asserts.size() + air.aux_asserts.size();
    w.u8_((u8)air.w); w.u8_((u8)air.aw); w.u8_((u8)air.nr); w.u8_((u8)log_n); w.u16_(0);
    w.u8_(8); w.u64_(GL_P);
    w.u8_((u8)o.num_queries); w.u8_((u8)o.blowup); w.u8_((u8)o.grinding); w.u8_((u8)o.ext); w.u8_((u8)o.folding);
    w.u8_((u8)o.rem_max_deg); w.u8_((u8)o.batch_c); w.u8_((u8)o.batch_d); w.u8_((u8)o.num_partitions); w.u8_((u8)o.hash_rate);
    w.usize(n_cons);
    w.u8_((u8)num_positions);
    w.u16_((uint16_t)commitments.v.size());
    w.bytes(commitments.v.data(), commitments.v.size());
}

template <int D>
int upload_ext(wf_ctx* ctx, const std::vector<GlExt<D>>& v, size_t first, size_t count, u64** out) {
    void* p;
    CKI(wf_dev_alloc(ctx, std::max(count, (size_t)1) * D * 8, &p));
    std::vector<u64> flat(count * D);
    for (size_t i = 0; i < count; i++) for (int q = 0; q < D; q++) flat[i * D + q] = v[first + i].v[q];
    CK(cudaMemcpyAsync(p, flat.data(), flat.size() * 8, cudaMemcpyHostToDevice, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));  // `flat` is a stack object
    *out = (u64*)p;
    return WF_OK;
}

// evaluate all columns of the coefficient matrices at z0 and z1 -> host vectors [cols][D]
// (out[2m] = mats[m] @ z0, out[2m+1] = mats[m] @ z1); one synchronisation for all matrices
template <int D>
int ood_eval(wf_ctx* ctx, const std::vector<const wf_mat*>& mats, const GlExt<D>& z0, const GlExt<D>& z1,
             std::vector<std::vector<GlExt<D>>>& out) {
    const int nm = (int)mats.size();
    DevScratch tmp(ctx);               // every buffer below returns to the pool on any exit
    std::vector<void*> part(nm);
    void* res;
    size_t total_cols = 0;
    for (auto* m : mats) total_cols += m->m.cols;
    out.assign(2 * nm, {});
    CKI(tmp.alloc(total_cols * 2 * D * 8, &res));
    size_t off = 0;
    std::vector<void*> zbs(nm, nullptr);
    for (int m = 0; m < nm; m++) {
        const size_t n = mats[m]->m.rows;
        const u32 chunks = (u32)((n + OOD_ROWS_PER_BLOCK - 1) / OOD_ROWS_PER_BLOCK);
        const u32 cols = mats[m]->m.cols;
        CKI(tmp.alloc((size_t)cols * chunks * 2 * D * 8, &part[m]));
        CKI(tmp.alloc((size_t)2 * chunks * D * 8, &zbs[m]));
        ood_pow_kernel<D><<<(2 * chunks + 127) / 128, 128, 0, ctx->st>>>(z0, z1, chunks, (u64*)zbs[m]);
        ood_partial_kernel<D><<<dim3(chunks, mats[m]->m.nseg()), 256, 0, ctx->st>>>(mats[m]->m, z0, z1, (const u64*)zbs[m], (u64*)part[m], chunks);
        ood_reduce_kernel<D><<<(2 * cols * 32 + 255) / 256, 256, 0, ctx->st>>>((const u64*)part[m], cols, chunks, (u64*)res + off);
        ctx->launches += 3;
        CK(cudaGetLastError());
        off += (size_t)cols * 2 * D;
    }
    std::vector<u64> host(total_cols * 2 * D);
    CK(cudaMemcpyAsync(host.data(), res, host.size() * 8, cudaMemcpyDeviceToHost, ctx->st));
    CK(cudaStreamSynchronize(ctx->st));
    off = 0;
    for (int m = 0; m < nm; m++) {
        const u32 cols = mats[m]->m.cols;
        out[2 * m].resize(cols);
        out[2 * m + 1].resize(cols);
        for (u32 j = 0; j < cols; j++)
            for (int pt = 0; pt < 2; pt++)
                for (int q = 0; q < D; q++) out[2 * m + pt][j].v[q] = host[off + ((size_t)j * 2 + pt) * D + q];
        off += (size_t)cols * 2 * D;
    }
    return WF_OK;
}

template <int D>
void write_elems(ByteVec& w, const std::vector<GlExt<D>>& v) {
    for (auto& e : v) for (int q = 0; q < D; q++) w.u64_(e.v[q]);
}

// Queries::new (air/src/proof/queries.rs:51-78) + Serializable (:138-146), from batched gathers
void write_queries(const GatherBatch& gb, size_t row_id, size_t dig_id, size_t nvals, ByteVec& w) {
    ByteVec proof;
    wf_open_finish(gb.digs[dig_id].plan, gb.digest_result(dig_id), nullptr, proof);
    w.usize(nvals * 8);
    w.bytes(gb.row_result(row_id), nvals * 8);
    w.usize(proof.v.size());
    w.bytes(proof.v.data(), proof.v.size());
}

// cycle lengths of a TransitionConstraintDegree must not exceed the trace length (get_evaluation_degree,
// air/src/air/transition/degree.rs:85-97, divides trace_length by each cycle)
static int validate_degrees(wf_ctx* ctx, const std::vector<std::pair<u32, std::vector<u32>>>& degs, size_t n) {
    for (auto& dg : degs)
        for (u32 cyc : dg.second)
            if (cyc < 2 || (cyc & (cyc - 1)) || cyc > n) return wf_fail(ctx, WF_ERR_INVALID, "constraint degree cycle %u does not fit a trace of %zu rows", cyc, n);
    return WF_OK;
}

// Assertion validity (air/src/air/assertions/mod.rs:62-120, :166-230 validate_*)
static int validate_assertions(wf_ctx* ctx, const std::vector<AirAssertion>& as, size_t n, size_t words_per_value, const char* what) {
    for (auto& a : as) {
        const size_t nv = a.values.size() / words_per_value;
        bool ok = a.first_step < n && nv >= 1;
        if (a.stride != 0) ok = ok && a.stride >= 2 && !(a.stride & (a.stride - 1)) && a.stride <= n && a.first_step < a.stride;
        if (nv > 1) ok = ok && a.stride != 0 && !(nv & (nv - 1)) && nv * a.stride == n;   // sequence: one value per asserted step
        if (!ok) return wf_fail(ctx, WF_ERR_INVALID, "invalid %s", what);
    }
    // no two assertions may cover the same cell (Assertion::overlaps_with, assertions/mod.rs:175-208;
    // prepare_assertions panics on it, boundary/mod.rs:205-210)
    auto overlaps = [](const AirAssertion& s, const AirAssertion& o) {
        if (s.column != o.column) return false;
        if (s.first_step == o.first_step) return true;
        if (s.stride == o.stride) return false;
        const AirAssertion& lo = s.first_step < o.first_step ? s : o;
        const AirAssertion& hi = s.first_step < o.first_step ? o : s;
        if (lo.stride == 0) return false;  // the earlier one is a single assertion
        if (hi.stride == 0 || lo.stride < hi.stride) return (hi.first_step - lo.first_step) % lo.stride == 0;
        return false;
    };
    for (size_t i = 0; i < as.size(); i++)
        for (size_t j = i + 1; j < as.size(); j++)
            if (overlaps(as[i], as[j])) return wf_fail(ctx, WF_ERR_INVALID, "%s %zu overlaps with %zu", what, j, i);
    return WF_OK;
}

// Value table of a sequence assertion over the CE domain (LargePolyConstraint::new,
// prover/src/constraints/evaluator/boundary.rs:400-425): interpolate the L values over the size-L
// subgroup (air/src/air/boundary/constraint.rs:58-68), then evaluate that polynomial at 7 * w_ce^i for
// all i (coefficient k scaled by 7^k, zero-padded, one plain NTT of size ce). The reference's
// SmallPolyConstraint (Horner at x * g^(-first_step), :340-375) yields the same values, so one path
// serves both; the x offset becomes the row shift (i - first_step * ce_blowup) mod ce (:428-445).
static int sequence_table(wf_ctx* ctx, const u64* values, size_t L, u32 words_per_value, u32 dcols, size_t ce, wf_mat** out) {
    std::vector<u64> cols((size_t)dcols * L);
    std::vector<const u64*> ptr(dcols);
    for (u32 q = 0; q < dcols; q++) {
        for (size_t k = 0; k < L; k++) cols[q * L + k] = values[k * words_per_value + q];
        ptr[q] = &cols[q * L];
    }
    wf_mat *vals, *poly, *padded;
    CKI(wf_mat_from_host_columns(ctx, ptr.data(), dcols, L, 1, 0, &vals));  // synchronous w.r.t. `cols`
    CKI(wf_mat_interpolate(ctx, vals, &poly));
    wf_mat_free(ctx, vals);
    CKI(wf_mat_alloc(ctx, ce, dcols, &padded));
    CK(cudaMemsetAsync(padded->m.base, 0, padded->m.words() * 8, ctx->st));
    // dcols <= 3 -> one segment: the first L rows of `padded` are the L rows of `poly`
    CK(cudaMemcpyAsync(padded->m.base, poly->m.base, poly->m.words() * 8, cudaMemcpyDeviceToDevice, ctx->st));
    wf_mat_free(ctx, poly);
    CK(layout_scale_rows_by_powers(padded->m, GL_GENERATOR, ctx->st));
    ctx->launches++;
    int r = wf_mat_evaluate(ctx, padded, out);
    wf_mat_free(ctx, padded);
    return r;
}

// DefaultConstraintEvaluator::evaluate (prover/src/constraints/evaluator/default.rs:60-118) fused with
// ConstraintEvaluationTable::combine (evaluation_table.rs:163-407): the combined, divisor-normalised
// constraint evaluations over the CE domain = CompositionPolyTrace, as a (n * ce_blowup) x D matrix.
// cc: main transition, aux transition, main assertions, aux assertions (sorted order).
template <int D>
int eval_constraints(wf_ctx* ctx, const AirHost& air, const wf_mat* lde, const wf_mat* alde, const std::vector<GlExt<D>>& cc,
                     const std::vector<u64>& rnd_flat, u32 log_n, u32 log_b, wf_mat** out, size_t row0 = 0, size_t ce_rows = 0) {
    // ce_rows != 0: row-sharded call — CE rows [row0, row0 + ce_rows) only; `lde` then holds the LDE rows of that range
    // followed by `blowup` halo rows (FibEvalParams::row0, GenEvalParams::row0)
    const size_t n = (size_t)1 << log_n;
    const u32 c = air.w, aw = air.aw, log_ceb = air.log_ce_blowup();
    const u32 n_atr = (u32)air.aux_degrees.size(), n_mtr = (u32)air.degrees.size(), n_mas = (u32)air.asserts.size();
    const u32 n_tr = n_mtr + n_atr;
    const size_t ce = n << log_ceb;
    wf_mat* comp;
    CKI(wf_mat_alloc(ctx, ce_rows ? ce_rows : ce, D, &comp));
    if (comp->m.W > D) CK(cudaMemsetAsync(comp->m.base, 0, comp->m.words() * 8, ctx->st));
    const u64 g_tr = gl_root_of_unity(log_n);
    std::vector<u64> zt((size_t)1 << log_ceb);  // ce_blowup <= blowup <= 128 entries
    {   // x^n over the CE domain takes ce_blowup values: (7 w_ce^i)^n = 7^n * w_ceb^i
        u64 o_n = gl_pow(GL_GENERATOR, n), w_ceb = gl_root_of_unity(log_ceb);
        for (u32 i = 0; i < (1u << log_ceb); i++) zt[i] = gl_inv(gl_sub(gl_mul(o_n, gl_pow(w_ceb, i)), 1));
    }
    // device buffers of this stage; `comp` too until it is handed to the caller (returned to the pool on every error path)
    struct StageBufs {
        DevScratch dev;
        wf_mat* comp;
        std::vector<wf_mat*> mats;
        StageBufs(wf_ctx* c, wf_mat* m) : dev(c), comp(m) {}
        ~StageBufs() { if (comp) wf_mat_free(dev.ctx, comp); for (wf_mat* t : mats) wf_mat_free(dev.ctx, t); }
    } stage(ctx, comp);
    auto upload = [&](const void* src, size_t bytes, void** out) -> int {
        void* p;
        CKI(stage.dev.alloc(std::max(bytes, (size_t)8), &p));
        // stream-ordered copy; the (pageable) source vectors stay alive until the synchronisation below
        if (bytes) CK(cudaMemcpyAsync(p, src, bytes, cudaMemcpyHostToDevice, ctx->st));
        *out = p;
        return WF_OK;
    };
    auto flat = [&](size_t first, size_t count) {
        std::vector<u64> f(count * D);
        for (size_t i = 0; i < count; i++) for (int q = 0; q < D; q++) f[i * D + q] = cc[first + i].v[q];
        return f;
    };
    if (air.is_fib) {
        // boundary coefficients follow the assertions sorted by (stride, first_step, column)
        // (air/src/air/assertions/mod.rs:301-315): 2k assertions at step 0, then k at step n-1
        const u32 k = air.fib_k;
        void* d_cf = nullptr;
        std::vector<u64> cf((size_t)k * 5 * D);
        GlExt<D> K0 = ext_zero<D>(), K1 = ext_zero<D>();
        for (u32 j = 0; j < k; j++) {
            const GlExt<D>&tc0 = cc[2 * j], &tc1 = cc[2 * j + 1], &b0a = cc[n_tr + 2 * j], &b0b = cc[n_tr + 2 * j + 1], &b1 = cc[n_tr + 2 * k + j];
            for (int q = 0; q < D; q++) {
                u64* o = &cf[(size_t)j * 5 * D];
                o[q] = tc0.v[q]; o[D + q] = tc1.v[q]; o[2 * D + q] = b0a.v[q]; o[3 * D + q] = b0b.v[q]; o[4 * D + q] = b1.v[q];
            }
            // asserted values: columns 2j and 2j+1 start at j + 1, column 2j+1 ends at results[j] (fib_air_host)
            K0 = ext_add(K0, ext_mul_base(ext_add(b0a, b0b), (u64)(j + 1)));
            K1 = ext_add(K1, ext_mul_base(b1, air.fib_results[j]));
        }
        CKI(upload(cf.data(), cf.size() * 8, &d_cf));
        FibEvalParams p;
        memset(&p, 0, sizeof(p));
        p.lde = lde->m; p.out = comp->m; p.k = k; p.log_n = log_n; p.log_blowup = log_b; p.log_ce_blowup = log_ceb;
        p.coef = (const u64*)d_cf;
        for (int q = 0; q < D; q++) { p.K0[q] = K0.v[q]; p.K1[q] = K1.v[q]; }
        CKI(wf_get_twiddles(ctx, log_n + log_ceb, &p.tw_ce));
        p.last = gl_pow(g_tr, n - 1);
        if (log_ceb > 3) return wf_fail(ctx, WF_ERR_STATE, "FibSmall has degree-1 constraints");  // FibEvalParams::zt[8]
        for (u32 i = 0; i < (1u << log_ceb); i++) p.zt[i] = zt[i];
        p.row0 = row0; p.ce_rows = ce_rows;
        const size_t rows_per_thread = D == 3 ? FIB_ROWS_D3 : 4;
        size_t threads = ((ce_rows ? ce_rows : ce) + rows_per_thread - 1) / rows_per_thread;
        fib_constraints_kernel<D><<<(unsigned)((threads + 255) / 256), 256, cf.size() * 8, ctx->st>>>(p);
        ctx->launches++;
        CK(cudaGetLastError());
    } else {
        GenEvalParams p;
        memset(&p, 0, sizeof(p));
        p.lde = lde->m; p.out = comp->m; p.w = c; p.log_n = log_n; p.log_blowup = log_b; p.log_ce_blowup = log_ceb;
        p.prog_len = (u32)(air.prog.size() / 4); p.num_regs = air.num_regs; p.num_periodic = (u32)air.periodic.size(); p.num_tc = n_mtr;
        void* dp = nullptr;
        CKI(upload(air.prog.data(), air.prog.size() * 4, &dp)); p.prog = (u32*)dp;
        CKI(upload(air.consts.data(), air.consts.size() * 8, &dp)); p.consts = (u64*)dp;
        // periodic value tables (evaluator/periodic_table.rs:24-76): poly_j over offset^(n/L) <w_(L*ceb)>
        std::vector<u64> ptab;
        std::vector<u32> poff, plen;
        for (auto& col : air.periodic) {
            const size_t L = col.size(), M = L << log_ceb;
            std::vector<u64> v = col;
            wf_host_dft(v, L, 1, true, 1);              // get_periodic_column_polys (air/mod.rs:325-360)
            v.resize(M, 0);
            wf_host_dft(v, M, 1, false, gl_pow(GL_GENERATOR, n / L));
            poff.push_back((u32)ptab.size()); plen.push_back((u32)M);
            ptab.insert(ptab.end(), v.begin(), v.end());
        }
        CKI(upload(ptab.data(), ptab.size() * 8, &dp)); p.ptab = (u64*)dp;
        CKI(upload(poff.data(), poff.size() * 4, &dp)); p.ptab_off = (u32*)dp;
        CKI(upload(plen.data(), plen.size() * 4, &dp)); p.ptab_len = (u32*)dp;
        auto f0 = flat(0, n_mtr);
        CKI(upload(f0.data(), f0.size() * 8, &dp)); p.tcoef = (u64*)dp;
        // boundary groups: BTreeMap keyed by (stride, first_step) (air/src/air/boundary/mod.rs:154),
        // coefficients assigned in sorted-assertion order; divisor x^a - g^(a*first_step) (divisor.rs:44-56)
        auto as = air.sorted_assertions();
        std::map<std::pair<u64, u64>, std::vector<size_t>> groups;
        for (size_t i = 0; i < as.size(); i++) groups[{as[i].stride, as[i].first_step}].push_back(i);
        std::vector<u32> goff = {0}, ecol, etstride, eshift;
        std::vector<u64> ga, gb, goa, eval, ecc;
        std::vector<const u64*> etab;
        std::vector<wf_mat*>& seq_tables = stage.mats;  // returned to the pool when the stage ends (stream-ordered: after the kernel)
        for (auto& kv : groups) {
            u64 a = kv.first.first == 0 ? 1 : n / kv.first.first;
            ga.push_back(a);
            gb.push_back(kv.first.second == 0 ? 1 : gl_pow(g_tr, a * kv.first.second));
            goa.push_back(gl_pow(GL_GENERATOR, a));
            for (size_t i : kv.second) {
                ecol.push_back((u32)as[i].column); eval.push_back(as[i].values[0]);
                for (int q = 0; q < D; q++) ecc.push_back(cc[n_tr + i].v[q]);
                if (as[i].values.size() > 1) {
                    wf_mat* t;
                    CKI(sequence_table(ctx, as[i].values.data(), as[i].values.size(), 1, 1, ce, &t));
                    seq_tables.push_back(t);
                    etab.push_back(t->m.base); etstride.push_back((u32)t->m.W);
                    eshift.push_back((u32)(((u64)as[i].first_step << log_ceb) & (ce - 1)));
                } else { etab.push_back(nullptr); etstride.push_back(0); eshift.push_back(0); }
            }
            goff.push_back((u32)ecol.size());
        }
        p.num_groups = (u32)ga.size();
        CKI(upload(goff.data(), goff.size() * 4, &dp)); p.g_off = (u32*)dp;
        CKI(upload(ga.data(), ga.size() * 8, &dp)); p.g_a = (u64*)dp;
        CKI(upload(gb.data(), gb.size() * 8, &dp)); p.g_b = (u64*)dp;
        CKI(upload(goa.data(), goa.size() * 8, &dp)); p.g_oa = (u64*)dp;
        CKI(upload(ecol.data(), ecol.size() * 4, &dp)); p.e_col = (u32*)dp;
        CKI(upload(eval.data(), eval.size() * 8, &dp)); p.e_val = (u64*)dp;
        CKI(upload(ecc.data(), ecc.size() * 8, &dp)); p.e_cc = (u64*)dp;
        CKI(upload(etab.data(), etab.size() * 8, &dp)); p.e_tab = (const u64* const*)dp;
        CKI(upload(etstride.data(), etstride.size() * 4, &dp)); p.e_tstride = (u32*)dp;
        CKI(upload(eshift.data(), eshift.size() * 4, &dp)); p.e_shift = (u32*)dp;
        CKI(wf_get_twiddles(ctx, log_n + log_ceb, &p.tw_ce));
        CKI(upload(zt.data(), zt.size() * 8, &dp)); p.zt = (const u64*)dp;
        p.num_exempt = air.exemptions;
        for (u32 e = 0; e < air.exemptions; e++) p.exempt[e] = gl_pow(g_tr, n - air.exemptions + e);  // divisor.rs:31-41
        p.row0 = row0; p.ce_rows = ce_rows;   // run-time parameters: the compiled kernel of an AIR serves every rank
        std::vector<u32> agoff = {0}, aecol, aetstride, aeshift;
        std::vector<u64> aga, agb, agoa, aeval, aecc, fa;
        std::vector<const u64*> aetab;
        if (aw) {
            p.alde = alde->m; p.aw = aw; p.nr = air.nr; p.aprog_len = (u32)(air.aux_prog.size() / 4);
            CKI(upload(air.aux_prog.data(), air.aux_prog.size() * 4, &dp)); p.aprog = (u32*)dp;
            CKI(upload(rnd_flat.data(), rnd_flat.size() * 8, &dp)); p.rnd = (u64*)dp;
            fa = flat(n_mtr, n_atr);
            CKI(upload(fa.data(), fa.size() * 8, &dp)); p.atcoef = (u64*)dp;
            auto aas = air.sorted_aux_assertions();
            std::map<std::pair<u64, u64>, std::vector<size_t>> agroups;
            for (size_t i = 0; i < aas.size(); i++) agroups[{aas[i].stride, aas[i].first_step}].push_back(i);
            for (auto& kv : agroups) {
                u64 a = kv.first.first == 0 ? 1 : n / kv.first.first;
                aga.push_back(a);
                agb.push_back(kv.first.second == 0 ? 1 : gl_pow(g_tr, a * kv.first.second));
                agoa.push_back(gl_pow(GL_GENERATOR, a));
                for (size_t i : kv.second) {
                    aecol.push_back((u32)aas[i].column);
                    for (int q = 0; q < D; q++) { aeval.push_back(aas[i].values[q]); aecc.push_back(cc[n_tr + n_mas + i].v[q]); }
                    if (aas[i].values.size() > 3) {
                        wf_mat* t;
                        CKI(sequence_table(ctx, aas[i].values.data(), aas[i].values.size() / 3, 3, D, ce, &t));
                        seq_tables.push_back(t);
                        aetab.push_back(t->m.base); aetstride.push_back((u32)t->m.W);
                        aeshift.push_back((u32)(((u64)aas[i].first_step << log_ceb) & (ce - 1)));
                    } else { aetab.push_back(nullptr); aetstride.push_back(0); aeshift.push_back(0); }
                }
                agoff.push_back((u32)aecol.size());
            }
            p.num_agroups = (u32)aga.size();
            CKI(upload(agoff.data(), agoff.size() * 4, &dp)); p.ag_off = (u32*)dp;
            CKI(upload(aga.data(), aga.size() * 8, &dp)); p.ag_a = (u64*)dp;
            CKI(upload(agb.data(), agb.size() * 8, &dp)); p.ag_b = (u64*)dp;
            CKI(upload(agoa.data(), agoa.size() * 8, &dp)); p.ag_oa = (u64*)dp;
            CKI(upload(aecol.data(), aecol.size() * 4, &dp)); p.ae_col = (u32*)dp;
            CKI(upload(aeval.data(), aeval.size() * 8, &dp)); p.ae_val = (u64*)dp;
            CKI(upload(aecc.data(), aecc.size() * 8, &dp)); p.ae_cc = (u64*)dp;
            CKI(upload(aetab.data(), aetab.size() * 8, &dp)); p.ae_tab = (const u64* const*)dp;
            CKI(upload(aetstride.data(), aetstride.size() * 4, &dp)); p.ae_tstride = (u32*)dp;
            CKI(upload(aeshift.data(), aeshift.size() * 4, &dp)); p.ae_shift = (u32*)dp;
        }
        // the kernel compiled for this AIR (NVRTC, jit.cu) when there is one, else the interpreter
        cudaKernel_t jk = nullptr;
        const bool jit = ctx->jit_enabled &&
                         wf_jit_get_kernel(ctx, wf_jit_source(D, air.w, (u32)air.periodic.size(), air.num_regs, air.prog, air.consts, aw, air.nr,
                                                              air.aux_num_regs, air.aux_prog), &jk) == WF_OK;
        const unsigned blocks = (unsigned)(((ce_rows ? ce_rows : ce) + 127) / 128);
        if (jit) {
            void* args[] = {&p};
            CK(cudaLaunchKernel((const void*)jk, dim3(blocks), dim3(128), args, 0, ctx->st));
        } else if (aw) {
            generic_constraints_kernel<D, true><<<blocks, 128, 0, ctx->st>>>(p);
        } else {
            generic_constraints_kernel<D, false><<<blocks, 128, 0, ctx->st>>>(p);
        }
        ctx->launches++;
        CK(cudaGetLastError());
    }
    CK(cudaStreamSynchronize(ctx->st));
    stage.comp = nullptr;   // the caller's now
    *out = comp;
    return WF_OK;
}

// DefaultConstraintCommitment::new (prover/src/constraints/commitment/default.rs:44-150): composition
// trace (CE-domain evaluations, ce x D) -> CompositionPoly columns (n x kc*D coefficient matrix,
// composition_poly.rs:58-78,128-140), their LDE (N x kc*D) and the row commitment.
// CompositionPoly::new (composition_poly.rs:58-78): CE-domain evaluations -> kc column polynomials of degree < n
int composition_polys(wf_ctx* ctx, const wf_mat* comp, u32 log_n, int D, u32 kc, wf_mat** polys_out) {
    const size_t n = (size_t)1 << log_n;
    if (comp->m.rows < n * kc || (int)comp->m.cols != D) return wf_fail(ctx, WF_ERR_INVALID, "composition trace shape");
    wf_mat *ccoefs, *cpolys;
    // The composition polynomial has degree < kc * n by the AIR's declared degrees (that is what kc is computed from), so the
    // evaluations on the sub-coset 7 <w_m>, m = the power of two >= kc * n — every (ce / m)-th row of the CE domain — already
    // determine it: the size-m inverse transform returns exactly the coefficients the reference reads out of its size-ce one
    // (whose upper ce - kc * n coefficients are zero, composition_poly.rs:64-70). For FibSmall m = ce / 2.
    size_t m = n;
    while (m < n * kc) m <<= 1;
    if (m < comp->m.rows && comp->m.nseg() == 1) {
        wf_mat* sub;
        CKI(wf_mat_alloc_w(ctx, m, comp->m.cols, comp->m.W, &sub));
        const size_t rb = (size_t)comp->m.W * 8, stride = comp->m.rows / m;
        cudaError_t e = cudaMemcpy2DAsync(sub->m.base, rb, comp->m.base, stride * rb, rb, m, cudaMemcpyDeviceToDevice, ctx->st);
        int rc = e == cudaSuccess ? wf_mat_interpolate_with_offset(ctx, sub, GL_GENERATOR, &ccoefs)
                                  : wf_fail(ctx, WF_ERR_CUDA, "composition sub-coset copy: %s", cudaGetErrorString(e));
        wf_mat_free(ctx, sub);
        if (rc != WF_OK) return rc;
    } else {
        CKI(wf_mat_interpolate_with_offset(ctx, comp, GL_GENERATOR, &ccoefs));
    }
    CKI(wf_mat_alloc(ctx, n, kc * D, &cpolys));
    if (cpolys->m.W > (int)(kc * D)) CK(cudaMemsetAsync(cpolys->m.base, 0, cpolys->m.words() * 8, ctx->st));
    comp_split_kernel<<<(unsigned)((n * kc * D + 255) / 256), 256, 0, ctx->st>>>(ccoefs->m, n, kc, D, cpolys->m);
    ctx->launches++;
    CK(cudaGetLastError());
    wf_mat_free(ctx, ccoefs);
    wf_mark(ctx, "composition_interpolate");
    *polys_out = cpolys;
    return WF_OK;
}
int composition_commit(wf_ctx* ctx, int h, const wf_mat* comp, u32 log_n, u32 log_b, int D, u32 kc, wf_mat** polys_out,
                       wf_mat** lde_out, wf_tree** tree_out, u32 partition_words = 0) {
    wf_mat *cpolys = nullptr, *clde = nullptr;
    CKI(composition_polys(ctx, comp, log_n, D, kc, &cpolys));
    int r = wf_mat_lde(ctx, cpolys, log_b, &clde);
    if (r == WF_OK) {
        wf_mark(ctx, "composition_lde");
        if (tree_out) r = wf_commit_rows_partitioned(ctx, h, clde, partition_words, tree_out);  // sharded proofs commit their own row range
    }
    if (r != WF_OK) { wf_mat_free(ctx, cpolys); wf_mat_free(ctx, clde); return r; }
    *polys_out = cpolys;
    *lde_out = clde;
    return WF_OK;
}

// DeepCompositionPoly::{add_trace_polys, add_composition_poly, evaluate} (prover/src/composer/mod.rs:67-210)
// in evaluation form over the LDE domain (see the header of this file). dc: c + aw + kc coefficients.
template <int D>
int deep_compose(wf_ctx* ctx, const wf_mat* lde, const wf_mat* alde, const wf_mat* clde, u32 kc, u32 log_N,
                 const std::vector<GlExt<D>>& dc, const GlExt<D>& z, const GlExt<D>& zg, const GlExt<D>& Sz, const GlExt<D>& Szg,
                 wf_mat** out, size_t row0 = 0, size_t nrows = 0) {
    // nrows != 0: row-sharded call — the matrices hold LDE rows [row0, row0 + nrows) only
    const u32 c = lde->m.cols, aw = alde ? alde->m.cols / D : 0, ct = c + aw;
    const size_t N = nrows ? nrows : ((size_t)1 << log_N);
    u64 *d_dt, *d_dq, *d_da;
    CKI(upload_ext<D>(ctx, dc, 0, ct + kc, &d_dt));  // one upload (one synchronisation) for all coefficients
    d_da = d_dt + (size_t)c * D;
    d_dq = d_dt + (size_t)ct * D;
    wf_mat* deep;
    CKI(wf_mat_alloc(ctx, N, D, &deep));
    if (deep->m.W > D) CK(cudaMemsetAsync(deep->m.base, 0, deep->m.words() * 8, ctx->st));
    DeepParams p;
    p.trace = lde->m; p.cons = clde->m; p.out = deep->m; p.c = c; p.kc = kc; p.log_N = log_N;
    p.row0 = row0; p.nrows = nrows;
    p.tcc = d_dt; p.ccc = d_dq; p.acc = d_da; p.aw = aw;
    p.aux = aw ? alde->m : lde->m;
    CKI(wf_get_twiddles(ctx, log_N, &p.tw_N));
    const size_t coef_bytes = (size_t)(c + aw + kc) * D * 8;
    deep_sum_kernel<D><<<(unsigned)((N + DEEP_SUM_THREADS - 1) / DEEP_SUM_THREADS), DEEP_SUM_THREADS, coef_bytes, ctx->st>>>(p);
    const size_t rows_per_thread = DEEP_ROWS;
    size_t threads = (N + rows_per_thread - 1) / rows_per_thread;
    DeepPoint<D> pz, pzg;
    if (!deep_point<D>(z, pz) || !deep_point<D>(zg, pzg)) return wf_fail(ctx, WF_ERR_STATE, "conjugates of the out-of-domain point are inconsistent");
    deep_div_kernel<D><<<(unsigned)((threads + 255) / 256), 256, 0, ctx->st>>>(p, pz, pzg, Sz, Szg);
    ctx->launches += 2;
    CK(cudaGetLastError());
    // the coefficient buffers are pool allocations on the same stream: safe to release after the launch
    wf_dev_free(ctx, d_dt);
    *out = deep;
    return WF_OK;
}

// Device objects of one proof: whatever is still registered when prove_air leaves (normally or through
// an error return) goes back to the context's pool.
struct ProofScope {
    wf_ctx* ctx;
    std::vector<wf_mat**> mats;
    std::vector<wf_tree**> trees;
    wf_fri** fri = nullptr;
    explicit ProofScope(wf_ctx* c) : ctx(c) {}
    void own(std::initializer_list<wf_mat**> l) { mats.insert(mats.end(), l); }
    void own(std::initializer_list<wf_tree**> l) { trees.insert(trees.end(), l); }
    void drop(wf_mat*& m) { wf_mat_free(ctx, m); m = nullptr; }
    ~ProofScope() {
        if (fri && *fri) wf_fri_free(ctx, *fri);
        for (wf_mat** m : mats) if (*m) wf_mat_free(ctx, *m);
        for (wf_tree** t : trees) if (*t) wf_tree_free(ctx, *t);
    }
};

template <int D>
int prove_air(wf_ctx* ctx, const AirHost& air_in, const uint64_t* const* trace_cols, const uint64_t* d_trace, int mont, u32 log_n,
              const Options& o, wf_aux_builder_fn aux_builder, void* aux_user, std::vector<u8>& proof_out,
              wf_aux_assertions_fn aux_assertions = nullptr) {
    AirHost air_dyn;                       // copy whose aux assertion values are rewritten from the random elements
    if (aux_assertions) air_dyn = air_in;  // (Air::get_aux_assertions(aux_rand_elements), air/src/air/mod.rs:279)
    const AirHost& air = aux_assertions ? air_dyn : air_in;
    const int h = o.hash_id;
    const size_t n = (size_t)1 << log_n;
    u32 log_b = 0;
    while ((1u << log_b) < o.blowup) log_b++;
    const size_t N = n << log_b;
    const u32 c = air.w, kc = air.num_comp_cols(n), log_ceb = air.log_ce_blowup();
    const u32 aw = air.aw, n_atr = (u32)air.aux_degrees.size(), n_aas = (u32)air.aux_asserts.size();
    const u32 n_mtr = (u32)air.degrees.size(), n_mas = (u32)air.asserts.size();
    const u32 n_tr = n_mtr + n_atr, n_as = n_mas + n_aas;  // context.rs:205-207, :223-225
    if (aw && !aux_builder) return wf_fail(ctx, WF_ERR_INVALID, "multi-segment AIR needs an aux trace builder");
    if (log_ceb > log_b) return wf_fail(ctx, WF_ERR_INVALID, "blowup factor too small for the constraint degrees");
    for (auto& col : air.periodic) if (col.size() > n) return wf_fail(ctx, WF_ERR_INVALID, "periodic column longer than the trace");
    CKI(validate_degrees(ctx, air.all_degrees(), n));
    CKI(validate_assertions(ctx, air.aux_asserts, n, 3, "aux assertion"));
    CKI(validate_assertions(ctx, air.asserts, n, 1, "assertion"));
    Channel<D> ch(h, channel_seed(air, n, o));

    // ---- 1. trace commitment (lib.rs:497-522) ----
    wf_mat *trace = nullptr, *polys = nullptr, *lde = nullptr, *apolys = nullptr, *alde = nullptr, *comp = nullptr, *cpolys = nullptr,
           *clde = nullptr, *deep = nullptr;
    wf_tree *ttree = nullptr, *atree = nullptr, *ctree = nullptr;
    wf_fri* fri = nullptr;
    ProofScope scope(ctx);
    scope.own({&trace, &polys, &lde, &apolys, &alde, &comp, &cpolys, &clde, &deep});
    scope.own({&ttree, &atree, &ctree});
    scope.fri = &fri;
    wf_mark(ctx, "start");
    if (d_trace) {
        CKI(wf_mat_from_device_columns(ctx, d_trace, c, n, &trace));
        wf_mark(ctx, "trace_upload_layout");
        CKI(wf_mat_interpolate(ctx, trace, &polys));
        scope.drop(trace);
        wf_mark(ctx, "trace_interpolate");
        CKI(wf_mat_lde(ctx, polys, log_b, &lde));
    } else {
        // host trace: upload, layout, iNTT and LDE pipelined per column chunk (capi.cu)
        CKI(wf_trace_lde_from_host(ctx, trace_cols, c, n, mont, log_b, &polys, &lde));
    }
    wf_mark(ctx, "trace_lde");
    CKI(wf_commit_rows_partitioned(ctx, h, lde, o.part_words(c, 1), &ttree));
    u8 root[32];
    CKI(wf_tree_root(ctx, ttree, root));
    wf_mark(ctx, "trace_commit");
    ch.commit(root);

    // ---- 1b. auxiliary segment (lib.rs:309-349; Air::get_aux_rand_elements air/src/air/mod.rs:292-306;
    //          DefaultTraceLde::set_aux_trace trace_lde/default/mod.rs:140-166) ----
    std::vector<u64> rnd_flat;  // [nr][D], canonical
    if (aw) {
        for (u32 i = 0; i < air.nr; i++) { GlExt<D> e = ch.draw(); for (int q = 0; q < D; q++) rnd_flat.push_back(e.v[q]); }
        std::vector<u64> rnd_user = rnd_flat;
        if (mont) for (u64& v : rnd_user) v = gl_mul(v, 0xFFFFFFFFULL);  // x * R, R = 2^64 mod p
        std::vector<u64> aux_host((size_t)aw * n * D);  // [aw][n][D]: ColMatrix<E>, one Vec<E> per column
        if (aux_builder(aux_user, rnd_user.data(), aux_host.data()) != 0) return wf_fail(ctx, WF_ERR_INVALID, "aux trace builder failed");
        if (aux_assertions) {
            size_t total = 0;
            for (auto& a : air_dyn.aux_asserts) total += a.values.size() / 3;
            std::vector<u64> vals(total * D);
            size_t q = 0;
            for (auto& a : air_dyn.aux_asserts)
                for (size_t i = 0; i < a.values.size() / 3; i++, q++)
                    for (int k = 0; k < D; k++) vals[q * D + k] = mont ? gl_mul(a.values[i * 3 + k], 0xFFFFFFFFULL) : a.values[i * 3 + k];
            if (aux_assertions(aux_user, rnd_user.data(), vals.data()) != 0) return wf_fail(ctx, WF_ERR_INVALID, "aux assertion callback failed");
            q = 0;
            for (auto& a : air_dyn.aux_asserts)
                for (size_t i = 0; i < a.values.size() / 3; i++, q++)
                    for (int k = 0; k < 3; k++) {
                        u64 v = k < D ? vals[q * D + k] : 0;
                        if (mont) v = gl_from_mont(v);
                        else if (v >= GL_P) return wf_fail(ctx, WF_ERR_INVALID, "aux assertion value is not a canonical field element");
                        a.values[i * 3 + k] = v;
                    }
        }
        // E column j -> D base columns j*D + q (rows of the LDE then serialise exactly like [E] rows)
        std::vector<const u64*> cols(aw);
        for (u32 j = 0; j < aw; j++) cols[j] = &aux_host[(size_t)j * n * D];
        wf_mat* atrace = nullptr;
        CKI(wf_mat_from_host_columns(ctx, cols.data(), aw, n, D, mont, &atrace));
        int ir = wf_mat_interpolate(ctx, atrace, &apolys);
        wf_mat_free(ctx, atrace);
        if (ir != WF_OK) return ir;
        CKI(wf_mat_lde(ctx, apolys, log_b, &alde));
        CKI(wf_commit_rows_partitioned(ctx, h, alde, o.part_words(aw, D), &atree));
        CKI(wf_tree_root(ctx, atree, root));
        wf_mark(ctx, "aux_commit");
        ch.commit(root);
    }

    // ---- 2. constraint evaluation (lib.rs:373-378) ----
    // coefficient order: main transition, aux transition (transition/mod.rs:63-72), main assertions,
    // aux assertions (boundary/mod.rs:108-110)
    std::vector<GlExt<D>> cc = ch.draw_coeffs(o.batch_c, n_tr + n_as);
    CKI(eval_constraints<D>(ctx, air, lde, alde, cc, rnd_flat, log_n, log_b, &comp));
    wf_mark(ctx, "constraint_eval");
    // ---- 3. composition polynomial + commitment (lib.rs:527-552) ----
    CKI(composition_commit(ctx, h, comp, log_n, log_b, D, kc, &cpolys, &clde, &ctree, o.part_words(kc, D)));
    scope.drop(comp);
    CKI(wf_tree_root(ctx, ctree, root));
    wf_mark(ctx, "composition_commit");
    ch.commit(root);

    // ---- 4. out-of-domain frames (lib.rs:392-401) ----
    GlExt<D> z = ch.draw();
    GlExt<D> zg = ext_mul_base(z, gl_root_of_unity(log_n));
    std::vector<std::vector<GlExt<D>>> ood;
    {
        std::vector<const wf_mat*> mats = {polys, cpolys};
        if (aw) mats.push_back(apolys);
        CKI(ood_eval<D>(ctx, mats, z, zg, ood));
    }
    std::vector<GlExt<D>>&t_cur = ood[0], &t_nxt = ood[1], &qb_cur = ood[2], &qb_nxt = ood[3];  // qb_*: per base component column
    // H_j(z) = sum_comp phi^comp * (component column evaluated at z)
    auto combine = [&](const std::vector<GlExt<D>>& comp_evals) {
        std::vector<GlExt<D>> r(comp_evals.size() / D);
        for (u32 j = 0; j < r.size(); j++) {
            GlExt<D> acc = ext_zero<D>();
            for (int q = 0; q < D; q++) {
                GlExt<D> basis = ext_zero<D>();
                basis.v[q] = 1;
                acc = ext_add(acc, ext_mul(basis, comp_evals[j * D + q]));
            }
            r[j] = acc;
        }
        return r;
    };
    std::vector<GlExt<D>> q_cur = combine(qb_cur), q_nxt = combine(qb_nxt);
    if (aw) {  // trace frame rows = main columns then aux columns (ood_frame.rs:40-72)
        auto a_cur = combine(ood[4]), a_nxt = combine(ood[5]);
        t_cur.insert(t_cur.end(), a_cur.begin(), a_cur.end());
        t_nxt.insert(t_nxt.end(), a_nxt.begin(), a_nxt.end());
    }
    const u32 ct = c + aw;
    ByteVec ood_t, ood_q;  // OodFrame (air/src/proof/ood_frame.rs:59-72, :95-108)
    ood_t.u8_(2); write_elems<D>(ood_t, t_cur); write_elems<D>(ood_t, t_nxt);
    ood_q.u8_(2); write_elems<D>(ood_q, q_cur); write_elems<D>(ood_q, q_nxt);
    {
        ByteVec m;  // merge_ood_evaluations (:335-349): cur(trace, quotient), next(trace, quotient)
        write_elems<D>(m, t_cur); write_elems<D>(m, q_cur); write_elems<D>(m, t_nxt); write_elems<D>(m, q_nxt);
        Digest dg = hh_hash_elements(h, (const u64*)m.v.data(), m.v.size() / 8);
        ch.coin.reseed(dg);  // channel.rs:109-112 (not added to the commitments)
    }
    wf_mark(ctx, "ood_frames");
    // ---- 5. DEEP composition (lib.rs:403-440), evaluation form ----
    std::vector<GlExt<D>> dc = ch.draw_coeffs(o.batch_d, ct + kc);
    GlExt<D> Sz = ext_zero<D>(), Szg = ext_zero<D>();  // S(z), S(zg): the constant terms composer/mod.rs:202-210 subtracts
    for (u32 j = 0; j < ct; j++) { Sz = ext_add(Sz, ext_mul(dc[j], t_cur[j])); Szg = ext_add(Szg, ext_mul(dc[j], t_nxt[j])); }
    for (u32 j = 0; j < kc; j++) { Sz = ext_add(Sz, ext_mul(dc[ct + j], q_cur[j])); Szg = ext_add(Szg, ext_mul(dc[ct + j], q_nxt[j])); }
    CKI(deep_compose<D>(ctx, lde, alde, clde, kc, log_n + log_b, dc, z, zg, Sz, Szg, &deep));
    wf_mark(ctx, "deep_composition");
    // ---- 6. FRI (lib.rs:442-448) ----
    {   // transcript replicated on the device: one synchronisation for the whole commit phase (capi.cu)
        std::vector<Digest> fri_roots;
        CKI(wf_fri_build_layers_coin(ctx, h, deep, D, o.folding, o.rem_max_deg, o.blowup, ch.coin, fri_roots, &fri));
        for (auto& r : fri_roots) ch.commitments.bytes(r.b, WF_DIGEST_BYTES(h));
    }
    scope.drop(deep);
    wf_mark(ctx, "fri_layers");
    // ---- 7. grinding + query positions (channel.rs:151-184; serial semantics: smallest nonce) ----
    u64 nonce;
    CKI(grind_on_device(ctx, h, ch.coin.seed, o.grinding, &nonce));
    if (ch.coin.check_leading_zeros(nonce) < o.grinding) return wf_fail(ctx, WF_ERR_STATE, "grinding self-check failed");
    std::vector<u64> pos;
    if (!ch.coin.draw_integers(o.num_queries, N, nonce, pos)) return wf_fail(ctx, WF_ERR_STATE, "failed to draw query positions");
    std::sort(pos.begin(), pos.end());
    pos.erase(std::unique(pos.begin(), pos.end()), pos.end());
    wf_mark(ctx, "grinding");
    // ---- 8. proof object (lib.rs:464-489; air/src/proof/mod.rs:189-200) ----
    ByteVec w;
    write_proof_head(w, air, log_n, o, pos.size(), ch.commitments);
    // every gather of the proof (trace rows, constraint rows, all FRI layers + their Merkle paths)
    // goes through one batch: one index upload, one download, one synchronisation
    GatherBatch gb;
    FriProofPlan fplan;
    size_t tr_rows = gb.add_rows(lde->m, pos), cr_rows = gb.add_rows(clde->m, pos), tr_dig, cr_dig;
    size_t ar_rows = 0, ar_dig = 0;
    if (aw) ar_rows = gb.add_rows(alde->m, pos);
    CKI(gb.add_opening(ctx, ttree, pos, &tr_dig));
    CKI(gb.add_opening(ctx, ctree, pos, &cr_dig));
    if (aw) CKI(gb.add_opening(ctx, atree, pos, &ar_dig));
    CKI(wf_fri_queue_proof(ctx, fri, pos, gb, fplan));
    CKI(gb.run(ctx));
    write_queries(gb, tr_rows, tr_dig, pos.size() * c, w);
    if (aw) write_queries(gb, ar_rows, ar_dig, pos.size() * aw * D, w);  // trace_lde/default/mod.rs:199-218
    write_queries(gb, cr_rows, cr_dig, pos.size() * kc * D, w);
    w.u16_((uint16_t)ood_t.v.size()); w.bytes(ood_t.v.data(), ood_t.v.size());
    w.u16_((uint16_t)ood_q.v.size()); w.bytes(ood_q.v.data(), ood_q.v.size());
    wf_fri_finish_proof(fri, gb, fplan, w);
    w.u64_(nonce);
    wf_mark(ctx, "queries_and_proof");
    proof_out.swap(w.v);
    // `scope` returns every device object of this proof to the pool
    return WF_OK;
}

// =================================================================================================
// One proof sharded over several GPUs (include/winterfell_b200.h: wf_comm, wf_prove_fib_sharded)
// =================================================================================================
// staging: [b cosets][rows_j][W] (per segment) -> natural order row j * b + k of the row shard
__global__ void __launch_bounds__(256) coset_interleave_kernel(SegMatrix src, SegMatrix dst, size_t rows_j, u32 b) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // (row of dst, word)
    const int W = dst.W;
    if (idx >= dst.rows * (size_t)W) return;
    const size_t row = idx / W;
    const u32 w = (u32)(idx % W), g = blockIdx.y;
    const size_t j = row / b, k = row % b;
    dst.base[(size_t)g * dst.seg_stride + idx] = src.base[(size_t)g * src.seg_stride + (k * rows_j + j) * W + w];
}

struct ShardCtx {
    wf_ctx* ctx;
    const wf_comm* cm;
    int G, r;
    u32 logG;
    double bytes_sent = 0, bytes_overlapped = 0, ncoll = 0, ms_small = 0;
    bool forked = false;
    // exchanges issued between fork() and join() run on the communicator's stream, behind the ctx stream's tail at fork time
    // (wf_comm::fork / join; without the callbacks they simply stay on the ctx stream)
    int fork() {
        if (cm->fork) { if (cm->fork(cm->user) != 0) return wf_fail(ctx, WF_ERR_STATE, "fork callback failed"); forked = true; }
        return WF_OK;
    }
    int join() {
        if (forked) { forked = false; if (cm->join(cm->user) != 0) return wf_fail(ctx, WF_ERR_STATE, "join callback failed"); }
        return WF_OK;
    }
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev;  // around every exchange on the ctx stream (not the overlapped ones)
    ~ShardCtx() { for (auto& e : ev) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); } }
    // send[i] -> rank sp[i], recv[i] <- rank rp[i], all `bytes` long; entries naming this rank are not allowed
    int exchange(const std::vector<int>& sp, const std::vector<const void*>& sv, const std::vector<int>& rp, const std::vector<void*>& rv,
                 size_t bytes) {
        cudaEvent_t a = nullptr, b = nullptr;
        if (!forked) {
            CK(cudaEventCreate(&a));
            CK(cudaEventCreate(&b));
            ev.push_back({a, b});
            CK(cudaEventRecord(a, ctx->st));
        }
        if (cm->exchange(cm->user, sp.size(), sp.data(), sv.data(), rp.size(), rp.data(), rv.data(), bytes) != 0)
            return wf_fail(ctx, WF_ERR_STATE, "exchange callback failed");
        if (!forked) CK(cudaEventRecord(b, ctx->st));
        (forked ? bytes_overlapped : bytes_sent) += (double)bytes * (double)sp.size();
        ncoll += 1;
        return WF_OK;
    }
    // every rank contributes `bytes` device bytes at `mine`; all[q * bytes ..] receives rank q's (all-gather over exchange)
    int all_gather_dev(const void* mine, void* all, size_t bytes) {
        std::vector<int> sp, rp;
        std::vector<const void*> sv;
        std::vector<void*> rv;
        for (int q = 0; q < G; q++) {
            if (q == r) continue;
            sp.push_back(q); sv.push_back(mine);
            rp.push_back(q); rv.push_back((u8*)all + (size_t)q * bytes);
        }
        if ((const u8*)mine != (u8*)all + (size_t)r * bytes)
            CK(cudaMemcpyAsync((u8*)all + (size_t)r * bytes, mine, bytes, cudaMemcpyDeviceToDevice, ctx->st));
        return exchange(sp, sv, rp, rv, bytes);
    }
    int gather_host(const void* send, void* recv, size_t bytes) {
        cudaEvent_t a, b;  // host-side wall time is what this costs (the stream is already drained by the caller)
        (void)a; (void)b;
        const auto t0 = std::chrono::steady_clock::now();
        if (cm->all_gather_host(cm->user, send, recv, bytes) != 0) return wf_fail(ctx, WF_ERR_STATE, "all_gather_host callback failed");
        ms_small += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        ncoll += 1;
        return WF_OK;
    }
    // Maps the buffer at `local_base` (a cudaMalloc allocation of the same size on every rank) of every other rank into this
    // process (cudaIpcGetMemHandle -> all-gather of the handles -> cudaIpcOpenMemHandle, cached in the context). Returns
    // WF_ERR_UNSUPPORTED when the driver refuses (ranks on different nodes, IPC disabled): the caller then falls back to the
    // communicator's exchange.
    int map_peers(void* local_base, std::vector<void*>& out) {
        out.assign(G, nullptr);
        if (const char* e = getenv("WF_PEER_PUSH")) if (atoi(e) == 0) return WF_ERR_UNSUPPORTED;
        cudaIpcMemHandle_t h;
        memset(&h, 0, sizeof(h));
        int ok = cudaIpcGetMemHandle(&h, local_base) == cudaSuccess ? 1 : 0;
        if (!ok) cudaGetLastError();
        struct Msg { cudaIpcMemHandle_t h; int ok; int pad; } mine{h, ok, 0};
        std::vector<Msg> all(G);
        CKI(gather_host(&mine, all.data(), sizeof(Msg)));
        for (int q = 0; q < G; q++) ok &= all[q].ok;
        if (!ok) return WF_ERR_UNSUPPORTED;
        int opened = 1;
        for (int q = 0; q < G; q++) {
            if (q == r) { out[q] = local_base; continue; }
            std::string key((const char*)&all[q].h, sizeof(cudaIpcMemHandle_t));
            auto it = ctx->ipc_opened.find(key);
            if (it != ctx->ipc_opened.end()) { out[q] = it->second; continue; }
            void* pp = nullptr;
            if (cudaIpcOpenMemHandle(&pp, all[q].h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); opened = 0; continue; }
            ctx->ipc_opened[key] = pp;
            out[q] = pp;
        }
        // every rank must take the same path: agree on the outcome
        std::vector<int> flags(G);
        CKI(gather_host(&opened, flags.data(), sizeof(int)));
        for (int q = 0; q < G; q++) if (!flags[q]) return WF_ERR_UNSUPPORTED;
        return WF_OK;
    }
    int host_barrier() {
        int one = 1;
        std::vector<int> all(G);
        return gather_host(&one, all.data(), sizeof(int));
    }
    double exchange_ms() {
        double t = 0;
        for (auto& e : ev) { float ms = 0; if (cudaEventElapsedTime(&ms, e.first, e.second) == cudaSuccess) t += ms; }
        return t;
    }
};

// A Merkle tree of n_global leaves held as one subtree per rank (this rank's: `local`) plus the top log2(G) levels,
// recomputed on every rank from the all-gathered subtree roots: exactly the reference's heap (crypto/src/merkle/mod.rs:
// 344-368) because rank r's leaves [r n/G, (r+1) n/G) are the leaves of node G + r.
struct ShardTree {
    wf_tree* local = nullptr;
    size_t n_global = 0;
    std::vector<Digest> top;  // [1, G): internal nodes; [G, 2G): subtree roots
};
static int shard_tree_finish(ShardCtx& sc, int h, ShardTree& t, Digest* root) {
    wf_ctx* ctx = sc.ctx;
    Digest mine;
    CKI(wf_tree_root(ctx, t.local, mine.b));
    std::vector<Digest> all(sc.G);
    CKI(sc.gather_host(mine.b, all.data(), 32));
    t.top.assign(2 * sc.G, Digest{});
    for (int q = 0; q < sc.G; q++) t.top[sc.G + q] = all[q];
    for (int i = sc.G - 1; i >= 1; i--) t.top[i] = hh_merge(h, t.top[2 * i], t.top[2 * i + 1]);
    *root = t.top[1];
    return WF_OK;
}

// Trace columns of rank `rank` of `world` in a sharded proof: the S = ceil(width / 8) segments of the whole trace split as
// evenly as possible, rank r owning segments [floor(r S / world), floor((r+1) S / world)), i.e. the columns
// [*first, *first + *count). Narrow traces leave some ranks without a column (*count = 0). When 8 * world divides the width
// this is the block [r * width / world, (r+1) * width / world) of every rank.
static bool shard_columns(u32 width, int world, int rank, u32* first, u32* count) {
    if (width == 0 || width > 255 || world < 2 || (world & (world - 1)) || rank < 0 || rank >= world) return false;
    const u64 S = (width + 7) / 8;
    const u32 s0 = (u32)((u64)rank * S / (u64)world), s1 = (u32)((u64)(rank + 1) * S / (u64)world);
    *first = std::min(8 * s0, width);
    *count = std::min(8 * s1, width) - *first;
    return true;
}

// What a sharded proof needs of its shape; the same on every rank, checked before any device work
static int sharded_shape_check(wf_ctx* ctx, const AirHost& air, u32 log_n, const Options& o, int G, int r) {
    if (G < 2 || (G & (G - 1)) || r < 0 || r >= G) return wf_fail(ctx, WF_ERR_INVALID, "world size must be a power of two >= 2");
    // the FibSmall entry point keeps its contract: every rank passes a block of whole 8-column segments
    if (air.is_fib && (air.w % (u32)G || (air.w / (u32)G) % 8))
        return wf_fail(ctx, WF_ERR_UNSUPPORTED, "each rank must own whole 8-column segments (2k / world a multiple of 8)");
    u32 log_b = 0;
    while ((1u << log_b) < o.blowup) log_b++;
    const u32 log_ceb = air.log_ce_blowup();
    if (log_ceb > log_b) return wf_fail(ctx, WF_ERR_INVALID, "blowup factor too small for the constraint degrees");
    const size_t rows_per = ((size_t)1 << (log_n + log_b)) / (size_t)G, ce_per = ((size_t)1 << (log_n + log_ceb)) / (size_t)G;
    if (rows_per < 64 * (size_t)o.blowup || ce_per < 64) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "trace too short to shard over %d ranks", G);
    return WF_OK;
}

// Column ownership of one trace segment (shard_columns), in segments of the WHOLE segment's width Wg: the row shard, the staging
// buffer and every rank's local LDE use that width, so local segment g of rank q is global segment sg0[q] + g and blocks move
// as whole segment rows
struct ShardSplit {
    u32 c, nsg;
    int Wg;
    std::vector<u32> col0, ncol, sg0, nsl;
    ShardSplit(u32 cols, int G) : c(cols), Wg(seg_width_for(cols)), col0(G), ncol(G), sg0(G), nsl(G) {
        nsg = (c + Wg - 1) / Wg;
        for (int q = 0; q < G; q++) {
            shard_columns(c, G, q, &col0[q], &ncol[q]);
            sg0[q] = col0[q] / Wg;
            nsl[q] = (ncol[q] + Wg - 1) / Wg;
        }
    }
};

// One trace segment from this rank's columns to its row shard: interpolate the local base columns, extend them coset by coset
// (no communication: columns are independent) and move every rank's rows to it. *shard_out = LDE rows [r N/G, (r+1) N/G) of
// every column of the segment followed by `blowup` halo rows (the first rows of rank r + 1); *polys_out = the local columns'
// polynomials (none when the rank owns no column). Columns: resident d_local, or host columns of d-component elements starting
// at component q0 (wf_trace_lde_cosetwise). *path = the transport that ran: 2 fused scatter, 1 peer copies, 0 exchange.
static int segment_to_row_shard(ShardCtx& sc, const ShardSplit& sp, const uint64_t* const* cols, const uint64_t* d_local, int d, u32 q0,
                                int mont, u32 log_n, u32 log_b, wf_mat** polys_out, wf_mat** shard_out, int* path, const char* mark_lde) {
    wf_ctx* ctx = sc.ctx;
    const int G = sc.G, r = sc.r, Wg = sp.Wg;
    const u32 c = sp.c, nsg = sp.nsg, cl = sp.ncol[r];
    const std::vector<u32>&sg0 = sp.sg0, &nsl = sp.nsl;
    const size_t n = (size_t)1 << log_n, b = (size_t)1 << log_b, N = n << log_b, rows_per = N / (size_t)G;
    //         Coset k is written coset-major, so that the rows of rank q's range (n / G points of the coset) are one contiguous
    //         block per segment: its exchange runs on the communicator's stream while coset k + 1 is being extended
    const size_t nj = n / (size_t)G;   // points of one coset inside one rank's row range
    const size_t blk = nj * (size_t)Wg * 8;   // bytes of one (segment, coset, row range) block
    wf_mat *&polys = *polys_out, *&shard = *shard_out, *lde = nullptr, *stage = nullptr;
    ProofScope tmp(ctx);   // this segment's local LDE and staging buffer
    tmp.own({&lde, &stage});
    CKI(wf_mat_alloc(ctx, rows_per + b, c, &shard));   // segment width Wg
    shard->m.rows = rows_per;  // seg_stride stays (rows_per + b) * Wg: rows [rows_per, rows_per + b) are the halo
    const size_t sstride = shard->m.seg_stride;
    // Transport 1 — the exchange fused into the LDE: every rank maps the others' row shards (CUDA IPC) and the last
    // pass of every coset's transform writes each row straight to its owner (and the first rows of a range also into the halo
    // of the rank before it) with stores over NVLink: natural order at the destination, no staging buffer, no copy kernel,
    // no interleaving pass, nothing left to overlap. Closed by one stream synchronisation + host barrier.
    std::vector<void*> peer_shard;
    u32 log_nj = 0;
    while (((size_t)1 << log_nj) < nj) log_nj++;
    // (measured at 2 GPUs, cfg3: the remote 64-byte stores stall the pass by about what the transfer costs — 37.4 ms LDE + 0.6 ms
    // exposed against 30.3 + 5.6 with copy-engine pushes and 28.1 + 8.1 with a blocking NCCL all-to-all — so the fused form is
    // opt-in, WF_FUSED_SCATTER=1, and the copy-engine push below is the default). The fused form places rank r's segments at
    // one offset per rank: it needs every rank to own the same number of whole 8-column segments; other splits take the push.
    const char* fused_env = getenv("WF_FUSED_SCATTER");
    const bool even = c % (8 * (u32)G) == 0;
    const bool scat = fused_env && atoi(fused_env) != 0 && even && G <= 8 && log_n <= 22 && sc.map_peers(shard->m.base, peer_shard) == WF_OK;
    bool push = false;
    if (scat) {
        LdeScatter sct;
        for (int q = 0; q < 8; q++) sct.peer[q] = q < G ? (u64*)peer_shard[q] : nullptr;
        sct.seg_stride = sstride; sct.seg0 = sg0[r]; sct.log_nj = log_nj; sct.world = (u32)G;
        CKI(wf_trace_lde_cosetwise(ctx, cols, d_local, cl, n, mont, log_b, &polys, nullptr, false, nullptr, &sct, d, q0));
        wf_mark(ctx, mark_lde);
        CK(cudaStreamSynchronize(ctx->st));   // my stores have landed; everybody's have when every rank says so
        CKI(sc.host_barrier());
        sc.ncoll += 1;
        sc.bytes_overlapped += (double)(G - 1) * nsl[r] * (double)rows_per * Wg * 8;
        *path = 2;
        return WF_OK;
    }
    if (cl) CKI(wf_mat_alloc_w(ctx, N, cl, Wg, &lde));   // mine, coset-major: [local segment][coset][n][Wg]
    CKI(wf_mat_alloc_w(ctx, rows_per, c, Wg, &stage));   // what arrives: [global segment][coset][nj][Wg]
    // Preferred transport: every rank maps the others' `stage` buffers (CUDA IPC) and PUSHES its blocks there with peer copies
    // on side streams — copy engines over NVLink, no SM taken from the NTT kernels they overlap (NCCL send/recv kernels on a
    // side stream were measured: they slow the LDE down by as much as they hide). Fallback: the communicator's exchange.
    std::vector<void*> peer_stage;
    push = sc.map_peers(stage->m.base, peer_stage) == WF_OK;
    if (push) {
        for (int i = 0; i < 4; i++) if (!ctx->push_st[i]) CK(cudaStreamCreateWithFlags(&ctx->push_st[i], cudaStreamNonBlocking));
        for (int i = 0; i < 16; i++) if (!ctx->push_ev[i]) CK(cudaEventCreateWithFlags(&ctx->push_ev[i], cudaEventDisableTiming));
    }
    // block of my local segment sg, coset k, that belongs to rank q's rows; the block's place in a stage buffer
    auto my_block = [&](u32 sg, u32 k, int q) { return lde->m.base + (size_t)sg * lde->m.seg_stride + ((size_t)k * n + (size_t)q * nj) * Wg; };
    auto stage_block = [&](u64* base, u32 gseg, u32 k) { return base + (size_t)gseg * stage->m.seg_stride + (size_t)k * nj * Wg; };
    const std::function<int(u32)> after_coset = [&](u32 k) -> int {   // coset k of every local column is enqueued: ship it
        if (push) {
            cudaEvent_t ev = ctx->push_ev[k % 16];
            CK(cudaEventRecord(ev, ctx->st));
            for (int dq = 1; dq < G && nsl[r]; dq++) {   // start with the next rank: no two ranks hit the same peer first
                const int q = (r + dq) % G;
                cudaStream_t ps = ctx->push_st[dq % 4];
                CK(cudaStreamWaitEvent(ps, ev, 0));
                for (u32 sg = 0; sg < nsl[r]; sg++)
                    CK(cudaMemcpyAsync(stage_block((u64*)peer_stage[q], sg0[r] + sg, k), my_block(sg, k, q), blk, cudaMemcpyDeviceToDevice, ps));
            }
            for (u32 sg = 0; sg < nsl[r]; sg++)
                CK(cudaMemcpyAsync(stage_block(stage->m.base, sg0[r] + sg, k), my_block(sg, k, r), blk, cudaMemcpyDeviceToDevice, ctx->st));
            sc.bytes_overlapped += (double)(G - 1) * nsl[r] * blk;
            return WF_OK;
        }
        // pairwise order: sender r -> q lists my segments ascending; receiver r <- q lists q's segments ascending
        std::vector<int> spk, rp;
        std::vector<const void*> sv;
        std::vector<void*> rv;
        for (u32 sg = 0; sg < nsl[r]; sg++)
            for (int q = 0; q < G; q++) {
                if (q == r) CK(cudaMemcpyAsync(stage_block(stage->m.base, sg0[r] + sg, k), my_block(sg, k, r), blk, cudaMemcpyDeviceToDevice, ctx->st));
                else { spk.push_back(q); sv.push_back(my_block(sg, k, q)); }
            }
        for (int q = 0; q < G; q++)
            for (u32 sg = 0; q != r && sg < nsl[q]; sg++) { rp.push_back(q); rv.push_back(stage_block(stage->m.base, sg0[q] + sg, k)); }
        CKI(sc.fork());
        return sc.exchange(spk, sv, rp, rv, blk);
    };
    // (upload ->) layout -> interpolate -> extend, pipelined per column chunk for host columns; the cosets of the last chunk
    // are extended one by one and after_coset(k) ships coset k while coset k + 1 is computed. A rank without columns only
    // takes part in the exchanges.
    if (cl) CKI(wf_trace_lde_cosetwise(ctx, cols, d_local, cl, n, mont, log_b, &polys, &lde, true, &after_coset, nullptr, d, q0));
    else for (u32 k = 0; k < (u32)b; k++) CKI(after_coset(k));
    wf_mark(ctx, mark_lde);
    if (push) {
        // my pushes have landed when my side streams drain; everybody's have when every rank says so
        for (int i = 0; i < 4; i++) CK(cudaStreamSynchronize(ctx->push_st[i]));
        CKI(sc.host_barrier());
        sc.ncoll += 1;
    } else {
        CKI(sc.join());
    }
    {   // coset-major -> natural order (row = b j + k) of my row range, every segment
        SegMatrix dstv = shard->m;
        dim3 grid((unsigned)((rows_per * Wg + 255) / 256), nsg);
        coset_interleave_kernel<<<grid, 256, 0, ctx->st>>>(stage->m, dstv, nj, (u32)b);
        ctx->launches++;
        CK(cudaGetLastError());
    }
    tmp.drop(lde);
    tmp.drop(stage);
    {   // halo: the first `blowup` rows of every segment of rank (r + 1) mod G
        void *pk, *pk2;
        const size_t hb = b * Wg * 8;
        CKI(wf_dev_alloc(ctx, hb * nsg, &pk));
        CKI(wf_dev_alloc(ctx, hb * nsg, &pk2));
        CK(cudaMemcpy2DAsync(pk, hb, shard->m.base, sstride * 8, hb, nsg, cudaMemcpyDeviceToDevice, ctx->st));
        CKI(sc.exchange({(r + G - 1) % G}, {pk}, {(r + 1) % G}, {pk2}, hb * nsg));
        CK(cudaMemcpy2DAsync(shard->m.base + rows_per * Wg, sstride * 8, pk2, hb, hb, nsg, cudaMemcpyDeviceToDevice, ctx->st));
        wf_dev_free(ctx, pk);
        wf_dev_free(ctx, pk2);
    }
    *path = push ? 1 : 0;
    return WF_OK;
}

// FNV-1a, for the agreement steps of a sharded proof: what must be equal on every rank is hashed and the hashes all-gathered
struct Fnv {
    u64 h = 0xcbf29ce484222325ULL;
    void mix(u64 v) { for (int i = 0; i < 8; i++) { h ^= (v >> (8 * i)) & 0xff; h *= 0x100000001b3ULL; } }
};

// One proof sharded over the ranks of `cm` (wf_prove_fib_sharded, wf_prove_air_sharded, wf_prove_air_aux_sharded). The
// arguments have been checked on every rank alike; this rank passes the main columns shard_columns assigns it (none is
// possible) and, for a two-segment AIR, builds the aux columns it owns with aux_builder.
template <int D>
int prove_sharded(wf_ctx* ctx, const wf_comm* cm, const AirHost& air_in, const uint64_t* const* local_cols, const uint64_t* d_local, int mont,
                  u32 log_n, const Options& o, std::vector<u8>& proof_out, double* stats, wf_aux_shard_builder_fn aux_builder = nullptr,
                  wf_aux_assertions_fn aux_assertions = nullptr, void* aux_user = nullptr) {
    AirHost air_dyn;                       // copy whose aux assertion values are rewritten from the random elements (as prove_air)
    if (aux_assertions) air_dyn = air_in;
    const AirHost& air = aux_assertions ? air_dyn : air_in;
    ShardCtx sc{ctx, cm, cm->world, cm->rank, 0};
    const int G = sc.G, r = sc.r;
    CKI(sharded_shape_check(ctx, air, log_n, o, G, r));
    while ((1 << sc.logG) < G) sc.logG++;
    const int h = o.hash_id;
    const size_t n = (size_t)1 << log_n;
    u32 log_b = 0;
    while ((1u << log_b) < o.blowup) log_b++;
    const size_t N = n << log_b;
    const u32 c = air.w, aw = air.aw;
    const u32 kc = air.num_comp_cols(n), log_ceb = air.log_ce_blowup();
    const size_t rows_per = N / (size_t)G, ce = n << log_ceb, ce_per = ce / (size_t)G;
    const ShardSplit tsp(c, G), asp(aw * D, G);   // main columns; aux BASE columns (component q of E column j = j D + q)
    const std::vector<u32>&col0 = tsp.col0, &ncol = tsp.ncol;
    const u32 cl = ncol[r], acl = aw ? asp.ncol[r] : 0;
    const u32 n_tr = (u32)(air.degrees.size() + air.aux_degrees.size()), n_as = (u32)(air.asserts.size() + air.aux_asserts.size());
    Channel<D> ch(h, channel_seed(air, n, o));  // every rank replays the whole transcript

    wf_mat *polys = nullptr, *shard = nullptr, *apolys = nullptr, *ashard = nullptr, *comp_l = nullptr, *comp = nullptr, *cpolys = nullptr,
           *clde = nullptr, *deep = nullptr, *fri_in = nullptr;
    ShardTree ttree, atree, ctree;
    wf_fri* fri = nullptr;
    ProofScope scope(ctx);   // holds the ADDRESSES of these pointers: every owned pointer lives as long as the scope
    scope.own({&polys, &shard, &apolys, &ashard, &comp_l, &comp, &cpolys, &clde, &deep, &fri_in});
    scope.own({&ttree.local, &atree.local, &ctree.local});
    scope.fri = &fri;
    struct SLayer { u64* vals; size_t m_l, m_g; ShardTree tree; };
    std::vector<SLayer> slayers;   // FRI layers folded on row shards
    std::vector<void*> owned;      // device buffers of the sharded FRI phase
    struct Cleanup {
        wf_ctx* ctx; std::vector<SLayer>& sl; std::vector<void*>& ow;
        ~Cleanup() { for (auto& l : sl) wf_tree_free(ctx, l.tree.local); for (void* p : ow) wf_dev_free(ctx, p); }
    } cleanup{ctx, slayers, owned};

    // ---- 1-2. main trace: local columns -> LDE -> row shard with halo ----
    wf_mark(ctx, "start");
    int tpath = 0, apath = 0;
    CKI(segment_to_row_shard(sc, tsp, local_cols, d_local, 1, 0, mont, log_n, log_b, &polys, &shard, &tpath, "trace_lde"));
    wf_mark(ctx, "trace_exchange");
    // ---- 3. leaves + subtree over my rows, all-gather of the subtree roots ----
    Digest root;
    CKI(wf_commit_rows_partitioned(ctx, h, shard, o.part_words(c, 1), &ttree.local));
    ttree.n_global = N;
    CKI(shard_tree_finish(sc, h, ttree, &root));
    wf_mark(ctx, "trace_commit");
    ch.commit(root.b);
    // ---- 3b. auxiliary segment (prove_air 1b): every rank draws the random elements and builds the E columns that cover its
    //          aux base columns (an E column split between two ranks is built by both), the ranks agree on the callbacks'
    //          outcome, then the segment goes the main trace's way: LDE, row shard with halo, subtree, commitment ----
    std::vector<u64> rnd_flat;  // [nr][D], canonical
    double cb_ms = 0;
    if (aw) {
        for (u32 i = 0; i < air.nr; i++) { GlExt<D> e = ch.draw(); for (int q = 0; q < D; q++) rnd_flat.push_back(e.v[q]); }
        std::vector<u64> rnd_user = rnd_flat;
        if (mont) for (u64& v : rnd_user) v = gl_mul(v, 0xFFFFFFFFULL);  // x * R, R = 2^64 mod p
        const u32 af = asp.col0[r], e0 = af / D, ne = acl ? (af + acl + D - 1) / D - e0 : 0;
        std::vector<u64> aux_host((size_t)ne * n * D);  // [ne][n][D]: E columns [e0, e0 + ne)
        int st = WF_OK;
        const auto t0 = std::chrono::steady_clock::now();
        if (ne && aux_builder(aux_user, rnd_user.data(), e0, ne, aux_host.data()) != 0)
            st = wf_fail(ctx, WF_ERR_INVALID, "aux trace builder failed (rank %d, columns [%u, %u))", r, e0, e0 + ne);
        if (st == WF_OK && aux_assertions) {
            size_t total = 0;
            for (auto& a : air_dyn.aux_asserts) total += a.values.size() / 3;
            std::vector<u64> vals(total * D);
            size_t q = 0;
            for (auto& a : air_dyn.aux_asserts)
                for (size_t i = 0; i < a.values.size() / 3; i++, q++)
                    for (int k = 0; k < D; k++) vals[q * D + k] = mont ? gl_mul(a.values[i * 3 + k], 0xFFFFFFFFULL) : a.values[i * 3 + k];
            if (aux_assertions(aux_user, rnd_user.data(), vals.data()) != 0) st = wf_fail(ctx, WF_ERR_INVALID, "aux assertion callback failed");
            q = 0;
            for (auto& a : air_dyn.aux_asserts)
                for (size_t i = 0; st == WF_OK && i < a.values.size() / 3; i++, q++)
                    for (int k = 0; st == WF_OK && k < 3; k++) {
                        u64 v = k < D ? vals[q * D + k] : 0;
                        if (mont) v = gl_from_mont(v);
                        else if (v >= GL_P) st = wf_fail(ctx, WF_ERR_INVALID, "aux assertion value is not a canonical field element");
                        a.values[i * 3 + k] = v;
                    }
        }
        cb_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        wf_mark(ctx, "aux_build");
        // agreement: every rank takes the same way out of here, even when only one rank's callback failed
        Fnv vh;
        for (auto& a : air.aux_asserts) for (u64 v : a.values) vh.mix(v);
        struct Vote { int32_t status, pad; u64 hash; } v{st, 0, vh.h};
        std::vector<Vote> all(G);
        CKI(sc.gather_host(&v, all.data(), sizeof(Vote)));
        for (int q = 0; q < G; q++) {   // the lowest failing rank's status, on every rank
            if (all[q].status == WF_OK) continue;
            if (q == r) return st;
            return wf_fail(ctx, all[q].status, "rank %d's aux callbacks failed", q);
        }
        for (int q = 0; q < G; q++)
            if (all[q].hash != vh.h) return wf_fail(ctx, WF_ERR_INVALID, "ranks %d and %d computed different aux assertion values", r, q);
        std::vector<const u64*> ecols(ne);   // E column e0 + j -> base columns (e0 + j) D + q; mine start at component af % D
        for (u32 j = 0; j < ne; j++) ecols[j] = &aux_host[(size_t)j * n * D];
        CKI(segment_to_row_shard(sc, asp, ne ? ecols.data() : nullptr, nullptr, D, af % D, mont, log_n, log_b, &apolys, &ashard, &apath,
                                 "aux_lde"));
        wf_mark(ctx, "aux_exchange");
        CKI(wf_commit_rows_partitioned(ctx, h, ashard, o.part_words(aw, D), &atree.local));
        atree.n_global = N;
        CKI(shard_tree_finish(sc, h, atree, &root));
        wf_mark(ctx, "aux_commit");
        ch.commit(root.b);
    }
    // ---- 4. constraint evaluation over my CE rows; coefficient order as prove_air's ----
    std::vector<GlExt<D>> cc = ch.draw_coeffs(o.batch_c, n_tr + n_as);
    CKI(eval_constraints<D>(ctx, air, shard, ashard, cc, rnd_flat, log_n, log_b, &comp_l, (size_t)r * ce_per, ce_per));
    wf_mark(ctx, "constraint_eval");
    // ---- 5. composition polynomial: all-gather the CE evaluations (a few hundred MiB at most), interpolate + extend on
    //         every rank (the transform is over the row index), commit my row range ----
    CKI(wf_mat_alloc(ctx, ce, D, &comp));
    CKI(sc.all_gather_dev(comp_l->m.base, comp->m.base, ce_per * comp->m.W * 8));
    scope.drop(comp_l);
    const size_t b = o.blowup;
    wf_mat cview;  // my rows of the composition LDE
    if (b % (size_t)G == 0) {
        // the composition polynomial has too few columns to shard by column: shard its LDE by COSET instead. Rank r extends
        // cosets [r b/G, (r+1) b/G) (coset-major), one exchange hands every rank the rows of its row range from every coset's
        // owner, one kernel interleaves them into natural order (row = b j + k).
        CKI(composition_polys(ctx, comp, log_n, D, kc, &cpolys));
        scope.drop(comp);
        const u32 kpr = (u32)(b / (size_t)G);
        const size_t nj = n / (size_t)G;     // points of every coset that fall into one rank's row range
        wf_mat *ccos = nullptr, *stage = nullptr;
        CKI(wf_mat_alloc_w(ctx, (size_t)kpr * n, cpolys->m.cols, cpolys->m.W, &ccos));
        int rc = wf_mat_lde_cosets(ctx, cpolys, log_b, (u32)r * kpr, (u32)(r + 1) * kpr, ccos);
        if (rc == WF_OK) rc = wf_mat_alloc_w(ctx, rows_per, cpolys->m.cols, cpolys->m.W, &stage);
        if (rc == WF_OK) rc = wf_mat_alloc_w(ctx, rows_per, cpolys->m.cols, cpolys->m.W, &clde);
        if (rc != WF_OK) { wf_mat_free(ctx, ccos); wf_mat_free(ctx, stage); return rc; }
        wf_mark(ctx, "composition_lde");
        {
            const int W = cpolys->m.W;
            const size_t blk = nj * W;       // words of one (coset, destination) block of one segment
            std::vector<int> sp, rp;
            std::vector<const void*> sv;
            std::vector<void*> rv;
            for (u32 sg = 0; sg < ccos->m.nseg(); sg++) {
                const u64* cb = ccos->m.base + (size_t)sg * ccos->m.seg_stride;
                u64* sb = stage->m.base + (size_t)sg * stage->m.seg_stride;
                for (u32 kl = 0; kl < kpr; kl++)
                    for (int q = 0; q < G; q++) {
                        const u64* src = cb + ((size_t)kl * n + (size_t)q * nj) * W;
                        if (q == r) CK(cudaMemcpyAsync(sb + ((size_t)r * kpr + kl) * blk, src, blk * 8, cudaMemcpyDeviceToDevice, ctx->st));
                        else { sp.push_back(q); sv.push_back(src); }
                    }
                for (u32 k = 0; k < (u32)b; k++) {
                    const int owner = (int)(k / kpr);
                    if (owner != r) { rp.push_back(owner); rv.push_back(sb + (size_t)k * blk); }
                }
            }
            // pairwise order: sender r -> q lists (segment, local coset) ascending; receiver q <- s lists (segment, coset) ascending
            rc = sc.exchange(sp, sv, rp, rv, blk * 8);
            if (rc == WF_OK) {
                dim3 grid((unsigned)((rows_per * W + 255) / 256), clde->m.nseg());
                coset_interleave_kernel<<<grid, 256, 0, ctx->st>>>(stage->m, clde->m, nj, (u32)b);
                ctx->launches++;
                if (cudaGetLastError() != cudaSuccess) rc = wf_fail(ctx, WF_ERR_CUDA, "coset_interleave_kernel launch failed");
            }
        }
        wf_mat_free(ctx, ccos);
        wf_mat_free(ctx, stage);
        if (rc != WF_OK) return rc;
        cview.m = clde->m;               // clde IS my row shard
    } else {
        CKI(composition_commit(ctx, h, comp, log_n, log_b, D, kc, &cpolys, &clde, nullptr));
        scope.drop(comp);
        cview.m = clde->m;
        cview.m.base += (size_t)r * rows_per * clde->m.W;
        cview.m.rows = rows_per;
    }
    const bool comp_sharded = b % (size_t)G == 0;
    CKI(wf_commit_rows_partitioned(ctx, h, &cview, o.part_words(kc, D), &ctree.local));
    ctree.n_global = N;
    CKI(shard_tree_finish(sc, h, ctree, &root));
    wf_mark(ctx, "composition_commit");
    ch.commit(root.b);
    // ---- 6. out-of-domain frames: my columns' polynomials, all-gathered (every rank's part padded to the largest rank's
    //         column count: the gather takes equal sizes); composition columns are replicated ----
    GlExt<D> z = ch.draw();
    GlExt<D> zg = ext_mul_base(z, gl_root_of_unity(log_n));
    std::vector<std::vector<GlExt<D>>> ood;   // [0], [1]: composition columns at z, zg; then my trace columns, my aux base columns
    std::vector<const wf_mat*> om = {cpolys};
    if (cl) om.push_back(polys);
    if (acl) om.push_back(apolys);
    CKI(ood_eval<D>(ctx, om, z, zg, ood));
    std::vector<GlExt<D>> t_cur(c), t_nxt(c), ab_cur((size_t)aw * D), ab_nxt((size_t)aw * D);   // ab_*: per aux base column
    {
        const u32 cmax = *std::max_element(ncol.begin(), ncol.end()), amax = *std::max_element(asp.ncol.begin(), asp.ncol.end());
        const u32 amx = aw ? amax : 0, per = cmax + amx;   // one rank's part: its main columns, then its aux base columns
        std::vector<u64> mine((size_t)per * 2 * D, 0), all((size_t)G * per * 2 * D);
        auto put = [&](u32 slot, const GlExt<D>& x0, const GlExt<D>& x1) {
            for (int q = 0; q < D; q++) { mine[((size_t)slot * 2) * D + q] = x0.v[q]; mine[((size_t)slot * 2 + 1) * D + q] = x1.v[q]; }
        };
        for (u32 j = 0; j < cl; j++) put(j, ood[2][j], ood[3][j]);
        const size_t ai = cl ? 4 : 2;
        for (u32 j = 0; j < acl; j++) put(cmax + j, ood[ai][j], ood[ai + 1][j]);
        CKI(sc.gather_host(mine.data(), all.data(), mine.size() * 8));
        for (int rq = 0; rq < G; rq++) {
            for (u32 j = 0; j < ncol[rq]; j++) {
                const u64* e = &all[((size_t)rq * per + j) * 2 * D];
                for (int q = 0; q < D; q++) { t_cur[col0[rq] + j].v[q] = e[q]; t_nxt[col0[rq] + j].v[q] = e[D + q]; }
            }
            for (u32 j = 0; aw && j < asp.ncol[rq]; j++) {
                const u64* e = &all[((size_t)rq * per + cmax + j) * 2 * D];
                for (int q = 0; q < D; q++) { ab_cur[asp.col0[rq] + j].v[q] = e[q]; ab_nxt[asp.col0[rq] + j].v[q] = e[D + q]; }
            }
        }
    }
    auto combine = [&](const std::vector<GlExt<D>>& comp_evals) {  // H_j(z) from its base-component columns
        std::vector<GlExt<D>> rr(comp_evals.size() / D);
        for (u32 j = 0; j < rr.size(); j++) {
            GlExt<D> acc = ext_zero<D>();
            for (int q = 0; q < D; q++) {
                GlExt<D> basis = ext_zero<D>();
                basis.v[q] = 1;
                acc = ext_add(acc, ext_mul(basis, comp_evals[j * D + q]));
            }
            rr[j] = acc;
        }
        return rr;
    };
    std::vector<GlExt<D>> q_cur = combine(ood[0]), q_nxt = combine(ood[1]);
    if (aw) {  // trace frame rows = main columns then aux columns; an E column's components may come from two ranks
        auto a_cur = combine(ab_cur), a_nxt = combine(ab_nxt);
        t_cur.insert(t_cur.end(), a_cur.begin(), a_cur.end());
        t_nxt.insert(t_nxt.end(), a_nxt.begin(), a_nxt.end());
    }
    const u32 ct = c + aw;
    ByteVec ood_t, ood_q;
    ood_t.u8_(2); write_elems<D>(ood_t, t_cur); write_elems<D>(ood_t, t_nxt);
    ood_q.u8_(2); write_elems<D>(ood_q, q_cur); write_elems<D>(ood_q, q_nxt);
    {
        ByteVec m;
        write_elems<D>(m, t_cur); write_elems<D>(m, q_cur); write_elems<D>(m, t_nxt); write_elems<D>(m, q_nxt);
        Digest dg = hh_hash_elements(h, (const u64*)m.v.data(), m.v.size() / 8);
        ch.coin.reseed(dg);
    }
    wf_mark(ctx, "ood_frames");
    // ---- 7. DEEP composition over my LDE rows (evaluation form is row-local) ----
    std::vector<GlExt<D>> dc = ch.draw_coeffs(o.batch_d, ct + kc);
    GlExt<D> Sz = ext_zero<D>(), Szg = ext_zero<D>();
    for (u32 j = 0; j < ct; j++) { Sz = ext_add(Sz, ext_mul(dc[j], t_cur[j])); Szg = ext_add(Szg, ext_mul(dc[j], t_nxt[j])); }
    for (u32 j = 0; j < kc; j++) { Sz = ext_add(Sz, ext_mul(dc[ct + j], q_cur[j])); Szg = ext_add(Szg, ext_mul(dc[ct + j], q_nxt[j])); }
    CKI(deep_compose<D>(ctx, shard, ashard, &cview, kc, log_n + log_b, dc, z, zg, Sz, Szg, &deep, (size_t)r * rows_per, rows_per));
    wf_mark(ctx, "deep_composition");
    // ---- 8. FRI: layers folded on shards while they are large. A layer of L points is held as contiguous position
    //         ranges; leaf i joins positions i, i + L/nf, ...: one exchange gives the owner of leaf range o (L/nf/G leaves)
    //         its nf pieces, which then look like a complete layer of nf * L/nf/G points to the hash and fold kernels ----
    const u32 nf = o.folding;
    const int ld = deep->m.W;
    const size_t max_rem = (size_t)(o.rem_max_deg + 1) * o.blowup;
    u64* cur = deep->m.base;  // my range of the current layer: L / G elements, ld words each
    size_t L = N;
    // a layer stays sharded while a rank's range has >= 2^17 elements (below that one exchange + two host round trips per
    // layer cost more than folding the whole layer everywhere); WF_SHARD_FRI_MIN_LOG lowers the bound for small tests
    u32 min_log = 17;
    if (const char* e = getenv("WF_SHARD_FRI_MIN_LOG")) min_log = (u32)atoi(e);
    while (L > max_rem && L / (size_t)G >= ((size_t)1 << min_log) && (L / nf) % (size_t)G == 0 && L / nf / (size_t)G >= 2) {
        SLayer sl;
        sl.m_g = L / nf;
        sl.m_l = sl.m_g / (size_t)G;
        void* vp;
        CKI(wf_dev_alloc(ctx, (size_t)nf * sl.m_l * ld * 8, &vp));
        owned.push_back(vp);
        sl.vals = (u64*)vp;
        std::vector<int> sp, rp;
        std::vector<const void*> sv;
        std::vector<void*> rv;
        for (u32 t = 0; t < nf; t++) {  // my range = pieces nf*r .. nf*r + nf - 1 of the layer; piece P belongs to leaf range P % G, slot P / G
            const size_t P = (size_t)nf * r + t;
            const int owner = (int)(P % (size_t)G);
            const size_t q = P / (size_t)G;
            const u64* src = cur + (size_t)t * sl.m_l * ld;
            if (owner == r) CK(cudaMemcpyAsync(sl.vals + q * sl.m_l * ld, src, sl.m_l * ld * 8, cudaMemcpyDeviceToDevice, ctx->st));
            else { sp.push_back(owner); sv.push_back(src); }
        }
        for (u32 q = 0; q < nf; q++) {
            const size_t P = (size_t)q * G + r;
            const int src_rank = (int)(P / nf);
            if (src_rank != r) { rp.push_back(src_rank); rv.push_back(sl.vals + (size_t)q * sl.m_l * ld); }
        }
        CKI(sc.exchange(sp, sv, rp, rv, sl.m_l * ld * 8));
        CKI(wf_fri_layer_tree(ctx, h, sl.vals, (size_t)nf * sl.m_l, D, ld, (int)nf, &sl.tree.local));
        sl.tree.n_global = sl.m_g;
        slayers.push_back(sl);
        CKI(shard_tree_finish(sc, h, slayers.back().tree, &root));
        ch.commit(root.b);              // commit_fri_layer, then draw_fri_alpha (prover/src/channel.rs:215-234)
        GlExt<D> alpha = ch.draw();
        u32 logL = 0;
        while (((size_t)1 << logL) < L) logL++;
        const u64* master;
        CKI(wf_get_twiddles(ctx, logL, &master));
        void* nx;
        CKI(wf_dev_alloc(ctx, sl.m_l * ld * 8, &nx));
        owned.push_back(nx);
        if (ld > D) CK(cudaMemsetAsync(nx, 0, sl.m_l * ld * 8, ctx->st));
        u64 av[3] = {0, 0, 0};
        for (int q = 0; q < D; q++) av[q] = alpha.v[q];
        CK(fri_fold_layer(sl.vals, (size_t)nf * sl.m_l, D, ld, (int)nf, av, master, (u64*)nx, ld, ctx->st, nullptr, (size_t)r * sl.m_l, logL));
        ctx->launches++;
        cur = (u64*)nx;
        L = sl.m_g;
    }
    // the rest of the commit phase on every rank: all-gather the current layer (small by now)
    CKI(wf_mat_alloc(ctx, L, D, &fri_in));
    CKI(sc.all_gather_dev(cur, fri_in->m.base, (L / (size_t)G) * ld * 8));
    scope.drop(deep);
    {
        std::vector<Digest> fri_roots;
        CKI(wf_fri_build_layers_coin(ctx, h, fri_in, D, o.folding, o.rem_max_deg, o.blowup, ch.coin, fri_roots, &fri));
        for (auto& rt : fri_roots) ch.commitments.bytes(rt.b, WF_DIGEST_BYTES(h));
    }
    scope.drop(fri_in);
    wf_mark(ctx, "fri_layers");
    // ---- 9. grinding + query positions (every rank; deterministic) ----
    u64 nonce;
    CKI(grind_on_device(ctx, h, ch.coin.seed, o.grinding, &nonce));
    if (ch.coin.check_leading_zeros(nonce) < o.grinding) return wf_fail(ctx, WF_ERR_STATE, "grinding self-check failed");
    std::vector<u64> pos;
    if (!ch.coin.draw_integers(o.num_queries, N, nonce, pos)) return wf_fail(ctx, WF_ERR_STATE, "failed to draw query positions");
    std::sort(pos.begin(), pos.end());
    pos.erase(std::unique(pos.begin(), pos.end()), pos.end());
    wf_mark(ctx, "grinding");
    // ---- 10. proof object: every rank queues the same gathers, contributes what it holds, the words are summed ----
    ByteVec w;
    write_proof_head(w, air, log_n, o, pos.size(), ch.commitments);
    GatherBatch gb;
    gb.comm = cm;
    const u64 NONE = ~(u64)0;
    auto owned_rows = [&](const std::vector<u64>& p, size_t per) {  // global row -> my local row, or NONE
        std::vector<u64> l(p.size(), NONE);
        for (size_t i = 0; i < p.size(); i++) if ((int)(p[i] / per) == r) l[i] = p[i] % per;
        return l;
    };
    std::vector<std::pair<size_t, u64>> top_t, top_a, top_c;
    size_t tr_rows = gb.add_rows(shard->m, owned_rows(pos, rows_per));
    size_t ar_rows = 0, ar_dig = 0;
    if (aw) ar_rows = gb.add_rows(ashard->m, owned_rows(pos, rows_per));
    size_t cr_rows = comp_sharded ? gb.add_rows(cview.m, owned_rows(pos, rows_per))
                                  : gb.add_rows(clde->m, r == 0 ? pos : std::vector<u64>(pos.size(), NONE));  // replicated: rank 0 contributes
    size_t tr_dig, cr_dig;
    CKI(gb.add_opening_sharded(ctx, ttree.local, N, G, r, pos, &tr_dig, &top_t));
    CKI(gb.add_opening_sharded(ctx, ctree.local, N, G, r, pos, &cr_dig, &top_c));
    if (aw) CKI(gb.add_opening_sharded(ctx, atree.local, N, G, r, pos, &ar_dig, &top_a));
    struct SQ { size_t row_id, dig_id, nq; std::vector<std::pair<size_t, u64>> top; };
    std::vector<SQ> sq;
    std::vector<u64> fpos = pos;
    for (auto& sl : slayers) {  // FriProver::build_proof (fri/src/prover/mod.rs:254-319) on the sharded layers
        std::vector<u64> fp;    // fold_positions (fri/src/folding/mod.rs:159-176)
        for (u64 p : fpos) { u64 q = p % sl.m_g; if (std::find(fp.begin(), fp.end(), q) == fp.end()) fp.push_back(q); }
        fpos = fp;
        std::vector<u64> gpos(fpos.size() * nf, NONE);
        for (size_t i = 0; i < fpos.size(); i++)
            if ((int)(fpos[i] / sl.m_l) == r)
                for (u32 j = 0; j < nf; j++) gpos[i * nf + j] = (u64)j * sl.m_l + fpos[i] % sl.m_l;
        SegMatrix lm;
        lm.base = sl.vals; lm.rows = (size_t)nf * sl.m_l; lm.cols = (u32)D; lm.W = ld; lm.seg_stride = lm.rows * ld;
        SQ e;
        e.row_id = gb.add_rows(lm, gpos);
        CKI(gb.add_opening_sharded(ctx, sl.tree.local, sl.m_g, G, r, fpos, &e.dig_id, &e.top));
        e.nq = fpos.size();
        sq.push_back(e);
    }
    FriProofPlan fplan;
    {
        const size_t r0 = gb.rows.size(), d0 = gb.digs.size();
        CKI(wf_fri_queue_proof(ctx, fri, fpos, gb, fplan));
        if (r != 0) {  // replicated layers: rank 0 contributes
            for (size_t i = r0; i < gb.rows.size(); i++) std::fill(gb.rows[i].pos.begin(), gb.rows[i].pos.end(), NONE);
            for (size_t i = d0; i < gb.digs.size(); i++) std::fill(gb.digs[i].idx.begin(), gb.digs[i].idx.end(), NONE);
        }
    }
    CKI(gb.run(ctx));
    auto patch = [&](size_t dig_id, const std::vector<std::pair<size_t, u64>>& slots, const ShardTree& t) {
        for (auto& se : slots) memcpy(gb.digest_words(dig_id) + se.first * 4, t.top[se.second].b, 32);
    };
    patch(tr_dig, top_t, ttree);
    patch(cr_dig, top_c, ctree);
    if (aw) patch(ar_dig, top_a, atree);
    for (size_t i = 0; i < sq.size(); i++) patch(sq[i].dig_id, sq[i].top, slayers[i].tree);
    write_queries(gb, tr_rows, tr_dig, pos.size() * c, w);
    if (aw) write_queries(gb, ar_rows, ar_dig, pos.size() * aw * D, w);
    write_queries(gb, cr_rows, cr_dig, pos.size() * kc * D, w);
    w.u16_((uint16_t)ood_t.v.size()); w.bytes(ood_t.v.data(), ood_t.v.size());
    w.u16_((uint16_t)ood_q.v.size()); w.bytes(ood_q.v.data(), ood_q.v.size());
    {   // FriProof (fri/src/proof.rs:149-163, 275-285): sharded layers, then the replicated ones
        w.u8_((u8)(slayers.size() + fri->layers.size()));
        for (size_t l = 0; l < sq.size(); l++) {
            const size_t nvals = sq[l].nq * nf * D;
            ByteVec paths;
            wf_open_finish(gb.digs[sq[l].dig_id].plan, gb.digest_result(sq[l].dig_id), nullptr, paths);
            w.u32_((u32)(nvals * 8));
            w.bytes(gb.row_result(sq[l].row_id), nvals * 8);
            w.u32_((u32)paths.v.size());
            w.bytes(paths.v.data(), paths.v.size());
        }
        for (size_t l = 0; l < fri->layers.size(); l++) {
            const size_t nvals = fplan.nq[l] * fri->folding * fri->d;
            ByteVec paths;
            wf_open_finish(gb.digs[fplan.dig_ids[l]].plan, gb.digest_result(fplan.dig_ids[l]), nullptr, paths);
            w.u32_((u32)(nvals * 8));
            w.bytes(gb.row_result(fplan.row_ids[l]), nvals * 8);
            w.u32_((u32)paths.v.size());
            w.bytes(paths.v.data(), paths.v.size());
        }
        w.u16_((uint16_t)(fri->remainder.size() * 8));
        w.bytes(fri->remainder.data(), fri->remainder.size() * 8);
        w.u8_(0);
    }
    w.u64_(nonce);
    wf_mark(ctx, "queries_and_proof");
    proof_out.swap(w.v);
    if (stats) {
        CK(cudaStreamSynchronize(ctx->st));
        stats[0] = sc.bytes_sent; stats[1] = sc.exchange_ms(); stats[2] = sc.ncoll + 1; stats[3] = sc.ms_small;
        for (int i = 4; i < 8; i++) stats[i] = 0;
        stats[4] = (double)slayers.size();
        stats[5] = sc.bytes_overlapped;
        stats[6] = (double)tpath;   // the main trace's transport (the aux segment's: its own split decides)
        stats[7] = cb_ms;
    }
    return WF_OK;
}

}  // namespace

extern "C" int wf_grind(wf_ctx* ctx, int hash_id, const uint8_t seed[32], uint32_t grinding, uint64_t* nonce) {
    if (!ctx || !seed || !nonce || grinding > 40) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    Digest d;
    memcpy(d.b, seed, 32);
    return grind_on_device(ctx, hash_id, d, grinding, nonce);
}

static int parse_options(wf_ctx* ctx, const uint32_t* opts, Options& o) {
    o.num_queries = opts[0]; o.blowup = opts[1]; o.grinding = opts[2]; o.ext = opts[3]; o.folding = opts[4];
    o.rem_max_deg = opts[5]; o.batch_c = opts[6]; o.batch_d = opts[7]; o.hash_id = (int)(opts[8] & 0xff);
    // ProofOptions::with_partitions (air/src/options.rs:193-200): opts[8] = hash_id | num_partitions << 8 | hash_rate << 16;
    // 0 in either field is the default PartitionOptions::new(1, 1)
    o.num_partitions = (opts[8] >> 8) & 0xff; o.hash_rate = (opts[8] >> 16) & 0xff;
    if (o.num_partitions == 0) o.num_partitions = 1;
    if (o.hash_rate == 0) o.hash_rate = 1;
    if (o.num_partitions > 16) return wf_fail(ctx, WF_ERR_INVALID, "at most 16 partitions (air/src/options.rs:413-414)");
    if (o.blowup < 2 || o.blowup > 128 || (o.blowup & (o.blowup - 1)) || o.num_queries == 0 || o.num_queries > 255 || o.batch_c > 2 ||
        o.batch_d > 2 || o.grinding > 32 || o.rem_max_deg > 255 || ((o.rem_max_deg + 1) & o.rem_max_deg) ||
        (o.folding != 2 && o.folding != 4 && o.folding != 8 && o.folding != 16) || o.ext < 1 || o.ext > 3)
        return wf_fail(ctx, WF_ERR_INVALID, "bad proof options");  // ProofOptions::new asserts (air/src/options.rs:132-190)
    if (!WF_HASH_IS_KNOWN(o.hash_id)) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "unknown hash %d", o.hash_id);
    return WF_OK;
}
static int prove_dispatch(wf_ctx* ctx, const AirHost& air, const uint64_t* const* trace_cols, const uint64_t* d_trace, int mont,
                          uint32_t log_n, const Options& o, uint8_t* proof, size_t* proof_len, wf_aux_builder_fn aux_builder = nullptr,
                          void* aux_user = nullptr, wf_aux_assertions_fn aux_assertions = nullptr) {
    std::vector<u8> out;
    int r;
    switch (o.ext) {
        case 1: r = prove_air<1>(ctx, air, trace_cols, d_trace, mont, log_n, o, aux_builder, aux_user, out, aux_assertions); break;
        case 2: r = prove_air<2>(ctx, air, trace_cols, d_trace, mont, log_n, o, aux_builder, aux_user, out, aux_assertions); break;
        case 3: r = prove_air<3>(ctx, air, trace_cols, d_trace, mont, log_n, o, aux_builder, aux_user, out, aux_assertions); break;
        default: return wf_fail(ctx, WF_ERR_UNSUPPORTED, "field extension %u", o.ext);
    }
    if (r != WF_OK) return r;
    if (out.size() > *proof_len) return wf_fail(ctx, WF_ERR_INVALID, "proof buffer too small (%zu needed)", out.size());
    memcpy(proof, out.data(), out.size());
    *proof_len = out.size();
    return WF_OK;
}
static int prove_fib_entry(wf_ctx* ctx, const uint64_t* const* trace_cols, const uint64_t* d_trace, int mont, uint32_t k,
                           uint32_t log_n, const uint64_t* results, const uint32_t* opts, uint8_t* proof, size_t* proof_len) {
    if (!ctx || (!trace_cols && !d_trace) || !results || !opts || !proof || !proof_len || k == 0 || 2 * k > 255 || log_n < 3)
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    Options o;
    CKI(parse_options(ctx, opts, o));
    AirHost air = fib_air_host(k, (size_t)1 << log_n, results);
    return prove_dispatch(ctx, air, trace_cols, d_trace, mont, log_n, o, proof, proof_len);
}
extern "C" int wf_prove_air(wf_ctx* ctx, const uint64_t* air_desc, size_t air_desc_len, const uint64_t* const* trace_cols, int mont,
                            uint32_t log_n, const uint32_t* opts, uint8_t* proof, size_t* proof_len) {
    if (!ctx || !air_desc || !trace_cols || !opts || !proof || !proof_len || log_n < 3)
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    Options o;
    CKI(parse_options(ctx, opts, o));
    AirHost air;
    if (!parse_air_host(air_desc, air_desc_len, air)) return wf_fail(ctx, WF_ERR_INVALID, "malformed AIR description");
    if (air.aw) return wf_fail(ctx, WF_ERR_INVALID, "multi-segment AIR: use wf_prove_air_aux");
    return prove_dispatch(ctx, air, trace_cols, nullptr, mont, log_n, o, proof, proof_len);
}
extern "C" int wf_prove_air_aux(wf_ctx* ctx, const uint64_t* air_desc, size_t air_desc_len, const uint64_t* const* trace_cols, int mont,
                                uint32_t log_n, const uint32_t* opts, wf_aux_builder_fn aux_builder, void* aux_user, uint8_t* proof,
                                size_t* proof_len) {
    if (!ctx || !air_desc || !trace_cols || !opts || !proof || !proof_len || log_n < 3)
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    Options o;
    CKI(parse_options(ctx, opts, o));
    AirHost air;
    if (!parse_air_host(air_desc, air_desc_len, air)) return wf_fail(ctx, WF_ERR_INVALID, "malformed AIR description");
    return prove_dispatch(ctx, air, trace_cols, nullptr, mont, log_n, o, proof, proof_len, aux_builder, aux_user);
}
extern "C" int wf_prove_air_aux_dyn(wf_ctx* ctx, const uint64_t* air_desc, size_t air_desc_len, const uint64_t* const* trace_cols, int mont,
                                    uint32_t log_n, const uint32_t* opts, wf_aux_builder_fn aux_builder,
                                    wf_aux_assertions_fn aux_assertions, void* aux_user, uint8_t* proof, size_t* proof_len) {
    if (!ctx || !air_desc || !trace_cols || !opts || !proof || !proof_len || log_n < 3 || !aux_assertions)
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    Options o;
    CKI(parse_options(ctx, opts, o));
    AirHost air;
    if (!parse_air_host(air_desc, air_desc_len, air)) return wf_fail(ctx, WF_ERR_INVALID, "malformed AIR description");
    return prove_dispatch(ctx, air, trace_cols, nullptr, mont, log_n, o, proof, proof_len, aux_builder, aux_user, aux_assertions);
}

// Compiles the constraint kernel of an AIR description; needs no device (a build-time / CI check of the JIT path and of the
// generated code). *cubin_bytes = size of the sm_100a cubin; `log` receives the compiler log (warnings or errors).
extern "C" int wf_jit_compile_air(const uint64_t* air_desc, size_t air_desc_len, uint32_t ext, size_t* cubin_bytes, char* log, size_t log_cap) {
    if (!air_desc || ext < 1 || ext > 3) return WF_ERR_INVALID;
    AirHost air;
    if (!parse_air_host(air_desc, air_desc_len, air)) return WF_ERR_INVALID;
    std::vector<char> cubin;
    std::string lg;
    const int rc = wf_jit_compile(wf_jit_source((int)ext, air.w, (u32)air.periodic.size(), air.num_regs, air.prog, air.consts, air.aw, air.nr,
                                                air.aux_num_regs, air.aux_prog), cubin, lg);
    if (log && log_cap) { strncpy(log, lg.c_str(), log_cap - 1); log[log_cap - 1] = 0; }
    if (cubin_bytes) *cubin_bytes = cubin.size();
    if (const char* dump = getenv("WF_JIT_DUMP")) if (rc == 0) { FILE* f = fopen(dump, "wb"); if (f) { fwrite(cubin.data(), 1, cubin.size(), f); fclose(f); } }
    return rc == 0 ? WF_OK : WF_ERR_UNSUPPORTED;
}

// The checks wf_prove_air / wf_eval_constraints run on an AIR description before touching the device, without a device:
// structure of the description, degrees against the blowup factor, periodic columns, assertion validity and overlaps
// (the panics of Air::new / BoundaryConstraints::new / prepare_assertions in the reference, returned as a status).
extern "C" int wf_air_check(const uint64_t* air_desc, size_t air_desc_len, uint32_t log_n, uint32_t blowup, char* msg, size_t msg_cap) {
    auto say = [&](const char* t) { if (msg && msg_cap) { strncpy(msg, t, msg_cap - 1); msg[msg_cap - 1] = 0; } };
    say("");
    if (!air_desc || log_n < 3 || log_n > 32 || blowup < 2 || blowup > 128 || (blowup & (blowup - 1))) { say("bad arguments"); return WF_ERR_INVALID; }
    AirHost air;
    if (!parse_air_host(air_desc, air_desc_len, air)) { say("malformed AIR description"); return WF_ERR_INVALID; }
    wf_ctx note{};   // carries the message of the shared validators, nothing else
    u32 log_b = 0;
    while ((1u << log_b) < blowup) log_b++;
    const size_t n = (size_t)1 << log_n;
    int r = WF_OK;
    if (air.log_ce_blowup() > log_b) r = wf_fail(&note, WF_ERR_INVALID, "blowup factor too small for the constraint degrees");
    for (auto& col : air.periodic) if (r == WF_OK && col.size() > n) r = wf_fail(&note, WF_ERR_INVALID, "periodic column longer than the trace");
    if (r == WF_OK) r = validate_degrees(&note, air.all_degrees(), n);
    if (r == WF_OK) r = validate_assertions(&note, air.aux_asserts, n, 3, "aux assertion");
    if (r == WF_OK) r = validate_assertions(&note, air.asserts, n, 1, "assertion");
    say(note.err.c_str());
    return r;
}

// ---- stepwise exports: the seams of prover/src/lib.rs:125-223 (ConstraintEvaluator, ConstraintCommitment)
//      and the concrete steps between them, for a host that keeps the transcript itself ----------------
template <int D>
static int eval_constraints_entry(wf_ctx* ctx, const AirHost& air, u32 log_n, u32 log_b, const wf_mat* lde, const wf_mat* alde,
                                  const uint64_t* coeffs, const uint64_t* aux_rand, wf_mat** out) {
    const size_t ncc = air.degrees.size() + air.aux_degrees.size() + air.asserts.size() + air.aux_asserts.size();
    std::vector<GlExt<D>> cc(ncc);
    for (size_t i = 0; i < ncc; i++) for (int q = 0; q < D; q++) cc[i].v[q] = coeffs[i * D + q];
    std::vector<u64> rnd;
    if (air.aw) rnd.assign(aux_rand, aux_rand + (size_t)air.nr * D);
    return eval_constraints<D>(ctx, air, lde, alde, cc, rnd, log_n, log_b, out);
}
extern "C" int wf_eval_constraints(wf_ctx* ctx, const uint64_t* air_desc, size_t air_desc_len, uint32_t log_n, uint32_t blowup,
                                   uint32_t ext, const wf_mat* main_lde, const wf_mat* aux_lde, const uint64_t* coeffs,
                                   const uint64_t* aux_rand, wf_mat** out) {
    if (!ctx || !air_desc || !main_lde || !coeffs || !out || log_n < 3 || blowup < 2 || (blowup & (blowup - 1)))
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    AirHost air;
    if (!parse_air_host(air_desc, air_desc_len, air)) return wf_fail(ctx, WF_ERR_INVALID, "malformed AIR description");
    u32 log_b = 0;
    while ((1u << log_b) < blowup) log_b++;
    const size_t N = (size_t)1 << (log_n + log_b);
    if (air.log_ce_blowup() > log_b) return wf_fail(ctx, WF_ERR_INVALID, "blowup factor too small for the constraint degrees");
    if (main_lde->m.rows != N || main_lde->m.cols != air.w) return wf_fail(ctx, WF_ERR_INVALID, "main LDE shape does not match the AIR");
    if (air.aw && (!aux_lde || !aux_rand || aux_lde->m.rows != N || aux_lde->m.cols != air.aw * ext))
        return wf_fail(ctx, WF_ERR_INVALID, "aux LDE / random elements missing or of the wrong shape");
    for (auto& col : air.periodic) if (col.size() > ((size_t)1 << log_n)) return wf_fail(ctx, WF_ERR_INVALID, "periodic column longer than the trace");
    CKI(validate_degrees(ctx, air.all_degrees(), (size_t)1 << log_n));
    CKI(validate_assertions(ctx, air.aux_asserts, (size_t)1 << log_n, 3, "aux assertion"));
    CKI(validate_assertions(ctx, air.asserts, (size_t)1 << log_n, 1, "assertion"));
    const wf_mat* al = air.aw ? aux_lde : nullptr;
    switch (ext) {
        case 1: return eval_constraints_entry<1>(ctx, air, log_n, log_b, main_lde, al, coeffs, aux_rand, out);
        case 2: return eval_constraints_entry<2>(ctx, air, log_n, log_b, main_lde, al, coeffs, aux_rand, out);
        case 3: return eval_constraints_entry<3>(ctx, air, log_n, log_b, main_lde, al, coeffs, aux_rand, out);
    }
    return wf_fail(ctx, WF_ERR_UNSUPPORTED, "field extension %u", ext);
}

extern "C" int wf_composition_commit(wf_ctx* ctx, int hash_id, const wf_mat* comp_trace, uint32_t log_n, uint32_t blowup, uint32_t ext,
                                     uint32_t num_cols, wf_mat** polys, wf_mat** lde, wf_tree** tree) {
    if (!ctx || !comp_trace || !polys || !lde || !tree || ext < 1 || ext > 3 || num_cols == 0 || blowup < 2 || (blowup & (blowup - 1)))
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    u32 log_b = 0;
    while ((1u << log_b) < blowup) log_b++;
    return composition_commit(ctx, hash_id, comp_trace, log_n, log_b, (int)ext, num_cols, polys, lde, tree);
}
extern "C" int wf_composition_commit_partitioned(wf_ctx* ctx, int hash_id, const wf_mat* comp_trace, uint32_t log_n, uint32_t blowup,
                                                 uint32_t ext, uint32_t num_cols, uint32_t partition_size, wf_mat** polys, wf_mat** lde,
                                                 wf_tree** tree) {
    if (!ctx || !comp_trace || !polys || !lde || !tree || ext < 1 || ext > 3 || num_cols == 0 || blowup < 2 || (blowup & (blowup - 1)))
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    u32 log_b = 0;
    while ((1u << log_b) < blowup) log_b++;
    return composition_commit(ctx, hash_id, comp_trace, log_n, log_b, (int)ext, num_cols, polys, lde, tree, partition_size);
}

template <int D>
static int evaluate_at_entry(wf_ctx* ctx, const wf_mat* polys, u32 col_ext, const uint64_t* z0, const uint64_t* z1, uint64_t* o0,
                             uint64_t* o1) {
    GlExt<D> a = ext_zero<D>(), b = ext_zero<D>();
    for (int q = 0; q < D; q++) { a.v[q] = z0[q]; b.v[q] = z1[q]; }
    std::vector<std::vector<GlExt<D>>> ev;
    CKI(ood_eval<D>(ctx, {polys}, a, b, ev));
    for (int pt = 0; pt < 2; pt++) {
        uint64_t* o = pt ? o1 : o0;
        const size_t cols = ev[pt].size() / col_ext;
        for (size_t j = 0; j < cols; j++) {
            GlExt<D> acc = ext_zero<D>();
            for (u32 q = 0; q < col_ext; q++) {  // column of E = sum_q phi^q * (component column q)
                GlExt<D> basis = ext_zero<D>();
                basis.v[q] = 1;
                acc = ext_add(acc, ext_mul(basis, ev[pt][j * col_ext + q]));
            }
            for (int q = 0; q < D; q++) o[j * D + q] = acc.v[q];
        }
    }
    return WF_OK;
}
extern "C" int wf_mat_evaluate_at(wf_ctx* ctx, const wf_mat* polys, uint32_t ext, uint32_t col_ext, const uint64_t* z0, const uint64_t* z1,
                                  uint64_t* out0, uint64_t* out1) {
    if (!ctx || !polys || !z0 || !z1 || !out0 || !out1 || (col_ext != 1 && col_ext != ext) || polys->m.cols % col_ext)
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    switch (ext) {
        case 1: return evaluate_at_entry<1>(ctx, polys, col_ext, z0, z1, out0, out1);
        case 2: return evaluate_at_entry<2>(ctx, polys, col_ext, z0, z1, out0, out1);
        case 3: return evaluate_at_entry<3>(ctx, polys, col_ext, z0, z1, out0, out1);
    }
    return wf_fail(ctx, WF_ERR_UNSUPPORTED, "field extension %u", ext);
}

template <int D>
static int deep_entry(wf_ctx* ctx, const wf_mat* lde, const wf_mat* alde, const wf_mat* clde, u32 log_n, const uint64_t* zw,
                      const uint64_t* coeffs, const uint64_t* ood_cur, const uint64_t* ood_next, wf_mat** out) {
    const u32 c = lde->m.cols, aw = alde ? alde->m.cols / D : 0, kc = clde->m.cols / D, tot = c + aw + kc;
    u32 log_N = 0;
    while (((size_t)1 << log_N) < lde->m.rows) log_N++;
    if (log_n > log_N) return wf_fail(ctx, WF_ERR_INVALID, "trace length exceeds the LDE domain");
    std::vector<GlExt<D>> dc(tot);
    GlExt<D> z = ext_zero<D>(), Sz = ext_zero<D>(), Szg = ext_zero<D>();
    for (int q = 0; q < D; q++) z.v[q] = zw[q];
    for (u32 i = 0; i < tot; i++) {
        GlExt<D> a = ext_zero<D>(), b = ext_zero<D>();
        for (int q = 0; q < D; q++) { dc[i].v[q] = coeffs[i * D + q]; a.v[q] = ood_cur[i * D + q]; b.v[q] = ood_next[i * D + q]; }
        Sz = ext_add(Sz, ext_mul(dc[i], a));
        Szg = ext_add(Szg, ext_mul(dc[i], b));
    }
    GlExt<D> zg = ext_mul_base(z, gl_root_of_unity(log_n));
    return deep_compose<D>(ctx, lde, alde, clde, kc, log_N, dc, z, zg, Sz, Szg, out);
}
extern "C" int wf_deep_compose(wf_ctx* ctx, uint32_t ext, const wf_mat* main_lde, const wf_mat* aux_lde, const wf_mat* cons_lde,
                               uint32_t log_n, const uint64_t* z, const uint64_t* coeffs, const uint64_t* ood_cur,
                               const uint64_t* ood_next, wf_mat** out) {
    if (!ctx || !main_lde || !cons_lde || !z || !coeffs || !ood_cur || !ood_next || !out || ext < 1 || ext > 3 ||
        cons_lde->m.cols % ext || cons_lde->m.rows != main_lde->m.rows || (aux_lde && (aux_lde->m.cols % ext || aux_lde->m.rows != main_lde->m.rows)))
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    switch (ext) {
        case 1: return deep_entry<1>(ctx, main_lde, aux_lde, cons_lde, log_n, z, coeffs, ood_cur, ood_next, out);
        case 2: return deep_entry<2>(ctx, main_lde, aux_lde, cons_lde, log_n, z, coeffs, ood_cur, ood_next, out);
        default: return deep_entry<3>(ctx, main_lde, aux_lde, cons_lde, log_n, z, coeffs, ood_cur, ood_next, out);
    }
}

static int prove_sharded_dispatch(wf_ctx* ctx, const wf_comm* comm, const AirHost& air, const uint64_t* const* local_cols,
                                  const uint64_t* d_local, int mont, uint32_t log_n, const Options& o, uint8_t* proof, size_t* proof_len,
                                  double* stats, wf_aux_shard_builder_fn aux_builder = nullptr,
                                  wf_aux_assertions_fn aux_assertions = nullptr, void* aux_user = nullptr) {
    std::vector<u8> out;
    int r;
    switch (o.ext) {
        case 1: r = prove_sharded<1>(ctx, comm, air, local_cols, d_local, mont, log_n, o, out, stats, aux_builder, aux_assertions, aux_user); break;
        case 2: r = prove_sharded<2>(ctx, comm, air, local_cols, d_local, mont, log_n, o, out, stats, aux_builder, aux_assertions, aux_user); break;
        default: r = prove_sharded<3>(ctx, comm, air, local_cols, d_local, mont, log_n, o, out, stats, aux_builder, aux_assertions, aux_user); break;
    }
    if (r != WF_OK) return r;
    if (out.size() > *proof_len) return wf_fail(ctx, WF_ERR_INVALID, "proof buffer too small (%zu needed)", out.size());
    memcpy(proof, out.data(), out.size());
    *proof_len = out.size();
    return WF_OK;
}
extern "C" int wf_prove_fib_sharded(wf_ctx* ctx, const wf_comm* comm, const uint64_t* const* local_cols, const uint64_t* d_local, int mont,
                                    uint32_t k, uint32_t log_n, const uint64_t* results, const uint32_t* opts, uint8_t* proof,
                                    size_t* proof_len, double* stats) {
    if (!ctx || !comm || !comm->exchange || !comm->all_gather_host || !comm->all_reduce_sum || (!local_cols && !d_local) || !results ||
        !opts || !proof || !proof_len || k == 0 || 2 * k > 255 || log_n < 3)
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
    Options o;
    CKI(parse_options(ctx, opts, o));
    const AirHost air = fib_air_host(k, (size_t)1 << log_n, results);
    return prove_sharded_dispatch(ctx, comm, air, local_cols, d_local, mont, log_n, o, proof, proof_len, stats);
}
extern "C" int wf_host_shard_columns(uint32_t width, int world, int rank, uint32_t* first, uint32_t* count) {
    if (!first || !count) return WF_ERR_INVALID;
    return shard_columns(width, world, rank, first, count) ? WF_OK : WF_ERR_INVALID;
}
// A sharded proof must not start unless every rank can go through with it: a rank that refused would otherwise leave the
// others waiting in a collective. So each rank checks its own arguments (no device work), hashes what must be equal on
// every rank, and one all-gather of (status, hash) decides for all of them. aux_entry: wf_prove_air_aux_sharded (the
// description must have an aux segment), else wf_prove_air_sharded (it must not).
static int prove_air_sharded_entry(wf_ctx* ctx, const wf_comm* comm, const uint64_t* air_desc, size_t air_desc_len,
                                   const uint64_t* const* local_cols, const uint64_t* d_local, int mont, uint32_t log_n,
                                   const uint32_t* opts, uint8_t* proof, size_t* proof_len, double* stats, bool aux_entry,
                                   wf_aux_shard_builder_fn aux_builder, wf_aux_assertions_fn aux_assertions, void* aux_user) {
    if (!ctx || !comm || !comm->exchange || !comm->all_gather_host || !comm->all_reduce_sum || comm->world < 1 || comm->rank < 0 ||
        comm->rank >= comm->world)
        return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");   // no communicator to agree over
    const int G = comm->world, r = comm->rank;
    Options o;
    AirHost air;
    auto own_checks = [&]() -> int {
        if (!air_desc || !opts || !proof || !proof_len || log_n < 3 || log_n > 32) return wf_fail(ctx, WF_ERR_INVALID, "bad arguments");
        CKI(parse_options(ctx, opts, o));
        if (!parse_air_host(air_desc, air_desc_len, air)) return wf_fail(ctx, WF_ERR_INVALID, "malformed AIR description");
        if (!aux_entry && air.aw) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "sharded proofs cover single-segment AIRs (this description has an auxiliary segment)");
        if (aux_entry && !air.aw) return wf_fail(ctx, WF_ERR_INVALID, "the description has no auxiliary segment: use wf_prove_air_sharded");
        if (aux_entry && !aux_builder) return wf_fail(ctx, WF_ERR_INVALID, "multi-segment AIR needs an aux trace builder");
        if (air.aw * o.ext > 255) return wf_fail(ctx, WF_ERR_UNSUPPORTED, "at most 255 aux base columns (aux width x field extension)");
        CKI(sharded_shape_check(ctx, air, log_n, o, G, r));
        const size_t n = (size_t)1 << log_n;
        for (auto& col : air.periodic) if (col.size() > n) return wf_fail(ctx, WF_ERR_INVALID, "periodic column longer than the trace");
        CKI(validate_degrees(ctx, air.all_degrees(), n));
        CKI(validate_assertions(ctx, air.aux_asserts, n, 3, "aux assertion"));
        CKI(validate_assertions(ctx, air.asserts, n, 1, "assertion"));
        u32 first = 0, count = 0;
        shard_columns(air.w, G, r, &first, &count);
        if (count && !local_cols && !d_local) return wf_fail(ctx, WF_ERR_INVALID, "rank %d owns columns [%u, %u) but passed none", r, first, first + count);
        if (!count && (local_cols || d_local)) return wf_fail(ctx, WF_ERR_INVALID, "rank %d owns no column but passed some", r);
        return WF_OK;
    };
    const int mine = own_checks();
    Fnv hsh;   // over the description, log_n, the options and the world size (and whether aux assertions are dynamic)
    hsh.mix(air_desc ? air_desc_len : ~(u64)0);
    for (size_t i = 0; air_desc && i < air_desc_len; i++) hsh.mix(air_desc[i]);
    hsh.mix(log_n);
    for (int i = 0; i < 9; i++) hsh.mix(opts ? opts[i] : ~(u64)0);
    hsh.mix((u64)G);
    if (aux_entry) hsh.mix(aux_assertions ? 1 : 0);
    struct Vote { int32_t status, pad; u64 hash; } v{mine, 0, hsh.h};
    std::vector<Vote> all(G);
    if (comm->all_gather_host(comm->user, &v, all.data(), sizeof(Vote)) != 0) return wf_fail(ctx, WF_ERR_STATE, "all_gather_host callback failed");
    for (int q = 0; q < G; q++) {   // the lowest refusing rank's status, on every rank
        if (all[q].status == WF_OK) continue;
        if (q == r) return mine;
        const std::string own = mine == WF_OK ? std::string() : "; this rank: " + ctx->err;
        return wf_fail(ctx, all[q].status, "rank %d refused the sharded proof%s", q, own.c_str());
    }
    for (int q = 0; q < G; q++)
        if (all[q].hash != hsh.h)
            return wf_fail(ctx, WF_ERR_INVALID, "ranks %d and %d were given different AIR descriptions, trace lengths, options or world sizes%s", r, q,
                           aux_entry ? " (or only one of them an aux assertion callback)" : "");
    return prove_sharded_dispatch(ctx, comm, air, local_cols, d_local, mont, log_n, o, proof, proof_len, stats, aux_builder, aux_assertions,
                                  aux_user);
}
extern "C" int wf_prove_air_sharded(wf_ctx* ctx, const wf_comm* comm, const uint64_t* air_desc, size_t air_desc_len,
                                    const uint64_t* const* local_cols, const uint64_t* d_local, int mont, uint32_t log_n,
                                    const uint32_t* opts, uint8_t* proof, size_t* proof_len, double* stats) {
    return prove_air_sharded_entry(ctx, comm, air_desc, air_desc_len, local_cols, d_local, mont, log_n, opts, proof, proof_len, stats, false,
                                   nullptr, nullptr, nullptr);
}
extern "C" int wf_prove_air_aux_sharded(wf_ctx* ctx, const wf_comm* comm, const uint64_t* air_desc, size_t air_desc_len,
                                        const uint64_t* const* local_cols, const uint64_t* d_local, int mont, uint32_t log_n,
                                        const uint32_t* opts, wf_aux_shard_builder_fn aux_builder, wf_aux_assertions_fn aux_assertions,
                                        void* aux_user, uint8_t* proof, size_t* proof_len, double* stats) {
    return prove_air_sharded_entry(ctx, comm, air_desc, air_desc_len, local_cols, d_local, mont, log_n, opts, proof, proof_len, stats, true,
                                   aux_builder, aux_assertions, aux_user);
}
extern "C" int wf_prove_fib(wf_ctx* ctx, const uint64_t* const* trace_cols, int mont, uint32_t k, uint32_t log_n,
                            const uint64_t* results, const uint32_t* opts, uint8_t* proof, size_t* proof_len) {
    return prove_fib_entry(ctx, trace_cols, nullptr, mont, k, log_n, results, opts, proof, proof_len);
}
extern "C" int wf_prove_fib_dev(wf_ctx* ctx, const uint64_t* d_trace, uint32_t k, uint32_t log_n, const uint64_t* results,
                                const uint32_t* opts, uint8_t* proof, size_t* proof_len) {
    return prove_fib_entry(ctx, nullptr, d_trace, 0, k, log_n, results, opts, proof, proof_len);
}
