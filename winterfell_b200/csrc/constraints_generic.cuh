// constraints_generic.cuh — the generic constraint evaluator kernel, one source for two builds:
//   * compiled with the library (nvcc): the AIR's transition programs are INTERPRETED from device memory, registers in a
//     local-memory array (any program, no compilation step);
//   * compiled at run time for ONE AIR (NVRTC, jit.cu; WF_JIT defined): jit.cu prepends the AIR's shape as macros and its
//     two programs as straight-line C++ (wf_jit_main / wf_jit_aux) — every register index is a literal, so the register file
//     lives in registers and constants are immediates. "Compiled to a device functor", SURVEY.md 8(f)3.
// Replaces DefaultConstraintEvaluator::evaluate_fragment_main / _full + ConstraintEvaluationTable::combine
// (prover/src/constraints/evaluator/default.rs:165-341, evaluation_table.rs:163-407) for AIRs given as programs
// (frame registers r[0..w) current row, r[w..2w) next row, then periodic values, then temporaries), any number of
// boundary groups (single, periodic and sequence assertions) and transition exemptions. One CE row per thread.
#pragma once
#include "commit.cuh"
#include "gl64.cuh"

template <int D>
__device__ __forceinline__ GlExt<D> ld_ext(const u64* p) {
    GlExt<D> r;
#pragma unroll
    for (int i = 0; i < D; i++) r.v[i] = p[i];
    return r;
}
__device__ __forceinline__ u64 seg_at(const SegMatrix& m, size_t row, u32 col) {
    return m.base[(size_t)(col / m.W) * m.seg_stride + row * m.W + (col % m.W)];
}

#define GEN_MAX_REGS 160
#define AUX_MAX_REGS 96
struct GenEvalParams {
    SegMatrix lde, out;
    u32 w, log_n, log_blowup, log_ce_blowup;
    const u32* prog;       // [prog_len][4]: op, dst, a, b
    u32 prog_len, num_regs, num_periodic, num_tc;
    const u64* consts;
    const u64* ptab;       // periodic tables, concatenated
    const u32* ptab_off;   // [num_periodic]
    const u32* ptab_len;   // [num_periodic]  (L_j * ce_blowup, a power of two)
    const u64* tcoef;      // [num_tc][D]
    u32 num_groups;
    const u32* g_off;      // [num_groups + 1] offsets into the entry arrays
    const u64* g_a;        // x^a - b divisor exponent (a divides n)
    const u64* g_b;
    const u64* g_oa;       // 7^a
    const u32* e_col;
    const u64* e_val;
    const u64* e_cc;       // [entries][D]
    // sequence assertions (Assertion::sequence): per entry the value polynomial evaluated over the CE
    // domain (LargePolyConstraint, evaluator/boundary.rs:389-445); nullptr for single-value entries
    const u64* const* e_tab;
    const u32* e_tstride;  // words per table row
    const u32* e_shift;    // (first_step * ce_blowup) mod ce
    const u64* tw_ce;      // w_ce^i, i < ce/2
    const u64* zt;         // [ce_blowup] 1 / (x^n - 1) at CE step i mod ce_blowup (device table: ce_blowup <= 128)
    u64 exempt[8];
    u32 num_exempt;
    // auxiliary segment (Air::evaluate_aux_transition, air/src/air/mod.rs:248-260): program over E
    // registers [main cur | main next | aux cur | aux next | periodic | random elements | temporaries]
    SegMatrix alde;        // N x aw*D
    u32 aw, nr, aprog_len, num_agroups;
    const u32* aprog;
    const u64* rnd;        // [nr][D]
    const u64* atcoef;     // [aux constraints][D]
    const u32* ag_off;     // aux boundary groups (air/src/air/boundary/mod.rs:121-128)
    const u64* ag_a;
    const u64* ag_b;
    const u64* ag_oa;
    const u32* ae_col;
    const u64* ae_val;     // [entries][D]
    const u64* ae_cc;      // [entries][D]
    const u64* const* ae_tab;
    const u32* ae_tstride;
    const u32* ae_shift;
    // row-sharded evaluation (multi-GPU): this launch covers CE rows [row0, row0 + ce_rows); `lde` (and `alde`) then hold the
    // LDE rows of that range followed by `blowup` halo rows, so the next-state row is local row + blowup without wrap-around,
    // and `out` holds the launch's rows only. ce_rows = 0: the whole domain.
    size_t row0, ce_rows;
};

#ifdef WF_JIT
// supplied by the generated prologue: WF_JIT_D, WF_JIT_AUX, WF_JIT_W, WF_JIT_NPER, WF_JIT_AW, WF_JIT_NR, WF_JIT_NREGS,
// WF_JIT_NAREGS and the two functions below (bodies = the programs)
template <int D> __device__ __forceinline__ void wf_jit_main(u64* r, const GenEvalParams& p, GlExt<D>& T);
template <int D> __device__ __forceinline__ void wf_jit_aux(GlExt<D>* ra, const GenEvalParams& p, GlExt<D>& T);
#endif

template <int D, bool AUX>
__device__ __forceinline__ void generic_constraints_row(const GenEvalParams& p) {
    const size_t ce = (size_t)1 << (p.log_n + p.log_ce_blowup);
    const size_t il = (size_t)blockIdx.x * blockDim.x + threadIdx.x;   // row of this launch: indexes lde / alde / out
    if (il >= (p.ce_rows ? p.ce_rows : ce)) return;
    const size_t i = il + p.row0;                                       // row of the CE domain: x, divisors, periodic and sequence tables
    const size_t N = (size_t)1 << (p.log_n + p.log_blowup);
    const size_t ls = il << (p.log_blowup - p.log_ce_blowup);
    const size_t nx = p.ce_rows ? ls + ((size_t)1 << p.log_blowup) : ((ls + ((size_t)1 << p.log_blowup)) & (N - 1));
    GlExt<D> T = ext_zero<D>();
#ifdef WF_JIT
    // compile-time shape: every index below is a literal after unrolling, r[] and ra[] are promoted to registers; the rows a
    // boundary constraint may address by a run-time column index are kept in the small arrays cur[] / acur[]
    u64 r[WF_JIT_NREGS];
    u64 cur[WF_JIT_W];
#pragma unroll
    for (u32 c = 0; c < WF_JIT_W; c++) { r[c] = seg_at(p.lde, ls, c); r[WF_JIT_W + c] = seg_at(p.lde, nx, c); cur[c] = r[c]; }
#pragma unroll
    for (u32 j = 0; j < WF_JIT_NPER; j++) r[2 * WF_JIT_W + j] = p.ptab[p.ptab_off[j] + (u32)(i & (p.ptab_len[j] - 1))];
    wf_jit_main<D>(r, p, T);
    GlExt<D> ra[AUX ? WF_JIT_NAREGS : 1];
    GlExt<D> acur[AUX ? WF_JIT_AW : 1];
    if constexpr (AUX) {
#pragma unroll
        for (u32 c = 0; c < 2 * WF_JIT_W; c++) ra[c] = ext_from_base<D>(r[c]);
#pragma unroll
        for (u32 j = 0; j < WF_JIT_AW; j++) {
#pragma unroll
            for (int q = 0; q < D; q++) {
                ra[2 * WF_JIT_W + j].v[q] = seg_at(p.alde, ls, j * D + q);
                ra[2 * WF_JIT_W + WF_JIT_AW + j].v[q] = seg_at(p.alde, nx, j * D + q);
            }
            acur[j] = ra[2 * WF_JIT_W + j];
        }
#pragma unroll
        for (u32 j = 0; j < WF_JIT_NPER; j++) ra[2 * WF_JIT_W + 2 * WF_JIT_AW + j] = ext_from_base<D>(r[2 * WF_JIT_W + j]);
#pragma unroll
        for (u32 j = 0; j < WF_JIT_NR; j++) ra[2 * WF_JIT_W + 2 * WF_JIT_AW + WF_JIT_NPER + j] = ld_ext<D>(p.rnd + (size_t)j * D);
        wf_jit_aux<D>(ra, p, T);
    }
#define WF_MAIN_CUR(col) cur[col]
#define WF_AUX_CUR(col) acur[col]
#else
    u64 r[GEN_MAX_REGS];
    for (u32 c = 0; c < p.w; c++) { r[c] = seg_at(p.lde, ls, c); r[p.w + c] = seg_at(p.lde, nx, c); }
    for (u32 j = 0; j < p.num_periodic; j++) r[2 * p.w + j] = p.ptab[p.ptab_off[j] + (u32)(i & (p.ptab_len[j] - 1))];
    for (u32 k = 0; k < p.prog_len; k++) {
        const u32 op = p.prog[4 * k], dst = p.prog[4 * k + 1], a = p.prog[4 * k + 2], b = p.prog[4 * k + 3];
        switch (op) {
            case 0: r[dst] = gl_add(r[a], r[b]); break;
            case 1: r[dst] = gl_sub(r[a], r[b]); break;
            case 2: r[dst] = gl_mul(r[a], r[b]); break;
            case 3: r[dst] = p.consts[a]; break;
            default: T = ext_add(T, ext_mul_base(ld_ext<D>(p.tcoef + (size_t)dst * D), r[a])); break;  // OUT
        }
    }
    GlExt<D> ra[AUX ? AUX_MAX_REGS : 1];
    if constexpr (AUX) {  // evaluator/default.rs:306-341 evaluate_aux_transition
        for (u32 c = 0; c < 2 * p.w; c++) ra[c] = ext_from_base<D>(r[c]);
        for (u32 j = 0; j < p.aw; j++) {
#pragma unroll
            for (int q = 0; q < D; q++) {
                ra[2 * p.w + j].v[q] = seg_at(p.alde, ls, j * D + q);
                ra[2 * p.w + p.aw + j].v[q] = seg_at(p.alde, nx, j * D + q);
            }
        }
        const u32 pb = 2 * p.w + 2 * p.aw;
        for (u32 j = 0; j < p.num_periodic; j++) ra[pb + j] = ext_from_base<D>(r[2 * p.w + j]);
        for (u32 j = 0; j < p.nr; j++) ra[pb + p.num_periodic + j] = ld_ext<D>(p.rnd + (size_t)j * D);
        for (u32 k = 0; k < p.aprog_len; k++) {
            const u32 op = p.aprog[4 * k], dst = p.aprog[4 * k + 1], a = p.aprog[4 * k + 2], b = p.aprog[4 * k + 3];
            switch (op) {
                case 0: ra[dst] = ext_add(ra[a], ra[b]); break;
                case 1: ra[dst] = ext_sub(ra[a], ra[b]); break;
                case 2: ra[dst] = ext_mul(ra[a], ra[b]); break;
                case 3: ra[dst] = ext_from_base<D>(p.consts[a]); break;
                default: T = ext_add(T, ext_mul(ra[a], ld_ext<D>(p.atcoef + (size_t)dst * D))); break;  // OUT
            }
        }
    }
#define WF_MAIN_CUR(col) r[col]
#define WF_AUX_CUR(col) ra[2 * p.w + (col)]
#endif
    const u32 half = (u32)(ce >> 1);
    const u32 cemask = (u32)(ce - 1);
    u64 w = p.tw_ce[i & (half - 1)];
    if (i & half) w = gl_neg(w);
    const u64 x = gl_mul(w, GL_GENERATOR);
    u64 ex = 1;
    for (u32 k = 0; k < p.num_exempt; k++) ex = gl_mul(ex, gl_sub(x, p.exempt[k]));
    GlExt<D> acc = ext_mul_base(T, gl_mul(p.zt[i & (((size_t)1 << p.log_ce_blowup) - 1)], ex));
    // boundary groups, WF_BGRP at a time sharing ONE field inversion (math::batch_inversion, math/src/utils/mod.rs:169; the
    // divisors are never zero on the coset 7 <w_ce>): an inversion is a 72-multiplication chain, the first version spent more
    // time in one gl_inv per group and row than in the transition program of a Rescue-sized AIR
    constexpr u32 WF_BGRP = 4;
    for (u32 g0 = 0; g0 < p.num_groups; g0 += WF_BGRP) {
        GlExt<D> Bs[WF_BGRP];
        u64 den[WF_BGRP], pre[WF_BGRP], run = 1;
#pragma unroll
        for (u32 t = 0; t < WF_BGRP; t++) {
            const u32 g = g0 + t;
            Bs[t] = ext_zero<D>();
            den[t] = 1;
            if (g < p.num_groups) {
                for (u32 e = p.g_off[g]; e < p.g_off[g + 1]; e++) {
                    u64 val = p.e_val[e];
                    if (const u64* tab = p.e_tab[e]) val = tab[(size_t)((u32)(i - p.e_shift[e]) & cemask) * p.e_tstride[e]];
                    Bs[t] = ext_add(Bs[t], ext_mul_base(ld_ext<D>(p.e_cc + (size_t)e * D), gl_sub(WF_MAIN_CUR(p.e_col[e]), val)));
                }
                // x^a = 7^a * w_ce^(i*a mod ce)
                u32 ia = (u32)(((u64)i * p.g_a[g]) & cemask);
                u64 wa = p.tw_ce[ia & (half - 1)];
                if (ia & half) wa = gl_neg(wa);
                den[t] = gl_sub(gl_mul(wa, p.g_oa[g]), p.g_b[g]);
            }
            pre[t] = run;
            run = gl_mul(run, den[t]);
        }
        run = gl_inv(run);
#pragma unroll
        for (int t = WF_BGRP - 1; t >= 0; t--) {
            const u64 inv = gl_mul(run, pre[t]);
            run = gl_mul(run, den[t]);
            acc = ext_add(acc, ext_mul_base(Bs[t], inv));
        }
    }
    if constexpr (AUX) {  // evaluator/boundary.rs: aux_single_value constraints, values and columns in E
        for (u32 g0 = 0; g0 < p.num_agroups; g0 += WF_BGRP) {
            GlExt<D> Bs[WF_BGRP];
            u64 den[WF_BGRP], pre[WF_BGRP], run = 1;
#pragma unroll
            for (u32 t = 0; t < WF_BGRP; t++) {
                const u32 g = g0 + t;
                Bs[t] = ext_zero<D>();
                den[t] = 1;
                if (g < p.num_agroups) {
                    for (u32 e = p.ag_off[g]; e < p.ag_off[g + 1]; e++) {
                        GlExt<D> val = ld_ext<D>(p.ae_val + (size_t)e * D);
                        if (const u64* tab = p.ae_tab[e]) val = ld_ext<D>(tab + (size_t)((u32)(i - p.ae_shift[e]) & cemask) * p.ae_tstride[e]);
                        Bs[t] = ext_add(Bs[t], ext_mul(ext_sub(WF_AUX_CUR(p.ae_col[e]), val), ld_ext<D>(p.ae_cc + (size_t)e * D)));
                    }
                    u32 ia = (u32)(((u64)i * p.ag_a[g]) & cemask);
                    u64 wa = p.tw_ce[ia & (half - 1)];
                    if (ia & half) wa = gl_neg(wa);
                    den[t] = gl_sub(gl_mul(wa, p.ag_oa[g]), p.ag_b[g]);
                }
                pre[t] = run;
                run = gl_mul(run, den[t]);
            }
            run = gl_inv(run);
#pragma unroll
            for (int t = WF_BGRP - 1; t >= 0; t--) {
                const u64 inv = gl_mul(run, pre[t]);
                run = gl_mul(run, den[t]);
                acc = ext_add(acc, ext_mul_base(Bs[t], inv));
            }
        }
    }
    u64* o = p.out.base + il * p.out.W;
#pragma unroll
    for (int q = 0; q < D; q++) o[q] = acc.v[q];
}

#ifdef WF_JIT
extern "C" __global__ void __launch_bounds__(128) wf_jit_constraints_kernel(GenEvalParams p) {
    generic_constraints_row<WF_JIT_D, (WF_JIT_AUX != 0)>(p);
}
#else
template <int D, bool AUX>
__global__ void __launch_bounds__(128) generic_constraints_kernel(GenEvalParams p) {
    generic_constraints_row<D, AUX>(p);
}
#endif
