// Arithmetic modulo a perfect square M = N^2 in "N-adic" Montgomery form.
//
// Every exponentiation modulo N^2 on the path (Paillier encrypt / homomorphic multiply, the u, v
// terms of the range and PDL proofs: /root/reference/src/utilities/mta/mod.rs:133-145,
// src/utilities/mta/range_proofs.rs:54,135,141, src/utilities/zk_pdl_with_slack/mod.rs:144-157)
// is 4096-bit arithmetic in the reference (GMP) and costs 2*(2K)^2 MACs per Montgomery product in
// exp_jobs_kernel<128,8>.  Here a residue x mod N^2 is kept as two digits x = x0 + x1*N
// (0 <= x0, x1 < N) and all work is done modulo N (K limbs, R = 2^(32K)):
//
//   X*Y*R^-1 mod N^2,  with  t = X0*Y0,  u' = (t + m*N)/R  (the Montgomery step, quotient number m):
//       Z0 = u' mod N,   Z1 = (X0*Y1 + X1*Y0 - m) * R^-1 + [u' >= N]   (mod N)
//
// (t = u'*R - m*N, so t*R^-1 = u' - N*(m*R^-1) mod N^2, and N*x mod N^2 only depends on x mod N.)
// Z1 is ONE interleaved Montgomery reduction over both cross products with -m folded into the
// starting accumulator, so a multiplication costs 2K^2 + 3K^2 = 5K^2 MACs and a squaring 4K^2
// (cross term X0 * (2*X1 mod N)), against 8K^2 for the direct 2K-limb Montgomery product.  The
// values are identical: operands come in and results go out as plain 2K-limb integers.  Per-key
// constants (digits of R, R^2, R^3 mod N^2) are built at key upload by nadic_setup_kernel.
#pragma once
#include "jobs.cuh"

// The row loop of a pass walks the TPI lanes of a group; its body (L rows) ends with the accumulator pairs rotated, which costs
// 2 L + 1 register moves per trip on the FMA-heavy pipe (ptxas emits IMAD.MOV; 7 % of the executed instructions,
// profiles/r02_ncu_nadic_summary.md).  Unrolling two lanes per trip halves the moves but MEASURED no faster on B200 (1190 vs
// 1190 ms per 8192-session batch), four lanes 6 % slower (instruction cache): profiles/r02_nadic_unroll_ab.md.  Default 1.
#ifndef NADIC_GROUP_UNROLL
#define NADIC_GROUP_UNROLL 1
#endif
constexpr int kNadicGroupUnroll = NADIC_GROUP_UNROLL;

namespace tecdsa {

template <int L> struct Dig { uint32_t d0[L], d1[L]; };

// (a + b) mod n, (a - b) mod n for canonical inputs
template <int TPI, int L>
__device__ __forceinline__ void mod_add(uint32_t (&r)[L], const uint32_t (&a)[L], const uint32_t (&b)[L], const uint32_t (&n)[L]) {
    uint32_t T[L];
#pragma unroll
    for (int j = 0; j < L; j++) T[j] = a[j];
    uint32_t cy = group_add_masked<TPI, L>(T, b, 0xffffffffu);
    reduce_once<TPI, L>(r, T, cy, n);
}
template <int TPI, int L>
__device__ __forceinline__ void mod_sub(uint32_t (&r)[L], const uint32_t (&a)[L], const uint32_t (&b)[L], const uint32_t (&n)[L]) {
    uint32_t T[L];
#pragma unroll
    for (int j = 0; j < L; j++) T[j] = a[j];
    uint32_t ge = group_sub_masked<TPI, L>(T, b, 0xffffffffu, 1u);       // a + ~b + 1; carry out == (a >= b)
    (void)group_add_masked<TPI, L>(T, n, ge ? 0u : 0xffffffffu);          // borrowed: add n back
#pragma unroll
    for (int j = 0; j < L; j++) r[j] = T[j];
}
template <int TPI, int L>
__device__ __forceinline__ void mod_inc(uint32_t (&r)[L], uint32_t c, const uint32_t (&n)[L]) {      // r = (r + c) mod n, c in {0,1}
    uint32_t one[L];
#pragma unroll
    for (int j = 0; j < L; j++) one[j] = 0;
    if (group_lane<TPI>() == 0) one[0] = c;
    mod_add<TPI, L>(r, r, one, n);
}

// One row of the fused product: the accumulator pair takes x0*b (and x1*b2 when THREE), then the Montgomery step.
template <int TPI, int L, bool THREE>
__device__ __forceinline__ uint32_t nadic_row(uint32_t (&A)[L + 2], uint32_t (&B)[L + 2], const uint32_t (&x0)[L], const uint32_t (&x1)[L],
                                              const uint32_t (&n)[L], uint32_t b, uint32_t b2, uint32_t n0inv, uint32_t inc, uint32_t& q_out) {
    B[L] = add_cc(B[L], inc);
    B[L + 1] = addc(0, 0);
    A[0] = add_cc(A[0], B[1]);
    madc_odd_rshift<L>(B, x0, b);
    mad_even<L>(A, x0, b);
    if (THREE) {
        mad_odd<L>(B, x1, b2);
        mad_even<L>(A, x1, b2);
    }
    uint32_t q = __shfl_sync(FULL, A[0] * n0inv, 0, TPI);
    q_out = q;
    mad_odd<L>(B, n, q);
    mad_even<L>(A, n, q);
    uint32_t dn = __shfl_down_sync(FULL, A[0], 1, TPI);
    return (group_lane<TPI>() == TPI - 1) ? 0u : dn;
}
// All K rows of one pass over accumulators E/O (pre-loaded by the caller): sum_i (x0*b[i] + [THREE] x1*b2[i] + q_i*n) 2^(32i),
// divided by R.  REC keeps the quotient digits (lane g its own L).  Result: T (K limbs), return = words above them.
template <int TPI, int L, bool THREE, bool REC>
__device__ __forceinline__ uint32_t nadic_pass(uint32_t (&T)[L], uint32_t (&E)[L + 2], uint32_t (&O)[L + 2], const uint32_t (&x0)[L],
                                               const uint32_t (&x1)[L], const uint32_t (&b)[L], const uint32_t (&b2)[L], const uint32_t (&n)[L],
                                               uint32_t n0inv, uint32_t (&m)[L]) {
    const int gl = group_lane<TPI>();
    uint32_t inc = 0;
#pragma unroll kNadicGroupUnroll
    for (int gi = 0; gi < TPI; gi++) {
        const bool rec = gi == gl;
#pragma unroll
        for (int li = 0; li < L; li += 2) {
            const uint32_t b0 = __shfl_sync(FULL, b[li], gi, TPI);
            const uint32_t b1 = __shfl_sync(FULL, b[li + 1], gi, TPI);
            uint32_t c0 = 0, c1 = 0;
            if (THREE) {
                c0 = __shfl_sync(FULL, b2[li], gi, TPI);
                c1 = __shfl_sync(FULL, b2[li + 1], gi, TPI);
            }
            uint32_t q0, q1;
            inc = nadic_row<TPI, L, THREE>(E, O, x0, x1, n, b0, c0, n0inv, inc, q0);
            inc = nadic_row<TPI, L, THREE>(O, E, x0, x1, n, b1, c1, n0inv, inc, q1);
            if (REC && rec) { m[li] = q0; m[li + 1] = q1; }
        }
    }
    return rows_finish<TPI, L>(T, E, O, inc);
}
// value = ov * R + T < 3N  ->  canonical T; returns how many times N was subtracted
template <int TPI, int L>
__device__ __forceinline__ uint32_t reduce_twice(uint32_t (&T)[L], uint32_t ov, const uint32_t (&n)[L]) {
    uint32_t cnt = 0;
#pragma unroll 1
    for (int r = 0; r < 2; r++) {
        uint32_t D[L];
#pragma unroll
        for (int j = 0; j < L; j++) D[j] = T[j];
        const uint32_t ge = group_sub_masked<TPI, L>(D, n, 0xffffffffu, 1u);
        const bool take = (ov | ge) != 0;
#pragma unroll
        for (int j = 0; j < L; j++) T[j] = take ? D[j] : T[j];
        if (take) { cnt++; if (!ge) ov--; }
    }
    return cnt;
}

// Z = X*Y*R^-1 mod N^2 in digits, in two passes of K rows:
//   pass 0:  u' = (X0*Y0 + m*N)/R, recording the quotient digits m;        Z0 = u' mod N, uc = [u' >= N]
//   pass 1:  (X0*Y1 + X1*Y0 - m) * R^-1 mod N in one interleaved reduction: the accumulator starts at ~m + 1
//            (T - m = T + ~m + 1 - R, and R*R^-1 = 1), so Z1 = redc(T + ~m + 1) - 1 + uc.
// Cost 5K^2 MACs; 4K^2 with `cross2` false, which drops the X1*Y0 term — valid when X1 == 0 (lifting a plain operand: X0
// may then be any value < R) or when the caller passes Y = (X0, 2*X1 mod N) to square X.  Y is canonical, X1 < N.
template <int TPI, int L>
__device__ __forceinline__ void nadic_mul(Dig<L>& Z, const Dig<L>& X, const Dig<L>& Y, bool cross2, const uint32_t (&n)[L], uint32_t n0inv) {
    const int gl = group_lane<TPI>();
    uint32_t u[L], m[L], T[L];
    uint32_t E[L + 2], O[L + 2];
#pragma unroll
    for (int j = 0; j < L; j++) m[j] = 0;
#pragma unroll
    for (int j = 0; j < L + 2; j++) { E[j] = 0; O[j] = 0; }
    uint32_t ov = nadic_pass<TPI, L, false, true>(u, E, O, X.d0, X.d1, Y.d0, Y.d0, n, n0inv, m);
    const uint32_t uc = reduce_twice<TPI, L>(u, ov, n);
#pragma unroll
    for (int j = 0; j < L; j++) { E[j] = ~m[j]; O[j] = 0; }
    E[L] = 0; E[L + 1] = 0; O[L] = 0; O[L + 1] = 0;
    if (gl == 0) O[1] = 1;                                     // enters column 0 with the first row
    if (cross2) ov = nadic_pass<TPI, L, true, false>(T, E, O, X.d0, X.d1, Y.d1, Y.d0, n, n0inv, m);
    else ov = nadic_pass<TPI, L, false, false>(T, E, O, X.d0, X.d1, Y.d1, Y.d0, n, n0inv, m);
    (void)reduce_twice<TPI, L>(T, ov, n);
    // Z1 = T - 1 + uc
    {
        uint32_t one[L];
#pragma unroll
        for (int j = 0; j < L; j++) one[j] = 0;
        if (gl == 0) one[0] = 1u - uc;
        mod_sub<TPI, L>(T, T, one, n);
    }
#pragma unroll
    for (int j = 0; j < L; j++) { Z.d0[j] = u[j]; Z.d1[j] = T[j]; }
}

// Y = (X0, 2*X1 mod N): nadic_mul(Z, X, Y, false) then squares X
template <int TPI, int L>
__device__ __forceinline__ void square_operand(Dig<L>& Y, const Dig<L>& X, const uint32_t (&n)[L]) {
#pragma unroll
    for (int j = 0; j < L; j++) Y.d0[j] = X.d0[j];
    mod_add<TPI, L>(Y.d1, X.d1, X.d1, n);
}

// (A + B) mod N^2 in digits
template <int TPI, int L>
__device__ __forceinline__ void dig_add(Dig<L>& Z, const Dig<L>& A, const Dig<L>& B, const uint32_t (&n)[L]) {
    uint32_t T[L], D[L];
#pragma unroll
    for (int j = 0; j < L; j++) T[j] = A.d0[j];
    const uint32_t cy = group_add_masked<TPI, L>(T, B.d0, 0xffffffffu);
#pragma unroll
    for (int j = 0; j < L; j++) D[j] = T[j];
    const uint32_t ge = group_sub_masked<TPI, L>(D, n, 0xffffffffu, 1u);
    const uint32_t c = (cy | ge) ? 1u : 0u;
    uint32_t hi[L];
    mod_add<TPI, L>(hi, A.d1, B.d1, n);
    mod_inc<TPI, L>(hi, c, n);
#pragma unroll
    for (int j = 0; j < L; j++) { Z.d0[j] = c ? D[j] : T[j]; Z.d1[j] = hi[j]; }
}

template <int TPI, int L>
__device__ __forceinline__ void load_dig(Dig<L>& D, const uint32_t* p) {
    constexpr int K = TPI * L;
    load_limbs<TPI, L>(D.d0, p);
    load_limbs<TPI, L>(D.d1, p + K);
}
template <int TPI, int L>
__device__ __forceinline__ void store_dig(uint32_t* p, const Dig<L>& D) {
    constexpr int K = TPI * L;
    store_limbs<TPI, L>(p, D.d0);
    store_limbs<TPI, L>(p + K, D.d1);
}

// per-key constants row, NADIC_CONST_K * K limbs: digits of R ("one") and of R^2 .. R^5 modulo N^2
static constexpr int NADIC_ONE = 0, NADIC_RR2 = 2;                    // offsets in units of K limbs; R^(2+h) at NADIC_RR2 + 2h
static constexpr int NADIC_CONST_K = 10;
static constexpr int NADIC_TABLE_ENTRIES = 2 * (1 << WINDOW_BITS) + 1;  // per lane group: two window tables + one parked value, 2K limbs each

// plain operand c = sum_h c_h R^h (up to 4K limbs, zero-extended from o.limbs, any value) -> Montgomery digits of c mod N^2:
// sum_h (c_h, 0) * R^(h+2) * R^-1
template <int TPI, int L>
__device__ __forceinline__ void to_nadic(Dig<L>& X, const Operand& o, int i, const uint32_t* consts, const uint32_t (&n)[L], uint32_t n0inv) {
    constexpr int K = TPI * L;
    Dig<L> a, c, part;
#pragma unroll
    for (int j = 0; j < L; j++) { a.d1[j] = 0; part.d0[j] = 0; part.d1[j] = 0; X.d0[j] = 0; X.d1[j] = 0; }
    int parts = ((int)o.limbs + K - 1) / K;                    // uniform per class
    if (parts > 4) parts = 4;
#pragma unroll 1
    for (int h = 0; h < parts; h++) {
        load_operand<TPI, L>(a.d0, o, i, (uint32_t)(h * K));
        load_dig<TPI, L>(c, consts + (NADIC_RR2 + 2 * h) * K);
        nadic_mul<TPI, L>(part, a, c, false, n, n0inv);        // a.d1 == 0: no X1*Y0 term
        dig_add<TPI, L>(X, X, part, n);
    }
}

// Same job semantics as exp_jobs_kernel (out = m1*m2*m3 * b1^e1 * b2^e2 mod N^2, plain 2K-limb operands and result), but
// `mod` names N (K limbs) and `nadic` the per-key constants row.  K is the width of N.
template <int K, int TPI, int MINB>
__global__ void __launch_bounds__(128, MINB)
nadic_jobs_kernel(const ExpLaunch* __restrict__ launch, uint32_t* __restrict__ tables, unsigned int* __restrict__ counter,
                  unsigned long long* __restrict__ work) {
    constexpr int L = K / TPI;
    constexpr int GPW = 32 / TPI;
    constexpr int TBL = 1 << WINDOW_BITS;
    const int lane = threadIdx.x & 31;
    const int gl = lane & (TPI - 1);
    const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t* my_tbl = tables + ((size_t)warp_global * GPW + lane / TPI) * (size_t)(NADIC_TABLE_ENTRIES * 2 * K);
    uint32_t* p_slot = my_tbl + (size_t)(2 * TBL) * 2 * K;    // product of the plain multipliers, parked during the exponentiation
    const int total = launch->total_items;
    const int ncls = launch->n_classes;

    while (true) {
        unsigned int item = 0;
        if (lane == 0) item = atomicAdd(counter, 1u);
        item = __shfl_sync(FULL, item, 0);
        if ((int)item >= total) break;
        int ci = 0;
        while (ci + 1 < ncls && launch->cls[ci + 1].item_begin <= (int)item) ci++;
        const ExpClass& c = launch->cls[ci];
        bool live;
        const int i = job_unit(c, ((int)item - c.item_begin) * GPW + lane / TPI, live);

        uint32_t n[L];
        load_operand<TPI, L>(n, c.mod, i);
        const uint32_t n0inv = neg_inv32(__shfl_sync(FULL, n[0], 0, TPI));
        const uint32_t* consts = operand_at(c.nadic, i);

        // operands 0..nbases-1 are bases (window tables), the rest plain multipliers (folded into P)
        Dig<L> acc, Y;
        {
            Dig<L> P;
            load_dig<TPI, L>(P, consts + NADIC_ONE * K);
            store_dig<TPI, L>(p_slot, P);
        }
#pragma unroll 1
        for (int k = 0; k < c.nbases + c.nmul; k++) {
            const bool is_base = k < c.nbases;
            Dig<L> xr;
            to_nadic<TPI, L>(xr, is_base ? c.base[k] : c.mul[k - c.nbases], i, consts, n, n0inv);
            uint32_t* tb = my_tbl + (size_t)k * TBL * 2 * K;
            const bool odd = k == 0 && c.keyexp;
            if (odd) {
                store_dig<TPI, L>(tb, xr);
                Y = xr;
            } else if (is_base) {
                load_dig<TPI, L>(Y, consts + NADIC_ONE * K);
                store_dig<TPI, L>(tb, Y);
                store_dig<TPI, L>(tb + 2 * K, xr);
                Y = xr;
            } else {
                load_dig<TPI, L>(Y, p_slot);
            }
            // base: Y runs through xr^2 .. xr^31 into the table; multiplier: one product P *= xr.  Key-exponent base 0: the
            // first product gives x^2, which becomes the step of the chain x^3 .. x^63 of odd powers (entry j = x^(2j+1)).
            const int steps = odd ? KEYEXP_TBL : is_base ? TBL - 2 : 1;
#pragma unroll 1
            for (int e = 0; e < steps; e++) {
                nadic_mul<TPI, L>(Y, Y, xr, true, n, n0inv);
                if (odd && e == 0) { xr = Y; load_dig<TPI, L>(Y, tb); }
                else if (is_base) store_dig<TPI, L>(tb + (size_t)(odd ? e : e + 2) * 2 * K, Y);
            }
            if (!is_base) store_dig<TPI, L>(p_slot, Y);
        }
        __syncwarp();
        // exponentiation; the multiplier product P and the exit from the Montgomery domain (times (1, 0)) are the two
        // last steps of the same loop
        load_dig<TPI, L>(acc, consts + NADIC_ONE * K);
        {
            // a keyexp class walks the sliding windows of the warp's key exponent (every lane group holds the same row)
            const uint32_t* e0 = operand_at(c.exp[0], c.keyexp ? __shfl_sync(FULL, i, 0) : i);
            const uint32_t* e1 = c.nbases > 1 ? operand_at(c.exp[1], i) : e0;
            const int nw0 = c.nbases > 0 ? (c.exp_limbs[0] * 32 + WINDOW_BITS - 1) / WINDOW_BITS : 0;
            const int nw1 = c.nbases > 1 ? (c.exp_limbs[1] * 32 + WINDOW_BITS - 1) / WINDOW_BITS : 0;
            const int nw = nw0 > nw1 ? nw0 : nw1;
            int w = nw - 1, ph = WINDOW_BITS;
            // keyexp: w is the bit position; ph = 8 * (next window of base 0, KeyWin) + the products pending at w (4 the squaring
            // into w, then 1 and 2 as keyexp_pending), one per trip.  One register for both keeps the kernel at 128 registers.
            if (c.keyexp) {
                KeyWin kw;
                kw.next(e0, c.exp_limbs[0] * 32 - 1);
                w = keyexp_start(kw, nw1);
                ph = kw.v * 8 + (w >= 0 ? keyexp_pending(kw, w, nw1) : 0);
                if (w < 0) w = -1;
            }
#pragma unroll 1
            while (w >= -2) {
                bool do_mul = true, cross2 = true;
                if (w == -1) { load_dig<TPI, L>(Y, p_slot); do_mul = c.nmul > 0; w = -2; }
                else if (w == -2) {
#pragma unroll
                    for (int j = 0; j < L; j++) { Y.d0[j] = 0; Y.d1[j] = 0; }
                    if (gl == 0) Y.d0[0] = 1;
                    w = -3;
                }
                else if (c.keyexp) {
                    KeyWin kw{ph >> 3};
                    int pend = ph & 7;
                    if (pend & 4) { square_operand<TPI, L>(Y, acc, n); cross2 = false; pend &= 3; }
                    else if (pend & 1) { load_dig<TPI, L>(Y, my_tbl + (size_t)kw.entry() * 2 * K); kw.next(e0, w - 1); pend &= 2; }
                    else {
                        load_dig<TPI, L>(Y, my_tbl + ((size_t)TBL + exp_window(e1, c.exp_limbs[1], w / WINDOW_BITS)) * 2 * K);
                        pend = 0;
                    }
                    if (!pend) {                        // position w done: square into w - 1, or leave for the multipliers
                        if (w > 0) { w--; pend = 4 | keyexp_pending(kw, w, nw1); }
                        else w = -1;
                    }
                    ph = kw.v * 8 + pend;
                }
                else if (ph < WINDOW_BITS) { square_operand<TPI, L>(Y, acc, n); cross2 = false; ph++; }
                else if (ph == WINDOW_BITS) {
                    if (w < nw0) load_dig<TPI, L>(Y, my_tbl + (size_t)exp_window(e0, c.exp_limbs[0], w) * 2 * K);
                    else do_mul = false;
                    ph++;
                } else {
                    if (w < nw1) load_dig<TPI, L>(Y, my_tbl + ((size_t)TBL + exp_window(e1, c.exp_limbs[1], w)) * 2 * K);
                    else do_mul = false;
                    ph = 0; w--;
                }
                if (do_mul) nadic_mul<TPI, L>(acc, acc, Y, cross2, n, n0inv);
            }
        }
        // plain value = d0 + d1 * N  (2K limbs)
        uint32_t lo[L], hi[L];
        group_mul_wide<TPI, L>(lo, hi, acc.d1, n);
        const uint32_t cy = group_add_masked<TPI, L>(lo, acc.d0, 0xffffffffu);
        {
            uint32_t one[L];
#pragma unroll
            for (int j = 0; j < L; j++) one[j] = 0;
            if (gl == 0) one[0] = cy;
            (void)group_add_masked<TPI, L>(hi, one, 0xffffffffu);
        }
        if (live) {
            uint32_t* o = c.out + (size_t)i * c.out_stride;
            store_limbs<TPI, L>(o, lo);
            store_limbs<TPI, L>(o + K, hi);
            if (gl == 0 && work) {
                // nadic_mul: 4K^2 + 2K without the second cross product (lifts, squarings), 5K^2 + 2K with it
                const unsigned long long m4 = 4ull * K * K + 2 * K, m5 = 5ull * K * K + 2 * K;
                unsigned long long macs = (unsigned long long)K * K + m5;                                    // exit: times (1, 0), then d0 + d1 * N
                int nwmax = 0, first_lo = -1;
                for (int k = 0; k < c.nbases + c.nmul; k++) {
                    const Operand& o2 = k < c.nbases ? c.base[k] : c.mul[k - c.nbases];
                    int parts = ((int)o2.limbs + K - 1) / K;
                    macs += (unsigned long long)(parts > 4 ? 4 : parts) * m4;
                    if (k == 0 && c.keyexp) {           // x^2 and 31 chain products, one product per window
                        macs += (unsigned long long)(KEYEXP_TBL + keyexp_count(operand_at(c.exp[0], i), c.exp_limbs[0] * 32, first_lo)) * m5;
                    } else if (k < c.nbases) {
                        const int nwb = (c.exp_limbs[k] * 32 + WINDOW_BITS - 1) / WINDOW_BITS;
                        macs += (unsigned long long)(TBL - 2 + nwb) * m5;
                        nwmax = nwb > nwmax ? nwb : nwmax;
                    } else macs += m5;
                }
                if (c.nmul > 0) macs += m5;
                const int top = (nwmax - 1) * WINDOW_BITS > first_lo ? (nwmax - 1) * WINDOW_BITS : first_lo;   // squarings
                if (top > 0) macs += (unsigned long long)top * m4;
                atomicAdd(work, macs);
            }
        }
        __syncwarp();
    }
}

// One lane-group per key row: digits of R, R^2 .. R^5 modulo N^2 (N odd, > 1).  R^2 = 2^(64K) comes from doubling (1, 0).
template <int K, int TPI>
__global__ void __launch_bounds__(128)
nadic_setup_kernel(const uint32_t* __restrict__ n_tab, uint32_t* __restrict__ out, int rows) {
    constexpr int L = K / TPI;
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) / TPI;
    const bool live = g < rows;
    const int row = live ? g : rows - 1;
    uint32_t n[L];
    load_limbs<TPI, L>(n, n_tab + (size_t)row * K);
    const uint32_t n0inv = neg_inv32(__shfl_sync(FULL, n[0], 0, TPI));
    Dig<L> t, rr2;
#pragma unroll
    for (int j = 0; j < L; j++) { t.d0[j] = 0; t.d1[j] = 0; }
    if (group_lane<TPI>() == 0) t.d0[0] = 1;
    rr2 = t;
#pragma unroll 1
    for (int i = 0; i < 64 * K; i++) dig_add<TPI, L>(rr2, rr2, rr2, n);
    uint32_t* o = out + (size_t)row * NADIC_CONST_K * K;
    if (live) store_dig<TPI, L>(o + NADIC_RR2 * K, rr2);
    // s = 0: (1, 0) * R^2 * R^-1 = R;   s >= 1: R^(s+1) * R^2 * R^-1 = R^(s+2)
    Dig<L> cur = rr2;
#pragma unroll 1
    for (int s = 0; s < 4; s++) {
        nadic_mul<TPI, L>(t, s ? cur : t, rr2, true, n, n0inv);
        if (s) cur = t;
        if (live) store_dig<TPI, L>(o + (s ? NADIC_RR2 + 2 * s : NADIC_ONE) * K, t);
    }
}

}  // namespace tecdsa
