// Job-list kernels: the batched round driver describes each round of the GG20 offline stage
// as a few "classes" of identical big-integer jobs (one instance per work unit) and runs a
// whole list of classes in ONE persistent launch per modulus width, so the SMs stay full even
// though a single class has only `units` instances.
//
//   out = m1 * m2 * b1^e1 * b2^e2  mod n          (any factor optional)
//
// covers every product of powers on the path: `(h1^a * h2^ro) % N_tilde`
// (/root/reference/src/utilities/mta/range_proofs.rs:52,57,129-132), `(alpha*N+1) * beta^N % NN`
// (:53-55), `r^e * beta % N` (:86), `gs1 * s^N * cipher_e_inv % NN` (:141), Paillier
// encrypt/mul/add (src/utilities/mta/mod.rs:133-145) and `commitment_unknown_order`
// (src/utilities/zk_pdl_with_slack/mod.rs:182-199).  The two powers share their squarings
// (Straus interleaving); multipliers m1, m2 are plain residues.
#pragma once
#include "keyexp.h"
#include "modexp.cuh"

namespace tecdsa {

// instance i of an operand lives at ptr + (idx ? idx[i*idx_stride] : i) * stride   (units: limbs)
struct Operand {
    const uint32_t* ptr;
    const uint32_t* idx;
    uint32_t stride;
    uint32_t idx_stride;
    uint32_t limbs;         // valid limbs at the address (multiple of 4); the rest of K reads as zero
};
__device__ __forceinline__ const uint32_t* operand_at(const Operand& o, int i) {
    size_t row = o.idx ? (size_t)__ldg(o.idx + (size_t)i * o.idx_stride) : (size_t)i;
    return o.ptr + row * o.stride;
}
// this lane's L limbs of a (possibly shorter than K) operand, zero-extended; `skip` limbs are
// skipped first (used to read the high half of a double-width value)
template <int TPI, int L>
__device__ __forceinline__ void load_operand(uint32_t (&x)[L], const Operand& o, int i, uint32_t skip = 0) {
    static_assert(L % 4 == 0, "vector loads need L % 4 == 0");
    const uint32_t* p = operand_at(o, i);
    const uint32_t first = skip + group_lane<TPI>() * L;
#pragma unroll
    for (int c = 0; c < L / 4; c++) {
        uint4 v = make_uint4(0, 0, 0, 0);
        if (first + 4 * c + 4 <= o.limbs) v = *reinterpret_cast<const uint4*>(p + first + 4 * c);
        x[4 * c] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
    }
}

struct ExpClass {
    Operand mod;            // K limbs
    Operand base[2];        // K limbs each
    Operand exp[2];         // exp_limbs[b] limbs each
    Operand mul[3];         // K limbs each (plain residues, any value < 2^(32K))
    uint32_t* out;          // K limbs per instance, out_stride apart
    uint32_t out_stride;
    int exp_limbs[2];
    int nbases;             // 0..2
    int nmul;               // 0..3
    int wide0;              // base[0] is 2K limbs wide and is reduced mod n first (c mod p^2, kzen-paillier decrypt)
    // fixed-base mode: both bases are per-key constants (h1, h2 of a DLogStatement) whose powers
    // base^(j * 2^(5w)) were tabulated at key upload; the job is then a pure product, no squarings.
    const uint32_t* fb;     // nullptr = off; else tables [row][2][FB_WINDOWS][FB_TBL][K] in Montgomery form
    Operand fb_row;         // idx -> key row of instance i (ptr unused)
    int fb_sel[2];          // which of the row's two tables base[b] is (0 = h1, 1 = h2)
    // N-adic mode (nadic.cuh, nadic_jobs_kernel only): the job is modulo N^2, `mod` names N and this the key's
    // constants row (digits of R, R^2, R^3 mod N^2)
    Operand nadic;
    // key-row order (keyexp.h): slot g runs unit order[g] & ~ORDER_PAD and stores only without the ORDER_PAD flag; count is
    // then the number of slots.  nullptr: slot g runs unit g.
    const uint32_t* order;
    int keyexp;             // exp[0] is a key-row exponent and the class is ordered: base 0 runs sliding windows over odd powers
    int count;              // instances
    int item_begin;         // first warp-item of this class in the launch (prefix sum)
};

static constexpr int MAX_CLASSES = 64;
static constexpr int FB_WINDOW_BITS = 8;        // fixed-base windows are wider than the 5-bit windows of variable bases: no squarings to amortise
static constexpr int FB_TBL = 1 << FB_WINDOW_BITS;
static constexpr int FB_WINDOWS = (92 * 32 + FB_WINDOW_BITS - 1) / FB_WINDOW_BITS;   // covers 92-limb (2944-bit) exponents
// window `w` (FB_WINDOW_BITS wide) of a little-endian limb array
__device__ __forceinline__ uint32_t fb_window(const uint32_t* __restrict__ e, int exp_limbs, int w) {
    const int bit = w * FB_WINDOW_BITS;
    const int limb = bit >> 5, off = bit & 31;
    const uint32_t lo = __ldg(e + limb);
    const uint32_t hi = (limb + 1 < exp_limbs) ? __ldg(e + limb + 1) : 0u;
    return (uint32_t)((((uint64_t)hi << 32) | lo) >> off) & (FB_TBL - 1);
}
struct ExpLaunch {
    ExpClass cls[MAX_CLASSES];
    int n_classes;
    int total_items;
};

// The unit slot g of class c runs; `live` is false for a slot that only does its warp's work and stores nothing (the tail of
// an unordered class, a padding slot of an ordered one: the latter repeats a unit of its key row).
__device__ __forceinline__ int job_unit(const ExpClass& c, int g, bool& live) {
    if (c.order) {
        const uint32_t u = __ldg(c.order + g);
        live = !(u & ORDER_PAD);
        return (int)(u & ~ORDER_PAD);
    }
    live = g < c.count;
    return live ? g : c.count - 1;
}

// Key-exponent loop state (keyexp classes), one register: the next window of base 0's exponent as lo * 64 + digit, lo = -1
// once there is none.
static_assert(KEYEXP_BITS <= 6, "the digit is packed in 6 bits");
struct KeyWin {
    int v;
    __device__ __forceinline__ int lo() const { return v >> 6; }
    __device__ __forceinline__ uint32_t entry() const { return (uint32_t)(v & 63) >> 1; }     // table entry of the odd digit
    __device__ __forceinline__ void next(const uint32_t* e, int from) {
        const int top = keyexp_top(e, from);
        uint32_t d = 0;
        v = top >= 0 ? keyexp_window(e, top, d) * 64 + (int)d : -64;
    }
};
// Highest bit position of a keyexp class's merged schedule: the first window of exp[0] or the top 5-bit window of exp[1].
__device__ __forceinline__ int keyexp_start(const KeyWin& kw, int nw1) {
    const int p1 = (nw1 - 1) * WINDOW_BITS;
    return kw.lo() > p1 ? kw.lo() : p1;
}
// Products pending at bit position p of the merged schedule: 1 = the digit of base 0 (a window ends at p), 2 = the window of
// base 1 (p is a multiple of 5).  Worked out once per position, so that every trip of the loop runs one product.
__device__ __forceinline__ int keyexp_pending(const KeyWin& kw, int p, int nw1) {
    return (p == kw.lo() ? 1 : 0) | (p % WINDOW_BITS == 0 && p / WINDOW_BITS < nw1 ? 2 : 0);
}

template <int K, int TPI>
__global__ void __launch_bounds__(128)          // (128, 4) caps at 128 registers with spills: measured 2 % slower
exp_jobs_kernel(const ExpLaunch* __restrict__ launch, uint32_t* __restrict__ tables, unsigned int* __restrict__ counter,
                unsigned long long* __restrict__ work) {
    constexpr int L = K / TPI;
    constexpr int GPW = 32 / TPI;                 // groups per warp
    constexpr int TBL = 1 << WINDOW_BITS;
    const int lane = threadIdx.x & 31;
    const int gl = lane & (TPI - 1);
    const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t* my_tbl = tables + ((size_t)warp_global * GPW + lane / TPI) * (size_t)(2 * TBL * K);
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

        MontCtx<L> m;
        load_operand<TPI, L>(m.n, c.mod, i);
        mont_setup<TPI, L>(m);

        uint32_t acc[L];
#pragma unroll
        for (int j = 0; j < L; j++) acc[j] = m.one[j];
        if (c.fb) {
            // fixed-base product: acc = prod_b prod_w T_b[w][window_w(e_b)]; the next entry is fetched while the current
            // product runs
            const size_t row = __ldg(c.fb_row.idx + (size_t)i * c.fb_row.idx_stride);
            uint32_t bb[L], nb[L];
#pragma unroll 1
            for (int b = 0; b < c.nbases; b++) {
                const uint32_t* tb = c.fb + (row * 2 + c.fb_sel[b]) * (size_t)FB_WINDOWS * FB_TBL * K;
                const uint32_t* e = operand_at(c.exp[b], i);
                const int nwb = (c.exp_limbs[b] * 32 + FB_WINDOW_BITS - 1) / FB_WINDOW_BITS;
                load_limbs<TPI, L>(bb, tb + (size_t)fb_window(e, c.exp_limbs[b], 0) * K);
#pragma unroll 1
                for (int w = 0; w < nwb; w++) {
                    const int wn = w + 1 < nwb ? w + 1 : w;
                    load_limbs<TPI, L>(nb, tb + ((size_t)wn * FB_TBL + fb_window(e, c.exp_limbs[b], wn)) * K);
                    mont_mul<TPI, L>(acc, acc, bb, m.n, m.n0inv);
#pragma unroll
                    for (int j = 0; j < L; j++) bb[j] = nb[j];
                }
            }
        } else {
        // window tables: base*R powers 0..31 for each base
        for (int b = 0; b < c.nbases; b++) {
            uint32_t x[L], xr[L], t[L];
            load_operand<TPI, L>(x, c.base[b], i);
            if (b == 0 && c.wide0) {
                // value = hi * R + lo: reduce both halves and add (mod n)
                uint32_t hi[L], one_p[L];
                load_operand<TPI, L>(hi, c.base[0], i, (uint32_t)K);
#pragma unroll
                for (int j = 0; j < L; j++) one_p[j] = 0;
                if (gl == 0) one_p[0] = 1;
                mont_mul<TPI, L>(hi, hi, m.rr, m.n, m.n0inv);          // hi * R mod n
                mont_mul<TPI, L>(x, x, m.rr, m.n, m.n0inv);
                mont_mul<TPI, L>(x, x, one_p, m.n, m.n0inv);           // lo mod n
                uint32_t cy = group_add_masked<TPI, L>(x, hi, 0xffffffffu);
                uint32_t D[L];
#pragma unroll
                for (int j = 0; j < L; j++) D[j] = x[j];
                uint32_t ge = group_sub_masked<TPI, L>(D, m.n, 0xffffffffu, 1u);
                if (cy | ge) {
#pragma unroll
                    for (int j = 0; j < L; j++) x[j] = D[j];
                }
            }
            mont_mul<TPI, L>(xr, x, m.rr, m.n, m.n0inv);
            uint32_t* tb = my_tbl + (size_t)b * TBL * K;
#pragma unroll
            for (int j = 0; j < L; j++) t[j] = xr[j];
            if (b == 0 && c.keyexp) {
                // odd powers: entry j = x^(2j+1), a chain with step x^2
                mont_mul<TPI, L>(x, xr, xr, m.n, m.n0inv);
                store_limbs<TPI, L>(tb, xr);
#pragma unroll 1
                for (int e = 1; e < KEYEXP_TBL; e++) {
                    mont_mul<TPI, L>(t, t, x, m.n, m.n0inv);
                    store_limbs<TPI, L>(tb + (size_t)e * K, t);
                }
                continue;
            }
            store_limbs<TPI, L>(tb, m.one);
            store_limbs<TPI, L>(tb + K, xr);
#pragma unroll 1
            for (int e = 2; e < TBL; e++) {
                mont_mul<TPI, L>(t, t, xr, m.n, m.n0inv);
                store_limbs<TPI, L>(tb + (size_t)e * K, t);
            }
        }
        __syncwarp();
        if (c.keyexp) {
            // sliding windows over the warp's key exponent (base 0) merged with the 5-bit windows of base 1: at each bit
            // position p a squaring, base 0's digit if a window ends at p, base 1's window if p is a multiple of 5; one product
            // per trip (trips without a product cost as much as the saved products on the 1024-bit jobs)
            const uint32_t* e0 = operand_at(c.exp[0], __shfl_sync(FULL, i, 0));
            const uint32_t* e1 = c.nbases > 1 ? operand_at(c.exp[1], i) : e0;
            const int nw1 = c.nbases > 1 ? (c.exp_limbs[1] * 32 + WINDOW_BITS - 1) / WINDOW_BITS : 0;
            KeyWin kw;
            kw.next(e0, c.exp_limbs[0] * 32 - 1);
            int p = keyexp_start(kw, nw1);
            int pend = p >= 0 ? keyexp_pending(kw, p, nw1) : 0;
            uint32_t bb[L];
#pragma unroll 1
            while (pend) {                              // pend: 4 the squaring into position p, then 1 and 2 as keyexp_pending
                if (pend & 4) {
#pragma unroll
                    for (int j = 0; j < L; j++) bb[j] = acc[j];
                    pend &= 3;
                } else if (pend & 1) {
                    load_limbs<TPI, L>(bb, my_tbl + (size_t)kw.entry() * K);
                    kw.next(e0, p - 1);
                    pend &= 2;
                } else {
                    load_limbs<TPI, L>(bb, my_tbl + (size_t)TBL * K + (size_t)exp_window(e1, c.exp_limbs[1], p / WINDOW_BITS) * K);
                    pend = 0;
                }
                mont_mul<TPI, L>(acc, acc, bb, m.n, m.n0inv);
                if (!pend && p > 0) { p--; pend = 4 | keyexp_pending(kw, p, nw1); }
            }
        } else if (c.nbases > 0) {
            const uint32_t* e0 = operand_at(c.exp[0], i);
            const uint32_t* e1 = c.nbases > 1 ? operand_at(c.exp[1], i) : e0;
            const int nw0 = (c.exp_limbs[0] * 32 + WINDOW_BITS - 1) / WINDOW_BITS;
            const int nw1 = c.nbases > 1 ? (c.exp_limbs[1] * 32 + WINDOW_BITS - 1) / WINDOW_BITS : 0;
            const int nw = nw0 > nw1 ? nw0 : nw1;
            // phases per window: WINDOW_BITS squarings, then one multiply per base that still has windows
            int w = nw - 1, ph = WINDOW_BITS;        // start at the multiply phase of the top window
            uint32_t bb[L];
#pragma unroll 1
            while (w >= 0) {
                bool do_mul = true;
                if (ph < WINDOW_BITS) {
#pragma unroll
                    for (int j = 0; j < L; j++) bb[j] = acc[j];
                    ph++;
                } else if (ph == WINDOW_BITS) {
                    if (w < nw0) load_limbs<TPI, L>(bb, my_tbl + (size_t)exp_window(e0, c.exp_limbs[0], w) * K);
                    else do_mul = false;
                    ph++;
                } else {
                    if (w < nw1) load_limbs<TPI, L>(bb, my_tbl + (size_t)TBL * K + (size_t)exp_window(e1, c.exp_limbs[1], w) * K);
                    else do_mul = false;
                    ph = 0; w--;
                }
                if (do_mul) mont_mul<TPI, L>(acc, acc, bb, m.n, m.n0inv);
            }
        }
        }
        // plain multipliers; the last Montgomery product also leaves the Montgomery domain
        uint32_t u[L];
        if (c.nmul == 0) {
#pragma unroll
            for (int j = 0; j < L; j++) u[j] = 0;
            if (gl == 0) u[0] = 1;
            mont_mul<TPI, L>(acc, acc, u, m.n, m.n0inv);
        } else {
            load_operand<TPI, L>(u, c.mul[0], i);
            mont_mul<TPI, L>(acc, acc, u, m.n, m.n0inv);              // plain acc * m1
#pragma unroll 1
            for (int k = 1; k < c.nmul; k++) {
                load_operand<TPI, L>(u, c.mul[k], i);
                mont_mul<TPI, L>(u, u, m.rr, m.n, m.n0inv);           // m_k * R   (rr < n keeps it canonical)
                mont_mul<TPI, L>(acc, acc, u, m.n, m.n0inv);
            }
        }
        if (live) store_limbs<TPI, L>(c.out + (size_t)i * c.out_stride, acc);
        if (live && gl == 0 && work) {
            unsigned long long products = setup_products(K) + (c.nmul == 0 ? 1 : 1 + 2 * (c.nmul - 1));
            if (c.fb) {
                for (int b = 0; b < c.nbases; b++) products += (c.exp_limbs[b] * 32 + FB_WINDOW_BITS - 1) / FB_WINDOW_BITS;
            } else if (c.nbases > 0) {
                int nwmax = 0, first_lo = -1;
                for (int b = 0; b < c.nbases; b++) {
                    const int nwb = (c.exp_limbs[b] * 32 + WINDOW_BITS - 1) / WINDOW_BITS;
                    const int wide = (b == 0 && c.wide0) ? 3 : 0;
                    if (b == 0 && c.keyexp) {           // x^2, 31 chain products, one product per window
                        products += 1 + KEYEXP_TBL + keyexp_count(operand_at(c.exp[0], i), c.exp_limbs[0] * 32, first_lo) + wide;
                        continue;
                    }
                    products += 1 + (TBL - 2) + nwb + wide;
                    nwmax = nwb > nwmax ? nwb : nwmax;
                }
                const int top = (nwmax - 1) * WINDOW_BITS > first_lo ? (nwmax - 1) * WINDOW_BITS : first_lo;   // squarings
                if (top > 0) products += (unsigned long long)top;
            }
            atomicAdd(work, products * mac_mont(K));
        }
        __syncwarp();
    }
}

// Fixed-base tables T[w][j] = base^(j * 2^(FB_WINDOW_BITS * w)) * R mod N_tilde, w < FB_WINDOWS, j < FB_TBL (entry 0 = R mod n),
// built once per key upload in two steps: the chain of window bases (sequential squarings, one lane-group per (row, base))
// and the fill of every window (one lane-group per (row, base, window)).
template <int K, int TPI>
__global__ void __launch_bounds__(128)
fb_chain_kernel(const uint32_t* __restrict__ mod_tab, const uint32_t* __restrict__ h1_tab, const uint32_t* __restrict__ h2_tab,
                uint32_t* __restrict__ fb, int rows) {
    constexpr int L = K / TPI;
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) / TPI;
    const bool live = g < rows * 2;
    const int gi = live ? g : rows * 2 - 1;
    const int row = gi >> 1, sel = gi & 1;
    MontCtx<L> m;
    load_limbs<TPI, L>(m.n, mod_tab + (size_t)row * K);
    mont_setup<TPI, L>(m);
    uint32_t x[L], bw[L];
    load_limbs<TPI, L>(x, (sel ? h2_tab : h1_tab) + (size_t)row * K);
    mont_mul<TPI, L>(bw, x, m.rr, m.n, m.n0inv);                 // base * R
    uint32_t* tb = fb + (size_t)gi * FB_WINDOWS * FB_TBL * K;
#pragma unroll 1
    for (int w = 0; w < FB_WINDOWS; w++) {
        uint32_t* tw = tb + (size_t)w * FB_TBL * K;
        if (live) { store_limbs<TPI, L>(tw, m.one); store_limbs<TPI, L>(tw + K, bw); }
#pragma unroll 1
        for (int sq = 0; sq < FB_WINDOW_BITS; sq++) mont_mul<TPI, L>(bw, bw, bw, m.n, m.n0inv);
    }
}
template <int K, int TPI>
__global__ void __launch_bounds__(128)
fb_fill_kernel(const uint32_t* __restrict__ mod_tab, uint32_t* __restrict__ fb, int rows) {
    constexpr int L = K / TPI;
    const int total = rows * 2 * FB_WINDOWS;
    const int g = (blockIdx.x * blockDim.x + threadIdx.x) / TPI;
    const bool live = g < total;
    const int gi = live ? g : total - 1;
    const int row = gi / (2 * FB_WINDOWS);
    uint32_t n[L], bw[L], t[L];
    load_limbs<TPI, L>(n, mod_tab + (size_t)row * K);
    const uint32_t n0inv = neg_inv32(__shfl_sync(FULL, n[0], 0, TPI));
    uint32_t* tw = fb + (size_t)gi * FB_TBL * K;
    load_limbs<TPI, L>(bw, tw + K);
#pragma unroll
    for (int j = 0; j < L; j++) t[j] = bw[j];
#pragma unroll 1
    for (int e = 2; e < FB_TBL; e++) {
        mont_mul<TPI, L>(t, t, bw, n, n0inv);
        if (live) store_limbs<TPI, L>(tw + (size_t)e * K, t);
    }
}

}  // namespace tecdsa
