// Batched round driver of the GG20 offline-signing stage (t = 1, n = 3, two signers per
// session): reproduces /root/reference/src/protocols/multi_party_ecdsa/gg_2020/state_machine/
// sign/rounds.rs Round0..Round6 for `units` parties at once.  Both parties of a session are
// resident on the same GPU, so the six message rounds are plain reads of the peer's arena
// fields.  Every round is: a glue kernel (EC / hashing / plain integers), one persistent
// job-list launch per kind of modulus (1024-bit: p, q; 2048-bit: N_tilde, N; p-adic: p^2, q^2;
// N-adic: N^2 — nadic.cuh), and, where the verifier needs `mod_inv`, an inversion launch.
#include "ctx.h"
#include "gg20_rounds.cuh"
#include "modinv.cuh"

#include <algorithm>
#include <cstdlib>
#include <string>
#include <thread>
#include <vector>

using namespace tecdsa;

namespace {

struct Builder {
    tecdsa_ctx* c;
    const tecdsa_keyset* ks;
    Arena A;
    int U;
    ExpLaunch L32, L64, L128, LPQ;      // 1024-bit, 2048-bit, N-adic mod N^2, p-adic mod p^2 / q^2
    InvLaunch I64, I128, I128H;        // I128H: modulo N^2 via the N-wide inversion + Hensel step
    const uint32_t* order[2];          // units ordered by own / peer key row (keyexp.h), order_len[r] slots each
    int order_len[2];

    Operand fld(int f, int limbs = 0) const {
        return Operand{A.base + (size_t)A.off[f] * U, nullptr, A.size[f], 0, (uint32_t)(limbs ? limbs : A.size[f])};
    }
    Operand peer(int f, int limbs = 0) const {
        return Operand{A.base + (size_t)A.off[f] * U, A.peer, A.size[f], 1, (uint32_t)(limbs ? limbs : A.size[f])};
    }
    // sub-field of the randomness record (own unit or peer unit)
    Operand rnd(int off, int limbs, bool of_peer = false) const {
        return Operand{A.base + (size_t)A.off[F_RND] * U + off, of_peer ? A.peer : nullptr, RND_LIMBS, 1, (uint32_t)limbs};
    }
    Operand key(int t, const uint32_t* rows) const { return Operand{A.key[t], rows, (uint32_t)KEY_SIZE[t], 1, (uint32_t)KEY_SIZE[t]}; }
    uint32_t* out(int f) const { return A.base + (size_t)A.off[f] * U; }

    static void reset(ExpLaunch& l) { l.n_classes = 0; l.total_items = 0; }
    static void reset(InvLaunch& l) { l.n_classes = 0; l.total_items = 0; }
    // Jobs modulo a square whose root the key tables hold (N^2, and the unit's own p^2 / q^2) are routed to the N-adic
    // lists (nadic.cuh: same value, about half the MACs of the double-width Montgomery product); `l` / `gpw` then only say
    // where the class would have gone otherwise.
    void exp_class(ExpLaunch& l, int gpw, Operand mod, int nb, Operand b0, Operand e0, int el0, Operand b1, Operand e1, int el1,
                   int nm, Operand m0, Operand m1, int out_field, int wide0 = 0, Operand m2 = Operand{nullptr, nullptr, 0, 0, 0}) {
        ExpLaunch* dst = &l;
        Operand nadic = Operand{nullptr, nullptr, 0, 0, 0};
        if (mod.ptr == A.key[KT_NN]) {
            dst = &L128; gpw = 32 / tecdsa_nadic_tpi();
            mod = key(KT_N, mod.idx); nadic = Operand{ks->nadic, mod.idx, NADIC_ROW * 64, 1, NADIC_ROW * 64};
        } else if (mod.ptr == A.key[KT_PP] || mod.ptr == A.key[KT_QQ]) {
            const bool is_p = mod.ptr == A.key[KT_PP];
            dst = &LPQ; gpw = 32 / tecdsa_nadic32_tpi(); wide0 = 0;      // operand width is handled by the lift (any width up to 4K)
            mod = key(is_p ? KT_P : KT_Q, mod.idx); nadic = Operand{is_p ? ks->nadic_p : ks->nadic_q, mod.idx, NADIC_ROW * 32, 1, NADIC_ROW * 32};
        }
        // base 0 raised to an exponent of the own or the peer key row: the class runs over the units ordered by that row, so
        // that its warps are key-uniform and can walk the row's sliding-window schedule
        int kx = -1;
        if (nb > 0 && (e0.idx == A.row_own || e0.idx == A.row_peer))
            for (int t : {KT_N, KT_P, KT_Q, KT_PM1, KT_QM1, KT_QMODPM1, KT_PMODQM1})
                if (e0.ptr == A.key[t]) kx = e0.idx == A.row_peer;
        ExpClass& k = dst->cls[dst->n_classes++];
        k.mod = mod; k.base[0] = b0; k.base[1] = b1; k.exp[0] = e0; k.exp[1] = e1; k.exp_limbs[0] = el0; k.exp_limbs[1] = el1;
        k.mul[0] = m0; k.mul[1] = m1; k.mul[2] = m2; k.nbases = nb; k.nmul = nm; k.wide0 = wide0;
        k.fb = nullptr; k.fb_row = Operand{nullptr, nullptr, 0, 0, 0}; k.fb_sel[0] = k.fb_sel[1] = 0;
        k.nadic = nadic;
        k.order = kx >= 0 ? order[kx] : nullptr; k.keyexp = kx >= 0;
        k.out = out(out_field); k.out_stride = A.size[out_field]; k.count = kx >= 0 ? order_len[kx] : U; k.item_begin = dst->total_items;
        dst->total_items += (k.count + gpw - 1) / gpw;
    }
    // out = [m0 *] h2^e_h2 * h1^e_h1 mod N_tilde(rows) through the per-key fixed-base tables
    void fb_class(ExpLaunch& l, int gpw, const uint32_t* rows, Operand e_h2, int el_h2, Operand e_h1, int el_h1, int nm, Operand m0, int out_field) {
        const Operand none = {nullptr, nullptr, 0, 0, 0};
        exp_class(l, gpw, key(KT_NT, rows), 2, none, e_h2, el_h2, none, e_h1, el_h1, nm, m0, none, out_field);
        ExpClass& k = l.cls[l.n_classes - 1];
        k.fb = ks->fb; k.fb_row = Operand{nullptr, rows, 0, 1, 0}; k.fb_sel[0] = 1; k.fb_sel[1] = 0;
    }
    // own-key power base^N mod N^2 (the unit knows its own p, q), slot s, in three stages (declared shortcut: identical
    // value): b^(pq) mod p^2 == ((b mod p)^(q mod (p-1)) mod p)^p mod p^2 because x^p mod p^2 depends only on x mod p.
    //   1. 1024-bit job list:  TP[s] = (b mod p)^(q mod (p-1)) mod p,   TQ[s] likewise          (crt_stage1)
    //   2. 2048-bit job list:  YP[s] = TP[s]^p mod p^2,  YQ[s] = TQ[s]^q mod q^2                (crt_stage2)
    //   3. gg20_crt recombines YP, YQ into XC[s] in [0, N^2)
    void crt_stage1(ExpLaunch& l32, int gpw32, const uint32_t* rows, int slot, Operand base64) {
        const Operand none = {nullptr, nullptr, 0, 0, 0};
        exp_class(l32, gpw32, key(KT_P, rows), 1, base64, key(KT_QMODPM1, rows), 32, none, none, 0, 0, none, none, F_TP0 + slot, 1);
        exp_class(l32, gpw32, key(KT_Q, rows), 1, base64, key(KT_PMODQM1, rows), 32, none, none, 0, 0, none, none, F_TQ0 + slot, 1);
    }
    void crt_stage2(ExpLaunch& l64, int gpw64, const uint32_t* rows, int slot) {
        const Operand none = {nullptr, nullptr, 0, 0, 0};
        exp_class(l64, gpw64, key(KT_PP, rows), 1, fld(F_TP0 + slot, 32), key(KT_P, rows), 32, none, none, 0, 0, none, none, F_YP0 + slot);
        exp_class(l64, gpw64, key(KT_QQ, rows), 1, fld(F_TQ0 + slot, 32), key(KT_Q, rows), 32, none, none, 0, 0, none, none, F_YQ0 + slot);
    }
    void inv_class(InvLaunch& l, int gpw, Operand mod, Operand in, int out_field, int flag_byte) {
        InvLaunch* dst = &l;
        Operand nadic = Operand{nullptr, nullptr, 0, 0, 0};
        if (mod.ptr == A.key[KT_NN] && tecdsa_hensel_inverse()) {     // inverse modulo N plus a Hensel step (nadic_inv.cuh)
            dst = &I128H; gpw = 32 / TPI_NADIC_INV;
            mod = key(KT_N, mod.idx); nadic = Operand{ks->nadic, mod.idx, NADIC_ROW * 64, 1, NADIC_ROW * 64};
        }
        InvLaunch& ll = *dst;
        InvClass& k = ll.cls[ll.n_classes++];
        k.nadic = nadic;
        k.mod = mod; k.in = in; k.out = out(out_field); k.out_stride = A.size[out_field];
        k.ok = reinterpret_cast<uint8_t*>(out(F_FLAGS)) + flag_byte; k.ok_stride = A.size[F_FLAGS] * 4;
        k.count = U; k.item_begin = ll.total_items;
        ll.total_items += (U + gpw - 1) / gpw;
    }
};

#define glue(c, kern, ...) glue_named(c, kern, #kern, __VA_ARGS__)
const Operand NONE = {nullptr, nullptr, 0, 0, 0};
constexpr int GPW32 = 32 / TPI_1024, GPW64 = 32 / TPI_2048, GPWI128 = 32 / TPI_4096;

template <typename Kern> int glue_named(tecdsa_ctx* c, Kern kern, const char* name, const Arena& A, int per_unit = 1) {
    int grid = (A.U * per_unit + 63) / 64;
    c->prof_begin(name);
    kern<<<grid, 64, 0, c->stream>>>(A);
    c->prof_end();
    c->count_launch();
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : tecdsa_fail(TECDSA_E_CUDA, "glue launch", e);
}

int glue_crt(tecdsa_ctx* c, const Arena& A, int first, int count) {
    c->prof_begin("gg20_crt");
    gg20_crt<<<(A.U + 63) / 64, 64, 0, c->stream>>>(A, first, count);
    c->prof_end();
    c->count_launch();
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : tecdsa_fail(TECDSA_E_CUDA, "crt launch", e);
}

}  // namespace

// ------------------------------------------------------------------------------------------ fixed-base point tables
int tecdsa_internal_fb_points_init(int device, cudaStream_t stream, const uint32_t** table_out) {
    static uint32_t* tables[64] = {};
    if (device < 0 || device >= 64) return tecdsa_fail(TECDSA_E_ARG, "fb_points: bad device");
    if (!tables[device]) {
        uint32_t* t = nullptr;
        CK(cudaMalloc(&t, (size_t)2 * secp::FBP_WINDOWS * secp::FBP_DIGITS * 16 * 4));
        secp::fb_points_build<<<(2 * secp::FBP_WINDOWS + 31) / 32, 32, 0, stream>>>(t);
        CK(cudaGetLastError());
        CK(cudaStreamSynchronize(stream));
        tables[device] = t;
    }
    const uint32_t* p = tables[device];
    CK(cudaMemcpyToSymbol(secp::g_fb_points, &p, sizeof(p)));
    *table_out = p;
    return 0;
}

// ------------------------------------------------------------------------------------------ keys
extern "C" int tecdsa_keys_upload(tecdsa_ctx* c, const tecdsa_keys* k, tecdsa_keyset** out) {
    if (!c || !k || !out) return tecdsa_fail(TECDSA_E_ARG, "keys_upload: null argument");
    if (k->n_keysets == 0 || !k->paillier_p || !k->paillier_q || !k->n_tilde || !k->h1 || !k->h2 || !k->x_i || !k->pk || !k->y)
        return tecdsa_fail(TECDSA_E_ARG, "keys_upload: missing table");
    CK(cudaSetDevice(c->device));
    const int rows = (int)k->n_keysets * 3;
    // every modulus must be odd (Montgomery domain): checked on the host copy BEFORE anything is allocated or launched
    for (int r = 0; r < rows; r++)
        if (!(k->paillier_p[(size_t)r * 32] & 1) || !(k->paillier_q[(size_t)r * 32] & 1) || !(k->n_tilde[(size_t)r * 64] & 1))
            return tecdsa_fail(TECDSA_E_ARG, "keys_upload: even modulus");
    tecdsa_keyset* ks = new tecdsa_keyset();
    ks->n_keysets = (int)k->n_keysets;
    // from here on every failure releases the partially built key set
#undef CK
#define CK(call)                                                                                             \
    do {                                                                                                     \
        cudaError_t _e = (call);                                                                             \
        if (_e != cudaSuccess) { int _rc = tecdsa_fail(TECDSA_E_CUDA, #call, _e); tecdsa_keys_free(c, ks); return _rc; } \
    } while (0)
    size_t total = 0;
    size_t offs[KT_COUNT];
    for (int t = 0; t < KT_COUNT; t++) { offs[t] = total; total += (size_t)rows * KEY_SIZE[t]; total = (total + 63) & ~size_t(63); }
    size_t y_off = total; total += (size_t)k->n_keysets * 16;
    total = (total + 63) & ~size_t(63);
    size_t ptr_off = total;
    CK(cudaMalloc(&ks->mem, total * 4 + KT_COUNT * sizeof(uint32_t*)));
    CK(cudaMemsetAsync(ks->mem, 0, total * 4, c->stream));
    for (int t = 0; t < KT_COUNT; t++) ks->tab[t] = ks->mem + offs[t];
    ks->ypk = ks->mem + y_off;
    struct { int t; const uint32_t* src; } in[] = {{KT_P, k->paillier_p}, {KT_Q, k->paillier_q}, {KT_NT, k->n_tilde}, {KT_H1, k->h1},
                                                   {KT_H2, k->h2}, {KT_XI, k->x_i}, {KT_PK, k->pk}};
    for (auto& i : in) CK(cudaMemcpyAsync(ks->tab[i.t], i.src, (size_t)rows * KEY_SIZE[i.t] * 4, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(ks->ypk, k->y, (size_t)k->n_keysets * 16 * 4, cudaMemcpyHostToDevice, c->stream));
    uint32_t** d_ptrs = reinterpret_cast<uint32_t**>(ks->mem + ptr_off);
    CK(cudaMemcpyAsync(d_ptrs, ks->tab, sizeof(ks->tab), cudaMemcpyHostToDevice, c->stream));
    gg20_key_setup<<<(rows + 31) / 32, 32, 0, c->stream>>>(d_ptrs, rows);
    c->count_launch();
    CK(cudaGetLastError());
    {   // fixed-base tables for (h1, h2) mod N_tilde of every key row
        const size_t fb_limbs = (size_t)rows * 2 * FB_WINDOWS * FB_TBL * 64;
        CK(cudaMalloc(&ks->fb, fb_limbs * 4));
        const int per_block = 128 / TPI_2048;
        fb_chain_kernel<64, TPI_2048><<<(rows * 2 + per_block - 1) / per_block, 128, 0, c->stream>>>(ks->tab[KT_NT], ks->tab[KT_H1], ks->tab[KT_H2], ks->fb, rows);
        c->count_launch();
        CK(cudaGetLastError());
        fb_fill_kernel<64, TPI_2048><<<(rows * 2 * FB_WINDOWS + per_block - 1) / per_block, 128, 0, c->stream>>>(ks->tab[KT_NT], ks->fb, rows);
        c->count_launch();
        CK(cudaGetLastError());
    }
    {   // N-adic constants of every Paillier modulus (KT_N was derived by gg20_key_setup above)
        CK(cudaMalloc(&ks->nadic, (size_t)rows * NADIC_ROW * 64 * 4));
        CK(cudaMalloc(&ks->nadic_p, (size_t)rows * NADIC_ROW * 32 * 4));
        CK(cudaMalloc(&ks->nadic_q, (size_t)rows * NADIC_ROW * 32 * 4));
        int rc = c->nadic_setup(ks->tab[KT_N], ks->nadic, rows, 64);
        if (!rc) rc = c->nadic_setup(ks->tab[KT_P], ks->nadic_p, rows, 32);
        if (!rc) rc = c->nadic_setup(ks->tab[KT_Q], ks->nadic_q, rows, 32);
        if (rc) { tecdsa_keys_free(c, ks); return rc; }
    }
    CK(cudaStreamSynchronize(c->stream));
#undef CK
#define CK(call)                                                               \
    do {                                                                       \
        cudaError_t _e = (call);                                               \
        if (_e != cudaSuccess) return tecdsa_fail(TECDSA_E_CUDA, #call, _e);   \
    } while (0)
    *out = ks;
    return 0;
}
extern "C" int tecdsa_keys_free(tecdsa_ctx* c, tecdsa_keyset* ks) {
    if (!ks) return 0;
    if (c) { cudaSetDevice(c->device); cudaStreamSynchronize(c->stream); }
    if (ks->mem) cudaFree(ks->mem);
    if (ks->fb) cudaFree(ks->fb);
    if (ks->nadic) cudaFree(ks->nadic);
    if (ks->nadic_p) cudaFree(ks->nadic_p);
    if (ks->nadic_q) cudaFree(ks->nadic_q);
    delete ks;
    return 0;
}
extern "C" int tecdsa_keys_table(tecdsa_ctx* c, const tecdsa_keyset* ks, int table, uint32_t* out_host) {
    if (!c || !ks || !out_host || table < 0 || table >= KT_COUNT) return tecdsa_fail(TECDSA_E_ARG, "keys_table: bad argument");
    CK(cudaMemcpyAsync(out_host, ks->tab[table], (size_t)ks->n_keysets * 3 * KEY_SIZE[table] * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// ------------------------------------------------------------------------------------------ job launches
static int run_exp(tecdsa_ctx* c, ExpLaunch& l, int K) {
    if (l.n_classes == 0) return 0;
    int rc = K == 128 ? c->launch_nadic(l, 64) : K == -32 ? c->launch_nadic(l, 32) : c->launch_exp(l, K);   // 128: N-adic mod N^2, -32: p-adic
    l.n_classes = 0; l.total_items = 0;
    return rc;
}
static int run_inv(tecdsa_ctx* c, InvLaunch& l, int K) {
    if (l.n_classes == 0) return 0;
    int rc = K == -128 ? c->launch_nadic_inv(l) : c->launch_inv(l, K);
    l.n_classes = 0; l.total_items = 0;
    return rc;
}

// ------------------------------------------------------------------------------------------ offline stage
// `h_sess` is always a HOST copy of the session descriptors; `mem` says where rnd and the outputs live
static int offline_impl(tecdsa_ctx* c, const tecdsa_keyset* ks, const uint32_t* h_sess, size_t n_sessions,
                        const uint32_t* rnd, uint8_t* status, uint32_t* R_out, uint32_t* sigma_out,
                        uint32_t* tvec_out, uint32_t* digest_out, int mem) {
    CK(cudaSetDevice(c->device));
    const int U = (int)n_sessions * 2;

    // ---- host-side unit tables (who am I, who is my peer, which key rows), then the units ordered by own and by peer key row,
    // each row's run padded to whole warps of every job kernel (groups per warp are powers of two: the largest covers all)
    const uint32_t nrows = (uint32_t)ks->n_keysets * 3;
    const size_t pad = (size_t)std::max({32 / tecdsa_nadic_tpi(), 32 / tecdsa_nadic32_tpi(), GPW32});
    const size_t order_cap = (size_t)U + std::min((size_t)nrows, (size_t)U) * (pad - 1);
    std::vector<uint32_t> idx((size_t)7 * U + 2 * order_cap);
    uint32_t *row_own = idx.data(), *row_peer = row_own + U, *row_st = row_peer + U, *peer = row_st + 3 * (size_t)U, *kset = peer + U;
    for (size_t s = 0; s < n_sessions; s++) {
        uint32_t k = h_sess[3 * s], a = h_sess[3 * s + 1], b = h_sess[3 * s + 2];
        if (k >= (uint32_t)ks->n_keysets || a > 2 || b > 2 || a == b) return tecdsa_fail(TECDSA_E_ARG, "gg20_offline: bad session descriptor");
        for (int p = 0; p < 2; p++) {
            size_t u = 2 * s + p;
            row_own[u] = k * 3 + (p ? b : a); row_peer[u] = k * 3 + (p ? a : b);
            for (int x = 0; x < 3; x++) row_st[(size_t)x * U + u] = k * 3 + x;
            peer[u] = (uint32_t)(u ^ 1); kset[u] = k;
        }
    }
    size_t order_len[2];
    {
        std::vector<uint32_t> scratch(nrows);
        for (int r = 0; r < 2; r++)
            order_len[r] = keyexp_order(r ? row_peer : row_own, (size_t)U, nrows, pad, scratch.data(), kset + U + (size_t)r * order_cap);
    }
    // ---- arena
    Builder B;
    B.c = c; B.ks = ks; B.U = U;
    Arena& A = B.A;
    size_t limbs = 0;
    for (int f = 0; f < F_COUNT; f++) { A.off[f] = (uint32_t)limbs; A.size[f] = (uint16_t)FIELD_SIZE[f]; limbs += FIELD_SIZE[f]; }
    const size_t arena_bytes = limbs * 4 * (size_t)U;
    const size_t idx_bytes = idx.size() * 4;
    int rc = c->reserve_arena(arena_bytes + idx_bytes + 4096 + (size_t)U);
    if (rc) return rc;
    A.base = reinterpret_cast<uint32_t*>(c->arena);
    A.U = U;
    uint32_t* d_idx = reinterpret_cast<uint32_t*>(c->arena + ((arena_bytes + 255) & ~size_t(255)));
    A.row_own = d_idx; A.row_peer = d_idx + U; A.row_st = d_idx + 2 * (size_t)U; A.peer = d_idx + 5 * (size_t)U; A.keyset = d_idx + 6 * (size_t)U;
    for (int r = 0; r < 2; r++) { B.order[r] = d_idx + 7 * (size_t)U + (size_t)r * order_cap; B.order_len[r] = (int)order_len[r]; }
    A.status = reinterpret_cast<uint8_t*>(d_idx + idx.size());
    for (int t = 0; t < KT_COUNT; t++) A.key[t] = ks->tab[t];
    A.ypk = ks->ypk;
    CK(cudaMemcpyAsync(d_idx, idx.data(), idx_bytes, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(A.status, 0, U, c->stream));
    CK(cudaMemsetAsync(B.out(F_FLAGS), 0, (size_t)U * A.size[F_FLAGS] * 4, c->stream));
    CK(cudaMemcpyAsync(B.out(F_RND), rnd, (size_t)U * RND_LIMBS * 4,
                       mem == TECDSA_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, c->stream));
    const int launches0 = (int)c->launches;
    CK(cudaEventRecord(c->ev0, c->stream));

    ExpLaunch &L32 = B.L32, &L64 = B.L64, &L128 = B.L128;
    InvLaunch &I64 = B.I64, &I128 = B.I128;
    Builder::reset(L32); Builder::reset(L64); Builder::reset(L128); Builder::reset(B.LPQ); Builder::reset(I64); Builder::reset(I128); Builder::reset(B.I128H);
    const int GPW128 = 0;        // classes modulo N^2 are routed (and sized) by Builder::exp_class
    const uint32_t *ro = A.row_own, *rp = A.row_peer;
    auto st_rows = [&](int x) { return A.row_st + (size_t)x * U; };
#define RUN(x) do { int _rc = (x); if (_rc) return _rc; } while (0)

    // ================= Round 0 (rounds.rs:68-104): MessageA::a with one AliceProof per statement
    RUN(glue(c, gg20_r0_pre, A));
    // c_k = (1 + k N) * r_k^N mod N^2 (mta/mod.rs:68-75) and u = (alpha N + 1) * beta^N mod N^2 (range_proofs.rs:53-55):
    // the N-th powers are under the unit's OWN key, so they run as CRT halves mod p^2 / q^2 (2048-bit)
    B.crt_stage1(L32, GPW32, ro, 0, B.rnd(RND_RK, 64));
    for (int x = 0; x < 3; x++) B.crt_stage1(L32, GPW32, ro, 1 + x, B.rnd(RND_AL + x * RND_AL_STRIDE + RND_AL_BETA, 64));
    RUN(run_exp(c, L32, 32));
    B.crt_stage2(L64, GPW64, ro, 0);
    for (int x = 0; x < 3; x++) {
        const int al = RND_AL + x * RND_AL_STRIDE;
        B.crt_stage2(L64, GPW64, ro, 1 + x);
        // w = h1^alpha * h2^gamma mod N_tilde                           (range_proofs.rs:56-57)
        B.fb_class(L64, GPW64, st_rows(x), B.rnd(al + RND_AL_GAMMA, 88), 88, B.rnd(al + RND_AL_ALPHA, 24), 24, 0, NONE, F_WP0 + x);
        // z = h1^a * h2^ro mod N_tilde                                  (range_proofs.rs:52)
        B.fb_class(L64, GPW64, st_rows(x), B.rnd(al + RND_AL_RHO, 72), 72, B.rnd(RND_K, 8), 8, 0, NONE, F_Z0 + x);
    }
    RUN(run_exp(c, B.LPQ, -32)); RUN(run_exp(c, L64, 64));
    RUN(glue_crt(c, A, 0, 4));
    B.exp_class(L128, GPW128, B.key(KT_NN, ro), 0, NONE, NONE, 0, NONE, NONE, 0, 2, B.fld(F_MK), B.fld(F_XC0), F_CK);
    for (int x = 0; x < 3; x++)
        B.exp_class(L128, GPW128, B.key(KT_NN, ro), 0, NONE, NONE, 0, NONE, NONE, 0, 2, B.fld(F_ALIN0 + x), B.fld(F_XC1 + x), F_U0 + x);
    RUN(run_exp(c, L128, 128));
    RUN(glue(c, gg20_r0_mid, A));
    for (int x = 0; x < 3; x++)    // s = r^e * beta mod N                (range_proofs.rs:86)
        B.exp_class(L64, GPW64, B.key(KT_N, ro), 1, B.rnd(RND_RK, 64), B.fld(F_E0 + x), 8, NONE, NONE, 0, 1,
                    B.rnd(RND_AL + x * RND_AL_STRIDE + RND_AL_BETA, 64), NONE, F_S0 + x);
    RUN(run_exp(c, B.LPQ, -32)); RUN(run_exp(c, L64, 64));

    // ================= Round 1 (rounds.rs:122-206): 2 x MessageB::b — the three AliceProof::verify
    // of the peer's MessageA are computed ONCE and used for both calls (declared de-duplication).
    RUN(glue(c, gg20_r1_pre, A));
    // (c^e)^-1 mod N^2 is evaluated as (c^-1)^e (the reference does the same in commitment_unknown_order,
    // zk_pdl_with_slack/mod.rs:191-193): ONE inversion of the peer's ciphertext serves the three proofs here and the
    // peer's PDL proof in round 5 (declared shortcut, identical value)
    B.inv_class(I128, GPWI128, B.key(KT_NN, rp), B.peer(F_CK), F_CINVP, 3);
    RUN(run_inv(c, I128, 128)); RUN(run_inv(c, B.I128H, -128));
    for (int x = 0; x < 3; x++)
        B.exp_class(L64, GPW64, B.key(KT_NT, st_rows(x)), 1, B.peer(F_Z0 + x), B.peer(F_E0 + x), 8, NONE, NONE, 0, 0, NONE, NONE, F_ZE0 + x);   // z^e (:122)
    RUN(run_exp(c, L64, 64));
    for (int x = 0; x < 3; x++) B.inv_class(I64, GPW64, B.key(KT_NT, st_rows(x)), B.fld(F_ZE0 + x), F_ZEI0 + x, x);
    RUN(run_inv(c, I64, 64));
    for (int x = 0; x < 3; x++) {
        // w' = h1^s1 * h2^s2 * (z^e)^-1 mod N_tilde                     (range_proofs.rs:129-132)
        B.fb_class(L64, GPW64, st_rows(x), B.peer(F_S20 + x), 92, B.peer(F_S10 + x), 28, 1, B.fld(F_ZEI0 + x), F_WV0 + x);
        // u' = (s1 N + 1) * s^N * (c^e)^-1 mod N^2                      (range_proofs.rs:134-141)
        // (c^-1)^e (:135) is the second base of the same product: its 256-bit exponent shares the squarings of s^N
        B.exp_class(L128, GPW128, B.key(KT_NN, rp), 2, B.peer(F_S0 + x, 64), B.key(KT_N, rp), 64, B.fld(F_CINVP), B.peer(F_E0 + x), 8, 1,
                    B.fld(F_GS10 + x), NONE, F_UV0 + x);
    }
    // c_b = c_a^b * Enc(beta'; r') mod N^2 for b = gamma_i and b = w_i  (mta/mod.rs:133-145)
    B.exp_class(L128, GPW128, B.key(KT_NN, rp), 2, B.rnd(RND_R_G, 64), B.key(KT_N, rp), 64, B.peer(F_CK), B.rnd(RND_GAMMA, 8), 8, 1, B.fld(F_LBG), NONE, F_CBG);
    B.exp_class(L128, GPW128, B.key(KT_NN, rp), 2, B.rnd(RND_R_W, 64), B.key(KT_N, rp), 64, B.peer(F_CK), B.fld(F_W), 8, 1, B.fld(F_LBW), NONE, F_CBW);
    RUN(run_exp(c, L128, 128)); RUN(run_exp(c, B.LPQ, -32)); RUN(run_exp(c, L64, 64));
    RUN(glue(c, gg20_r1_post_hash, A, 3));
    RUN(glue(c, gg20_r1_post_dlog, A, 4));

    // ================= Round 2 (rounds.rs:234-317): Paillier decrypt of the peer's two MessageB
    B.exp_class(L64, GPW64, B.key(KT_PP, ro), 1, B.peer(F_CBG), B.key(KT_PM1, ro), 32, NONE, NONE, 0, 0, NONE, NONE, F_DPG, 1);
    B.exp_class(L64, GPW64, B.key(KT_QQ, ro), 1, B.peer(F_CBG), B.key(KT_QM1, ro), 32, NONE, NONE, 0, 0, NONE, NONE, F_DQG, 1);
    B.exp_class(L64, GPW64, B.key(KT_PP, ro), 1, B.peer(F_CBW), B.key(KT_PM1, ro), 32, NONE, NONE, 0, 0, NONE, NONE, F_DPW, 1);
    B.exp_class(L64, GPW64, B.key(KT_QQ, ro), 1, B.peer(F_CBW), B.key(KT_QM1, ro), 32, NONE, NONE, 0, 0, NONE, NONE, F_DQW, 1);
    RUN(run_exp(c, B.LPQ, -32)); RUN(run_exp(c, L64, 64));
    RUN(glue(c, gg20_r2_check, A, 7));
    RUN(glue(c, gg20_r2_finish, A));
    // ================= Round 3 (rounds.rs:347-402)
    RUN(glue(c, gg20_r3_check, A, 2));
    RUN(glue(c, gg20_r3_finish, A));
    // ================= Round 4 (rounds.rs:431-498): R, R_dash, PDLwSlackProof::prove against the peer's statement
    RUN(glue(c, gg20_r4_pre, A));
    B.fb_class(L64, GPW64, rp, B.rnd(RND_PDL_RHO, 72), 72, B.rnd(RND_K, 8), 8, 0, NONE, F_PZ);                  // z  (:78-84)
    B.fb_class(L64, GPW64, rp, B.rnd(RND_PDL_GAMMA, 88), 88, B.rnd(RND_PDL_ALPHA, 24), 24, 0, NONE, F_PU3);     // u3 (:93-99)
    // u2 = (N+1)^alpha * beta^N mod N^2, with (N+1)^alpha == 1 + alpha N (declared shortcut, identical value) (:86-92);
    // beta^N under the own key through CRT halves
    B.crt_stage1(L32, GPW32, ro, 4, B.rnd(RND_PDL_BETA, 64));
    RUN(run_exp(c, L32, 32));
    B.crt_stage2(L64, GPW64, ro, 4);
    RUN(run_exp(c, B.LPQ, -32)); RUN(run_exp(c, L64, 64));
    RUN(glue_crt(c, A, 4, 1));
    B.exp_class(L128, GPW128, B.key(KT_NN, ro), 0, NONE, NONE, 0, NONE, NONE, 0, 2, B.fld(F_PLIN), B.fld(F_XC4), F_PU2);
    RUN(run_exp(c, L128, 128));
    RUN(glue(c, gg20_r4_mid, A));
    B.exp_class(L64, GPW64, B.key(KT_N, ro), 1, B.rnd(RND_RK, 64), B.fld(F_PE), 8, NONE, NONE, 0, 1, B.rnd(RND_PDL_BETA, 64), NONE, F_PS2);   // s2 = r^e * beta mod N (:113)
    RUN(run_exp(c, B.LPQ, -32)); RUN(run_exp(c, L64, 64));

    // ================= Round 5 (rounds.rs:525-592): verify both signers' PDL proofs (own one included)
    RUN(glue(c, gg20_r5_pre, A));
    B.inv_class(I128, GPWI128, B.key(KT_NN, ro), B.fld(F_CK), F_CINVO, 8);          // own ciphertext (proof j = 0); the peer's inverse is CINVP
    RUN(run_inv(c, I128, 128)); RUN(run_inv(c, B.I128H, -128));
    for (int j = 0; j < 2; j++) {
        const uint32_t* stmt = j ? ro : rp;              // whose (N_tilde, h1, h2) the proof was made against
        Operand z = j ? B.peer(F_PZ) : B.fld(F_PZ);
        B.exp_class(L64, GPW64, B.key(KT_NT, stmt), 1, z, B.fld(F_VE0 + j), 8, NONE, NONE, 0, 0, NONE, NONE, F_VZE0 + j);       // z^e; (z^-1)^e == (z^e)^-1 (:166-172)
    }
    B.crt_stage1(L32, GPW32, ro, 5, B.fld(F_PS2, 64));       // own proof's s2^N mod N^2_own through the CRT stages
    RUN(run_exp(c, L32, 32));
    B.crt_stage2(L64, GPW64, ro, 5);
    RUN(run_exp(c, B.LPQ, -32)); RUN(run_exp(c, L64, 64));
    RUN(glue_crt(c, A, 5, 1));
    for (int j = 0; j < 2; j++) B.inv_class(I64, GPW64, B.key(KT_NT, j ? ro : rp), B.fld(F_VZE0 + j), F_VZEI0 + j, 6 + j);
    RUN(run_inv(c, I64, 64));
    for (int j = 0; j < 2; j++) {
        const uint32_t* prover = j ? rp : ro;
        const uint32_t* stmt = j ? ro : rp;
        Operand s1 = j ? B.peer(F_PS1) : B.fld(F_PS1), s2 = j ? B.peer(F_PS2, 64) : B.fld(F_PS2, 64), s3 = j ? B.peer(F_PS3) : B.fld(F_PS3);
        // u3' = h1^s1 * h2^s3 * z^-e mod N_tilde                         (:158-172)
        B.fb_class(L64, GPW64, stmt, s3, 92, s1, 28, 1, B.fld(F_VZEI0 + j), F_VU30 + j);
        // u2' = (N+1)^s1 * s2^N * c^-e mod N^2                           (:144-157); (c^-1)^e (:151-157) is a base of the same
        // product.  The own proof's s2^N came through the CRT stages (XC5); the peer's shares its squarings with (c^-1)^e.
        if (j == 0) B.exp_class(L128, GPW128, B.key(KT_NN, prover), 1, B.fld(F_CINVO), B.fld(F_VE0), 8, NONE, NONE, 0, 2, B.fld(F_VLIN0), B.fld(F_XC5), F_VU20);
        else B.exp_class(L128, GPW128, B.key(KT_NN, prover), 2, s2, B.key(KT_N, prover), 64, B.fld(F_CINVP), B.fld(F_VE1), 8, 1, B.fld(F_VLIN1), NONE, F_VU21);
    }
    RUN(run_exp(c, L128, 128)); RUN(run_exp(c, B.LPQ, -32)); RUN(run_exp(c, L64, 64));
    RUN(glue(c, gg20_r5_check, A, 2));
    RUN(glue(c, gg20_r5_finish, A));
    // ================= Round 6 (rounds.rs:612-636) + result records
    RUN(glue(c, gg20_r6_check, A, 2));
    RUN(glue(c, gg20_r6, A));
#undef RUN
    CK(cudaEventRecord(c->ev1, c->stream));
    c->last_launches = (int)c->launches - launches0;

    // ---- outputs
    const cudaMemcpyKind kind = mem == TECDSA_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    CK(cudaMemcpyAsync(status, A.status, U, kind, c->stream));
    if (R_out) CK(cudaMemcpyAsync(R_out, B.out(F_R), (size_t)U * 16 * 4, kind, c->stream));
    if (sigma_out) CK(cudaMemcpyAsync(sigma_out, B.out(F_SIGMA), (size_t)U * 8 * 4, kind, c->stream));
    if (digest_out) CK(cudaMemcpyAsync(digest_out, B.out(F_DIGEST), (size_t)U * 8 * 4, kind, c->stream));
    if (tvec_out) {
        // t_vec[u] = (T of signer position 0, T of signer position 1) of the session
        CK(cudaMemcpy2DAsync(tvec_out, 64 * 4, B.out(F_T), 32 * 4, 32 * 4, n_sessions, kind, c->stream));        // even units
        CK(cudaMemcpy2DAsync(tvec_out + 32, 64 * 4, B.out(F_T), 32 * 4, 32 * 4, n_sessions, kind, c->stream));   // odd units
    }
    c->last_U = U;
    memcpy(c->last_off, A.off, sizeof(A.off));
    if (mem == TECDSA_HOST) CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// Batches of at least SPLIT_MIN sessions run as two half-batches on two private streams, driven by two host threads: units
// are independent, so the results are those of the single-stream run, while the tail of each persistent job-list launch
// and the latency-bound glue kernels of one half overlap the job lists of the other.  TECDSA_SPLIT=0 turns it off.
static size_t split_min_sessions() {
    static const size_t v = [] {
        const char* e = getenv("TECDSA_SPLIT");
        return (e && atoi(e) == 0) ? (size_t)-1 : (size_t)2048;
    }();
    return v;
}
extern "C" int tecdsa_gg20_offline_batch(tecdsa_ctx* c, const tecdsa_keyset* ks, const uint32_t* sessions, size_t n_sessions,
                                         const uint32_t* rnd, uint8_t* status, uint32_t* R_out, uint32_t* sigma_out,
                                         uint32_t* tvec_out, uint32_t* digest_out, int mem) {
    if (!c || !ks || !sessions || !rnd || !status) return tecdsa_fail(TECDSA_E_ARG, "gg20_offline: null argument");
    if (mem != TECDSA_HOST && mem != TECDSA_DEVICE) return tecdsa_fail(TECDSA_E_ARG, "gg20_offline: bad mem");
    if (n_sessions == 0) return 0;
    if (n_sessions > (1u << 22)) return tecdsa_fail(TECDSA_E_ARG, "gg20_offline: too many sessions");
    CK(cudaSetDevice(c->device));
    std::vector<uint32_t> h_copy;
    if (mem == TECDSA_DEVICE) {                     // the host builds the per-unit index tables from the descriptors
        h_copy.resize(n_sessions * 3);
        CK(cudaMemcpyAsync(h_copy.data(), sessions, h_copy.size() * 4, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
        sessions = h_copy.data();
    }
    return tecdsa_internal_offline(c, ks, sessions, n_sessions, rnd, status, R_out, sigma_out, tvec_out, digest_out, mem);
}

int tecdsa_internal_offline(tecdsa_ctx* c, const tecdsa_keyset* ks, const uint32_t* sessions, size_t n_sessions,
                            const uint32_t* rnd, uint8_t* status, uint32_t* R_out, uint32_t* sigma_out,
                            uint32_t* tvec_out, uint32_t* digest_out, int mem) {
    if (n_sessions < split_min_sessions() || c->profiling) return offline_impl(c, ks, sessions, n_sessions, rnd, status, R_out, sigma_out, tvec_out, digest_out, mem);

    for (int h = 0; h < 2; h++) {
        if (c->child[h]) continue;
        cudaStream_t s = nullptr;
        cudaEvent_t ev = nullptr;
        CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));           // the join event exists before the child context is published
        cudaError_t se = cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        if (se != cudaSuccess) { cudaEventDestroy(ev); return tecdsa_fail(TECDSA_E_CUDA, "gg20_offline: stream for a half-batch", se); }
        tecdsa_ctx* child = nullptr;
        int rc = tecdsa_ctx_create(&child, c->device, s);
        if (rc) { cudaStreamDestroy(s); cudaEventDestroy(ev); return rc; }
        child->owns_stream = true;
        c->ev_join[h] = ev;
        c->child[h] = child;
    }
    if (!c->ev_fork) CK(cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming));
    // fork: both halves start after everything already queued on the caller's stream (device-resident inputs)
    CK(cudaEventRecord(c->ev0, c->stream));
    CK(cudaEventRecord(c->ev_fork, c->stream));
    const size_t n0 = n_sessions / 2;
    int rcs[2] = {0, 0};
    std::string errs[2];
    auto half = [&](int h) {
        tecdsa_ctx* cc = c->child[h];
        const size_t s0 = h ? n0 : 0, ns = h ? n_sessions - n0 : n0, u0 = 2 * s0;
        cudaSetDevice(cc->device);
        cudaError_t e = cudaStreamWaitEvent(cc->stream, c->ev_fork, 0);
        int rc = e == cudaSuccess ? 0 : tecdsa_fail(TECDSA_E_CUDA, "gg20_offline: fork", e);
        if (!rc) rc = offline_impl(cc, ks, sessions + 3 * s0, ns, rnd + u0 * RND_LIMBS, status + u0, R_out ? R_out + u0 * 16 : nullptr,
                                   sigma_out ? sigma_out + u0 * 8 : nullptr, tvec_out ? tvec_out + s0 * 64 : nullptr,
                                   digest_out ? digest_out + u0 * 8 : nullptr, mem);
        if (!rc) {
            e = cudaEventRecord(c->ev_join[h], cc->stream);
            if (e != cudaSuccess) rc = tecdsa_fail(TECDSA_E_CUDA, "gg20_offline: join", e);
        }
        rcs[h] = rc;
        if (rc) errs[h] = tecdsa_last_error();
    };
    const uint64_t l0 = c->child[0]->launches + c->child[1]->launches;
    bool threaded = true;
    std::thread other;
    try { other = std::thread(half, 1); } catch (...) { threaded = false; }      // no thread available: queue the halves one after the other
    half(0);
    if (threaded) other.join(); else half(1);
    for (int h = 0; h < 2; h++) {
        if (rcs[h]) { cudaDeviceSynchronize(); return tecdsa_fail(rcs[h], errs[h].c_str()); }
        CK(cudaStreamWaitEvent(c->stream, c->ev_join[h], 0));
    }
    CK(cudaEventRecord(c->ev1, c->stream));
    const uint64_t dl = c->child[0]->launches + c->child[1]->launches - l0;
    c->launches += dl;
    c->last_launches = (int)dl;
    c->last_U = 0;                                  // debug_field addresses one arena: not available for split batches
    if (mem == TECDSA_HOST) CK(cudaStreamSynchronize(c->stream));
    return 0;
}

// Debug / test access: copy one arena field of the last gg20_offline batch to the host.
extern "C" int tecdsa_gg20_debug_field(tecdsa_ctx* c, const char* name, uint32_t* out_host, size_t* limbs_per_unit) {
    if (!c || !name) return tecdsa_fail(TECDSA_E_ARG, "debug_field: null argument");
    if (c->last_U == 0) return tecdsa_fail(TECDSA_E_ARG, "debug_field: no batch has run");
    for (int f = 0; f < F_COUNT; f++) {
        if (strcmp(name, FIELD_NAME[f]) == 0) {
            if (limbs_per_unit) *limbs_per_unit = FIELD_SIZE[f];
            if (out_host) {
                CK(cudaMemcpyAsync(out_host, reinterpret_cast<uint32_t*>(c->arena) + (size_t)c->last_off[f] * c->last_U,
                                   (size_t)c->last_U * FIELD_SIZE[f] * 4, cudaMemcpyDeviceToHost, c->stream));
                CK(cudaStreamSynchronize(c->stream));
            }
            return 0;
        }
    }
    return tecdsa_fail(TECDSA_E_ARG, "debug_field: unknown field");
}
