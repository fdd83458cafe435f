// Shared host-side plumbing of the stand-alone batch entry points (l12.cu, keygen.cu, ecops.cu): stream-ordered staging of
// caller buffers and the job-class builders over the job-list kernels of jobs.cuh / nadic.cuh / modinv.cuh.
#pragma once
#include "ctx.h"
#include "gg20_glue.cuh"
#include "modinv.cuh"

#include <vector>

using namespace tecdsa;      // internal header, included by .cu files only
namespace {

// Stream-ordered staging of caller buffers: HOST pointers are copied to device scratch (and
// results copied back by finish()), DEVICE pointers are used in place.
struct Stage {
    tecdsa_ctx* c;
    int mem;
    struct Scratch { void* p; size_t bytes; };
    std::vector<Scratch> scratch;
    struct Back { void* host; void* dev; size_t bytes; };
    std::vector<Back> back;
    int err = 0;
    Stage(tecdsa_ctx* ctx, int m) : c(ctx), mem(m) {}
    void* alloc(size_t bytes) {
        void* p = nullptr;
        if (cudaMallocAsync(&p, bytes ? bytes : 16, c->stream) != cudaSuccess) { err = tecdsa_fail(TECDSA_E_NOMEM, "cudaMallocAsync"); return nullptr; }
        scratch.push_back({p, bytes ? bytes : 16});
        return p;
    }
    template <typename T> const T* in(const T* p, size_t n) {
        if (!p || mem == TECDSA_DEVICE) return p;
        T* d = static_cast<T*>(alloc(n * sizeof(T)));
        if (d && cudaMemcpyAsync(d, p, n * sizeof(T), cudaMemcpyHostToDevice, c->stream) != cudaSuccess) err = tecdsa_fail(TECDSA_E_CUDA, "H2D copy");
        return d;
    }
    template <typename T> T* out(T* p, size_t n) {
        if (!p || mem == TECDSA_DEVICE) return p;
        T* d = static_cast<T*>(alloc(n * sizeof(T)));
        if (d) back.push_back({p, d, n * sizeof(T)});
        return d;
    }
    template <typename T> T* tmp(size_t n) { return static_cast<T*>(alloc(n * sizeof(T))); }
    int finish() {
        for (auto& b : back)
            if (cudaMemcpyAsync(b.host, b.dev, b.bytes, cudaMemcpyDeviceToHost, c->stream) != cudaSuccess) err = tecdsa_fail(TECDSA_E_CUDA, "D2H copy");
        // staged inputs, intermediates and results can all hold secrets (nonces, shares, plaintexts): wipe before the memory goes
        // back to the stream-ordered pool, as the reference zeroizes its witnesses on drop (range_proofs.rs:26-27)
        for (const Scratch& b : scratch) { cudaMemsetAsync(b.p, 0, b.bytes, c->stream); cudaFreeAsync(b.p, c->stream); }
        scratch.clear();
        if (mem == TECDSA_HOST) {
            cudaError_t e = cudaStreamSynchronize(c->stream);
            if (e != cudaSuccess) err = tecdsa_fail(TECDSA_E_CUDA, "stream sync after batch", e);
        }
        return err;
    }
};

const Operand NONE = {nullptr, nullptr, 0, 0, 0};
Operand arr(const uint32_t* p, uint32_t limbs) { return Operand{p, nullptr, limbs, 0, limbs}; }
Operand tab(const uint32_t* p, const uint32_t* idx, uint32_t limbs) { return Operand{p, idx, limbs, 1, limbs}; }

struct Launches {
    ExpLaunch e64, e128;
    InvLaunch i64, i128;
    Launches() { e64.n_classes = e64.total_items = e128.n_classes = e128.total_items = 0; i64.n_classes = i64.total_items = i128.n_classes = i128.total_items = 0; }
};
void add_exp(ExpLaunch& l, int K, int count, Operand mod, int nb, Operand b0, Operand e0, int el0, Operand b1, Operand e1, int el1,
             int nm, Operand m0, Operand m1, uint32_t* out, uint32_t out_stride) {
    const int gpw = 32 / (K == 64 ? TPI_2048 : TPI_4096);
    ExpClass& k = l.cls[l.n_classes++];
    k.mod = mod; k.base[0] = b0; k.base[1] = b1; k.exp[0] = e0; k.exp[1] = e1; k.exp_limbs[0] = el0; k.exp_limbs[1] = el1;
    k.mul[0] = m0; k.mul[1] = m1; k.mul[2] = NONE; k.nbases = nb; k.nmul = nm; k.wide0 = 0;
    k.fb = nullptr; k.fb_row = NONE; k.fb_sel[0] = k.fb_sel[1] = 0; k.nadic = NONE; k.order = nullptr; k.keyexp = 0;
    k.out = out; k.out_stride = out_stride; k.count = count; k.item_begin = l.total_items;
    l.total_items += (count + gpw - 1) / gpw;
}
// class modulo N^2 through the N-adic kernel (nadic.cuh): `N` names the K = 64 limb modulus, `consts` its constants row
void add_nn(ExpLaunch& l, int count, Operand N, Operand consts, int nb, Operand b0, Operand e0, int el0, Operand b1, Operand e1, int el1,
            int nm, Operand m0, Operand m1, uint32_t* out, uint32_t out_stride) {
    add_exp(l, 128, count, N, nb, b0, e0, el0, b1, e1, el1, nm, m0, m1, out, out_stride);
    ExpClass& k = l.cls[l.n_classes - 1];
    const int gpw = N.limbs == 32 ? 32 / tecdsa_nadic32_tpi() : 32 / tecdsa_nadic_tpi();
    k.nadic = consts;
    l.total_items = k.item_begin + (count + gpw - 1) / gpw;
}
Operand key_n(const tecdsa_keyset* ks, const uint32_t* rows) { return tab(ks->tab[KT_N], rows, 64); }
Operand key_nadic(const tecdsa_keyset* ks, const uint32_t* rows) { return tab(ks->nadic, rows, NADIC_ROW * 64); }
void add_fb(ExpLaunch& l, int count, const tecdsa_keyset* ks, const uint32_t* rows, Operand e_h2, int el_h2, Operand e_h1, int el_h1,
            int nm, Operand m0, uint32_t* out) {
    add_exp(l, 64, count, tab(ks->tab[KT_NT], rows, 64), 2, NONE, e_h2, el_h2, NONE, e_h1, el_h1, nm, m0, NONE, out, 64);
    ExpClass& k = l.cls[l.n_classes - 1];
    k.fb = ks->fb; k.fb_row = Operand{nullptr, rows, 0, 1, 0}; k.fb_sel[0] = 1; k.fb_sel[1] = 0;
}
void add_inv(InvLaunch& l, int K, int count, Operand mod, Operand in, uint32_t* out, uint8_t* ok) {
    const int gpw = 32 / (K == 64 ? TPI_2048 : TPI_4096);
    InvClass& k = l.cls[l.n_classes++];
    k.mod = mod; k.in = in; k.out = out; k.out_stride = K; k.ok = ok; k.ok_stride = 1; k.nadic = NONE; k.count = count; k.item_begin = l.total_items;
    l.total_items += (count + gpw - 1) / gpw;
}
int run(tecdsa_ctx* c, ExpLaunch& l, int K) {
    if (!l.n_classes) return 0;
    int rc = c->launch_exp(l, K);
    l.n_classes = l.total_items = 0;
    return rc;
}
int run_nn(tecdsa_ctx* c, ExpLaunch& l, int K = 64) {
    if (!l.n_classes) return 0;
    int rc = c->launch_nadic(l, K);
    l.n_classes = l.total_items = 0;
    return rc;
}
int run(tecdsa_ctx* c, InvLaunch& l, int K) {
    if (!l.n_classes) return 0;
    int rc = c->launch_inv(l, K);
    l.n_classes = l.total_items = 0;
    return rc;
}
int check_bits(int mod_bits) { return (mod_bits == 2048 || mod_bits == 4096) ? 0 : tecdsa_fail(TECDSA_E_UNSUPPORTED, "mod_bits must be 2048 or 4096"); }

inline Arena key_arena(const tecdsa_keyset* ks) {
    Arena A;
    memset(&A, 0, sizeof(A));
    for (int t = 0; t < KT_COUNT; t++) A.key[t] = ks->tab[t];
    A.ypk = ks->ypk;
    return A;
}
inline int grid_for(size_t count) { return (int)((count + 63) / 64); }

}  // namespace

#define RUN(x) do { int _rc = (x); if (_rc) { S.finish(); return _rc; } } while (0)
#define KCHECK() do { c->count_launch(); cudaError_t _e = cudaGetLastError(); if (_e != cudaSuccess) { S.finish(); return tecdsa_fail(TECDSA_E_CUDA, "kernel launch", _e); } } while (0)
#define SIMPLE_PROLOGUE(name)                                                        \
    if (!c) return tecdsa_fail(TECDSA_E_ARG, name ": null ctx");                     \
    if (count == 0) return 0;                                                        \
    CK(cudaSetDevice(c->device));                                                    \
    const int n = (int)count;                                                        \
    Stage S(c, mem);
