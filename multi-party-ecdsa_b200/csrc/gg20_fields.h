// Per-unit arena layout of the batched GG20 offline stage (t = 1, two signers per session).
// One "unit" = one party's OfflineStage Round0..Round6
// (/root/reference/src/protocols/multi_party_ecdsa/gg_2020/state_machine/sign/rounds.rs:68-636).
// Field f of unit u lives at arena + off[f]*U + u*size[f] (limbs): every field is an
// operand-major array over the units, so the job-list kernels read it with coalesced
// 16-byte loads.  All sizes are multiples of 4 limbs.
#pragma once
#include <cstdint>

namespace tecdsa {

// ---- randomness record (input; see include/tecdsa_b200.h TECDSA_RND_*) ------------------
enum : int {
    RND_GAMMA = 0, RND_K = 8, RND_BLIND = 16, RND_RK = 24,
    RND_AL = 88,             // 3 x { alpha 24, beta 64, gamma 88, rho 72 }
    RND_AL_STRIDE = 248, RND_AL_ALPHA = 0, RND_AL_BETA = 24, RND_AL_GAMMA = 88, RND_AL_RHO = 176,
    RND_BT_G = 832, RND_R_G = 896, RND_NB_G = 960, RND_NBT_G = 968,
    RND_BT_W = 976, RND_R_W = 1040, RND_NB_W = 1104, RND_NBT_W = 1112,
    RND_L = 1120, RND_PED_S1 = 1128, RND_PED_S2 = 1136,
    RND_PDL_ALPHA = 1144, RND_PDL_BETA = 1168, RND_PDL_RHO = 1232, RND_PDL_GAMMA = 1304,
    RND_HEG_S1 = 1392, RND_HEG_S2 = 1400,
    RND_LIMBS = 1408
};

#define TECDSA_FIELDS(X)                                                                         \
    X(RND, RND_LIMBS)                                                                             \
    X(W, 8) X(GG, 16) X(COM, 8) X(MK, 128)                                                        \
    X(ALIN0, 128) X(ALIN1, 128) X(ALIN2, 128)                                                     \
    X(CK, 128) X(U0, 128) X(U1, 128) X(U2, 128)                                                   \
    X(Z0, 64) X(Z1, 64) X(Z2, 64) X(WP0, 64) X(WP1, 64) X(WP2, 64)                                \
    X(E0, 8) X(E1, 8) X(E2, 8) X(S10, 28) X(S11, 28) X(S12, 28) X(S20, 92) X(S21, 92) X(S22, 92)   \
    X(S0, 64) X(S1, 64) X(S2, 64)                                                                 \
    /* round 1: verification of the peer's three range proofs + the two MessageB */               \
    X(ZE0, 64) X(ZE1, 64) X(ZE2, 64) X(CINVP, 128) X(CINVO, 128)   /* c_peer^-1, c_own^-1 mod N^2 */  \
    X(ZEI0, 64) X(ZEI1, 64) X(ZEI2, 64)                                                           \
    X(GS10, 128) X(GS11, 128) X(GS12, 128)                                                        \
    X(WV0, 64) X(WV1, 64) X(WV2, 64) X(UV0, 128) X(UV1, 128) X(UV2, 128)                          \
    X(LBG, 128) X(LBW, 128) X(CBG, 128) X(CBW, 128)                                               \
    X(BETA_G, 8) X(NU, 8) X(BTG_FE, 8) X(BTW_FE, 8)                                               \
    X(DL0, 40) X(DL1, 40) X(DL2, 40) X(DL3, 40)     /* pk 16 | T 16 | response 8 */              \
    /* round 2 */                                                                                 \
    X(DPG, 64) X(DQG, 64) X(DPW, 64) X(DQW, 64) X(APLG, 64) X(APLW, 64)   /* alpha' plaintexts */      \
    X(ALPHA, 8) X(MU, 8) X(DELTA, 8) X(SIGMA, 8) X(T, 16)                                         \
    X(PED, 64)                                      /* e 8 | a1 16 | a2 16 | z1 8 | z2 8 | pad */ \
    X(DINV, 8)                                                                                    \
    /* round 4 */                                                                                 \
    X(R, 16) X(RD, 16) X(PZ, 64) X(PU1, 16) X(PU2, 128) X(PU3, 64) X(PLIN, 128)                   \
    X(PE, 8) X(PS1, 28) X(PS2, 64) X(PS3, 92)                                                     \
    /* round 5: j = 0 own proof, j = 1 the peer's proof */                                        \
    X(VE0, 8) X(VE1, 8) X(VLIN0, 128) X(VLIN1, 128) X(VZE0, 64) X(VZE1, 64) \
    X(VZEI0, 64) X(VZEI1, 64) X(VU20, 128) X(VU21, 128) X(VU30, 64) X(VU31, 64)                    \
    X(SI, 16) X(HEG, 48)                            /* T 16 | A3 16 | z1 8 | z2 8 */             \
    X(DIGEST, 8)                                                                                  \
    X(FLAGS, 8)                                     /* one ok byte per check, see gg20_glue.cuh */          \
    X(DBG, 256)                                     /* scratch for tools/debug_gg20.py */            \
    /* own-key powers b^N mod N^2 through CRT: halves mod p^2 / q^2 and the recombined value */      \
    X(YP0, 64) X(YP1, 64) X(YP2, 64) X(YP3, 64) X(YP4, 64) X(YP5, 64)                              \
    X(YQ0, 64) X(YQ1, 64) X(YQ2, 64) X(YQ3, 64) X(YQ4, 64) X(YQ5, 64)                              \
    X(XC0, 128) X(XC1, 128) X(XC2, 128) X(XC3, 128) X(XC4, 128) X(XC5, 128)                          \
    /* 1024-bit stage: (b mod p)^(q mod (p-1)) mod p and the q-side twin */                          \
    X(TP0, 32) X(TP1, 32) X(TP2, 32) X(TP3, 32) X(TP4, 32) X(TP5, 32)                              \
    X(TQ0, 32) X(TQ1, 32) X(TQ2, 32) X(TQ3, 32) X(TQ4, 32) X(TQ5, 32)

enum Field : int {
#define X(name, size) F_##name,
    TECDSA_FIELDS(X)
#undef X
    F_COUNT
};

static const int FIELD_SIZE[F_COUNT] = {
#define X(name, size) size,
    TECDSA_FIELDS(X)
#undef X
};
static const char* const FIELD_NAME[F_COUNT] = {
#define X(name, size) #name,
    TECDSA_FIELDS(X)
#undef X
};

// ---- per-key-row tables (row = keyset*3 + party) ------------------------------------------
enum KeyTable : int {
    KT_N = 0,        // 64   Paillier modulus
    KT_NN,           // 128  N^2
    KT_NT,           // 64   N_tilde
    KT_H1, KT_H2,    // 64
    KT_PP, KT_QQ,    // 64   p^2, q^2
    KT_PM1, KT_QM1,  // 32   p-1, q-1
    KT_P, KT_Q,      // 32
    KT_PINV2, KT_QINV2,  // 32   p^-1, q^-1 mod 2^1024 (exact division in the L-function)
    KT_HPR, KT_HQR,  // 32   hp*R mod p, hq*R mod q  (R = 2^1024; hp = L_p((1-N) mod p^2)^-1 mod p)
    KT_PINVQR,       // 32   (p^-1 mod q) * R mod q
    KT_PPINVQQR,     // 64   ((p^2)^-1 mod q^2) * 2^2048 mod q^2  (CRT recombination of own-key N^2 powers)
    KT_QMODPM1, KT_PMODQM1,   // 32   q mod (p-1), p mod (q-1): exponents of the 1024-bit stage of an own-key N-th power
    KT_XI,           // 8    x_i
    KT_PK,           // 16   X_i affine
    KT_COUNT
};
static const int KEY_SIZE[KT_COUNT] = {64, 128, 64, 64, 64, 64, 64, 32, 32, 32, 32, 32, 32, 32, 32, 32, 64, 32, 32, 8, 16};

}  // namespace tecdsa
