/*
 * dpf_core.cuh -- arithmetic core of the DPF evaluation engine.
 *
 * Everything here is `host + device`: the same functions are compiled by nvcc
 * into the sm_100a kernels (dpf_kernels.cu) and by g++ into the host library
 * (keygen / eval_cpu in dpf_host.cpp) and the CPU lane-emulator used by the
 * tests.  Device builds pick the hardware instruction (funnel shift, PRMT,
 * carry-chain adds, ld.shared with immediate offsets); host builds use a
 * portable expression of the same function.
 *
 * What is computed (reference semantics, cited per function):
 *   PRF(seed, pos) for the four reference PRFs, always for BOTH children
 *   pos = 0 and pos = 1 of one GGM node at once, because they share work:
 *     - Salsa20/ChaCha12: three of the four first-round quarter rounds do not
 *       touch the position word and are common to both children;
 *     - AES-128: the key schedule (10 S-box rounds) is common, and the first
 *       cipher round of the second child differs in one table lookup.
 *   The LEAF flavour only produces the low 32 bits of each child: the fused
 *   inner product keeps nothing else (dpf_wrapper.cu:182), which lets the
 *   compiler drop the unused tail of the last round.
 */
#pragma once

#include <stdint.h>

#if defined(__CUDACC__)
#define DPF_HD __host__ __device__ __forceinline__
#else
#define DPF_HD inline __attribute__((always_inline))
#endif

#if defined(__CUDA_ARCH__)
#define DPF_UNROLL _Pragma("unroll")
#else
#define DPF_UNROLL
#endif

#if defined(__CUDA_ARCH__)
#define DPF_DEVICE_CODE 1
#else
#define DPF_DEVICE_CODE 0
#endif

namespace b200dpf {

enum : int { PRF_DUMMY = 0, PRF_SALSA20 = 1, PRF_CHACHA20 = 2, PRF_AES128 = 3 };

/* 128-bit value as four 32-bit words, x = bits 0..31 (the word order of the
 * reference's uint128_t_gpu, dpf_gpu/utils.h:16-25). */
struct Seed {
    uint32_t x, y, z, w;
};

DPF_HD Seed make_seed(uint32_t x, uint32_t y, uint32_t z, uint32_t w)
{
    Seed s; s.x = x; s.y = y; s.z = z; s.w = w; return s;
}

/* ---- primitive ops ------------------------------------------------------ */

DPF_HD uint32_t rotl(uint32_t v, int r)
{
#if DPF_DEVICE_CODE
    return __funnelshift_l(v, v, r);
#else
    return (v << r) | (v >> (32 - r));
#endif
}

/* Rotate through the FMA pipe: x*2^r as a 64-bit product has the rotated word
 * split across its halves (low = x<<r, high = x>>(32-r)), which do not overlap.
 * One IMAD.WIDE + one add, no ALU-pipe slot: used for a fraction of the
 * Salsa/ChaCha rotates because those kernels saturate the ALU pipe (LOP3/SHF)
 * while the FMA pipe idles (profiles/r1_ncu_full_chacha20_*). */
#ifndef DPF_FMA_ROT_MASK
#define DPF_FMA_ROT_MASK 0
#endif
template <int R>
DPF_HD uint32_t rotl_fma(uint32_t v)
{
#if DPF_DEVICE_CODE
    uint32_t lo, hi;
    asm("{\n\t.reg .u64 t;\n\tmul.wide.u32 t, %2, %3;\n\tmov.b64 {%0,%1}, t;\n\t}"
        : "=r"(lo), "=r"(hi) : "r"(v), "n"(1u << R));
    return lo + hi;
#else
    return (v << R) | (v >> (32 - R));
#endif
}
/* rotate number `SLOT` (0..3) of a quarter round: FMA pipe if its mask bit is set */
template <int SLOT, int R>
DPF_HD uint32_t rot_sel(uint32_t v)
{
    return ((DPF_FMA_ROT_MASK >> SLOT) & 1) ? rotl_fma<R>(v) : rotl(v, R);
}

/* PRMT: pick 4 bytes out of the 8 bytes {a (0-3), b (4-7)}; selector nibbles
 * 0-7 only (no sign replication), least significant nibble -> byte 0. */
DPF_HD uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
#if DPF_DEVICE_CODE
    return __byte_perm(a, b, sel);
#else
    uint64_t ab = ((uint64_t)b << 32) | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; i++) {
        uint32_t n = (sel >> (4 * i)) & 7u;
        r |= (uint32_t)((ab >> (8 * n)) & 0xffu) << (8 * i);
    }
    return r;
#endif
}

/* 128-bit add with carry propagation (dpf_gpu/utils.h:45-56, dpf_base/dpf.h:373). */
DPF_HD Seed add128(const Seed &a, const Seed &b)
{
    Seed r;
#if DPF_DEVICE_CODE
    asm("add.cc.u32 %0, %4, %8;\n\t"
        "addc.cc.u32 %1, %5, %9;\n\t"
        "addc.cc.u32 %2, %6, %10;\n\t"
        "addc.u32 %3, %7, %11;"
        : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
        : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w));
#else
    uint64_t c = (uint64_t)a.x + b.x;
    r.x = (uint32_t)c; c >>= 32;
    c += (uint64_t)a.y + b.y; r.y = (uint32_t)c; c >>= 32;
    c += (uint64_t)a.z + b.z; r.z = (uint32_t)c; c >>= 32;
    c += (uint64_t)a.w + b.w; r.w = (uint32_t)c;
#endif
    return r;
}

/* ---- DUMMY PRF ---------------------------------------------------------- */
/* dpf_base/dpf.h:72-74, dpf_gpu/prf/prf.cu:30-35: seed*(4242+pos) + (4242+pos)
 * mod 2^128.  Test-only PRF of the reference (id 0). */
DPF_HD Seed dummy_prf(const Seed &s, uint32_t pos)
{
    const uint64_t k = 4242ull + pos;
    Seed r;
    uint64_t t = (uint64_t)s.x * k + k;
    r.x = (uint32_t)t; t >>= 32;
    t += (uint64_t)s.y * k; r.y = (uint32_t)t; t >>= 32;
    t += (uint64_t)s.z * k; r.z = (uint32_t)t; t >>= 32;
    t += (uint64_t)s.w * k; r.w = (uint32_t)t;
    return r;
}

/* ---- Salsa20/12 and ChaCha/12 ------------------------------------------- */
/* The four constant words exactly as the reference spells them
 * (dpf_base/dpf.h:102-105,163-166; dpf_gpu/prf/prf.cu:63-66,124-127). */
#define DPF_SIGMA0 0x65787061u
#define DPF_SIGMA1 0x6e642033u
#define DPF_SIGMA2 0x322d6279u
#define DPF_SIGMA3 0x7465206bu

#define DPF_SALSA_QR(a, b, c, d)      \
    do {                              \
        b ^= rot_sel<0, 7>(a + d);    \
        c ^= rot_sel<1, 9>(b + a);    \
        d ^= rot_sel<2, 13>(c + b);   \
        a ^= rot_sel<3, 18>(d + c);   \
    } while (0)

#define DPF_CHACHA_QR(a, b, c, d)     \
    do {                              \
        a += b; d = rot_sel<0, 16>(d ^ a);  \
        c += d; b = rot_sel<1, 12>(b ^ c);  \
        a += b; d = rot_sel<2, 8>(d ^ a);   \
        c += d; b = rot_sel<3, 7>(b ^ c);   \
    } while (0)

/*
 * Salsa20 core, 12 rounds (dpf_base/dpf.h:84-135).  Key words sit MSW first in
 * in[1..4], the position in in[9]; the PRF value is words 1..4 of core(in)+in
 * with word 1 the most significant.  LEAF: only the low word (word 4) is made.
 */
template <bool LEAF>
DPF_HD Seed salsa12(const Seed &s, uint32_t pos)
{
    const uint32_t i1 = s.w, i2 = s.z, i3 = s.y, i4 = s.x;
    uint32_t x0 = DPF_SIGMA0, x1 = i1, x2 = i2, x3 = i3, x4 = i4, x5 = DPF_SIGMA1, x6 = 0, x7 = 0,
             x8 = 0, x9 = pos, x10 = DPF_SIGMA2, x11 = 0, x12 = 0, x13 = 0, x14 = 0, x15 = DPF_SIGMA3;
DPF_UNROLL
    for (int r = 0; r < 6; r++) {
        DPF_SALSA_QR(x0, x4, x8, x12);
        DPF_SALSA_QR(x5, x9, x13, x1);
        DPF_SALSA_QR(x10, x14, x2, x6);
        DPF_SALSA_QR(x15, x3, x7, x11);
        DPF_SALSA_QR(x0, x1, x2, x3);
        DPF_SALSA_QR(x5, x6, x7, x4);
        DPF_SALSA_QR(x10, x11, x8, x9);
        DPF_SALSA_QR(x15, x12, x13, x14);
    }
    Seed o;
    o.x = x4 + i4;
    if (LEAF) { o.y = 0; o.z = 0; o.w = 0; }
    else { o.y = x3 + i3; o.z = x2 + i2; o.w = x1 + i1; }
    return o;
}

/*
 * ChaCha core, 12 rounds (dpf_base/dpf.h:145-196).  Key words MSW first in
 * in[4..7], position in in[13]; PRF value = words 4..7 of core(in)+in, word 4
 * most significant.
 */
template <bool LEAF>
DPF_HD Seed chacha12(const Seed &s, uint32_t pos)
{
    const uint32_t i4 = s.w, i5 = s.z, i6 = s.y, i7 = s.x;
    uint32_t x0 = DPF_SIGMA0, x1 = DPF_SIGMA1, x2 = DPF_SIGMA2, x3 = DPF_SIGMA3, x4 = i4, x5 = i5, x6 = i6,
             x7 = i7, x8 = 0, x9 = 0, x10 = 0, x11 = 0, x12 = 0, x13 = pos, x14 = 0, x15 = 0;
DPF_UNROLL
    for (int r = 0; r < 6; r++) {
        DPF_CHACHA_QR(x0, x4, x8, x12);
        DPF_CHACHA_QR(x1, x5, x9, x13);
        DPF_CHACHA_QR(x2, x6, x10, x14);
        DPF_CHACHA_QR(x3, x7, x11, x15);
        DPF_CHACHA_QR(x0, x5, x10, x15);
        DPF_CHACHA_QR(x1, x6, x11, x12);
        DPF_CHACHA_QR(x2, x7, x8, x13);
        DPF_CHACHA_QR(x3, x4, x9, x14);
    }
    Seed o;
    o.x = x7 + i7;
    if (LEAF) { o.y = 0; o.z = 0; o.w = 0; }
    else { o.y = x6 + i6; o.z = x5 + i5; o.w = x4 + i4; }
    return o;
}

/* ---- AES-128 ------------------------------------------------------------- */
/*
 * FIPS-197 AES-128 with key = the 16 little-endian bytes of the seed and
 * plaintext = the 16 little-endian bytes of pos (dpf_base/dpf.h:198-219 ->
 * dpf_base/aes_core.h:579-603,645-672; dpf_gpu/prf/prf.cu:159-184).
 *
 * State columns are little-endian words (column c = bytes 4c..4c+3, byte 4c in
 * bits 0..7), so seed.x is round-key word 0 and the PRF value's .x is output
 * column 0.  One round is four T-table lookups per column with
 *     Te0[v] = 2S | S<<8 | S<<16 | 3S<<24,   Te_k = rotl(Te0, 8k),  S = sbox[v].
 *
 * The lookup itself is behind a policy `TA` so device code can use its
 * conflict-free shared-memory layout and host code a plain array:
 *     uint32_t TA::te<K>(uint32_t word, BYTE) const  ->  Te_K[(word >> 8*BYTE) & 0xff]
 */
struct AesHostTables {
    const uint32_t *te0;   /* 256 entries of Te0 */
    template <int K, int BYTE>
    DPF_HD uint32_t te(uint32_t word) const
    {
        uint32_t v = te0[(word >> (8 * BYTE)) & 0xffu];
        return K == 0 ? v : rotl(v, 8 * K);
    }
};

/* S-box bytes laid out by position: (S[a1], S[a2], S[a3], S[a0]) style merges.
 * Te2 and Te3 carry S in byte 0, Te3/Te0 in byte 1, Te0/Te1 in byte 2 and
 * Te1/Te2 in byte 3, so a word of four S-box outputs is three PRMTs. */
template <class TA, int B0, int B1, int B2, int B3>
DPF_HD uint32_t aes_sub4(const TA &ta, uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3)
{
    /* result byte0 = S[byte B0 of w0], byte1 = S[byte B1 of w1], ... */
    const uint32_t a = ta.template te<2, B0>(w0);   /* S in byte 0 */
    const uint32_t b = ta.template te<3, B1>(w1);   /* S in byte 1 */
    const uint32_t c = ta.template te<0, B2>(w2);   /* S in byte 2 */
    const uint32_t d = ta.template te<1, B3>(w3);   /* S in byte 3 */
    const uint32_t ab = prmt(a, b, 0x0050);         /* byte0 <- a.0, byte1 <- b.1 */
    const uint32_t cd = prmt(c, d, 0x7200);         /* byte2 <- c.2, byte3 <- d.3 */
    return prmt(ab, cd, 0x7610);
}

/* next round key: w <- FIPS-197 key expansion step with round constant rc */
template <class TA>
DPF_HD void aes_next_rk(const TA &ta, uint32_t &k0, uint32_t &k1, uint32_t &k2, uint32_t &k3, uint32_t rc)
{
    /* SubWord(RotWord(k3)): bytes (S[b1], S[b2], S[b3], S[b0]) of k3 */
    const uint32_t t = aes_sub4<TA, 1, 2, 3, 0>(ta, k3, k3, k3, k3);
    k0 ^= t ^ rc;
    k1 ^= k0;
    k2 ^= k1;
    k3 ^= k2;
}

template <class TA>
DPF_HD void aes_round(const TA &ta, uint32_t &s0, uint32_t &s1, uint32_t &s2, uint32_t &s3,
                      uint32_t k0, uint32_t k1, uint32_t k2, uint32_t k3)
{
    const uint32_t t0 = ta.template te<0, 0>(s0) ^ ta.template te<1, 1>(s1) ^ ta.template te<2, 2>(s2) ^ ta.template te<3, 3>(s3) ^ k0;
    const uint32_t t1 = ta.template te<0, 0>(s1) ^ ta.template te<1, 1>(s2) ^ ta.template te<2, 2>(s3) ^ ta.template te<3, 3>(s0) ^ k1;
    const uint32_t t2 = ta.template te<0, 0>(s2) ^ ta.template te<1, 1>(s3) ^ ta.template te<2, 2>(s0) ^ ta.template te<3, 3>(s1) ^ k2;
    const uint32_t t3 = ta.template te<0, 0>(s3) ^ ta.template te<1, 1>(s0) ^ ta.template te<2, 2>(s1) ^ ta.template te<3, 3>(s2) ^ k3;
    s0 = t0; s1 = t1; s2 = t2; s3 = t3;
}

/*
 * First cipher round fused with the first key-schedule step.  The state entering
 * round 1 is plaintext ^ rk0 = (k0 ^ pos, k1, k2, k3), so the four lookups that
 * index the bytes of column 3 (= k3) are the same S-box reads the key schedule
 * needs for SubWord(RotWord(k3)): they are done once and their S bytes picked
 * out with PRMTs (4 fewer lookups per node).  In: rk0 in k0..k3.  Out: rk1 in
 * k0..k3, the state after round 1 in a0..a3, and in `col0_te0` the lookup
 * Te0[byte 0 of column 0] (the only one the sibling with pos^1 does not share).
 */
template <class TA>
DPF_HD void aes_first_round(const TA &ta, uint32_t pos, uint32_t &k0, uint32_t &k1, uint32_t &k2, uint32_t &k3,
                            uint32_t &a0, uint32_t &a1, uint32_t &a2, uint32_t &a3, uint32_t &col0_te0)
{
    const uint32_t s0 = k0 ^ pos;
    const uint32_t l00 = ta.template te<0, 0>(s0), l11 = ta.template te<1, 1>(k1), l22 = ta.template te<2, 2>(k2), l33 = ta.template te<3, 3>(k3);
    const uint32_t l01 = ta.template te<0, 0>(k1), l12 = ta.template te<1, 1>(k2), l23 = ta.template te<2, 2>(k3), l30 = ta.template te<3, 3>(s0);
    const uint32_t l02 = ta.template te<0, 0>(k2), l13 = ta.template te<1, 1>(k3), l20 = ta.template te<2, 2>(s0), l31 = ta.template te<3, 3>(k1);
    const uint32_t l03 = ta.template te<0, 0>(k3), l10 = ta.template te<1, 1>(s0), l21 = ta.template te<2, 2>(k1), l32 = ta.template te<3, 3>(k2);
    /* SubWord(RotWord(k3)) = (S[b1], S[b2], S[b3], S[b0]) of k3:
     *   l13 = Te1[b1] has S in bytes 2,3;  l23 = Te2[b2] in bytes 0,3;
     *   l33 = Te3[b3] in bytes 0,1;        l03 = Te0[b0] in bytes 1,2 */
    const uint32_t ab = prmt(l13, l23, 0x0042);   /* byte0 <- l13.2, byte1 <- l23.0 */
    const uint32_t cd = prmt(l33, l03, 0x5000);   /* byte2 <- l33.0, byte3 <- l03.1 */
    const uint32_t t = prmt(ab, cd, 0x7610);
    k0 ^= t ^ 1u;
    k1 ^= k0;
    k2 ^= k1;
    k3 ^= k2;
    a0 = l00 ^ l11 ^ l22 ^ l33 ^ k0;
    a1 = l01 ^ l12 ^ l23 ^ l30 ^ k1;
    a2 = l02 ^ l13 ^ l20 ^ l31 ^ k2;
    a3 = l03 ^ l10 ^ l21 ^ l32 ^ k3;
    col0_te0 = l00;
}

/* Both children of one node: AES_seed(0) and AES_seed(1).  LEAF: .x only. */
template <bool LEAF, class TA>
DPF_HD void aes128_pair(const TA &ta, const Seed &s, Seed &c0, Seed &c1)
{
    uint32_t k0 = s.x, k1 = s.y, k2 = s.z, k3 = s.w;
    uint32_t a0, a1, a2, a3, l00;
    /* the children's plaintexts are 0 and 1: they differ in byte 0 of column 0,
     * which after ShiftRows+MixColumns lands in output column 0 alone */
    const uint32_t sib = ta.template te<0, 0>(k0 ^ 1u);
    aes_first_round(ta, 0u, k0, k1, k2, k3, a0, a1, a2, a3, l00);
    uint32_t b0 = a0 ^ l00 ^ sib, b1 = a1, b2 = a2, b3 = a3;
    uint32_t rc = 2;
DPF_UNROLL
    for (int r = 2; r <= 9; r++) {
        aes_next_rk(ta, k0, k1, k2, k3, rc);
        rc = (rc << 1) ^ ((rc & 0x80u) ? 0x11bu : 0u);
        aes_round(ta, a0, a1, a2, a3, k0, k1, k2, k3);
        aes_round(ta, b0, b1, b2, b3, k0, k1, k2, k3);
    }
    aes_next_rk(ta, k0, k1, k2, k3, rc);
    /* final round: SubBytes + ShiftRows + AddRoundKey */
    c0.x = aes_sub4<TA, 0, 1, 2, 3>(ta, a0, a1, a2, a3) ^ k0;
    c1.x = aes_sub4<TA, 0, 1, 2, 3>(ta, b0, b1, b2, b3) ^ k0;
    if (LEAF) {
        c0.y = c0.z = c0.w = 0;
        c1.y = c1.z = c1.w = 0;
    } else {
        c0.y = aes_sub4<TA, 0, 1, 2, 3>(ta, a1, a2, a3, a0) ^ k1;
        c0.z = aes_sub4<TA, 0, 1, 2, 3>(ta, a2, a3, a0, a1) ^ k2;
        c0.w = aes_sub4<TA, 0, 1, 2, 3>(ta, a3, a0, a1, a2) ^ k3;
        c1.y = aes_sub4<TA, 0, 1, 2, 3>(ta, b1, b2, b3, b0) ^ k1;
        c1.z = aes_sub4<TA, 0, 1, 2, 3>(ta, b2, b3, b0, b1) ^ k2;
        c1.w = aes_sub4<TA, 0, 1, 2, 3>(ta, b3, b0, b1, b2) ^ k3;
    }
}

/* One child only (used on the root-to-subtree walk, where the branch taken is
 * known): AES_seed(pos), pos in {0,1}. */
template <class TA>
DPF_HD Seed aes128_one(const TA &ta, const Seed &s, uint32_t pos)
{
    uint32_t k0 = s.x, k1 = s.y, k2 = s.z, k3 = s.w;
    uint32_t a0, a1, a2, a3, l00;
    aes_first_round(ta, pos, k0, k1, k2, k3, a0, a1, a2, a3, l00);
    uint32_t rc = 2;
DPF_UNROLL
    for (int r = 2; r <= 9; r++) {
        aes_next_rk(ta, k0, k1, k2, k3, rc);
        rc = (rc << 1) ^ ((rc & 0x80u) ? 0x11bu : 0u);
        aes_round(ta, a0, a1, a2, a3, k0, k1, k2, k3);
    }
    aes_next_rk(ta, k0, k1, k2, k3, rc);
    Seed c;
    c.x = aes_sub4<TA, 0, 1, 2, 3>(ta, a0, a1, a2, a3) ^ k0;
    c.y = aes_sub4<TA, 0, 1, 2, 3>(ta, a1, a2, a3, a0) ^ k1;
    c.z = aes_sub4<TA, 0, 1, 2, 3>(ta, a2, a3, a0, a1) ^ k2;
    c.w = aes_sub4<TA, 0, 1, 2, 3>(ta, a3, a0, a1, a2) ^ k3;
    return c;
}

/* ---- PRF dispatch -------------------------------------------------------- */

/* PRF(parent, 0) and PRF(parent, 1), correction words NOT yet added.
 * (dpf_base/dpf.h:226-235 PRF_SELECT; dpf_gpu/prf/prf.cu:186-201). */
template <int PRF, bool LEAF, class TA>
DPF_HD void expand_pair(const TA &ta, const Seed &parent, Seed &c0, Seed &c1)
{
    if (PRF == PRF_DUMMY) {
        c0 = dummy_prf(parent, 0);
        c1 = dummy_prf(parent, 1);
    } else if (PRF == PRF_SALSA20) {
        c0 = salsa12<LEAF>(parent, 0);
        c1 = salsa12<LEAF>(parent, 1);
    } else if (PRF == PRF_CHACHA20) {
        c0 = chacha12<LEAF>(parent, 0);
        c1 = chacha12<LEAF>(parent, 1);
    } else {
        aes128_pair<LEAF>(ta, parent, c0, c1);
    }
}

template <int PRF, class TA>
DPF_HD Seed expand_one(const TA &ta, const Seed &parent, uint32_t pos)
{
    if (PRF == PRF_DUMMY) return dummy_prf(parent, pos);
    if (PRF == PRF_SALSA20) return salsa12<false>(parent, pos);
    if (PRF == PRF_CHACHA20) return chacha12<false>(parent, pos);
    return aes128_one(ta, parent, pos);
}

/* ---- tree traversal ------------------------------------------------------ */
/*
 * Tree conventions (dpf_base/dpf.h:362-377, EvaluateFlat): the root consumes
 * the LSB of the index; the step that consumes index bit k uses correction
 * words cw[2*level + bit] with level = depth-1-k, taken from bank cw_1 when the
 * PARENT seed is even and cw_2 when it is odd; child = PRF(parent, bit) + cw
 * with a full 128-bit add.  Leaf position p (path bits MSB first) therefore
 * holds index bitrev_depth(p), the order the table is stored in on the device.
 *
 * `Env` supplies storage (all per thread / per lane):
 *     Seed     cw(level, bank, bit)      correction word
 *     uint32_t cw_lo(bank, bit)          low word of the level-0 correction word
 *     void     push(h, Seed), Seed pop(h) pending right child of height h
 *     void     leaf_prefetch(local_pos)      called before the leaf pair is expanded
 *     void     leaf_pair(local_pos, v0, v1)  consume leaves local_pos, local_pos+1
 *     void     node_pair(local_pos, c0, c1)  (FULL mode) consume whole seeds
 *     ta                                 AES table policy
 */

/* Walk `steps` levels down from `seed`, whose children are produced with
 * correction-word level `first_level`; the branch taken at step k is bit
 * (steps-1-k) of `q`.  From the key's root (first_level = depth-1) with
 * steps = depth-s this reaches the root of the 2^s-leaf subtree with
 * breadth-first index q.  `q` is the same for every lane of a warp, so the
 * branch bits are warp-uniform. */
template <int PRF, class Env>
DPF_HD Seed walk_down(Env &env, Seed seed, int first_level, int steps, uint32_t q)
{
    for (int k = 0; k < steps; k++) {
        const uint32_t bit = (q >> (steps - 1 - k)) & 1u;
        const int level = first_level - k;
        const uint32_t bank = seed.x & 1u;
        seed = add128(expand_one<PRF>(env.ta, seed, bit), env.cw(level, bank, bit));
    }
    return seed;
}

DPF_HD int ctz32(uint32_t v)
{
#if DPF_DEVICE_CODE
    return __ffs((int)v) - 1;
#else
    return __builtin_ctz(v);
#endif
}

/*
 * Depth-first expansion of a complete subtree with 2^s leaves, one node pair at
 * a time, keeping only the pending right siblings (one per height).  A node of
 * height h has 2^h leaves below it; expanding it uses correction-word level
 * level_base + h - 1 (level_base = 0 when the subtree's leaves are the leaves
 * of the whole tree).  Leaves come out in increasing position order, two per
 * step:
 *   FULL = false: only their low 32 bits (the fused inner product / share
 *                 vector needs nothing else, dpf_wrapper.cu:182) via
 *                 env.leaf_pair(local_pos, v0, v1); requires level_base == 0;
 *   FULL = true : whole 128-bit seeds via env.node_pair(local_pos, c0, c1) --
 *                 used to materialise an interior frontier of the tree.
 */
template <int PRF, bool FULL, class Env>
DPF_HD void eval_subtree(Env &env, Seed seed, int s, int level_base)
{
    int h = s;
    /* AES: the pending right child of height 1 is taken right after the next leaf pair, so it stays
     * in registers instead of going through env.push/pop -- one 16-byte store and load fewer on the
     * shared-memory pipe that binds the AES kernel, per height-2 node.  The selects that cost are
     * extra issue slots, which is what binds Salsa/ChaCha, so they keep the stack. */
    constexpr bool REG_SIBLING = (PRF == PRF_AES128);
    Seed right1 = seed;
    const uint32_t npairs = 1u << (s - 1);
    for (uint32_t i = 0; i < npairs; i++) {
        while (h > 1) {
            Seed c0, c1;
            expand_pair<PRF, false>(env.ta, seed, c0, c1);
            const uint32_t bank = seed.x & 1u;
            const int level = level_base + h - 1;
            c1 = add128(c1, env.cw(level, bank, 1));
            if (REG_SIBLING && h == 2) right1 = c1;
            else env.push(h - 1, c1);
            seed = add128(c0, env.cw(level, bank, 0));
            h--;
        }
        Seed l0, l1;
        const uint32_t bank = seed.x & 1u;
        if (FULL) {
            expand_pair<PRF, false>(env.ta, seed, l0, l1);
            env.node_pair(2 * i, add128(l0, env.cw(level_base, bank, 0)), add128(l1, env.cw(level_base, bank, 1)));
        } else {
            env.leaf_prefetch(2 * i);
            expand_pair<PRF, true>(env.ta, seed, l0, l1);
            env.leaf_pair(2 * i, l0.x + env.cw_lo(bank, 0), l1.x + env.cw_lo(bank, 1));
        }
        h = ctz32(i + 1) + 1;
        if (REG_SIBLING && h == 1 && s > 1) seed = right1;
        else if (h < s) seed = env.pop(h);
    }
}

}  // namespace b200dpf
