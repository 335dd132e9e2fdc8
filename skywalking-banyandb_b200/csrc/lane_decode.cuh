// lane_decode.cuh -- the per-lane part of the fast varint decoders of scan_kernels.cu.
//
// Everything here is a plain function of one lane's registers (no shuffles, no shared memory), so the very same source is
// also compiled for the host: tests/native/lane_decode_test.cc runs it against a byte-at-a-time reference decoder
// (full chunks, chunks with bytes outside the page, and the two-chain experiment) without a GPU.
#pragma once

#include <cstdint>

#if defined(__CUDACC__)
#define BYDB_LANE_FN __host__ __device__ __forceinline__
#else
#include <vector_functions.h>  // uint4 / make_uint4 for a plain host compiler
#include <vector_types.h>
#define BYDB_LANE_FN inline
#endif

namespace bydb {

BYDB_LANE_FN uint32_t lane_popc(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return static_cast<uint32_t>(__popc(x));
#else
    return static_cast<uint32_t>(__builtin_popcount(x));
#endif
}
BYDB_LANE_FN int lane_clz(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __clz(static_cast<int>(x));
#else
    return x ? __builtin_clz(x) : 32;
#endif
}
BYDB_LANE_FN int lane_ffs(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __ffs(static_cast<int>(x));
#else
    return __builtin_ffs(static_cast<int>(x));
#endif
}
BYDB_LANE_FN uint32_t lane_byte_perm(uint32_t a, uint32_t b, uint32_t sel) {
#if defined(__CUDA_ARCH__)
    return __byte_perm(a, b, sel);
#else
    const uint64_t src = (static_cast<uint64_t>(b) << 32) | a;  // PRMT without the sign-replicate modes
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) r |= static_cast<uint32_t>((src >> (8 * ((sel >> (4 * i)) & 7))) & 0xff) << (8 * i);
    return r;
#endif
}

BYDB_LANE_FN uint32_t msb4(uint32_t x) {  // gathers the 4 byte-MSBs of x into bits 0..3
    // bit 8j+7 times 2^(21-7j) lands on bit 28+j; no two partial products share a bit, so nothing carries
    return ((x & 0x80808080u) * 0x00204081u) >> 28;
}

// one lane's 32 bytes: local prefix P of its deltas folded over the active rows.
// kFull: all 32 bytes are valid (interior chunk) -> no per-byte validity logic.
// kNeed: bit0 = sum wanted, bit1 = min/max wanted.
enum { kNeedSum = 1, kNeedMinMax = 2 };
constexpr uint32_t kFastLaneBytes = 32;
constexpr uint32_t kFastChunkBytes = 32 * kFastLaneBytes;  // 1 KB per warp iteration

BYDB_LANE_FN uint32_t low_bits(uint32_t n) { return n >= 32 ? 0xffffffffu : ((1u << n) - 1u); }

// 32-bit multiply-add that stays a multiply-add: IMAD runs on the FMA pipe, which this integer kernel otherwise
// leaves idle while LOP3/SHF/SEL/IADD3 saturate the ALU pipe (ncu r01h: alu 82 %, fma 17 %).  Written as inline PTX
// so that neither the front end nor ptxas turns a multiply by a 0/1 flag back into logic ops.
BYDB_LANE_FN uint32_t imad_u32(uint32_t a, uint32_t b, uint32_t c) {
    uint32_t d;
#if defined(__CUDA_ARCH__)
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
#else
    d = a * b + c;
#endif
    return d;
}
BYDB_LANE_FN int32_t imad_s32(int32_t a, int32_t b, int32_t c) {
    int32_t d;
#if defined(__CUDA_ARCH__)
    asm("mad.lo.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
#else
    d = static_cast<int32_t>(static_cast<uint32_t>(a) * static_cast<uint32_t>(b) + static_cast<uint32_t>(c));
#endif
    return d;
}

// Interior chunk (all 32 bytes valid): the per-byte state machine with its selects, masks and shifts rewritten as
// multiply-adds by 0/1 flags so that the work splits about evenly between the ALU and the FMA pipe.
//   accv += b * mul                (mul = 128^k inside a varint, back to 1 after its terminator)
//   v     = h - s * accv           (zig-zag: accv = 2h + s)
//   P    += v * t ; sumP += P * (t & active)
#ifndef BYDB_UNROLL
#define BYDB_UNROLL 2
#endif
#define BYDB_PRAGMA_(x) _Pragma(#x)
#define BYDB_PRAGMA(x) BYDB_PRAGMA_(x)
#define BYDB_UNROLL_WORDS BYDB_PRAGMA(unroll BYDB_UNROLL)

// kMasked: the chunk holds bytes outside the page (first / last chunk): `reset` = term | ~valid restarts the varint
// state at those bytes too, their payload is zeroed by the caller, and only real terminators (term) count as rows.
template <int kNeed, bool kMasked>
BYDB_LANE_FN void fast_lane_decode_imad(const uint4 &wa, const uint4 &wb, uint32_t term, uint32_t reset, uint32_t aw, uint32_t &accv,
                                                      uint32_t &sh, int32_t &P, int32_t &sumP, int32_t &minP, int32_t &maxP) {
    // 8 words x 4 bytes: the word loop stays rolled so that the body (the hottest code of the whole
    // path) stays resident in the instruction caches of every scheduler
    uint32_t w0 = wa.x, w1 = wa.y, w2 = wa.z, w3 = wa.w, w4 = wb.x, w5 = wb.y, w6 = wb.z, w7 = wb.w;
    uint32_t tm = term, rm = reset;
    uint32_t mul = 1u << sh;
    BYDB_UNROLL_WORDS
    for (int q8 = 0; q8 < 8; ++q8) {
        const uint32_t p = w0 & 0x7f7f7f7fu;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t b = j == 3 ? (p >> 24) : (j == 0 ? (p & 0xffu) : lane_byte_perm(p, 0u, 0x4440u + j));
            const uint32_t t = (tm >> j) & 1u;
            const uint32_t nr = (kMasked ? ((rm >> j) & 1u) : t) ^ 1u;
            accv = imad_u32(b, mul, accv);
            const uint32_t h = accv >> 1, s = accv & 1u;
            const int32_t v = imad_s32(static_cast<int32_t>(s), static_cast<int32_t>(0u - accv), static_cast<int32_t>(h));
            P = imad_s32(v, static_cast<int32_t>(t), P);
            const uint32_t at = aw & t;  // terminator of an active row
            if (kNeed & kNeedSum) sumP = imad_s32(P, static_cast<int32_t>(at), sumP);
            if (kNeed & kNeedMinMax) {
                // candidate = P at an active terminator, the neutral element otherwise
                const int32_t lo_c = static_cast<int32_t>(imad_u32(at, static_cast<uint32_t>(P) - 0x7fffffffu, 0x7fffffffu));
                const int32_t hi_c = static_cast<int32_t>(imad_u32(at, static_cast<uint32_t>(P) - 0x80000000u, 0x80000000u));
                minP = lo_c < minP ? lo_c : minP;
                maxP = hi_c > maxP ? hi_c : maxP;
            }
            aw >>= t;
            accv = imad_u32(accv, nr, 0u);
            mul = imad_u32(mul, imad_u32(nr, 128u, 0u), nr ^ 1u);
        }
        w0 = w1;
        w1 = w2;
        w2 = w3;
        w3 = w4;
        w4 = w5;
        w5 = w6;
        w6 = w7;
        tm >>= 4;
        if (kMasked) rm >>= 4;
    }
    sh = 31u - static_cast<uint32_t>(lane_clz(mul));
}

BYDB_LANE_FN int32_t head_delta(uint32_t w0, uint32_t term, uint32_t prev_acc, uint32_t prev_sh);

// ------------------------------------------------------------------------------------------------
// SWAR sum decoder: every row active, SUM/MEAN/COUNT only (BASELINE config 3: group-by sum over all rows).
//
// For a page first, d_1 .. d_{n-1} the sum over all rows of value_r = first + sum_{j<=r} d_j is
//     n*first + sum_j d_j * (n - j),
// and a zig-zag varint is LINEAR in its payload bytes once its sign is known:
//     d = sigma * ( (b0+1)>>1  +  64*b1  +  8192*b2 ),   sigma = 1 - 2*(b0 & 1)          (b_k = 7-bit payloads, <= 3 bytes)
// so the whole page sum is  sum over BYTES of  (class scale) * sigma * payload * (n - 1 - #terminators before the byte):
// no value is ever assembled, no prefix is carried along the bytes, and a varint that straddles two lanes (or two chunks)
// needs no correction -- each of its bytes is accounted where it lies.  Per 4-byte word the lane builds, with byte
// permutes (PRMT with sign replication) and bitwise selects,
//     M1 / M2   0xff where the previous / second previous byte is a continuation  -> class of the byte (0, 1, 2)
//     Sm        0xff where the byte belongs to a negative varint (bit 0 of the varint's first byte)
//     rank1     1 + number of terminators before the byte inside the lane (a SWAR prefix sum by one multiply)
// and feeds six 4-way byte dot products (IDP.4A): T_k += payload_k . (+-1), R_k += payload_k . (+-rank1).
// The class-0 payload carries its own sign instead:  (b0 ^ Sm) as int8 = b0 (even, positive) or -(b0+1) = 2 * d's
// class-0 part, so T0 / R0 hold twice their value (always even).  Lane result:
//     T = T0/2 + 64*T1 + 8192*T2 = sum of the lane's byte contributions,  R' = same with weights rank+1,
// page sum += (A + 1) * T - R'   with A = n - 1 - (terminators before the lane).
// Class 2 only exists in varints of 3 or more bytes (|delta| >= 8192 units of the last decimal), which metric columns at a fixed
// precision almost never hold: the scan runs the two-class form of the word (kTwoClass, five dot products) and decodes a chunk again
// with the three-class form only when its guard says a class-2 byte is there.
// ------------------------------------------------------------------------------------------------
BYDB_LANE_FN uint32_t lane_prmt(uint32_t a, uint32_t b, uint32_t sel) {  // PTX prmt.b32, default mode (bit 3 of a selector nibble = replicate the byte's msb)
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
#else
    const uint64_t src = (static_cast<uint64_t>(b) << 32) | a;
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) {
        const uint32_t n = (sel >> (4 * i)) & 0xfu;
        uint32_t byte = static_cast<uint32_t>((src >> (8 * (n & 7u))) & 0xffu);
        if (n & 8u) byte = (byte & 0x80u) ? 0xffu : 0x00u;
        r |= byte << (8 * i);
    }
    return r;
#endif
}
// 4-way byte dot products with 32-bit accumulate: a signed x b unsigned, a unsigned x b signed
BYDB_LANE_FN int32_t dp4a_su(uint32_t a, uint32_t b, int32_t c) {
#if defined(__CUDA_ARCH__)
    int32_t d;
    asm("dp4a.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
#else
    for (int i = 0; i < 4; ++i) c += static_cast<int32_t>(static_cast<int8_t>((a >> (8 * i)) & 0xff)) * static_cast<int32_t>((b >> (8 * i)) & 0xff);
    return c;
#endif
}
BYDB_LANE_FN int32_t dp4a_us(uint32_t a, uint32_t b, int32_t c) {
#if defined(__CUDA_ARCH__)
    int32_t d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
#else
    for (int i = 0; i < 4; ++i) c += static_cast<int32_t>((a >> (8 * i)) & 0xff) * static_cast<int32_t>(static_cast<int8_t>((b >> (8 * i)) & 0xff));
    return c;
#endif
}

BYDB_LANE_FN uint32_t mulhi_u32(uint32_t a, uint32_t b) {  // IMAD.HI: a right shift by a constant done on the FMA pipe
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("mul.hi.u32 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
#else
    return static_cast<uint32_t>((static_cast<uint64_t>(a) * b) >> 32);
#endif
}

struct SwarLane {
    int32_t T0, T1, T2, R0, R1, R2;
    uint32_t wide;     // msb set in some byte <=> a varint of 4 or more bytes was seen (three-class words only)
    uint32_t guard;    // msb set in some byte <=> the byte after it is of class 2 (two-class words only)
    int32_t nterm;     // 1 + terminators seen so far in this lane
    uint32_t prev_w;   // the word before the current one (the previous lane's last word for the first)
};
BYDB_LANE_FN void swar_begin(SwarLane &s, uint32_t prev_w) {
    s.T0 = s.T1 = s.T2 = s.R0 = s.R1 = s.R2 = 0;
    s.wide = s.guard = 0;
    s.nterm = 1;
    s.prev_w = prev_w;
}
// kMasked: first / last chunk of a page -- vm is 0xff for the bytes of the word that belong to the page; the others
// neither terminate, nor carry payload, nor continue anything.
// kTwoClass: the word as if no byte were of class 2 -- class 1 = every continued byte, its sign S1 -- which drops M2, S2, the
// S12 select and the two class-2 dot products.  The guard collects w & M1 instead: an msb there = a continuation byte after
// a continuation byte, so the NEXT byte is of class 2 (the third byte of a varint of 3 or more bytes) and the chunk has to be
// decoded again by the three-class word.  Without class-2 bytes both forms give the same T, R' and terminator count, bit for bit.
// Pipe balance (ncu r01: this integer kernel is bound by the ALU pipe, LOP3/PRMT/SHF, while the FMA pipe idles): everything
// that can be a multiply-add is one -- the shifts by constants (IMAD / IMAD.HI), the in-word prefix sum, the running
// terminator count (a dot product with 1s) and its broadcast.
template <bool kMasked, bool kTwoClass = false>
BYDB_LANE_FN void swar_word(SwarLane &s, uint32_t w_in, uint32_t vm) {
    const uint32_t w = kMasked ? (w_in & vm) : w_in;
    const uint32_t pw = s.prev_w;
    const uint32_t p = w & 0x7f7f7f7fu;
    const uint32_t M1 = lane_prmt(w, pw, 0xA98Fu);   // byte i <- msb of byte i-1, replicated: 0xff = not the first byte of a varint
    const uint32_t sb = imad_u32(w, 128u, 0u);       // bit 0 of every byte moved to its msb (the low bits are don't-care)
    const uint32_t psb = imad_u32(pw, 128u, 0u);
    const uint32_t S0 = lane_prmt(sb, 0u, 0xBA98u);  // sign of a varint that starts at this byte
    const uint32_t S1 = lane_prmt(sb, psb, 0xA98Fu); // ... that started one byte earlier
    const uint32_t x0 = (p ^ S0) & ~M1;              // class 0: int8 = 2 * (signed class-0 part); 0 elsewhere
    uint32_t p1, S12, q2 = 0;
    if (kTwoClass) {
        p1 = p & M1;                                 // class 1 payloads
        S12 = S1;
        s.guard |= w & M1;
    } else {
        const uint32_t M2 = lane_prmt(w, pw, 0x98FEu);    // byte i <- msb of byte i-2
        const uint32_t S2 = lane_prmt(sb, psb, 0x98FEu);  // sign of a varint that started two bytes earlier
        S12 = (M2 & S2) | (~M2 & S1);                     // sign of the varint a class-1 / class-2 byte belongs to
        p1 = p & M1 & ~M2;                                // class 1 payloads
        q2 = w & M1 & M2;                                 // class 2 payloads; an msb here = a fourth byte follows (wide: the page bails out)
    }
    const uint32_t wT = S12 | 0x01010101u;           // +-1 (only read where p1 / q2 are non-zero, i.e. on class 1 / 2 bytes)
    uint32_t t01 = ~mulhi_u32(w, 1u << 25) & 0x01010101u;  // 1 where the byte terminates a varint
    if (kMasked) t01 &= vm;
    const uint32_t base = imad_u32(static_cast<uint32_t>(s.nterm), 0x01010101u, 0u);
    const uint32_t rinc = imad_u32(t01, 0x01010101u, base);    // inclusive terminator count + 1
    const uint32_t rank1 = imad_u32(t01, 0xffffffffu, rinc);   // exclusive count + 1, in [1, 33]
    s.nterm = dp4a_su(0x01010101u, t01, s.nterm);
    const uint32_t wR = imad_u32(S12 & 0x01010101u, 1u, rank1 ^ S12);  // +-rank1 as int8 (rank1 >= 1: the +1 never carries)
    s.T0 = dp4a_su(x0, 0x01010101u, s.T0);
    s.R0 = dp4a_su(x0, rank1, s.R0);
    s.T1 = dp4a_us(p1, wT, s.T1);
    s.R1 = dp4a_us(p1, wR, s.R1);
    if (!kTwoClass) {
        s.T2 = dp4a_us(q2, wT, s.T2);
        s.R2 = dp4a_us(q2, wR, s.R2);
        s.wide |= q2;
    }
    s.prev_w = w;
}
// The word before a chunk ends in two continuation bytes: the chunk's first byte is of class 2, which the guard of the
// chunk's own words cannot see (it lies behind the previous chunk's last byte).
BYDB_LANE_FN bool swar_opens_class2(uint32_t last_w) { return ((last_w & (last_w << 8)) >> 31) != 0; }
// -> number of terminators of the lane; T and R' as defined above
BYDB_LANE_FN uint32_t swar_end(const SwarLane &s, int32_t &T, int32_t &Rp) {
    T = (s.T0 >> 1) + 64 * s.T1 + 8192 * s.T2;
    Rp = (s.R0 >> 1) + 64 * s.R1 + 8192 * s.R2;
    return static_cast<uint32_t>(s.nterm - 1);
}

// ------------------------------------------------------------------------------------------------
// Sparse masked decode (delta_page_sparse in scan_kernels.cu): when a row predicate / time range leaves most 64-byte lane
// windows of a page without an active row, the warp first runs a LIGHT pass over every window -- the byte-linear sum T of the
// SWAR decoder without the rank weights, the terminator count and the unfinished tail -- which is all that is needed to know
// every window's first row and the value in front of it; only the windows that hold an active row are then decoded value by
// value (fast_lane_decode, started from the previous window's tail), 32 of them at a time, one per lane.
// ------------------------------------------------------------------------------------------------
struct SwarLite {
    int32_t T0, T1, T2;
    uint32_t wide;
    int32_t nterm;     // terminators seen so far in this lane
    uint32_t prev_w;
};
BYDB_LANE_FN void swar_lite_begin(SwarLite &s, uint32_t prev_w) {
    s.T0 = s.T1 = s.T2 = 0;
    s.wide = 0;
    s.nterm = 0;
    s.prev_w = prev_w;
}
template <bool kMasked>
BYDB_LANE_FN void swar_lite_word(SwarLite &s, uint32_t w_in, uint32_t vm) {
    const uint32_t w = kMasked ? (w_in & vm) : w_in;
    const uint32_t pw = s.prev_w;
    const uint32_t p = w & 0x7f7f7f7fu;
    const uint32_t M1 = lane_prmt(w, pw, 0xA98Fu);
    const uint32_t M2 = lane_prmt(w, pw, 0x98FEu);
    const uint32_t sb = imad_u32(w, 128u, 0u);
    const uint32_t psb = imad_u32(pw, 128u, 0u);
    const uint32_t S0 = lane_prmt(sb, 0u, 0xBA98u);
    const uint32_t S1 = lane_prmt(sb, psb, 0xA98Fu);
    const uint32_t S2 = lane_prmt(sb, psb, 0x98FEu);
    const uint32_t S12 = (M2 & S2) | (~M2 & S1);
    const uint32_t x0 = (p ^ S0) & ~M1;
    const uint32_t p1 = p & M1 & ~M2;
    const uint32_t q2 = w & M1 & M2;
    const uint32_t wT = S12 | 0x01010101u;
    uint32_t t01 = ~mulhi_u32(w, 1u << 25) & 0x01010101u;
    if (kMasked) t01 &= vm;
    s.nterm = dp4a_su(0x01010101u, t01, s.nterm);
    s.T0 = dp4a_su(x0, 0x01010101u, s.T0);
    s.T1 = dp4a_us(p1, wT, s.T1);
    s.T2 = dp4a_us(q2, wT, s.T2);
    s.wide |= q2;
    s.prev_w = w;
}
BYDB_LANE_FN uint32_t swar_lite_end(const SwarLite &s, int32_t &T) {
    T = (s.T0 >> 1) + 64 * s.T1 + 8192 * s.T2;
    return static_cast<uint32_t>(s.nterm);
}
// The unfinished varint at the end of a lane (narrow pages: at most its first two bytes), from the lane's last word as the
// decoder saw it (bytes outside the page zeroed): payload bits gathered so far, their count (0 / 7 / 14), and what those
// bytes contributed to the lane's byte-linear sum T -- so that  T + pv(previous lane) - pv(this lane)  is the sum of the
// deltas of the values that END in this lane.
BYDB_LANE_FN void swar_tail(uint32_t lw, uint32_t &accv, uint32_t &sh, int32_t &pv) {
    const uint32_t b3 = lw >> 24, b2 = (lw >> 16) & 0xffu;
    accv = 0;
    sh = 0;
    pv = 0;
    if (b3 & 0x80u) {
        const bool two = (b2 & 0x80u) != 0;
        const uint32_t p0 = (two ? b2 : b3) & 0x7fu;
        const uint32_t p1 = two ? (b3 & 0x7fu) : 0u;
        accv = p0 | (p1 << 7);
        sh = two ? 14u : 7u;
        const int32_t mag = static_cast<int32_t>((p0 >> 1) + (p0 & 1u) + 64u * p1);
        pv = (p0 & 1u) ? -mag : mag;
    }
}

// ------------------------------------------------------------------------------------------------
// SWAR sum decoder under a row mask (delta_page_sum_masked in scan_kernels.cu): SUM / MEAN / COUNT over the ACTIVE rows only.
//     sum over active rows r of value_r  =  A * first + sum_j d_j * W_j ,   W_j = number of active rows >= j,
// so the byte weights of the all-rows decoder,  (n - 1) - #terminators before the byte,  become
//     (A - a_0) - #ACTIVE terminators before the byte
// (A = active rows, a_0 = row 0 active): the same dot products with the rank taken over active terminators only.  The lane
// brings the activity of the rows that end in it as a bit string (bit i = i-th terminator of the lane is an active row); per
// word the next <= 4 bits are deposited onto the word's terminator bytes with one byte gather (PRMT): byte j takes bit e_j of
// the nibble, e_j = terminators before byte j inside the word.
// ------------------------------------------------------------------------------------------------
struct SwarMasked {
    int32_t T0, T1, T2, R0, R1, R2;
    uint32_t wide, guard;  // as in SwarLane
    int32_t nact;      // 1 + ACTIVE terminators seen so far in this lane
    uint32_t prev_w;
    uint32_t aw_lo, aw_hi;  // activity bits of the terminators still to come in this lane
};
BYDB_LANE_FN void swar_masked_begin(SwarMasked &s, uint32_t prev_w, uint32_t aw_lo, uint32_t aw_hi) {
    s.T0 = s.T1 = s.T2 = s.R0 = s.R1 = s.R2 = 0;
    s.wide = s.guard = 0;
    s.nact = 1;
    s.prev_w = prev_w;
    s.aw_lo = aw_lo;
    s.aw_hi = aw_hi;
}
// kTwoClass: as in swar_word.
template <bool kMasked, bool kTwoClass = false>
BYDB_LANE_FN void swar_masked_word(SwarMasked &s, uint32_t w_in, uint32_t vm) {
    const uint32_t w = kMasked ? (w_in & vm) : w_in;
    const uint32_t pw = s.prev_w;
    const uint32_t p = w & 0x7f7f7f7fu;
    const uint32_t M1 = lane_prmt(w, pw, 0xA98Fu);
    const uint32_t sb = imad_u32(w, 128u, 0u);
    const uint32_t psb = imad_u32(pw, 128u, 0u);
    const uint32_t S0 = lane_prmt(sb, 0u, 0xBA98u);
    const uint32_t S1 = lane_prmt(sb, psb, 0xA98Fu);
    const uint32_t x0 = (p ^ S0) & ~M1;
    uint32_t p1, S12, q2 = 0;
    if (kTwoClass) {
        p1 = p & M1;
        S12 = S1;
        s.guard |= w & M1;
    } else {
        const uint32_t M2 = lane_prmt(w, pw, 0x98FEu);
        const uint32_t S2 = lane_prmt(sb, psb, 0x98FEu);
        S12 = (M2 & S2) | (~M2 & S1);
        p1 = p & M1 & ~M2;
        q2 = w & M1 & M2;
    }
    const uint32_t wT = S12 | 0x01010101u;
    uint32_t t01 = ~mulhi_u32(w, 1u << 25) & 0x01010101u;  // 1 where the byte terminates a varint
    if (kMasked) t01 &= vm;
    // ---- the word's terminators that are active rows: byte j <- bit e_j of the next activity bits
    const uint32_t e = imad_u32(t01, 0x01010100u, 0u);                  // byte j = terminators before byte j inside the word (0..3)
    const uint32_t a4 = imad_u32(s.aw_lo & 15u, 0x00204081u, 0u) & 0x01010101u;  // bits 0..3 of the activity string as four 0/1 bytes
    // the e_j (<= 3 each) as selector nibbles: x = e | e >> 4 holds (e_0, e_1) in byte 0 and (e_2, e_3) in byte 2
    const uint32_t sel = lane_prmt(e | (e >> 4), 0u, 0x4420u);
    const uint32_t a01 = lane_prmt(a4, 0u, sel) & t01;                  // 1 where an ACTIVE row ends
    const uint32_t ntw = (e >> 24) + (t01 >> 24);                       // terminators in this word (bytes 0..2, plus byte 3)
    // shift the activity string by the terminators consumed (<= 4)
    const uint64_t aw = ((static_cast<uint64_t>(s.aw_hi) << 32) | s.aw_lo) >> ntw;
    s.aw_lo = static_cast<uint32_t>(aw);
    s.aw_hi = static_cast<uint32_t>(aw >> 32);
    const uint32_t base = imad_u32(static_cast<uint32_t>(s.nact), 0x01010101u, 0u);
    const uint32_t rinc = imad_u32(a01, 0x01010101u, base);    // inclusive active count + 1
    const uint32_t rank1 = imad_u32(a01, 0xffffffffu, rinc);   // exclusive active count + 1
    s.nact = dp4a_su(0x01010101u, a01, s.nact);
    const uint32_t wR = imad_u32(S12 & 0x01010101u, 1u, rank1 ^ S12);
    s.T0 = dp4a_su(x0, 0x01010101u, s.T0);
    s.R0 = dp4a_su(x0, rank1, s.R0);
    s.T1 = dp4a_us(p1, wT, s.T1);
    s.R1 = dp4a_us(p1, wR, s.R1);
    if (!kTwoClass) {
        s.T2 = dp4a_us(q2, wT, s.T2);
        s.R2 = dp4a_us(q2, wR, s.R2);
        s.wide |= q2;
    }
    s.prev_w = w;
}
// -> ACTIVE terminators of the lane; T and R' (active ranks)
BYDB_LANE_FN uint32_t swar_masked_end(const SwarMasked &s, int32_t &T, int32_t &Rp) {
    T = (s.T0 >> 1) + 64 * s.T1 + 8192 * s.T2;
    Rp = (s.R0 >> 1) + 64 * s.R1 + 8192 * s.R2;
    return static_cast<uint32_t>(s.nact - 1);
}
// terminators among the 64 bytes of a lane (first pass: the lanes' row offsets must be known before the activity bits can be cut)
BYDB_LANE_FN uint32_t count_terminators(uint32_t w, uint32_t vm) { return lane_popc(~w & 0x80808080u & vm); }

// 4 bits -> 4 byte masks (bit j -> 0xff in byte j): bit j times 2^(7j) lands on bit 8j, nothing else does
BYDB_LANE_FN uint32_t expand4(uint32_t n) { return (((n & 0xfu) * 0x00204081u) & 0x01010101u) * 0xffu; }

template <bool kFull, int kNeed>
BYDB_LANE_FN void fast_lane_decode(const uint4 &wa, const uint4 &wb, uint32_t valid, uint32_t term, uint32_t aw, uint32_t &accv,
                                                 uint32_t &sh, int32_t &P, int32_t &sumP, int32_t &minP, int32_t &maxP) {
    if (kFull) {
        fast_lane_decode_imad<kNeed, false>(wa, wb, term, term, aw, accv, sh, P, sumP, minP, maxP);
    } else {
        const uint4 ma = make_uint4(wa.x & expand4(valid), wa.y & expand4(valid >> 4), wa.z & expand4(valid >> 8), wa.w & expand4(valid >> 12));
        const uint4 mb = make_uint4(wb.x & expand4(valid >> 16), wb.y & expand4(valid >> 20), wb.z & expand4(valid >> 24), wb.w & expand4(valid >> 28));
        fast_lane_decode_imad<kNeed, true>(ma, mb, term, term | ~valid, aw, accv, sh, P, sumP, minP, maxP);
    }
}

// what the previous lane's unfinished tail adds to this lane's first value (narrow mode: the value's own
// bytes are the first <= 3 bytes of the lane, its low bits are prev_acc)
BYDB_LANE_FN int32_t head_delta(uint32_t w0, uint32_t term, uint32_t prev_acc, uint32_t prev_sh) {
    const uint32_t fp = static_cast<uint32_t>(lane_ffs(term) - 1);                 // <= 2
    const uint32_t x = w0 & (0xffffffu >> (8u * (2u - fp)));                     // bytes 0..fp
    const uint32_t hx = (x & 0x7fu) | ((x >> 1) & 0x3f80u) | ((x >> 2) & 0x1fc000u);
    const uint32_t full = prev_acc | (hx << prev_sh);
    const int32_t v_true = static_cast<int32_t>(full >> 1) ^ -static_cast<int32_t>(full & 1u);
    const int32_t v_own = static_cast<int32_t>(hx >> 1) ^ -static_cast<int32_t>(hx & 1u);
    return v_true - v_own;
}


}  // namespace bydb
