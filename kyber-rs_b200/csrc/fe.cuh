// fe.cuh — GF(2^255-19) arithmetic for sm_100a: 8 saturated 32-bit limbs, products built
// from IMAD.WIDE.U32(.X) carry chains (PTX mad.lo.cc / madc.hi.cc pairs, which ptxas fuses).
//
// Replaces the reference's field layer src/group/edwards25519/fe.rs (10 signed 25.5-bit limbs,
// i64 products).  Internal limb values are NOT the reference's; only what is observable
// through fe_to_bytes / fe_is_negative / fe_is_zero has to match (SURVEY §A4), and does.
//
// Representation invariant: an fe is any integer in [0, 2^256) congruent to the field
// element mod p = 2^255-19 ("loosely reduced").  Every routine accepts and returns that.
//
// The same source compiles as plain host C++ when KB_HOST_EMU is defined; that build exists
// ONLY so tests/ can exercise the per-thread math on a machine without a GPU.  The product
// library never contains it (see csrc/Makefile) and has no CPU code path.
#pragma once
#include <stdint.h>

#if defined(KB_HOST_EMU)
#define KB_FN static inline
#define KB_UNROLL
#define KB_NOUNROLL
#else
#define KB_FN __device__ __forceinline__
#define KB_UNROLL _Pragma("unroll")
#define KB_NOUNROLL _Pragma("unroll 1")
#endif

struct fe {
    uint32_t v[8];
};

// ---------------------------------------------------------------------------------------
// carry-chain primitives
// ---------------------------------------------------------------------------------------

// acc[0..7] += {a0,a1,a2,a3} * b, product k landing on the word pair (2k, 2k+1); the carry
// out of word 7 is added to `top`.  8 PTX mads -> 4 IMAD.WIDE.U32.X.
KB_FN void kb_cmad4(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b, uint32_t& top)
{
#if defined(KB_HOST_EMU)
    const uint32_t a[4] = {a0, a1, a2, a3};
    uint64_t carry = 0;
    for (int k = 0; k < 4; k++) {
        uint64_t p = (uint64_t)a[k] * b;
        uint64_t lo = (uint64_t)acc[2 * k] + (uint32_t)p + carry;
        acc[2 * k] = (uint32_t)lo;
        uint64_t hi = (uint64_t)acc[2 * k + 1] + (p >> 32) + (lo >> 32);
        acc[2 * k + 1] = (uint32_t)hi;
        carry = hi >> 32;
    }
    top += (uint32_t)carry;
#else
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, %8, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(top)
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
#endif
}

// Two variants for rows whose surroundings are known to be FRESH words, so that no accumulator register has to be
// zeroed beforehand and no needless carry is captured (ptxas places both kinds of instruction on the multiplier pipe):
// kb_cmad4_top: like kb_cmad4, but `top` is a fresh word — it RECEIVES the carry out of word 7 (0 or 1).
KB_FN void kb_cmad4_top(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b, uint32_t& top)
{
#if defined(KB_HOST_EMU)
    top = 0;
    kb_cmad4(acc, a0, a1, a2, a3, b, top);
#else
    asm("mad.lo.cc.u32 %0, %9, %13, %0;\n\t"
        "madc.hi.cc.u32 %1, %9, %13, %1;\n\t"
        "madc.lo.cc.u32 %2, %10, %13, %2;\n\t"
        "madc.hi.cc.u32 %3, %10, %13, %3;\n\t"
        "madc.lo.cc.u32 %4, %11, %13, %4;\n\t"
        "madc.hi.cc.u32 %5, %11, %13, %5;\n\t"
        "madc.lo.cc.u32 %6, %12, %13, %6;\n\t"
        "madc.hi.cc.u32 %7, %12, %13, %7;\n\t"
        "addc.u32 %8, 0, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "=r"(top)
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
#endif
}
// kb_cmad4_hi: like kb_cmad4, but word 7 is a fresh word (it receives the high half of the last product plus the
// carry, which cannot overflow) and nothing is carried further.
KB_FN void kb_cmad4_hi(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    acc[7] = 0;
    kb_cmad4(acc, a0, a1, a2, a3, b, top);
#else
    asm("mad.lo.cc.u32 %0, %8, %12, %0;\n\t"
        "madc.hi.cc.u32 %1, %8, %12, %1;\n\t"
        "madc.lo.cc.u32 %2, %9, %12, %2;\n\t"
        "madc.hi.cc.u32 %3, %9, %12, %3;\n\t"
        "madc.lo.cc.u32 %4, %10, %12, %4;\n\t"
        "madc.hi.cc.u32 %5, %10, %12, %5;\n\t"
        "madc.lo.cc.u32 %6, %11, %12, %6;\n\t"
        "madc.hi.u32 %7, %11, %12, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "=r"(acc[7])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
#endif
}

// Same, for N = 1..3 products (used by the squaring's triangular rows).
KB_FN void kb_cmad3(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t b, uint32_t& top)
{
#if defined(KB_HOST_EMU)
    const uint32_t a[3] = {a0, a1, a2};
    uint64_t carry = 0;
    for (int k = 0; k < 3; k++) {
        uint64_t p = (uint64_t)a[k] * b;
        uint64_t lo = (uint64_t)acc[2 * k] + (uint32_t)p + carry;
        acc[2 * k] = (uint32_t)lo;
        uint64_t hi = (uint64_t)acc[2 * k + 1] + (p >> 32) + (lo >> 32);
        acc[2 * k + 1] = (uint32_t)hi;
        carry = hi >> 32;
    }
    top += (uint32_t)carry;
#else
    asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t"
        "madc.hi.cc.u32 %1, %7, %10, %1;\n\t"
        "madc.lo.cc.u32 %2, %8, %10, %2;\n\t"
        "madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "madc.lo.cc.u32 %4, %9, %10, %4;\n\t"
        "madc.hi.cc.u32 %5, %9, %10, %5;\n\t"
        "addc.u32 %6, %6, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(top)
        : "r"(a0), "r"(a1), "r"(a2), "r"(b));
#endif
}
KB_FN void kb_cmad2(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t b, uint32_t& top)
{
#if defined(KB_HOST_EMU)
    const uint32_t a[2] = {a0, a1};
    uint64_t carry = 0;
    for (int k = 0; k < 2; k++) {
        uint64_t p = (uint64_t)a[k] * b;
        uint64_t lo = (uint64_t)acc[2 * k] + (uint32_t)p + carry;
        acc[2 * k] = (uint32_t)lo;
        uint64_t hi = (uint64_t)acc[2 * k + 1] + (p >> 32) + (lo >> 32);
        acc[2 * k + 1] = (uint32_t)hi;
        carry = hi >> 32;
    }
    top += (uint32_t)carry;
#else
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t"
        "madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %7, %2;\n\t"
        "madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, %4, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(top)
        : "r"(a0), "r"(a1), "r"(b));
#endif
}
KB_FN void kb_cmad1(uint32_t* acc, uint32_t a0, uint32_t b, uint32_t& top)
{
#if defined(KB_HOST_EMU)
    uint64_t p = (uint64_t)a0 * b;
    uint64_t lo = (uint64_t)acc[0] + (uint32_t)p;
    acc[0] = (uint32_t)lo;
    uint64_t hi = (uint64_t)acc[1] + (p >> 32) + (lo >> 32);
    acc[1] = (uint32_t)hi;
    top += (uint32_t)(hi >> 32);
#else
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t"
        "madc.hi.cc.u32 %1, %3, %4, %1;\n\t"
        "addc.u32 %2, %2, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(top)
        : "r"(a0), "r"(b));
#endif
}

// the same two fresh-word variants (see kb_cmad4_top / kb_cmad4_hi) for the squaring's triangular rows
KB_FN void kb_cmad3_top(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t b, uint32_t& top)
{
#if defined(KB_HOST_EMU)
    top = 0;
    kb_cmad3(acc, a0, a1, a2, b, top);
#else
    asm("mad.lo.cc.u32 %0, %7, %10, %0;\n\t"
        "madc.hi.cc.u32 %1, %7, %10, %1;\n\t"
        "madc.lo.cc.u32 %2, %8, %10, %2;\n\t"
        "madc.hi.cc.u32 %3, %8, %10, %3;\n\t"
        "madc.lo.cc.u32 %4, %9, %10, %4;\n\t"
        "madc.hi.cc.u32 %5, %9, %10, %5;\n\t"
        "addc.u32 %6, 0, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "=r"(top)
        : "r"(a0), "r"(a1), "r"(a2), "r"(b));
#endif
}
KB_FN void kb_cmad3_hi(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t b)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    acc[5] = 0;
    kb_cmad3(acc, a0, a1, a2, b, top);
#else
    asm("mad.lo.cc.u32 %0, %6, %9, %0;\n\t"
        "madc.hi.cc.u32 %1, %6, %9, %1;\n\t"
        "madc.lo.cc.u32 %2, %7, %9, %2;\n\t"
        "madc.hi.cc.u32 %3, %7, %9, %3;\n\t"
        "madc.lo.cc.u32 %4, %8, %9, %4;\n\t"
        "madc.hi.u32 %5, %8, %9, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "=r"(acc[5])
        : "r"(a0), "r"(a1), "r"(a2), "r"(b));
#endif
}
KB_FN void kb_cmad2_top(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t b, uint32_t& top)
{
#if defined(KB_HOST_EMU)
    top = 0;
    kb_cmad2(acc, a0, a1, b, top);
#else
    asm("mad.lo.cc.u32 %0, %5, %7, %0;\n\t"
        "madc.hi.cc.u32 %1, %5, %7, %1;\n\t"
        "madc.lo.cc.u32 %2, %6, %7, %2;\n\t"
        "madc.hi.cc.u32 %3, %6, %7, %3;\n\t"
        "addc.u32 %4, 0, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "=r"(top)
        : "r"(a0), "r"(a1), "r"(b));
#endif
}
KB_FN void kb_cmad2_hi(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t b)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    acc[3] = 0;
    kb_cmad2(acc, a0, a1, b, top);
#else
    asm("mad.lo.cc.u32 %0, %4, %6, %0;\n\t"
        "madc.hi.cc.u32 %1, %4, %6, %1;\n\t"
        "madc.lo.cc.u32 %2, %5, %6, %2;\n\t"
        "madc.hi.u32 %3, %5, %6, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "=r"(acc[3])
        : "r"(a0), "r"(a1), "r"(b));
#endif
}
KB_FN void kb_cmad1_top(uint32_t* acc, uint32_t a0, uint32_t b, uint32_t& top)
{
#if defined(KB_HOST_EMU)
    top = 0;
    kb_cmad1(acc, a0, b, top);
#else
    asm("mad.lo.cc.u32 %0, %3, %4, %0;\n\t"
        "madc.hi.cc.u32 %1, %3, %4, %1;\n\t"
        "addc.u32 %2, 0, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "=r"(top)
        : "r"(a0), "r"(b));
#endif
}
KB_FN void kb_cmad1_hi(uint32_t* acc, uint32_t a0, uint32_t b)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    acc[1] = 0;
    kb_cmad1(acc, a0, b, top);
#else
    asm("mad.lo.cc.u32 %0, %2, %3, %0;\n\t"
        "madc.hi.u32 %1, %2, %3, 0;"
        : "+r"(acc[0]), "=r"(acc[1])
        : "r"(a0), "r"(b));
#endif
}

// acc[0..2N) = {a0, ...} * b on FRESH word pairs: N independent IMAD.WIDE.U32 with no addend — no zeroed
// accumulator registers to set up, no carry chain, no carry to capture (used for the first row of a product)
KB_FN void kb_cmul4(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b)
{
    const uint64_t p0 = (uint64_t)a0 * b, p1 = (uint64_t)a1 * b, p2 = (uint64_t)a2 * b, p3 = (uint64_t)a3 * b;
    acc[0] = (uint32_t)p0; acc[1] = (uint32_t)(p0 >> 32);
    acc[2] = (uint32_t)p1; acc[3] = (uint32_t)(p1 >> 32);
    acc[4] = (uint32_t)p2; acc[5] = (uint32_t)(p2 >> 32);
    acc[6] = (uint32_t)p3; acc[7] = (uint32_t)(p3 >> 32);
}
KB_FN void kb_cmul3(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t b)
{
    const uint64_t p0 = (uint64_t)a0 * b, p1 = (uint64_t)a1 * b, p2 = (uint64_t)a2 * b;
    acc[0] = (uint32_t)p0; acc[1] = (uint32_t)(p0 >> 32);
    acc[2] = (uint32_t)p1; acc[3] = (uint32_t)(p1 >> 32);
    acc[4] = (uint32_t)p2; acc[5] = (uint32_t)(p2 >> 32);
}

// ---------------------------------------------------------------------------------------
// Rows whose top pair is FRESH, and rows that ripple their carry into an EXISTING pair.
// An IMAD.WIDE adds a 64-bit addend held in a register PAIR.  When a row ends on (a word holding a captured carry,
// a fresh word), ptxas has to materialise the fresh half as a zeroed register — one IMAD.MOV per row, on the
// multiplier pipe (ncu, round 2: 46 of the 78 register zeroings of the verify loop).  Ordering the rows so that the
// row which CREATES a pair runs first (its top pair is completely fresh: addend RZ) and the row below it then
// ripples its carry into that existing pair (two IADD3.X on the ALU pipe) needs no zeroed registers at all.
// ---------------------------------------------------------------------------------------
// acc[0..2(N-1)) += {a..} * b on existing pairs; the top pair (acc[2N-2], acc[2N-1]) is fresh: it takes the last
// product plus the carry (cannot overflow)
KB_FN void kb_cmad4_new(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    acc[6] = acc[7] = 0;
    kb_cmad4(acc, a0, a1, a2, a3, b, top);
#else
    asm("mad.lo.cc.u32 %0, %8, %12, %0;\n\t"
        "madc.hi.cc.u32 %1, %8, %12, %1;\n\t"
        "madc.lo.cc.u32 %2, %9, %12, %2;\n\t"
        "madc.hi.cc.u32 %3, %9, %12, %3;\n\t"
        "madc.lo.cc.u32 %4, %10, %12, %4;\n\t"
        "madc.hi.cc.u32 %5, %10, %12, %5;\n\t"
        "madc.lo.cc.u32 %6, %11, %12, 0;\n\t"
        "madc.hi.u32 %7, %11, %12, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "=r"(acc[6]), "=r"(acc[7])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
#endif
}
KB_FN void kb_cmad3_new(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t b)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    acc[4] = acc[5] = 0;
    kb_cmad3(acc, a0, a1, a2, b, top);
#else
    asm("mad.lo.cc.u32 %0, %6, %9, %0;\n\t"
        "madc.hi.cc.u32 %1, %6, %9, %1;\n\t"
        "madc.lo.cc.u32 %2, %7, %9, %2;\n\t"
        "madc.hi.cc.u32 %3, %7, %9, %3;\n\t"
        "madc.lo.cc.u32 %4, %8, %9, 0;\n\t"
        "madc.hi.u32 %5, %8, %9, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "=r"(acc[4]), "=r"(acc[5])
        : "r"(a0), "r"(a1), "r"(a2), "r"(b));
#endif
}
KB_FN void kb_cmad2_new(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t b)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    acc[2] = acc[3] = 0;
    kb_cmad2(acc, a0, a1, b, top);
#else
    asm("mad.lo.cc.u32 %0, %4, %6, %0;\n\t"
        "madc.hi.cc.u32 %1, %4, %6, %1;\n\t"
        "madc.lo.cc.u32 %2, %5, %6, 0;\n\t"
        "madc.hi.u32 %3, %5, %6, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "=r"(acc[2]), "=r"(acc[3])
        : "r"(a0), "r"(a1), "r"(b));
#endif
}
// acc[0..2N) += {a..} * b on existing pairs; the carry out ripples into the existing pair (r0, r1) above them
// (callers guarantee it cannot leave r1)
KB_FN void kb_cmad4_rip(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b, uint32_t& r0, uint32_t& r1)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    kb_cmad4(acc, a0, a1, a2, a3, b, top);
    const uint64_t c = (uint64_t)r0 + top;
    r0 = (uint32_t)c;
    r1 += (uint32_t)(c >> 32);
#else
    asm("mad.lo.cc.u32 %0, %10, %14, %0;\n\t"
        "madc.hi.cc.u32 %1, %10, %14, %1;\n\t"
        "madc.lo.cc.u32 %2, %11, %14, %2;\n\t"
        "madc.hi.cc.u32 %3, %11, %14, %3;\n\t"
        "madc.lo.cc.u32 %4, %12, %14, %4;\n\t"
        "madc.hi.cc.u32 %5, %12, %14, %5;\n\t"
        "madc.lo.cc.u32 %6, %13, %14, %6;\n\t"
        "madc.hi.cc.u32 %7, %13, %14, %7;\n\t"
        "addc.cc.u32 %8, %8, 0;\n\t"
        "addc.u32 %9, %9, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(r0), "+r"(r1)
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b));
#endif
}
KB_FN void kb_cmad3_rip(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t b, uint32_t& r0, uint32_t& r1)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    kb_cmad3(acc, a0, a1, a2, b, top);
    const uint64_t c = (uint64_t)r0 + top;
    r0 = (uint32_t)c;
    r1 += (uint32_t)(c >> 32);
#else
    asm("mad.lo.cc.u32 %0, %8, %11, %0;\n\t"
        "madc.hi.cc.u32 %1, %8, %11, %1;\n\t"
        "madc.lo.cc.u32 %2, %9, %11, %2;\n\t"
        "madc.hi.cc.u32 %3, %9, %11, %3;\n\t"
        "madc.lo.cc.u32 %4, %10, %11, %4;\n\t"
        "madc.hi.cc.u32 %5, %10, %11, %5;\n\t"
        "addc.cc.u32 %6, %6, 0;\n\t"
        "addc.u32 %7, %7, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(r0), "+r"(r1)
        : "r"(a0), "r"(a1), "r"(a2), "r"(b));
#endif
}
KB_FN void kb_cmad2_rip(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t b, uint32_t& r0, uint32_t& r1)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    kb_cmad2(acc, a0, a1, b, top);
    const uint64_t c = (uint64_t)r0 + top;
    r0 = (uint32_t)c;
    r1 += (uint32_t)(c >> 32);
#else
    asm("mad.lo.cc.u32 %0, %6, %8, %0;\n\t"
        "madc.hi.cc.u32 %1, %6, %8, %1;\n\t"
        "madc.lo.cc.u32 %2, %7, %8, %2;\n\t"
        "madc.hi.cc.u32 %3, %7, %8, %3;\n\t"
        "addc.cc.u32 %4, %4, 0;\n\t"
        "addc.u32 %5, %5, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(r0), "+r"(r1)
        : "r"(a0), "r"(a1), "r"(b));
#endif
}
KB_FN void kb_cmad1_rip(uint32_t* acc, uint32_t a0, uint32_t b, uint32_t& r0, uint32_t& r1)
{
#if defined(KB_HOST_EMU)
    uint32_t top = 0;
    kb_cmad1(acc, a0, b, top);
    const uint64_t c = (uint64_t)r0 + top;
    r0 = (uint32_t)c;
    r1 += (uint32_t)(c >> 32);
#else
    asm("mad.lo.cc.u32 %0, %4, %5, %0;\n\t"
        "madc.hi.cc.u32 %1, %4, %5, %1;\n\t"
        "addc.cc.u32 %2, %2, 0;\n\t"
        "addc.u32 %3, %3, 0;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(r0), "+r"(r1)
        : "r"(a0), "r"(b));
#endif
}
KB_FN void kb_cmul1(uint32_t* acc, uint32_t a0, uint32_t b)
{
    const uint64_t p0 = (uint64_t)a0 * b;
    acc[0] = (uint32_t)p0; acc[1] = (uint32_t)(p0 >> 32);
}
// The merge of the squaring's two column sets, doubled:  t[1..16) = 2 * (ev[1..16) + od[0..15))  where ev[0] = ev[1] =
// ev[14] = ev[15] = od[14] = 0 are never materialised (t[1] = 2 od[0], t[14] = 2 (od[13] + carry), ...).  t[0] is not
// written (it is 0).
KB_FN void kb_sq_merge_dbl(uint32_t* t, const uint32_t* ev, const uint32_t* od)
{
#if defined(KB_HOST_EMU)
    uint32_t m[16];
    uint64_t c = 0;
    m[1] = od[0];
    for (int i = 2; i <= 13; i++) {
        c += (uint64_t)ev[i] + od[i - 1];
        m[i] = (uint32_t)c;
        c >>= 32;
    }
    c += od[13];
    m[14] = (uint32_t)c;
    m[15] = (uint32_t)(c >> 32);
    uint32_t cy = 0;
    for (int i = 1; i < 16; i++) {
        const uint32_t n = m[i] >> 31;
        t[i] = (m[i] << 1) | cy;
        cy = n;
    }
#else
    uint32_t m2, m3, m4, m5, m6, m7, m8, m9, m10, m11, m12, m13, m14, m15;
    asm("add.cc.u32 %0, %14, %26;\n\t"
        "addc.cc.u32 %1, %15, %27;\n\t"
        "addc.cc.u32 %2, %16, %28;\n\t"
        "addc.cc.u32 %3, %17, %29;\n\t"
        "addc.cc.u32 %4, %18, %30;\n\t"
        "addc.cc.u32 %5, %19, %31;\n\t"
        "addc.cc.u32 %6, %20, %32;\n\t"
        "addc.cc.u32 %7, %21, %33;\n\t"
        "addc.cc.u32 %8, %22, %34;\n\t"
        "addc.cc.u32 %9, %23, %35;\n\t"
        "addc.cc.u32 %10, %24, %36;\n\t"
        "addc.cc.u32 %11, %25, %37;\n\t"
        "addc.cc.u32 %12, %38, 0;\n\t"
        "addc.u32 %13, 0, 0;"
        : "=&r"(m2), "=&r"(m3), "=&r"(m4), "=&r"(m5), "=&r"(m6), "=&r"(m7), "=&r"(m8), "=&r"(m9), "=&r"(m10), "=&r"(m11), "=&r"(m12), "=&r"(m13), "=&r"(m14), "=&r"(m15)
        : "r"(ev[2]), "r"(ev[3]), "r"(ev[4]), "r"(ev[5]), "r"(ev[6]), "r"(ev[7]), "r"(ev[8]), "r"(ev[9]), "r"(ev[10]), "r"(ev[11]), "r"(ev[12]), "r"(ev[13]),
          "r"(od[1]), "r"(od[2]), "r"(od[3]), "r"(od[4]), "r"(od[5]), "r"(od[6]), "r"(od[7]), "r"(od[8]), "r"(od[9]), "r"(od[10]), "r"(od[11]), "r"(od[12]), "r"(od[13]));
    asm("add.cc.u32 %0, %15, %15;\n\t"
        "addc.cc.u32 %1, %16, %16;\n\t"
        "addc.cc.u32 %2, %17, %17;\n\t"
        "addc.cc.u32 %3, %18, %18;\n\t"
        "addc.cc.u32 %4, %19, %19;\n\t"
        "addc.cc.u32 %5, %20, %20;\n\t"
        "addc.cc.u32 %6, %21, %21;\n\t"
        "addc.cc.u32 %7, %22, %22;\n\t"
        "addc.cc.u32 %8, %23, %23;\n\t"
        "addc.cc.u32 %9, %24, %24;\n\t"
        "addc.cc.u32 %10, %25, %25;\n\t"
        "addc.cc.u32 %11, %26, %26;\n\t"
        "addc.cc.u32 %12, %27, %27;\n\t"
        "addc.cc.u32 %13, %28, %28;\n\t"
        "addc.u32 %14, %29, %29;"
        : "=&r"(t[1]), "=&r"(t[2]), "=&r"(t[3]), "=&r"(t[4]), "=&r"(t[5]), "=&r"(t[6]), "=&r"(t[7]), "=&r"(t[8]), "=&r"(t[9]), "=&r"(t[10]), "=&r"(t[11]), "=&r"(t[12]), "=&r"(t[13]), "=&r"(t[14]), "=&r"(t[15])
        : "r"(od[0]), "r"(m2), "r"(m3), "r"(m4), "r"(m5), "r"(m6), "r"(m7), "r"(m8), "r"(m9), "r"(m10), "r"(m11), "r"(m12), "r"(m13), "r"(m14), "r"(m15));
#endif
}
// acc[0..15) += x[0..15) (no carry out: callers guarantee it fits)
KB_FN void kb_acc15(uint32_t* acc, const uint32_t* x)
{
#if defined(KB_HOST_EMU)
    uint64_t c = 0;
    for (int i = 0; i < 15; i++) {
        c += (uint64_t)acc[i] + x[i];
        acc[i] = (uint32_t)c;
        c >>= 32;
    }
#else
    asm("add.cc.u32 %0, %0, %15;\n\t"
        "addc.cc.u32 %1, %1, %16;\n\t"
        "addc.cc.u32 %2, %2, %17;\n\t"
        "addc.cc.u32 %3, %3, %18;\n\t"
        "addc.cc.u32 %4, %4, %19;\n\t"
        "addc.cc.u32 %5, %5, %20;\n\t"
        "addc.cc.u32 %6, %6, %21;\n\t"
        "addc.cc.u32 %7, %7, %22;\n\t"
        "addc.cc.u32 %8, %8, %23;\n\t"
        "addc.cc.u32 %9, %9, %24;\n\t"
        "addc.cc.u32 %10, %10, %25;\n\t"
        "addc.cc.u32 %11, %11, %26;\n\t"
        "addc.cc.u32 %12, %12, %27;\n\t"
        "addc.cc.u32 %13, %13, %28;\n\t"
        "addc.u32 %14, %14, %29;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7]), "+r"(acc[8]), "+r"(acc[9]), "+r"(acc[10]), "+r"(acc[11]), "+r"(acc[12]), "+r"(acc[13]), "+r"(acc[14])
        : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(x[3]), "r"(x[4]), "r"(x[5]), "r"(x[6]), "r"(x[7]), "r"(x[8]), "r"(x[9]), "r"(x[10]), "r"(x[11]), "r"(x[12]), "r"(x[13]), "r"(x[14]));
#endif
}
// acc[0..8) += x[0..8) (no carry out: callers guarantee it fits)
KB_FN void kb_acc8(uint32_t* acc, const uint32_t* x)
{
#if defined(KB_HOST_EMU)
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) {
        c += (uint64_t)acc[i] + x[i];
        acc[i] = (uint32_t)c;
        c >>= 32;
    }
#else
    asm("add.cc.u32 %0, %0, %8;\n\t"
        "addc.cc.u32 %1, %1, %9;\n\t"
        "addc.cc.u32 %2, %2, %10;\n\t"
        "addc.cc.u32 %3, %3, %11;\n\t"
        "addc.cc.u32 %4, %4, %12;\n\t"
        "addc.cc.u32 %5, %5, %13;\n\t"
        "addc.cc.u32 %6, %6, %14;\n\t"
        "addc.u32 %7, %7, %15;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6]), "+r"(acc[7])
        : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(x[3]), "r"(x[4]), "r"(x[5]), "r"(x[6]), "r"(x[7]));
#endif
}
// t[0..16) <<= 1 (top bit must be clear)
KB_FN void kb_dbl16(uint32_t* t)
{
#if defined(KB_HOST_EMU)
    uint32_t c = 0;
    for (int i = 0; i < 16; i++) {
        uint32_t n = t[i] >> 31;
        t[i] = (t[i] << 1) | c;
        c = n;
    }
#else
    asm("add.cc.u32 %0, %0, %0;\n\t"
        "addc.cc.u32 %1, %1, %1;\n\t"
        "addc.cc.u32 %2, %2, %2;\n\t"
        "addc.cc.u32 %3, %3, %3;\n\t"
        "addc.cc.u32 %4, %4, %4;\n\t"
        "addc.cc.u32 %5, %5, %5;\n\t"
        "addc.cc.u32 %6, %6, %6;\n\t"
        "addc.cc.u32 %7, %7, %7;\n\t"
        "addc.cc.u32 %8, %8, %8;\n\t"
        "addc.cc.u32 %9, %9, %9;\n\t"
        "addc.cc.u32 %10, %10, %10;\n\t"
        "addc.cc.u32 %11, %11, %11;\n\t"
        "addc.cc.u32 %12, %12, %12;\n\t"
        "addc.cc.u32 %13, %13, %13;\n\t"
        "addc.cc.u32 %14, %14, %14;\n\t"
        "addc.u32 %15, %15, %15;"
        : "+r"(t[0]), "+r"(t[1]), "+r"(t[2]), "+r"(t[3]), "+r"(t[4]), "+r"(t[5]), "+r"(t[6]), "+r"(t[7]), "+r"(t[8]), "+r"(t[9]), "+r"(t[10]), "+r"(t[11]), "+r"(t[12]), "+r"(t[13]), "+r"(t[14]), "+r"(t[15]));
#endif
}
// r = a + b over 8 words (each asm chain is ONE statement so the compiler cannot split it); returns the carry
KB_FN uint32_t kb_add8(uint32_t* r, const uint32_t* a, const uint32_t* b)
{
#if defined(KB_HOST_EMU)
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) {
        c += (uint64_t)a[i] + b[i];
        r[i] = (uint32_t)c;
        c >>= 32;
    }
    return (uint32_t)c;
#else
    uint32_t t[8], c;
    asm("add.cc.u32 %0, %9, %17;\n\t"
        "addc.cc.u32 %1, %10, %18;\n\t"
        "addc.cc.u32 %2, %11, %19;\n\t"
        "addc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\t"
        "addc.cc.u32 %5, %14, %22;\n\t"
        "addc.cc.u32 %6, %15, %23;\n\t"
        "addc.cc.u32 %7, %16, %24;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=&r"(t[0]), "=&r"(t[1]), "=&r"(t[2]), "=&r"(t[3]), "=&r"(t[4]), "=&r"(t[5]), "=&r"(t[6]), "=&r"(t[7]), "=&r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    KB_UNROLL
    for (int i = 0; i < 8; i++) r[i] = t[i];
    return c & 1;
#endif
}
// r = a - b over 8 words; returns the borrow (0/1)
KB_FN uint32_t kb_sub8(uint32_t* r, const uint32_t* a, const uint32_t* b)
{
#if defined(KB_HOST_EMU)
    uint64_t br = 0;
    for (int i = 0; i < 8; i++) {
        uint64_t d = (uint64_t)a[i] - b[i] - br;
        r[i] = (uint32_t)d;
        br = (d >> 32) & 1;
    }
    return (uint32_t)br;
#else
    uint32_t t[8], c;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(t[0]), "=&r"(t[1]), "=&r"(t[2]), "=&r"(t[3]), "=&r"(t[4]), "=&r"(t[5]), "=&r"(t[6]), "=&r"(t[7]), "=&r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    KB_UNROLL
    for (int i = 0; i < 8; i++) r[i] = t[i];
    return c & 1;
#endif
}
// r = a - b over 8 words; returns the borrow as a MASK (0 / 0xffffffff): `mask & 38` is one ALU instruction where
// `38 * borrow` is an IMAD on the multiplier pipe
KB_FN uint32_t kb_sub8m(uint32_t* r, const uint32_t* a, const uint32_t* b)
{
#if defined(KB_HOST_EMU)
    return 0u - kb_sub8(r, a, b);
#else
    uint32_t t[8], c;
    asm("sub.cc.u32 %0, %9, %17;\n\t"
        "subc.cc.u32 %1, %10, %18;\n\t"
        "subc.cc.u32 %2, %11, %19;\n\t"
        "subc.cc.u32 %3, %12, %20;\n\t"
        "subc.cc.u32 %4, %13, %21;\n\t"
        "subc.cc.u32 %5, %14, %22;\n\t"
        "subc.cc.u32 %6, %15, %23;\n\t"
        "subc.cc.u32 %7, %16, %24;\n\t"
        "subc.u32 %8, 0, 0;"
        : "=&r"(t[0]), "=&r"(t[1]), "=&r"(t[2]), "=&r"(t[3]), "=&r"(t[4]), "=&r"(t[5]), "=&r"(t[6]), "=&r"(t[7]), "=&r"(c)
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]), "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
    KB_UNROLL
    for (int i = 0; i < 8; i++) r[i] = t[i];
    return c;
#endif
}
// r[0..8) += k (a 32-bit value), returns the carry out.
KB_FN uint32_t kb_add_small(uint32_t* r, uint32_t k)
{
#if defined(KB_HOST_EMU)
    uint64_t c = k;
    for (int i = 0; i < 8; i++) {
        c += r[i];
        r[i] = (uint32_t)c;
        c >>= 32;
    }
    return (uint32_t)c;
#else
    uint32_t c;
    asm("add.cc.u32 %0, %0, %9;\n\t"
        "addc.cc.u32 %1, %1, 0;\n\t"
        "addc.cc.u32 %2, %2, 0;\n\t"
        "addc.cc.u32 %3, %3, 0;\n\t"
        "addc.cc.u32 %4, %4, 0;\n\t"
        "addc.cc.u32 %5, %5, 0;\n\t"
        "addc.cc.u32 %6, %6, 0;\n\t"
        "addc.cc.u32 %7, %7, 0;\n\t"
        "addc.u32 %8, 0, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=&r"(c)
        : "r"(k));
    return c;
#endif
}
// r[0..8) -= k, returns the borrow as a mask
KB_FN uint32_t kb_sub_smallm(uint32_t* r, uint32_t k)
{
#if defined(KB_HOST_EMU)
    uint64_t br = k;
    for (int i = 0; i < 8; i++) {
        uint64_t d = (uint64_t)r[i] - br;
        r[i] = (uint32_t)d;
        br = (d >> 32) & 1;
    }
    return 0u - (uint32_t)br;
#else
    uint32_t c;
    asm("sub.cc.u32 %0, %0, %9;\n\t"
        "subc.cc.u32 %1, %1, 0;\n\t"
        "subc.cc.u32 %2, %2, 0;\n\t"
        "subc.cc.u32 %3, %3, 0;\n\t"
        "subc.cc.u32 %4, %4, 0;\n\t"
        "subc.cc.u32 %5, %5, 0;\n\t"
        "subc.cc.u32 %6, %6, 0;\n\t"
        "subc.cc.u32 %7, %7, 0;\n\t"
        "subc.u32 %8, 0, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=&r"(c)
        : "r"(k));
    return c;
#endif
}
// r[0..8) -= k, returns the borrow (0/1).
KB_FN uint32_t kb_sub_small(uint32_t* r, uint32_t k)
{
#if defined(KB_HOST_EMU)
    uint64_t br = k;
    for (int i = 0; i < 8; i++) {
        uint64_t d = (uint64_t)r[i] - br;
        r[i] = (uint32_t)d;
        br = (d >> 32) & 1;
    }
    return (uint32_t)br;
#else
    uint32_t c;
    asm("sub.cc.u32 %0, %0, %9;\n\t"
        "subc.cc.u32 %1, %1, 0;\n\t"
        "subc.cc.u32 %2, %2, 0;\n\t"
        "subc.cc.u32 %3, %3, 0;\n\t"
        "subc.cc.u32 %4, %4, 0;\n\t"
        "subc.cc.u32 %5, %5, 0;\n\t"
        "subc.cc.u32 %6, %6, 0;\n\t"
        "subc.cc.u32 %7, %7, 0;\n\t"
        "subc.u32 %8, 0, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "=&r"(c)
        : "r"(k));
    return c & 1;
#endif
}

// t[0..16) += a[i]^2 on word pairs (2i, 2i+1), one 16-instruction chain (8 IMAD.WIDE.U32.X).
KB_FN void kb_sqr_acc8(uint32_t* t, const uint32_t* a)
{
#if defined(KB_HOST_EMU)
    uint64_t carry = 0;
    for (int k = 0; k < 8; k++) {
        uint64_t p = (uint64_t)a[k] * a[k];
        uint64_t lo = (uint64_t)t[2 * k] + (uint32_t)p + carry;
        t[2 * k] = (uint32_t)lo;
        uint64_t hi = (uint64_t)t[2 * k + 1] + (p >> 32) + (lo >> 32);
        t[2 * k + 1] = (uint32_t)hi;
        carry = hi >> 32;
    }
#else
    asm("mad.lo.cc.u32 %0, %16, %16, %0;\n\t"
        "madc.hi.cc.u32 %1, %16, %16, %1;\n\t"
        "madc.lo.cc.u32 %2, %17, %17, %2;\n\t"
        "madc.hi.cc.u32 %3, %17, %17, %3;\n\t"
        "madc.lo.cc.u32 %4, %18, %18, %4;\n\t"
        "madc.hi.cc.u32 %5, %18, %18, %5;\n\t"
        "madc.lo.cc.u32 %6, %19, %19, %6;\n\t"
        "madc.hi.cc.u32 %7, %19, %19, %7;\n\t"
        "madc.lo.cc.u32 %8, %20, %20, %8;\n\t"
        "madc.hi.cc.u32 %9, %20, %20, %9;\n\t"
        "madc.lo.cc.u32 %10, %21, %21, %10;\n\t"
        "madc.hi.cc.u32 %11, %21, %21, %11;\n\t"
        "madc.lo.cc.u32 %12, %22, %22, %12;\n\t"
        "madc.hi.cc.u32 %13, %22, %22, %13;\n\t"
        "madc.lo.cc.u32 %14, %23, %23, %14;\n\t"
        "madc.hi.u32 %15, %23, %23, %15;"
        : "+r"(t[0]), "+r"(t[1]), "+r"(t[2]), "+r"(t[3]), "+r"(t[4]), "+r"(t[5]), "+r"(t[6]), "+r"(t[7]),
          "+r"(t[8]), "+r"(t[9]), "+r"(t[10]), "+r"(t[11]), "+r"(t[12]), "+r"(t[13]), "+r"(t[14]), "+r"(t[15])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
#endif
}

// t[0..16) = t[1..16) (t[0] absent = 0) + the squares a[i]^2 on word pairs (2i, 2i+1).  a[0]^2 is a plain product (its
// low word IS t[0]); its high word opens the carry chain with one add, the other seven squares follow as IMAD.WIDE.X.
KB_FN void kb_sqr_acc8_fresh0(uint32_t* t, const uint32_t* a)
{
#if defined(KB_HOST_EMU)
    t[0] = 0;
    kb_sqr_acc8(t, a);
#else
    const uint64_t p0 = (uint64_t)a[0] * a[0];
    t[0] = (uint32_t)p0;
    const uint32_t p0h = (uint32_t)(p0 >> 32);
    asm("add.cc.u32 %0, %0, %15;\n\t"
        "madc.lo.cc.u32 %1, %16, %16, %1;\n\t"
        "madc.hi.cc.u32 %2, %16, %16, %2;\n\t"
        "madc.lo.cc.u32 %3, %17, %17, %3;\n\t"
        "madc.hi.cc.u32 %4, %17, %17, %4;\n\t"
        "madc.lo.cc.u32 %5, %18, %18, %5;\n\t"
        "madc.hi.cc.u32 %6, %18, %18, %6;\n\t"
        "madc.lo.cc.u32 %7, %19, %19, %7;\n\t"
        "madc.hi.cc.u32 %8, %19, %19, %8;\n\t"
        "madc.lo.cc.u32 %9, %20, %20, %9;\n\t"
        "madc.hi.cc.u32 %10, %20, %20, %10;\n\t"
        "madc.lo.cc.u32 %11, %21, %21, %11;\n\t"
        "madc.hi.cc.u32 %12, %21, %21, %12;\n\t"
        "madc.lo.cc.u32 %13, %22, %22, %13;\n\t"
        "madc.hi.u32 %14, %22, %22, %14;"
        : "+r"(t[1]), "+r"(t[2]), "+r"(t[3]), "+r"(t[4]), "+r"(t[5]), "+r"(t[6]), "+r"(t[7]), "+r"(t[8]),
          "+r"(t[9]), "+r"(t[10]), "+r"(t[11]), "+r"(t[12]), "+r"(t[13]), "+r"(t[14]), "+r"(t[15])
        : "r"(p0h), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]));
#endif
}

// ---------------------------------------------------------------------------------------
// reduction of a 512-bit product: t[0..16) -> r[0..8), using 2^256 = 38 (mod p)
// ---------------------------------------------------------------------------------------
// upper word of (hi:lo) << s, 0 < s < 32 — a funnel shift (ALU pipe; a plain shift may become IMAD.SHL on the multiplier pipe)
KB_FN uint32_t kb_fshl(uint32_t lo, uint32_t hi, uint32_t s)
{
#if defined(KB_HOST_EMU)
    return (hi << s) | (lo >> (32 - s));
#else
    return __funnelshift_l(lo, hi, s);
#endif
}
// The same reduction WITHOUT multiplications: 38 H = 2 (H + 2H + 16H) by funnel shifts and carry chains, so that the eight
// IMAD.WIDE of the fold leave the multiplier pipe (about 50 ALU instructions instead).  -DKB_FE_FOLD_SHIFT selects it for
// every kernel: bit-exact, 12 % fewer multiplies, 24 % more instructions, every kernel about 20 % slower (DESIGN 7.1).
KB_FN void fe_reduce512_shift(fe& r, const uint32_t* t)
{
    const uint32_t* H = t + 8;
    uint32_t s1[8], s4[8], u[8];
    s1[0] = kb_fshl(0u, H[0], 1);
    s4[0] = kb_fshl(0u, H[0], 4);
    KB_UNROLL
    for (int k = 1; k < 8; k++) {
        s1[k] = kb_fshl(H[k - 1], H[k], 1);
        s4[k] = kb_fshl(H[k - 1], H[k], 4);
    }
    uint32_t top = kb_fshl(H[7], 0u, 1) + kb_fshl(H[7], 0u, 4);   // H[7] >> 31, H[7] >> 28
    top += kb_add8(u, H, s1);
    top += kb_add8(u, u, s4);      // (top : u) = 19 H < 2^261
    uint32_t S[8];
    S[0] = kb_fshl(0u, u[0], 1);
    KB_UNROLL
    for (int k = 1; k < 8; k++) S[k] = kb_fshl(u[k - 1], u[k], 1);
    uint32_t w8 = kb_fshl(u[7], top, 1);   // word 8 of 38 H, < 2^6
    w8 += kb_add8(r.v, t, S);
    uint32_t c = kb_add_small(r.v, w8 * 38u);
    r.v[0] += 38u * c;
}
// the fold of fe_reduce512_mul: r[0..8) + 2^256 * (returned word, < 2^7) = t[0..16) (mod p)
KB_FN uint32_t fe_reduce512_fold(fe& r, uint32_t* t)
{
    // even high words: (t0..t7) += 38 * {t8,t10,t12,t14}, carry into r8
    uint32_t r8;
    kb_cmad4_top(t, t[8], t[10], t[12], t[14], 38u, r8);
    // odd high words: 38*t9, 38*t11, 38*t13, 38*t15 land on word pairs (1,2) (3,4) (5,6) (7,8)
    uint32_t o[8];
    KB_UNROLL
    for (int k = 0; k < 4; k++) {
        uint64_t p = (uint64_t)t[9 + 2 * k] * 38u;
        o[2 * k] = (uint32_t)p;
        o[2 * k + 1] = (uint32_t)(p >> 32);
    }
    uint32_t hi[8];
    KB_UNROLL
    for (int k = 0; k < 7; k++) hi[k] = t[k + 1];
    hi[7] = r8;
    kb_acc8(hi, o);  // cannot carry: total < 39 * 2^256
    // fold word 8 (< 2^7): value = t0 + 2^32*hi[0..7) + 2^256*hi[7]
    r.v[0] = t[0];
    KB_UNROLL
    for (int k = 0; k < 7; k++) r.v[k + 1] = hi[k];
    return hi[7];
}
KB_FN void fe_reduce512_mul(fe& r, uint32_t* t)
{
    const uint32_t top = fe_reduce512_fold(r, t);
    uint32_t c = kb_add_small(r.v, top * 38u);
    // a second wrap leaves a value < 38*2^7, so adding 38 once more cannot carry
    r.v[0] += 38u * c;
}
KB_FN void fe_reduce512(fe& r, uint32_t* t)
{
#if defined(KB_FE_FOLD_SHIFT)
    fe_reduce512_shift(r, t);
#else
    fe_reduce512_mul(r, t);
#endif
}

// ev[0..16) = f * g (ev has room for 17 words), rows in natural order
KB_FN void fe_mul_rows_wide(uint32_t* ev, const fe& f, const fe& g)
{
    uint32_t od[16];
    const uint32_t* a = f.v;
    const uint32_t* b = g.v;
    // Operand scanning over b; products a[j]*b[i] with i+j even accumulate in ev (word i+j),
    // those with i+j odd in od (od[k] is word k+1), so every IMAD.WIDE is pair-aligned.
    // Row 0 lands on fresh words: plain products, nothing to zero and no carries.
    kb_cmul4(&ev[0], a[0], a[2], a[4], a[6], b[0]);
    kb_cmul4(&od[0], a[1], a[3], a[5], a[7], b[0]);
    // Later rows: an even row ends on a fresh word that takes its carry (kb_cmad4_top); an odd row's last product
    // lands on (a word holding at most that carry, a fresh word) and cannot carry out (kb_cmad4_hi).  ev[16] and
    // od[15] are never touched.  Only ev[8] has to be zeroed.
    ev[8] = 0;
    kb_cmad4_hi(&ev[2], a[1], a[3], a[5], a[7], b[1]);              // words 2..9
    kb_cmad4_top(&od[0], a[0], a[2], a[4], a[6], b[1], od[8]);      // words 1..8, carry -> 9
    kb_cmad4_top(&ev[2], a[0], a[2], a[4], a[6], b[2], ev[10]);
    kb_cmad4_hi(&od[2], a[1], a[3], a[5], a[7], b[2]);
    kb_cmad4_hi(&ev[4], a[1], a[3], a[5], a[7], b[3]);
    kb_cmad4_top(&od[2], a[0], a[2], a[4], a[6], b[3], od[10]);
    kb_cmad4_top(&ev[4], a[0], a[2], a[4], a[6], b[4], ev[12]);
    kb_cmad4_hi(&od[4], a[1], a[3], a[5], a[7], b[4]);
    kb_cmad4_hi(&ev[6], a[1], a[3], a[5], a[7], b[5]);
    kb_cmad4_top(&od[4], a[0], a[2], a[4], a[6], b[5], od[12]);
    kb_cmad4_top(&ev[6], a[0], a[2], a[4], a[6], b[6], ev[14]);
    kb_cmad4_hi(&od[6], a[1], a[3], a[5], a[7], b[6]);
    kb_cmad4_hi(&ev[8], a[1], a[3], a[5], a[7], b[7]);
    kb_cmad4_top(&od[6], a[0], a[2], a[4], a[6], b[7], od[14]);
    kb_acc15(&ev[1], &od[0]);
}
// h = f * g   (fe.rs:299 fe_mul), rows in natural order
KB_FN void fe_mul_rows(fe& h, const fe& f, const fe& g)
{
    uint32_t ev[17];
    fe_mul_rows_wide(ev, f, g);
    fe_reduce512(h, ev);
}

// ev[0..16) = f * g, rows ordered so that no register has to be zeroed (see kb_cmad4_new / kb_cmad4_rip)
KB_FN void fe_mul_rip_wide(uint32_t* ev, const fe& f, const fe& g)
{
    uint32_t od[15];
    const uint32_t* a = f.v;
    const uint32_t* b = g.v;
    // Operand scanning over b; products a[j]*b[i] with i+j even accumulate in ev (word i+j),
    // those with i+j odd in od (od[k] is word k+1), so every IMAD.WIDE is pair-aligned.
    // Row 0 lands on fresh words: plain products, nothing to zero and no carries.
    kb_cmul4(&ev[0], a[0], a[2], a[4], a[6], b[0]);
    kb_cmul4(&od[0], a[1], a[3], a[5], a[7], b[0]);
    // Two consecutive rows touch the same four pairs of a column set and together open ONE new pair.  The row that
    // opens it runs first (kb_cmad4_new: the new pair takes product + carry, addend RZ), the other one then ripples
    // its carry into that pair (kb_cmad4_rip) — no zeroed registers, no captured carries (see the primitives).
    // Bounds: after rows 0..r the partial sum of a column set is < 2^(256 + 32 (r+1)), so a ripple never leaves its pair.
    kb_cmad4_new(&ev[2], a[1], a[3], a[5], a[7], b[1]);                   // words 2..9
    kb_cmad4_new(&od[2], a[1], a[3], a[5], a[7], b[2]);                   // words 3..10
    kb_cmad4_rip(&od[0], a[0], a[2], a[4], a[6], b[1], od[8], od[9]);     // words 1..8, carry -> 9, 10
    kb_cmad4_new(&ev[4], a[1], a[3], a[5], a[7], b[3]);                   // words 4..11
    kb_cmad4_rip(&ev[2], a[0], a[2], a[4], a[6], b[2], ev[10], ev[11]);   // words 2..9, carry -> 10, 11
    kb_cmad4_new(&od[4], a[1], a[3], a[5], a[7], b[4]);                   // words 5..12
    kb_cmad4_rip(&od[2], a[0], a[2], a[4], a[6], b[3], od[10], od[11]);
    kb_cmad4_new(&ev[6], a[1], a[3], a[5], a[7], b[5]);                   // words 6..13
    kb_cmad4_rip(&ev[4], a[0], a[2], a[4], a[6], b[4], ev[12], ev[13]);
    kb_cmad4_new(&od[6], a[1], a[3], a[5], a[7], b[6]);                   // words 7..14
    kb_cmad4_rip(&od[4], a[0], a[2], a[4], a[6], b[5], od[12], od[13]);
    kb_cmad4_new(&ev[8], a[1], a[3], a[5], a[7], b[7]);                   // words 8..15
    kb_cmad4_rip(&ev[6], a[0], a[2], a[4], a[6], b[6], ev[14], ev[15]);
    kb_cmad4_top(&od[6], a[0], a[2], a[4], a[6], b[7], od[14]);           // words 7..14, carry -> word 15 (a plain word)
    kb_acc15(&ev[1], &od[0]);
}
// h = f * g, rows ordered so that no register has to be zeroed
KB_FN void fe_mul_rip(fe& h, const fe& f, const fe& g)
{
    uint32_t ev[16];
    fe_mul_rip_wide(ev, f, g);
    fe_reduce512(h, ev);
}

// ev[0..16) = f^2 (ev has room for 17 words), rows in natural order: 28 cross products, doubled, plus 8 squares
KB_FN void fe_sq_rows_wide(uint32_t* ev, const fe& f)
{
    uint32_t od[16];
    const uint32_t* a = f.v;
    // row i: a[j]*a[i] for j > i, word i+j; row 0 lands on fresh words (plain products, no zeroing, no carries)
    kb_cmul4(&od[0], a[1], a[3], a[5], a[7], a[0]);          // words 1,3,5,7
    kb_cmul3(&ev[2], a[2], a[4], a[6], a[0]);                // words 2,4,6
    // later rows end either on a fresh word that takes the carry (_top) or on (at most a carry, a fresh word) and
    // cannot carry out (_hi); only the six words no product reaches are zeroed
    ev[0] = ev[1] = ev[8] = ev[14] = ev[15] = 0;
    od[14] = 0;
    kb_cmad3_top(&od[2], a[2], a[4], a[6], a[1], od[8]);     // words 3,5,7
    kb_cmad3_hi(&ev[4], a[3], a[5], a[7], a[1]);             // words 4,6,8
    kb_cmad3_hi(&od[4], a[3], a[5], a[7], a[2]);             // words 5,7,9
    kb_cmad2_top(&ev[6], a[4], a[6], a[2], ev[10]);          // words 6,8
    kb_cmad2_top(&od[6], a[4], a[6], a[3], od[10]);          // words 7,9
    kb_cmad2_hi(&ev[8], a[5], a[7], a[3]);                   // words 8,10
    kb_cmad2_hi(&od[8], a[5], a[7], a[4]);                   // words 9,11
    kb_cmad1_top(&ev[10], a[6], a[4], ev[12]);               // word 10
    kb_cmad1_top(&od[10], a[6], a[5], od[12]);               // word 11
    kb_cmad1_hi(&ev[12], a[7], a[5]);                        // word 12
    kb_cmad1_hi(&od[12], a[7], a[6]);                        // word 13
    kb_acc15(&ev[1], &od[0]);
    kb_dbl16(ev);        // double the cross terms (top bit is clear: sum < 2^511)
    kb_sqr_acc8(ev, a);  // add the squares a[i]^2 on word pairs (2i, 2i+1)
}
// h = f^2   (fe.rs:544 fe_square), rows in natural order
KB_FN void fe_sq_rows(fe& h, const fe& f)
{
    uint32_t ev[17];
    fe_sq_rows_wide(ev, f);
    fe_reduce512(h, ev);
}

// t[0..16) = f^2, rows ordered so that no register has to be zeroed: 28 cross products, doubled, plus 8 squares
KB_FN void fe_sq_rip_wide(uint32_t* t, const fe& f)
{
    uint32_t ev[16], od[14];
    const uint32_t* a = f.v;
    // row i: a[j]*a[i] for j > i, word i+j; the rows are ordered as in fe_mul_inl — the row that opens a pair first
    // (or a plain product where nothing precedes it), the row below it ripples its carry in.  ev[0], ev[1], ev[14],
    // ev[15] and od[14] hold no cross product and are never materialised (kb_sq_merge_dbl).
    kb_cmul4(&od[0], a[1], a[3], a[5], a[7], a[0]);                  // words 1,3,5,7
    kb_cmul3(&ev[2], a[2], a[4], a[6], a[0]);                        // words 2,4,6
    kb_cmad3_new(&ev[4], a[3], a[5], a[7], a[1]);                    // words 4,6,8
    kb_cmad3_new(&od[4], a[3], a[5], a[7], a[2]);                    // words 5,7,9
    kb_cmad3_rip(&od[2], a[2], a[4], a[6], a[1], od[8], od[9]);      // words 3,5,7, carry -> 9, 10
    kb_cmad2_new(&ev[8], a[5], a[7], a[3]);                          // words 8,10
    kb_cmad2_rip(&ev[6], a[4], a[6], a[2], ev[10], ev[11]);          // words 6,8, carry -> 10, 11
    kb_cmad2_new(&od[8], a[5], a[7], a[4]);                          // words 9,11
    kb_cmad2_rip(&od[6], a[4], a[6], a[3], od[10], od[11]);          // words 7,9, carry -> 11, 12
    kb_cmul1(&ev[12], a[7], a[5]);                                   // word 12
    kb_cmad1_rip(&ev[10], a[6], a[4], ev[12], ev[13]);               // word 10, carry -> 12, 13
    kb_cmul1(&od[12], a[7], a[6]);                                   // word 13
    kb_cmad1_rip(&od[10], a[6], a[5], od[12], od[13]);               // word 11, carry -> 13, 14
    kb_sq_merge_dbl(t, ev, od);   // t[1..16) = doubled cross terms (sum < 2^511: the top bit is clear)
    kb_sqr_acc8_fresh0(t, a);     // add the squares a[i]^2 on word pairs (2i, 2i+1)
}
// h = f^2, rows ordered so that no register has to be zeroed
KB_FN void fe_sq_rip(fe& h, const fe& f)
{
    uint32_t t[16];
    fe_sq_rip_wide(t, f);
    fe_reduce512(h, t);
}

// Which bodies a translation unit uses (all are bit-exact; tests/emu runs every one):  MEASURED, round 2 — the
// zero-free row order (-DKB_FE_MUL_RIP / -DKB_FE_SQ_RIP) and the borrow-mask wrap of fe_sub (-DKB_FE_SUBMASK) shift the
// balance ptxas strikes between the ALU and the multiplier pipe differently in every kernel, see DESIGN §7.1.
#if defined(KB_FE_MUL_RIP)
KB_FN void fe_mul_inl(fe& h, const fe& f, const fe& g) { fe_mul_rip(h, f, g); }
#else
KB_FN void fe_mul_inl(fe& h, const fe& f, const fe& g) { fe_mul_rows(h, f, g); }
#endif
#if defined(KB_FE_SQ_RIP)
KB_FN void fe_sq_inl(fe& h, const fe& f) { fe_sq_rip(h, f); }
#else
KB_FN void fe_sq_inl(fe& h, const fe& f) { fe_sq_rows(h, f); }
#endif

// ---------------------------------------------------------------------------------------
// One level of (subtractive) Karatsuba for h = f * g: three 4 x 4-limb products (48 IMAD.WIDE) instead of 64.
//   a = a0 + 2^128 a1, b = b0 + 2^128 b1:   a b = z0 + 2^128 (z0 + z2 - (a0 - a1)(b0 - b1)) + 2^256 z2
// The differences are taken in absolute value (4 limbs, no overflow) with their signs tracked.  The IMAD.WIDE that
// does the products holds the multiplier pipe 4 cycles per warp instruction, the additions this costs (about 70
// more than the schoolbook form) run on the ALU pipe at 2 — in the point formulas the ALU pipe has that room.
// ---------------------------------------------------------------------------------------
KB_FN void kb_cmul2(uint32_t* acc, uint32_t a0, uint32_t a1, uint32_t b)
{
    const uint64_t p0 = (uint64_t)a0 * b, p1 = (uint64_t)a1 * b;
    acc[0] = (uint32_t)p0; acc[1] = (uint32_t)(p0 >> 32);
    acc[2] = (uint32_t)p1; acc[3] = (uint32_t)(p1 >> 32);
}
// acc[0..7) += x[0..7) (no carry out: callers guarantee it fits)
KB_FN void kb_acc7(uint32_t* acc, const uint32_t* x)
{
#if defined(KB_HOST_EMU)
    uint64_t c = 0;
    for (int i = 0; i < 7; i++) {
        c += (uint64_t)acc[i] + x[i];
        acc[i] = (uint32_t)c;
        c >>= 32;
    }
#else
    asm("add.cc.u32 %0, %0, %7;\n\t"
        "addc.cc.u32 %1, %1, %8;\n\t"
        "addc.cc.u32 %2, %2, %9;\n\t"
        "addc.cc.u32 %3, %3, %10;\n\t"
        "addc.cc.u32 %4, %4, %11;\n\t"
        "addc.cc.u32 %5, %5, %12;\n\t"
        "addc.u32 %6, %6, %13;"
        : "+r"(acc[0]), "+r"(acc[1]), "+r"(acc[2]), "+r"(acc[3]), "+r"(acc[4]), "+r"(acc[5]), "+r"(acc[6])
        : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(x[3]), "r"(x[4]), "r"(x[5]), "r"(x[6]));
#endif
}
// r[0..8) = a[0..4) * b[0..4): the even / odd column split of fe_mul_inl on 4 limbs (16 IMAD.WIDE, one 7-word merge)
KB_FN void kb_mul4x4(uint32_t* r, const uint32_t* a, const uint32_t* b)
{
    uint32_t od[7];
    kb_cmul2(&r[0], a[0], a[2], b[0]);                     // words 0..3
    kb_cmul2(&od[0], a[1], a[3], b[0]);                    // words 1..4
    r[4] = 0;
    kb_cmad2_hi(&r[2], a[1], a[3], b[1]);                  // words 2..5
    kb_cmad2_top(&od[0], a[0], a[2], b[1], od[4]);         // words 1..4, carry -> 5
    kb_cmad2_top(&r[2], a[0], a[2], b[2], r[6]);           // words 2..5, carry -> 6
    kb_cmad2_hi(&od[2], a[1], a[3], b[2]);                 // words 3..6
    kb_cmad2_hi(&r[4], a[1], a[3], b[3]);                  // words 4..7
    kb_cmad2_top(&od[2], a[0], a[2], b[3], od[6]);         // words 3..6, carry -> 7
    kb_acc7(&r[1], &od[0]);
}
// d[0..4) = |x - y| on 4 limbs; returns 0xffffffff if x < y, else 0
KB_FN uint32_t kb_absdiff4(uint32_t* d, const uint32_t* x, const uint32_t* y)
{
    uint32_t m;
#if defined(KB_HOST_EMU)
    uint64_t br = 0;
    for (int i = 0; i < 4; i++) {
        const uint64_t t = (uint64_t)x[i] - y[i] - br;
        d[i] = (uint32_t)t;
        br = (t >> 32) & 1u;
    }
    m = 0u - (uint32_t)br;
    uint64_t c = br;
    for (int i = 0; i < 4; i++) {
        c += (uint64_t)(d[i] ^ m);
        d[i] = (uint32_t)c;
        c >>= 32;
    }
#else
    asm("sub.cc.u32 %0, %5, %9;\n\t"
        "subc.cc.u32 %1, %6, %10;\n\t"
        "subc.cc.u32 %2, %7, %11;\n\t"
        "subc.cc.u32 %3, %8, %12;\n\t"
        "subc.u32 %4, 0, 0;"
        : "=&r"(d[0]), "=&r"(d[1]), "=&r"(d[2]), "=&r"(d[3]), "=&r"(m)
        : "r"(x[0]), "r"(x[1]), "r"(x[2]), "r"(x[3]), "r"(y[0]), "r"(y[1]), "r"(y[2]), "r"(y[3]));
    d[0] ^= m; d[1] ^= m; d[2] ^= m; d[3] ^= m;
    // (d ^ m) - m on 128 bits: + 1 when m is all ones
    asm("sub.cc.u32 %0, %0, %4;\n\t"
        "subc.cc.u32 %1, %1, %4;\n\t"
        "subc.cc.u32 %2, %2, %4;\n\t"
        "subc.u32 %3, %3, %4;"
        : "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
        : "r"(m));
#endif
    return m;
}
// t[0..16) = z0 + 2^128 (z0 + z2 -+ zm) + 2^256 z2 with z0 = t[0..8), z2 = t[8..16) on entry; nm = all ones to
// SUBTRACT zm, 0 to add it
KB_FN void kb_karatsuba_join(uint32_t* t, const uint32_t* zm, uint32_t nm)
{
#if defined(KB_HOST_EMU)
    uint32_t mid[9];
    uint64_t c = 0;
    for (int i = 0; i < 8; i++) {
        c += (uint64_t)t[i] + t[8 + i];
        mid[i] = (uint32_t)c;
        c >>= 32;
    }
    mid[8] = (uint32_t)c;
    c = nm & 1u;
    for (int i = 0; i < 8; i++) {
        c += (uint64_t)mid[i] + (zm[i] ^ nm);
        mid[i] = (uint32_t)c;
        c >>= 32;
    }
    mid[8] = (uint32_t)(mid[8] + nm + c);
    c = 0;
    for (int i = 0; i < 9; i++) {
        c += (uint64_t)t[4 + i] + mid[i];
        t[4 + i] = (uint32_t)c;
        c >>= 32;
    }
    for (int i = 13; i < 16; i++) {
        c += t[i];
        t[i] = (uint32_t)c;
        c >>= 32;
    }
#else
    uint32_t m0, m1, m2, m3, m4, m5, m6, m7, m8;
    asm("add.cc.u32 %0, %9, %17;\n\t"
        "addc.cc.u32 %1, %10, %18;\n\t"
        "addc.cc.u32 %2, %11, %19;\n\t"
        "addc.cc.u32 %3, %12, %20;\n\t"
        "addc.cc.u32 %4, %13, %21;\n\t"
        "addc.cc.u32 %5, %14, %22;\n\t"
        "addc.cc.u32 %6, %15, %23;\n\t"
        "addc.cc.u32 %7, %16, %24;\n\t"
        "addc.u32 %8, 0, 0;"
        : "=&r"(m0), "=&r"(m1), "=&r"(m2), "=&r"(m3), "=&r"(m4), "=&r"(m5), "=&r"(m6), "=&r"(m7), "=&r"(m8)
        : "r"(t[0]), "r"(t[1]), "r"(t[2]), "r"(t[3]), "r"(t[4]), "r"(t[5]), "r"(t[6]), "r"(t[7]),
          "r"(t[8]), "r"(t[9]), "r"(t[10]), "r"(t[11]), "r"(t[12]), "r"(t[13]), "r"(t[14]), "r"(t[15]));
    const uint32_t x0 = zm[0] ^ nm, x1 = zm[1] ^ nm, x2 = zm[2] ^ nm, x3 = zm[3] ^ nm, x4 = zm[4] ^ nm, x5 = zm[5] ^ nm, x6 = zm[6] ^ nm, x7 = zm[7] ^ nm;
    uint32_t scratch;
    // carry-in = nm & 1 (nm + 1 overflows exactly when nm is all ones); the ninth word takes the sign extension
    asm("add.cc.u32 %9, %18, 1;\n\t"
        "addc.cc.u32 %0, %0, %10;\n\t"
        "addc.cc.u32 %1, %1, %11;\n\t"
        "addc.cc.u32 %2, %2, %12;\n\t"
        "addc.cc.u32 %3, %3, %13;\n\t"
        "addc.cc.u32 %4, %4, %14;\n\t"
        "addc.cc.u32 %5, %5, %15;\n\t"
        "addc.cc.u32 %6, %6, %16;\n\t"
        "addc.cc.u32 %7, %7, %17;\n\t"
        "addc.u32 %8, %8, %18;"
        : "+r"(m0), "+r"(m1), "+r"(m2), "+r"(m3), "+r"(m4), "+r"(m5), "+r"(m6), "+r"(m7), "+r"(m8), "=&r"(scratch)
        : "r"(x0), "r"(x1), "r"(x2), "r"(x3), "r"(x4), "r"(x5), "r"(x6), "r"(x7), "r"(nm));
    asm("add.cc.u32 %0, %0, %12;\n\t"
        "addc.cc.u32 %1, %1, %13;\n\t"
        "addc.cc.u32 %2, %2, %14;\n\t"
        "addc.cc.u32 %3, %3, %15;\n\t"
        "addc.cc.u32 %4, %4, %16;\n\t"
        "addc.cc.u32 %5, %5, %17;\n\t"
        "addc.cc.u32 %6, %6, %18;\n\t"
        "addc.cc.u32 %7, %7, %19;\n\t"
        "addc.cc.u32 %8, %8, %20;\n\t"
        "addc.cc.u32 %9, %9, 0;\n\t"
        "addc.cc.u32 %10, %10, 0;\n\t"
        "addc.u32 %11, %11, 0;"
        : "+r"(t[4]), "+r"(t[5]), "+r"(t[6]), "+r"(t[7]), "+r"(t[8]), "+r"(t[9]), "+r"(t[10]), "+r"(t[11]), "+r"(t[12]), "+r"(t[13]), "+r"(t[14]), "+r"(t[15])
        : "r"(m0), "r"(m1), "r"(m2), "r"(m3), "r"(m4), "r"(m5), "r"(m6), "r"(m7), "r"(m8));
#endif
}
KB_FN void fe_mul_karatsuba(fe& h, const fe& f, const fe& g)
{
    uint32_t t[16], zm[8], da[4], db[4];
    const uint32_t sa = kb_absdiff4(da, f.v, f.v + 4);
    const uint32_t sb = kb_absdiff4(db, g.v, g.v + 4);
    kb_mul4x4(&t[0], f.v, g.v);
    kb_mul4x4(&t[8], f.v + 4, g.v + 4);
    kb_mul4x4(zm, da, db);
    // (a0 - a1)(b0 - b1) = +zm when the signs agree: the middle term is then z0 + z2 - zm
    kb_karatsuba_join(t, zm, ~(sa ^ sb));
    fe_reduce512(h, t);
}

// Code-size knob.  With every multiplication inlined, the verify kernel is ~29 k instructions and
// its window loop alone (75 KB) overflows the 32 KB L1.5 instruction cache: ncu reports
// "no_instruction" as the largest stall reason.  With KB_FE_CALLS the two big bodies exist ONCE per
// kernel and are reached by CALL with operands and result passed BY VALUE — the ABI keeps a
// 32-byte struct in registers (checked in SASS: MOVs + CALL.REL, 0 bytes of stack), so a call
// costs ~26 register moves and no memory traffic.
#if defined(KB_FE_CALLS) && !defined(KB_HOST_EMU)
__device__ __noinline__ fe fe_mul_call(fe f, fe g)
{
    fe h;
    fe_mul_inl(h, f, g);
    return h;
}
__device__ __noinline__ fe fe_sq_call(fe f)
{
    fe h;
    fe_sq_inl(h, f);
    return h;
}
KB_FN void fe_mul(fe& h, const fe& f, const fe& g) { h = fe_mul_call(f, g); }
KB_FN void fe_sq(fe& h, const fe& f) { h = fe_sq_call(f); }
#elif defined(KB_FE_KARATSUBA)
KB_FN void fe_mul(fe& h, const fe& f, const fe& g) { fe_mul_karatsuba(h, f, g); }
KB_FN void fe_sq(fe& h, const fe& f) { fe_sq_inl(h, f); }
#else
KB_FN void fe_mul(fe& h, const fe& f, const fe& g) { fe_mul_inl(h, f, g); }
KB_FN void fe_sq(fe& h, const fe& f) { fe_sq_inl(h, f); }
#endif

// ---------------------------------------------------------------------------------------
// linear operations (fe.rs: fe_add, fe_sub, fe_neg, fe_c_move)
// ---------------------------------------------------------------------------------------
KB_FN void fe_add(fe& h, const fe& f, const fe& g)
{
    uint32_t c = kb_add8(h.v, f.v, g.v);
    c = kb_add_small(h.v, 38u * c);  // 2^256 = 38
    h.v[0] += 38u * c;               // after a second wrap the value is < 38: cannot carry
}
KB_FN void fe_sub(fe& h, const fe& f, const fe& g)
{
#if defined(KB_FE_SUBMASK)
    uint32_t m = kb_sub8m(h.v, f.v, g.v);
    m = kb_sub_smallm(h.v, m & 38u);  // -2^256 = -38
    h.v[0] -= m & 38u;                // after a second wrap the value is >= 2^256-38: cannot borrow
#else
    uint32_t b = kb_sub8(h.v, f.v, g.v);
    b = kb_sub_small(h.v, 38u * b);  // -2^256 = -38
    h.v[0] -= 38u * b;               // after a second wrap the value is >= 2^256-38: cannot borrow
#endif
}
KB_FN void fe_set(fe& h, uint32_t x)
{
    h.v[0] = x;
    KB_UNROLL
    for (int i = 1; i < 8; i++) h.v[i] = 0;
}
KB_FN void fe_neg(fe& h, const fe& f)
{
    fe z;
    fe_set(z, 0);
    fe_sub(h, z, f);
}
// f = b ? g : f   (b in {0,1}); no branch on b
KB_FN void fe_cmov(fe& f, const fe& g, uint32_t b)
{
    uint32_t m = 0u - b;
    KB_UNROLL
    for (int i = 0; i < 8; i++) f.v[i] ^= m & (f.v[i] ^ g.v[i]);
}
KB_FN void fe_dbl(fe& h, const fe& f) { fe_add(h, f, f); }

// ---------------------------------------------------------------------------------------
// Short-wrap bodies, for code whose inputs are all public (the verifiers' k_verify_half_prep / k_verify_half_main).
// Every body above ends by adding a small k (38 * carry, or 38 * the fold's top word < 38 * 2^7) into word 0 and
// rippling the carry through all eight words, then wrapping a second time: one chain of 9 dependent instructions and
// a multiply.  The carry leaves word 0 with probability below 2^-19.8 and word 1 below 2^-52, so the bodies below stop
// the ripple at word 1 and ADD the carry (or borrow) out of word 1 to a per-thread counter `ovf` instead.
//
// Invariant: if `ovf` is still 0 after a sequence of short-wrap operations, every output equals the exact body's output
// bit for bit (the exact ripple stops at word 1 as well, and its second wrap adds 38 * 0).  When it is not 0, the
// caller recomputes with the exact bodies.  `ovf` counts: a few thousand operations per thread cannot wrap it around.
// Nothing here is constant-time — the flag depends on the data.
// ---------------------------------------------------------------------------------------
// r[0..2) += k; the carry out of word 1 is added to ovf (words 2..7 are not touched)
KB_FN void kb_add_small2(uint32_t* r, uint32_t k, uint32_t& ovf)
{
#if defined(KB_HOST_EMU)
    uint64_t c = (uint64_t)r[0] + k;
    r[0] = (uint32_t)c;
    c = (c >> 32) + r[1];
    r[1] = (uint32_t)c;
    ovf += (uint32_t)(c >> 32);
#else
    asm("add.cc.u32 %0, %0, %3;\n\t"
        "addc.cc.u32 %1, %1, 0;\n\t"
        "addc.u32 %2, %2, 0;"
        : "+r"(r[0]), "+r"(r[1]), "+r"(ovf)
        : "r"(k));
#endif
}
// r[0..2) -= k; the borrow out of word 1 is added to ovf (words 2..7 are not touched)
KB_FN void kb_sub_small2(uint32_t* r, uint32_t k, uint32_t& ovf)
{
#if defined(KB_HOST_EMU)
    uint64_t d = (uint64_t)r[0] - k;
    r[0] = (uint32_t)d;
    d = (uint64_t)r[1] - ((d >> 32) & 1u);
    r[1] = (uint32_t)d;
    ovf += (uint32_t)((d >> 32) & 1u);
#else
    uint32_t m;
    asm("sub.cc.u32 %0, %0, %3;\n\t"
        "subc.cc.u32 %1, %1, 0;\n\t"
        "subc.u32 %2, 0, 0;"
        : "+r"(r[0]), "+r"(r[1]), "=r"(m)
        : "r"(k));
    ovf -= m;   // m = 0 or all ones
#endif
}
KB_FN void fe_reduce512_sw(fe& r, uint32_t* t, uint32_t& ovf)
{
#if defined(KB_FE_FOLD_SHIFT)
    (void)ovf;
    fe_reduce512_shift(r, t);
#else
    const uint32_t top = fe_reduce512_fold(r, t);
    kb_add_small2(r.v, top * 38u, ovf);
#endif
}
// the row order of fe_mul_inl / fe_sq_inl (KB_FE_MUL_RIP, KB_FE_SQ_RIP), always inlined
KB_FN void fe_mul_sw(fe& h, const fe& f, const fe& g, uint32_t& ovf)
{
    uint32_t t[17];
#if defined(KB_FE_MUL_RIP)
    fe_mul_rip_wide(t, f, g);
#else
    fe_mul_rows_wide(t, f, g);
#endif
    fe_reduce512_sw(h, t, ovf);
}
KB_FN void fe_sq_sw(fe& h, const fe& f, uint32_t& ovf)
{
    uint32_t t[17];
#if defined(KB_FE_SQ_RIP)
    fe_sq_rip_wide(t, f);
#else
    fe_sq_rows_wide(t, f);
#endif
    fe_reduce512_sw(h, t, ovf);
}
KB_FN void fe_add_sw(fe& h, const fe& f, const fe& g, uint32_t& ovf)
{
    const uint32_t c = kb_add8(h.v, f.v, g.v);
    kb_add_small2(h.v, 38u * c, ovf);   // 2^256 = 38
}
KB_FN void fe_sub_sw(fe& h, const fe& f, const fe& g, uint32_t& ovf)
{
#if defined(KB_FE_SUBMASK)
    const uint32_t m = kb_sub8m(h.v, f.v, g.v);
    kb_sub_small2(h.v, m & 38u, ovf);   // -2^256 = -38
#else
    const uint32_t b = kb_sub8(h.v, f.v, g.v);
    kb_sub_small2(h.v, 38u * b, ovf);
#endif
}
KB_FN void fe_dbl_sw(fe& h, const fe& f, uint32_t& ovf) { fe_add_sw(h, f, f, ovf); }

// Two sets of field operations for code written once for both kinds of body (ge.cuh, ops.cuh): the last argument picks
// the exact bodies (fe_ex) or the short-wrap bodies and their counter (fe_sw).
struct fe_ex {};
struct fe_sw {
    uint32_t ovf;
};
KB_FN void fe_mul(fe& h, const fe& f, const fe& g, fe_ex&) { fe_mul(h, f, g); }
KB_FN void fe_sq(fe& h, const fe& f, fe_ex&) { fe_sq(h, f); }
KB_FN void fe_add(fe& h, const fe& f, const fe& g, fe_ex&) { fe_add(h, f, g); }
KB_FN void fe_sub(fe& h, const fe& f, const fe& g, fe_ex&) { fe_sub(h, f, g); }
KB_FN void fe_dbl(fe& h, const fe& f, fe_ex&) { fe_dbl(h, f); }
KB_FN void fe_mul(fe& h, const fe& f, const fe& g, fe_sw& s) { fe_mul_sw(h, f, g, s.ovf); }
KB_FN void fe_sq(fe& h, const fe& f, fe_sw& s) { fe_sq_sw(h, f, s.ovf); }
KB_FN void fe_add(fe& h, const fe& f, const fe& g, fe_sw& s) { fe_add_sw(h, f, g, s.ovf); }
KB_FN void fe_sub(fe& h, const fe& f, const fe& g, fe_sw& s) { fe_sub_sw(h, f, g, s.ovf); }
KB_FN void fe_dbl(fe& h, const fe& f, fe_sw& s) { fe_dbl_sw(h, f, s.ovf); }
template <class F>
KB_FN void fe_neg(fe& h, const fe& f, F& fo)
{
    fe z;
    fe_set(z, 0);
    fe_sub(h, z, f, fo);
}

// ---------------------------------------------------------------------------------------
// canonical form and byte I/O (fe.rs:67 fe_from_bytes, :147 fe_to_bytes, :240, :246)
// ---------------------------------------------------------------------------------------
// words = little-endian 32-bit words of the 32-byte encoding; bit 255 is dropped and values
// >= p are NOT rejected (fe.rs:67-77).
KB_FN void fe_from_words(fe& h, const uint32_t* w)
{
    KB_UNROLL
    for (int i = 0; i < 8; i++) h.v[i] = w[i];
    h.v[7] &= 0x7fffffffu;
}
// fully reduced representative in [0, p)
KB_FN void fe_canon(fe& h, const fe& f)
{
    fe t = f;
    // fold bit 255: t < 2^255 + 19
    uint32_t top = t.v[7] >> 31;
    t.v[7] &= 0x7fffffffu;
    kb_add_small(t.v, 19u * top);
    // t >= p  <=>  t + 19 >= 2^255
    fe u = t;
    kb_add_small(u.v, 19u);
    uint32_t ge = u.v[7] >> 31;
    u.v[7] &= 0x7fffffffu;
    fe_cmov(t, u, ge);
    h = t;
}
KB_FN void fe_to_words(uint32_t* w, const fe& f)
{
    fe t;
    fe_canon(t, f);
    KB_UNROLL
    for (int i = 0; i < 8; i++) w[i] = t.v[i];
}
KB_FN uint32_t fe_is_negative(const fe& f)
{
    fe t;
    fe_canon(t, f);
    return t.v[0] & 1u;
}
KB_FN uint32_t fe_is_zero(const fe& f)
{
    fe t;
    fe_canon(t, f);
    uint32_t x = 0;
    KB_UNROLL
    for (int i = 0; i < 8; i++) x |= t.v[i];
    return x == 0;
}

// ---------------------------------------------------------------------------------------
// exponentiations (fe.rs:857 fe_invert, :946 fe_pow22523)
// ---------------------------------------------------------------------------------------
KB_FN void fe_sqn(fe& h, const fe& f, int n)
{
    fe_sq(h, f);
    KB_NOUNROLL
    for (int i = 1; i < n; i++) fe_sq(h, h);
}
// t = z^(2^250-1), z11 = z^11
KB_FN void fe_pow_2_250_1(fe& t, fe& z11, const fe& z)
{
    fe t0, t1, t2, t3;
    fe_sq(t0, z);
    fe_sqn(t1, t0, 2);
    fe_mul(t1, z, t1);   // z^9
    fe_mul(t0, t0, t1);  // z^11
    z11 = t0;
    fe_sq(t2, t0);       // z^22
    fe_mul(t1, t1, t2);  // 2^5 - 1
    fe_sqn(t2, t1, 5);
    fe_mul(t1, t2, t1);  // 2^10 - 1
    fe_sqn(t2, t1, 10);
    fe_mul(t2, t2, t1);  // 2^20 - 1
    fe_sqn(t3, t2, 20);
    fe_mul(t2, t3, t2);  // 2^40 - 1
    fe_sqn(t2, t2, 10);
    fe_mul(t1, t2, t1);  // 2^50 - 1
    fe_sqn(t2, t1, 50);
    fe_mul(t2, t2, t1);  // 2^100 - 1
    fe_sqn(t3, t2, 100);
    fe_mul(t2, t3, t2);  // 2^200 - 1
    fe_sqn(t2, t2, 50);
    fe_mul(t, t2, t1);   // 2^250 - 1
}
KB_FN void fe_invert(fe& out, const fe& z)
{
    fe t, z11;
    fe_pow_2_250_1(t, z11, z);
    fe_sqn(t, t, 5);
    fe_mul(out, t, z11);  // z^(2^255-21)
}
KB_FN void fe_pow22523(fe& out, const fe& z)
{
    fe t, z11;
    fe_pow_2_250_1(t, z11, z);
    fe_sqn(t, t, 2);
    fe_mul(out, t, z);  // z^(2^252-3)
}

// curve constants (constants.rs:56,60,65) as 32-bit little-endian words
#define KB_FE_D      {{0x135978a3u, 0x75eb4dcau, 0x4141d8abu, 0x00700a4du, 0x7779e898u, 0x8cc74079u, 0x2b6ffe73u, 0x52036ceeu}}
#define KB_FE_D2     {{0x26b2f159u, 0xebd69b94u, 0x8283b156u, 0x00e0149au, 0xeef3d130u, 0x198e80f2u, 0x56dffce7u, 0x2406d9dcu}}
#define KB_FE_SQRTM1 {{0x4a0ea0b0u, 0xc4ee1b27u, 0xad2fe478u, 0x2f431806u, 0x3dfbd7a7u, 0x2b4d0099u, 0x4fc1df0bu, 0x2b832480u}}
#define KB_FE_BX     {{0x8f25d51au, 0xc9562d60u, 0x9525a7b2u, 0x692cc760u, 0xfdd6dc5cu, 0xc0a4e231u, 0xcd6e53feu, 0x216936d3u}}
#define KB_FE_BY     {{0x66666658u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u, 0x66666666u}}
#define KB_FE_BT     {{0xa5b7dda3u, 0x6dde8ab3u, 0x775152f5u, 0x20f09f80u, 0x64abe37du, 0x66ea4e8eu, 0xd78b7665u, 0x67875f0fu}}
