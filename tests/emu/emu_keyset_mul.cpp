// tests/emu/emu_keyset_mul.cpp — HOST EMULATION of the keyed scalar multiplication (ops.cuh ge_keyset_mul,
// kb_keyset_mul_one).  TEST INFRASTRUCTURE ONLY.  It builds on tests/emu/emu.cpp (the same headers compiled with
// KB_HOST_EMU) by including it, and adds the entry point of tests/test_emu_keyset_mul.py.  Never linked into
// libkyber_b200.so.
#include "emu.cpp"

extern "C" {
// out = compress(a * A) for the key pk from its comb, built as k_keyset_build builds it (the last key's comb is kept).
// direct = 1: ge_keyset_mul<ct> over the comb whatever the key's facts; direct = 0: the item as k_keyset_mul composes it
// (kb_keyset_mul_one<ct>).  Returns the item's status (0, or 1 when the key does not decode).
int emu_keyset_mul(uint8_t* out, const uint8_t* pk, const uint8_t* scalar, int ct, int direct)
{
    static std::vector<ge_precomp> ktab;
    static uint8_t kpk[32];
    static uint32_t kf;
    uint32_t pw[8], s[8], o[8];
    ld(pw, pk, 8);
    ld(s, scalar, 8);
    if (ktab.empty() || memcmp(kpk, pk, 32) != 0) {
        ge_p3 A;
        kf = kb_key_facts(A, pw);
        ktab.resize(KB_KEY_ENTRIES);
        for (int p = 0; p < KB_KEY_POS; p++) kb_key_row(ktab.data() + (size_t)p * KB_KEY_HALF, A, p);
        memcpy(kpk, pk, 32);
    }
    int8_t e[64];
    sc_recode16(e, s);
    ge_p3 h;
    uint32_t status = 0;
    if (direct) {
        if (ct) ge_keyset_mul<true>(h, e, ktab.data());
        else ge_keyset_mul<false>(h, e, ktab.data());
    } else {
        status = ct ? kb_keyset_mul_one<true>(h, kf, pw, e, ktab.data()) : kb_keyset_mul_one<false>(h, kf, pw, e, ktab.data());
    }
    ge_compress(o, h);
    st(out, o, 8);
    return (int)status;
}
}  // extern "C"
