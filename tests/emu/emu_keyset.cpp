// tests/emu/emu_keyset.cpp — HOST EMULATION of the key-set device math (ops.cuh kb_key_*, sig_keyset_*).  TEST
// INFRASTRUCTURE ONLY.  It builds on tests/emu/emu.cpp (the same headers compiled with KB_HOST_EMU, the host-built base
// tables and fixed-base comb) by including it, and adds the entry points of tests/test_emu_keyset.py.  Never linked into
// libkyber_b200.so.
#include "emu.cpp"

extern "C" {
// key sets (ops.cuh kb_key_*): row p of the key comb of pk as out[128 x 96] = canonical (y+x, y-x, 2dxy) words per entry;
// returns the key's facts (KB_F_AC | KB_F_AS | KB_F_AOK)
int emu_keyset_row(uint8_t* out, const uint8_t* pk, int p)
{
    uint32_t pw[8], w[8];
    ld(pw, pk, 8);
    ge_p3 A;
    const uint32_t f = kb_key_facts(A, pw);
    std::vector<ge_precomp> row(KB_KEY_HALF);
    kb_key_row(row.data(), A, p);
    for (int j = 0; j < KB_KEY_HALF; j++) {
        fe_to_words(w, row[j].ypx); st(out + 96 * j, w, 8);
        fe_to_words(w, row[j].ymx); st(out + 96 * j + 32, w, 8);
        fe_to_words(w, row[j].xy2d); st(out + 96 * j + 64, w, 8);
    }
    return (int)f;
}
// the keyed verifier composed as k_keyset_verify + k_verify_stage2 do it, with the comb of pk (the last key's comb is kept)
int emu_keyset_verify(int schnorr, const uint8_t* pk, const uint8_t* msg, uint64_t mlen, const uint8_t* sig)
{
    static std::vector<ge_precomp> ktab;
    static uint8_t kpk[32];
    static uint32_t kf;
    comb_init();
    if (ktab.empty() || memcmp(kpk, pk, 32) != 0) {
        uint32_t pw[8];
        ld(pw, pk, 8);
        ge_p3 A;
        kf = kb_key_facts(A, pw);
        ktab.resize(KB_KEY_ENTRIES);
        for (int p = 0; p < KB_KEY_POS; p++) kb_key_row(ktab.data() + (size_t)p * KB_KEY_HALF, A, p);
        memcpy(kpk, pk, 32);
    }
    uint32_t pw[8], sw[16], enc[8];
    ld(pw, pk, 8); ld(sw, sig, 16);
    ge_p3 Q;
    const uint32_t f = schnorr ? sig_keyset_stage1<true>(Q, kf, pw, sw, msg, mlen, g_comb.data(), ktab.data()) : sig_keyset_stage1<false>(Q, kf, pw, sw, msg, mlen, g_comb.data(), ktab.data());
    ge_compress(enc, Q);
    return schnorr ? (int)sig_finish<true>(f, enc, sw) : (int)sig_finish<false>(f, enc, sw);
}
}  // extern "C"
