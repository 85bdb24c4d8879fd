// tests/emu/emu_dkg_columns.cpp — HOST EMULATION of the share checks of a verifier range (dkgcol.cuh).  TEST
// INFRASTRUCTURE ONLY.  It builds on tests/emu/emu.cpp (the same headers compiled with KB_HOST_EMU) and composes the
// per-thread bodies the kernels inline the way the kernels compose them.  Never linked into libkyber_b200.so.
#include "emu.cpp"
#include "../../kyber-rs_b200/csrc/dkgcol.cuh"

#include <algorithm>

// e[8 j ..] = x^j mod 8L and dig[KB_COL_WINDOWS j + k] its digits for j < t, stepped as k_col_digits steps them (one
// power-chain start per chunk of KB_RC_POW_J exponents)
static void col_exponents(uint64_t x, size_t t, std::vector<uint32_t>& e, std::vector<int16_t>& dig)
{
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0}, xw[8] = {(uint32_t)x, (uint32_t)(x >> 32), 0, 0, 0, 0, 0, 0};
    e.assign(8 * t, 0);
    dig.assign(KB_COL_WINDOWS * t, 0);
    for (size_t j0 = 0; j0 < t; j0 += KB_RC_POW_J) {
        uint32_t a[8], r8;
        kb_col_power(a, r8, x, j0);
        for (size_t j = j0; j < t && j < j0 + KB_RC_POW_J; j++) {
            kb_col_exponent(&e[8 * j], a, r8);
            kb_col_recode(&dig[KB_COL_WINDOWS * j], &e[8 * j]);
            sc_muladd(a, a, xw, zero);
            r8 = (r8 * (uint32_t)x) & 7u;
        }
    }
}
// W = sum_j e_j C_j as k_rc_sort, k_col_msm and k_col_check compute it, with nch chunks per window
static void col_eval(ge_p3& W, const std::vector<ge_p3>& C, uint64_t x, size_t nch)
{
    const size_t t = C.size();
    std::vector<uint32_t> e;
    std::vector<int16_t> dig;
    col_exponents(x, t, e, dig);
    std::vector<ge_p3> parts((size_t)KB_COL_WINDOWS * nch);
    for (int k = 0; k < KB_COL_WINDOWS; k++) {
        std::vector<std::pair<int, uint32_t>> v;
        for (size_t j = 0; j < t; j++) {
            const int d = dig[KB_COL_WINDOWS * j + k];
            if (d) v.push_back({d < 0 ? -d : d, (uint32_t)j | (d < 0 ? 0x80000000u : 0u)});
        }
        std::stable_sort(v.begin(), v.end(), [](const std::pair<int, uint32_t>& a, const std::pair<int, uint32_t>& b) { return a.first > b.first; });
        std::vector<uint32_t> ent;
        std::vector<uint8_t> bkt;
        for (auto& q : v) {
            bkt.push_back((uint8_t)q.first);
            ent.push_back(q.second);
        }
        const size_t m = ent.size();
        for (size_t c = 0; c < nch; c++)
            kb_rc_chunk(parts[(size_t)k * nch + c], ent.data(), bkt.data(), m * c / nch, m * (c + 1) / nch, [&](uint32_t j, ge_p3& P) { P = C[j]; });
    }
    kb_rc_fold<KB_COL_WINDOWS>(W, nch, [&](size_t k, size_t c, ge_p3& P) { P = parts[k * nch + c]; });
}
static bool col_decode(std::vector<ge_p3>& C, const uint8_t* commits, size_t t)
{
    C.resize(t);
    for (size_t j = 0; j < t; j++) {
        uint32_t w[8];
        ld(w, commits + 32 * j, 8);
        if (!ge_decompress(C[j], w)) return false;
    }
    return true;
}

extern "C" {
void emu_col_exponents(uint64_t x, size_t t, uint8_t* e32, int16_t* dig)
{
    std::vector<uint32_t> e;
    std::vector<int16_t> d;
    col_exponents(x, t, e, d);
    st(e32, e.data(), 8 * (int)t);
    memcpy(dig, d.data(), sizeof(int16_t) * d.size());
}
void emu_col_recode(const uint8_t* e32, int16_t* dig)
{
    uint32_t e[8];
    ld(e, e32, 8);
    kb_col_recode(dig, e);
}
// out = encoding of sum_j (x^j mod 8L) C_j; 0 if a commitment does not decode
int emu_col_eval(uint8_t* out, const uint8_t* commits, size_t t, uint64_t x, size_t nch)
{
    std::vector<ge_p3> C;
    if (!col_decode(C, commits, t)) return 0;
    ge_p3 W;
    col_eval(W, C, x, nch);
    uint32_t o[8];
    ge_compress(o, W);
    st(out, o, 8);
    return 1;
}
// the verdict of k_col_check for one (column, dealer): eval(x) == s B with the base multiplication on the raw share bytes
int emu_col_check(const uint8_t* commits, size_t t, uint64_t x, const uint8_t* share, size_t nch)
{
    base_init();
    std::vector<ge_p3> C;
    if (!col_decode(C, commits, t)) return 0;
    ge_p3 W, h;
    col_eval(W, C, x, nch);
    uint32_t s[8];
    int8_t es[64];
    ld(s, share, 8);
    sc_recode16(es, s);
    ge_scalarmult_base<true>(h, es, g_base);
    return (int)kb_col_same(W, h);
}
}  // extern "C"
