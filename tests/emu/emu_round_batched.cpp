// tests/emu/emu_round_batched.cpp — HOST EMULATION of the batched share checks of a DKG round (dkgrlc.cuh).  TEST
// INFRASTRUCTURE ONLY.  It builds on tests/emu/emu.cpp (the same headers compiled with KB_HOST_EMU) and composes the
// per-thread bodies the kernels inline the way the kernels compose them.  Never linked into libkyber_b200.so.
#include "emu.cpp"
#include "../../kyber-rs_b200/csrc/dkgrlc.cuh"

#include <algorithm>

// z[16 i ..] = z_i, w[32 j ..] = w_j = sum_i z_i x_i^j mod L, summed as k_rc_weights sums them (64-bit words per j, one
// power-chain start per chunk of KB_RC_POW_J weights)
static void rc_weights(size_t n, size_t t, const kb_rc_seed& seed, std::vector<uint32_t>& z, std::vector<uint32_t>& w)
{
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    std::vector<uint64_t> acc(8 * t, 0);
    z.assign(8 * n, 0);
    for (size_t i = 0; i < n; i++) kb_rc_z(&z[8 * i], seed, i);
    for (size_t j0 = 0; j0 < t; j0 += KB_RC_POW_J)
        for (size_t i = 0; i < n; i++) {
            const uint64_t x = (uint64_t)i + 1;
            const uint32_t xw[8] = {(uint32_t)x, (uint32_t)(x >> 32), 0, 0, 0, 0, 0, 0};
            uint32_t y[8];
            kb_rc_pow_times(y, &z[8 * i], x, j0);
            for (size_t j = j0; j < t && j < j0 + KB_RC_POW_J; j++) {
                for (int k = 0; k < 8; k++) acc[8 * j + k] += y[k];
                sc_muladd(y, y, xw, zero);
            }
        }
    w.assign(8 * t, 0);
    for (size_t j = 0; j < t; j++) kb_rc_weight(&w[8 * j], &acc[8 * j]);
}

extern "C" {
void emu_rc_weights(size_t n, size_t t, const uint8_t* seed32, uint8_t* z16, uint8_t* w32)
{
    kb_rc_seed seed;
    ld(seed.w, seed32, 8);
    std::vector<uint32_t> z, w;
    rc_weights(n, t, seed, z, w);
    for (size_t i = 0; i < n; i++) st(z16 + 16 * i, &z[8 * i], 4);
    st(w32, w.data(), 8 * (int)t);
}
// signed radix-256 digits of one weight
void emu_rc_recode(const uint8_t* w32, int16_t* e)
{
    uint32_t w[8];
    ld(w, w32, 8);
    kb_rc_recode256(e, w);
}
// bit r = the torsion part of eval(x) vanishes for x = r (mod 8), from the [L] images of A_even, A_odd, C_0, C_1, C_2
uint32_t emu_rc_torsion_mask(size_t t, const uint8_t* commits)
{
    ge_p3 C, P[5], tl[5];
    ge_cached c;
    for (int q = 0; q < 5; q++) ge_identity(P[q]);
    for (size_t j = 0; j < t; j++) {
        uint32_t w[8];
        ld(w, commits + 32 * j, 8);
        if (!ge_decompress(C, w)) return 0xFFFFFFFFu;
        ge_to_cached(c, C);
        ge_add<true>(P[j & 1], P[j & 1], c);
        if (j < 3) P[2 + j] = C;
    }
    for (int q = 0; q < 5; q++) kb_rc_mul_l(tl[q], P[q]);
    return kb_rc_torsion_mask(tl);
}
// The state word of one dealer (KB_RC_PASS | ok mask, or KB_RC_FALLBACK) as k_rc_msm, k_rc_shares and k_rc_dealer compute
// it, with nch chunks per window; s_out = S_d.  Returns 0xFFFFFFFF for an undecodable commitment.
uint32_t emu_rc_dealer(size_t n, size_t t, const uint8_t* commits, const uint8_t* shares, const uint8_t* seed32, size_t nch, uint8_t* s_out)
{
    base_init();
    kb_rc_seed seed;
    ld(seed.w, seed32, 8);
    std::vector<uint32_t> z, w;
    rc_weights(n, t, seed, z, w);
    std::vector<ge_p3> C(t);
    for (size_t j = 0; j < t; j++) {
        uint32_t cw[8];
        ld(cw, commits + 32 * j, 8);
        if (!ge_decompress(C[j], cw)) return 0xFFFFFFFFu;
    }
    // per window: the j by bucket from the top down, then the chunks
    std::vector<ge_p3> parts((size_t)KB_RC_WINDOWS * nch);
    std::vector<int16_t> dig((size_t)KB_RC_WINDOWS * t);
    for (size_t j = 0; j < t; j++) {
        int16_t e[KB_RC_WINDOWS];
        kb_rc_recode256(e, &w[8 * j]);
        for (int k = 0; k < KB_RC_WINDOWS; k++) dig[(size_t)k * t + j] = e[k];
    }
    for (int k = 0; k < KB_RC_WINDOWS; k++) {
        std::vector<uint32_t> ent;
        std::vector<uint8_t> bkt;
        std::vector<std::pair<int, uint32_t>> v;
        for (size_t j = 0; j < t; j++) {
            const int d = dig[(size_t)k * t + j];
            if (d) v.push_back({d < 0 ? -d : d, (uint32_t)j | (d < 0 ? 0x80000000u : 0u)});
        }
        std::stable_sort(v.begin(), v.end(), [](const std::pair<int, uint32_t>& a, const std::pair<int, uint32_t>& b) { return a.first > b.first; });
        for (auto& e : v) {
            bkt.push_back((uint8_t)e.first);
            ent.push_back(e.second);
        }
        const size_t m = ent.size();
        for (size_t c = 0; c < nch; c++)
            kb_rc_chunk(parts[(size_t)k * nch + c], ent.data(), bkt.data(), m * c / nch, m * (c + 1) / nch, [&](uint32_t j, ge_p3& P) { P = C[j]; });
    }
    ge_p3 W, sb;
    kb_rc_fold(W, nch, [&](size_t k, size_t c, ge_p3& P) { P = parts[k * nch + c]; });
    uint32_t S[8] = {0, 0, 0, 0, 0, 0, 0, 0}, s[8], hi = 0;
    for (size_t i = 0; i < n; i++) {
        ld(s, shares + 32 * i, 8);
        hi |= s[7] >> 31;
        sc_muladd(S, &z[8 * i], s, S);
    }
    st(s_out, S, 8);
    int8_t es[64];
    sc_recode16(es, S);
    ge_scalarmult_base<true>(sb, es, g_base);
    const uint32_t pass = kb_rc_combination_ok(W, sb);
    const uint32_t okm = emu_rc_torsion_mask(t, commits);
    return (pass && !hi) ? (KB_RC_PASS | okm) : KB_RC_FALLBACK;
}
}  // extern "C"
