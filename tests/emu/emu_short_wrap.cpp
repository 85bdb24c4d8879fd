// tests/emu/emu_short_wrap.cpp — HOST EMULATION of the verifier as k_verify_half_main runs it with the short-wrap field
// bodies (fe.cuh fe_sw) and the exact redo behind them.  TEST INFRASTRUCTURE ONLY.  It builds on tests/emu/emu.cpp
// (the same headers compiled with KB_HOST_EMU, the host-built comb) by including it, and adds the entry points of
// tests/test_verify_short_wrap.py.  Never linked into libkyber_b200.so.
#include "emu.cpp"

extern "C" {
// One signature as k_verify_half_prep (exact bodies) and k_verify_half_main run it: the table build and the loop with the
// short-wrap bodies, redone with the exact bodies when the counter is not 0.  force = 1 starts the counter at 1 (what
// KB_VERIFY_FORCE_REDO does for a thread).  *ovf_out = the counter before any redo.
int emu_sig_verify_half_sw(int schnorr, const uint8_t* pk, const uint8_t* msg, uint64_t mlen, const uint8_t* sig, int min_windows, int force, uint32_t* ovf_out)
{
    uint32_t pw[8], sw[16];
    comb_init();
    ld(pw, pk, 8); ld(sw, sig, 16);
    if (min_windows < KB_HALF_MIN_WINDOWS) min_windows = KB_HALF_MIN_WINDOWS;
    kb_half_rec rec;
    if (schnorr) sig_half_prep<true>(rec, pw, sw, msg, mlen);
    else sig_half_prep<false>(rec, pw, sw, msg, mlen);
    kb_comb_digit dw[KB_COMB_POS];
    ge_cached tbl[KB_JOINT_SLOTS];
    uint32_t uk[8], vk[8];
    const int np0 = sc_joint4_pairs(rec.u, rec.v);
    const int np = np0 < 2 * min_windows ? 2 * min_windows : np0;
    fe_sw fm = {force ? 1u : 0u};
    sig_half_setup_joint(dw, uk, vk, tbl, rec, fm);
    ge_p3 W;
    ge_triple_scalarmult_joint<true>(W, np, dw, uk, vk, tbl, g_comb.data(), fm);
    *ovf_out = fm.ovf;
    if (fm.ovf) {
        fe_ex ex;
        sig_half_setup_joint(dw, uk, vk, tbl, rec, ex);
        ge_triple_scalarmult_joint<false>(W, np, dw, uk, vk, tbl, g_comb.data(), ex);
    }
    return schnorr ? (int)sig_half_finish<true>(rec.f, W) : (int)sig_half_finish<false>(rec.f, W);
}
}  // extern "C"
