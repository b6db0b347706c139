// CPU emulation harness for the backward kernel bodies (tests only, never shipped): the STFT adjoint on the inverse
// bodies (istft_core.cuh, aux_core.cuh) and the spectral / decibel VJP bodies (grad_core.cuh), compiled with
// KB_HOST_EMU so every barrier-free phase runs as a loop over the CTA's threads.
#define KB_HOST_EMU 1
#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <vector>
#include "../../kapre_b200/csrc/kb_tables.h"
#include "../../kapre_b200/csrc/stft_core.cuh"
#include "../../kapre_b200/csrc/istft_core.cuh"
#include "../../kapre_b200/csrc/aux_core.cuh"
#include "../../kapre_b200/csrc/grad_core.cuh"

template <int Q>
static void run_istft2_adjoint(const KbIstftParams& p, int n_cta) {
    const KbIstft2Smem L = kb_istft2_smem_layout(Q, p.n_fft, p.hop, p.win, p.n_warps);
    std::vector<char> smem(L.total + 64);
    for (int cta = 0; cta < n_cta; ++cta) {
        std::fill(smem.begin(), smem.end(), (char)0x7f);  // poison: catches reads of unwritten smem
        kb_istft2_cta<Q, true>(p, smem.data(), cta, n_cta);
    }
}

extern "C" {

// ---- backward kernel bodies (grad_core.cuh, and the inverse bodies as the STFT adjoint) --------------------------
// STFT adjoint: seg > 0 runs the streaming body (n_fft in {256..2048}) with tiles of seg hops, seg == 0 the direct body.
int kb_emu_stft_adjoint(const float* G, long long g_sb, long long g_sc, long long g_st, long long g_sk, int B, int C, int T,
                        int n_fft, int win_length, int hop, const float* window, int pad_left, int L, float* y,
                        long long y_sb, long long y_sc, long long y_sl, int seg, int n_warps, int n_cta) {
    const int win = win_length < n_fft ? win_length : n_fft;
    const long long out_len = (long long)pad_left + L;
    std::vector<float> wa(win), dn(win);
    for (int m = 0; m < win; ++m) {
        wa[m] = (float)(0.5 * (double)n_fft * (double)window[m]);
        dn[m] = (float)(0.5 * (double)window[m]);
    }
    if (seg > 0) {
        const int Q = kb_q_for_nfft(n_fft);
        if (!Q || T < 1) return -1;
        std::vector<float> adj;
        std::vector<float2> twp, twn;
        kb_make_dual(wa.data(), win, n_fft, adj);
        kb_make_twp(Q, twp);
        kb_make_twn(n_fft, twn);
        KbIstftParams p{};
        p.X = reinterpret_cast<const float2*>(G); p.x_sb = g_sb; p.x_sc = g_sc; p.x_st = g_st; p.x_sk = g_sk;
        p.B = B; p.C = C; p.T = T; p.n_fft = n_fft; p.hop = hop; p.win = win;
        p.out_len = (int)out_len;
        p.dual = adj.data(); p.twp = twp.data(); p.twn = twn.data();
        p.y = y; p.y_sb = y_sb; p.y_sc = y_sc; p.y_sl = y_sl;
        p.R = (win + hop - 1) / hop; p.seg = seg;
        const long long hops = (out_len + hop - 1) / hop;
        p.n_tiles_t = (int)((hops + seg - 1) / seg);
        p.n_warps = n_warps;
        p.y_off = pad_left; p.edge2 = 1;
        switch (Q) {
            case 4: run_istft2_adjoint<4>(p, n_cta); break;
            case 8: run_istft2_adjoint<8>(p, n_cta); break;
            case 16: run_istft2_adjoint<16>(p, n_cta); break;
            case 32: run_istft2_adjoint<32>(p, n_cta); break;
        }
        return 0;
    }
    std::vector<float2> tw(n_fft);
    for (int r = 0; r < n_fft; ++r) {
        const double a = 2.0 * M_PI * (double)r / (double)n_fft;
        tw[r] = make_float2((float)cos(a), (float)sin(a));
    }
    KbIdftParams p{};
    p.X = reinterpret_cast<const float2*>(G); p.x_sb = g_sb; p.x_sc = g_sc; p.x_st = g_st; p.x_sk = g_sk;
    p.B = B; p.C = C; p.T = T; p.n_fft = n_fft; p.hop = hop; p.win = win;
    p.out_len = (int)out_len; p.dualn = dn.data(); p.tw = tw.data();
    p.y = y; p.y_sb = y_sb; p.y_sc = y_sc; p.y_sl = y_sl;
    p.y_off = pad_left; p.edge2 = 1;
    p.n_warps = 8; p.n_tiles_s = (int)((out_len + 255) / 256);
    std::vector<char> smem((size_t)n_fft * 8 + 64);
    for (int cta = 0; cta < n_cta; ++cta) {
        std::fill(smem.begin(), smem.end(), (char)0x7f);
        kb_idft_cta(p, smem.data(), cta, n_cta);
    }
    return 0;
}

// Decibel statistics (kb_dbstat_cta) over (n_items, d1, d2, d3) views; stats: 4 floats per item.  Runs the CTAs of
// each item in the order given by `order` (a permutation of the n_items * chunks CTAs) to show the combine does not
// depend on the arrival order.
int kb_emu_dbstat(const float* y, long long y_s0, long long y_s1, long long y_s2, long long y_s3, const float* g,
                  long long g_s0, long long g_s1, long long g_s2, long long g_s3, int n_items, int d1, int d2, int d3,
                  int chunks, float dyn_range, const int* order, float* stats) {
    std::vector<KbDbStats> part((size_t)n_items * chunks);
    std::vector<unsigned int> arrive(n_items, 0u);
    KbDbStatParams q{};
    q.y = y; q.y_s0 = y_s0; q.y_s1 = y_s1; q.y_s2 = y_s2; q.y_s3 = y_s3;
    q.g = g; q.g_s0 = g_s0; q.g_s1 = g_s1; q.g_s2 = g_s2; q.g_s3 = g_s3;
    q.n_items = n_items; q.d1 = d1; q.d2 = d2; q.d3 = d3; q.chunks = chunks; q.dyn_range = dyn_range;
    q.part = part.data(); q.arrive = arrive.data(); q.stats = reinterpret_cast<KbDbStats*>(stats);
    std::vector<char> smem(KB_DBS_THREADS * sizeof(KbDbStats) + 16);
    for (int i = 0; i < n_items * chunks; ++i) kb_dbstat_cta(q, smem.data(), order[i], n_items * chunks);
    for (int i = 0; i < n_items; ++i)
        if (arrive[i] != 0u) return -2;     // the counters must be left at zero
    return 0;
}

// Spectral VJP (kb_specvjp_cta), channels_first / channels_last by strides; stats as kb_emu_dbstat wrote them.
int kb_emu_specvjp(const float* X, long long x_sb, long long x_sc, long long x_st, long long x_sk, const float* g,
                   long long g_sb, long long g_sc, long long g_st, long long g_sk, const float* y, long long y_sb,
                   long long y_sc, long long y_st, long long y_sk, int B, int C, int T, int F, const float* fb, int n_bands,
                   int db, float amin, const float* stats, float* G, int n_warps, int n_cta) {
    std::vector<KbBand> bands, bandsT;
    std::vector<float> w, wT;
    const int fbm = fb != nullptr;
    if (fbm) {
        kb_make_bands(fb, F, n_bands, bands, w);
        std::vector<float> fbT((size_t)F * n_bands);
        for (int k = 0; k < F; ++k)
            for (int m = 0; m < n_bands; ++m) fbT[(size_t)m * F + k] = fb[(size_t)k * n_bands + m];
        kb_make_bands(fbT.data(), n_bands, F, bandsT, wT);
    }
    KbSpecVjpParams p{};
    p.X = reinterpret_cast<const float2*>(X); p.x_sb = x_sb; p.x_sc = x_sc; p.x_st = x_st; p.x_sk = x_sk;
    p.G = reinterpret_cast<float2*>(G); p.G_sb = x_sb; p.G_sc = x_sc; p.G_st = x_st; p.G_sk = x_sk;
    p.g = g; p.g_sb = g_sb; p.g_sc = g_sc; p.g_st = g_st; p.g_sk = g_sk;
    p.y = y; p.y_sb = y_sb; p.y_sc = y_sc; p.y_st = y_st; p.y_sk = y_sk;
    p.B = B; p.C = C; p.T = T; p.F = F; p.K = fbm ? n_bands : F;
    p.fb = fbm; p.db = db;
    if (fbm) { p.bands = bands.data(); p.fbw = w.data(); p.bandsT = bandsT.data(); p.fbwT = wT.data(); }
    p.amin = amin; p.stats = reinterpret_cast<const KbDbStats*>(stats); p.n_warps = n_warps;
    const KbSpecVjpSmem L_ = kb_specvjp_smem_layout(F, p.K);
    std::vector<char> smem(L_.total + 64);
    for (int cta = 0; cta < n_cta; ++cta) {
        std::fill(smem.begin(), smem.end(), (char)0x7f);
        kb_specvjp_cta(p, smem.data(), cta, n_cta);
    }
    return 0;
}

}  // extern "C"
