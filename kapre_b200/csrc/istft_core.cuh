// Inverse STFT kernel body: complex-to-real FFT + dual window + overlap-add.
//
// Replaces tf.signal.inverse_stft as called at kapre/time_frequency.py:307-314
// (irfft(n_fft) -> keep the first win_length samples -> * inverse_stft_window_fn window
// (kapre/time_frequency.py:278-280) -> overlap_and_add), plus the layout transposes of
// kapre/time_frequency.py:304-305,316-317 via element strides.
//
// Gather formulation, no atomics: a tile owns `hops_out` output hops of one (batch, channel)
// signal and recomputes the R-1 halo frames that overlap into it.  Frames are processed in
// R = ceil(win/hop) classes (t mod R); frames of one class never overlap, so the
// shared-memory overlap-add is a plain read-modify-write, with a CTA barrier between classes.
//
// irfft of length N via one complex FFT of length P = N/2 (same register FFT as the forward
// kernel, run on conj(Z) to invert):  Z[k] = E[k] + i O[k],
//   E[k] = (X[k] + conj X[P-k]) / 2,  O[k] = exp(+2 pi i k / N) (X[k] - conj X[P-k]) / 2,
// z = IFFT_P(Z) gives x[2n] = Re z[n], x[2n+1] = Im z[n].  The 1/2, the 1/P and the sign of
// the odd samples are folded into the dual-window table.
#pragma once
#include "stft_core.cuh"

struct KbIstftSmem {
    int dual, twp, twn, ola, ex, total;
    int ola_len;
};

KB_HD KbIstftSmem kb_istft_smem_layout(int Q, int n_fft, int hop, int win, int TFc, int n_warps) {
    KbIstftSmem s;
    const int P = 32 * Q;
    int off = 0;
    s.dual = off; off += kb_align16((win + 2) * 4);
    s.twp = off;  off += kb_align16(Q * 33 * 8);
    s.twn = off;  off += kb_align16((P / 2) * 8);
    s.ola_len = TFc * hop + win + 2;
    s.ola = off;  off += kb_align16(s.ola_len * 4);
    s.ex = off;   off += n_warps * (32 * 33 * 8);
    s.total = off;
    (void)n_fft;
    return s;
}

KB_HD int kb_istft_tiles(int T, int hop, int win_length, int hops_out) {
    const int out_len = (T - 1) * hop + win_length;
    const int hops = (out_len + hop - 1) / hop;
    return (hops + hops_out - 1) / hops_out;
}


template <int Q>
#if defined(KB_HOST_EMU)
inline void kb_istft_cta(const KbIstftParams& p, char* smem, int cta, int n_cta)
#else
__device__ __forceinline__ void kb_istft_cta(const KbIstftParams& p, char* smem, int cta, int n_cta)
#endif
{
    constexpr int P = 32 * Q;
    constexpr int FPW = 32 / Q;
    constexpr int ZSTR = P + Q;
    constexpr int EXW = 32 * 33;
    const int NW = p.n_warps;
    const int kb_nt = NW * 32;
    (void)kb_nt;
    const int H = p.hop, TFc = p.TFc, R_ = p.R, win = p.win;
    const KbIstftSmem L = kb_istft_smem_layout(Q, p.n_fft, H, win, TFc, NW);
    float* dual_s = reinterpret_cast<float*>(smem + L.dual);
    cpx* twp_s = reinterpret_cast<cpx*>(smem + L.twp);
    cpx* twn_s = reinterpret_cast<cpx*>(smem + L.twn);
    float* ola_s = reinterpret_cast<float*>(smem + L.ola);
    cpx* ex_s = reinterpret_cast<cpx*>(smem + L.ex);
    const int FR = NW * FPW;
    const int n_tiles = p.B * p.C * p.n_tiles_t;

#if defined(KB_HOST_EMU)
    std::vector<KbThreadRegs> kb_regs(kb_nt);
#else
    KbThreadRegs kb_regs;
#endif

    KB_PHASE_BEGIN
        (void)R;
        for (int i = tid; i < win + 2; i += kb_nt) dual_s[i] = p.dual[i];
        for (int i = tid; i < Q * 33; i += kb_nt) { float2 t = p.twp[i]; twp_s[i] = cmake(t.x, t.y); }
        for (int i = tid; i < P / 2; i += kb_nt) { float2 t = p.twn[i]; twn_s[i] = cmake(t.x, t.y); }
    KB_PHASE_END
    KB_SYNC_CTA;

    for (int tile = cta; tile < n_tiles; tile += n_cta) {
        const int sig = tile / p.n_tiles_t;
        const int tt = tile - sig * p.n_tiles_t;
        const int b = sig / p.C, c = sig - b * p.C;
        const int h0 = tt * p.hops_out;          // first output hop of the tile
        const int tf0 = h0 - (R_ - 1);           // first (possibly negative) frame computed
        const float2* Xsig = p.X + (long long)b * p.x_sb + (long long)c * p.x_sc;

        KB_PHASE_BEGIN
            (void)R;
            for (int i = tid; i < L.ola_len; i += kb_nt) ola_s[i] = 0.0f;
        KB_PHASE_END
        KB_SYNC_CTA;

        for (int cl = 0; cl < R_; ++cl) {
            const int n_in_class = (TFc - cl + R_ - 1) / R_;   // frames fi = cl + R*idx < TFc
            const int n_rounds = (n_in_class + FR - 1) / FR;
            for (int round = 0; round < n_rounds; ++round) {
                // ---- phase 1: X[k], X[P-k] -> conj(2 Z[k]), conj(2 Z[P-k]) in natural order ----
                KB_PHASE_BEGIN
                    (void)R;
                    const int warp = tid >> 5, lane = tid & 31;
                    // all of the round's global loads are issued before the first use (FPW frames x Q/2 bin pairs)
                    float2 xa[FPW][Q / 2], xb[FPW][Q / 2], xm[FPW];
                    bool live[FPW];
#pragma unroll
                    for (int gg = 0; gg < FPW; ++gg) {
                        const int idx = round * FR + warp * FPW + gg;
                        const int fi = cl + R_ * idx;
                        const int t = tf0 + fi;
                        live[gg] = !(fi >= TFc || t < 0 || t >= p.T);
                        xm[gg] = make_float2(0.0f, 0.0f);
                        if (live[gg]) {
                            const float2* Xf = Xsig + (long long)t * p.x_st;
#pragma unroll
                            for (int i = 0; i < Q / 2; ++i) {
                                const int k = lane + 32 * i;
                                xa[gg][i] = Xf[(long long)k * p.x_sk];
                                xb[gg][i] = Xf[(long long)(P - k) * p.x_sk];
                            }
                            if (lane == 0) xm[gg] = Xf[(long long)(P / 2) * p.x_sk];
                        }
                    }
#pragma unroll
                    for (int gg = 0; gg < FPW; ++gg) {
                        if (!live[gg]) continue;
                        cpx* zf = ex_s + warp * EXW + gg * ZSTR;
#pragma unroll
                        for (int i = 0; i < Q / 2; ++i) {
                            const int k = lane + 32 * i;
                            float2 a = xa[gg][i];
                            float2 bq = xb[gg][i];
                            if (k == 0) { a.y = 0.0f; bq.y = 0.0f; }  // C2R ignores Im of DC / Nyquist
                            const cpx W = twn_s[k];
                            const float Er = a.x + bq.x, Ei = a.y - bq.y;
                            const float dr = a.x - bq.x, di = a.y + bq.y;
                            const float Or = W.re * dr + W.im * di;
                            const float Oi = W.re * di - W.im * dr;
                            zf[k] = cmake(Er - Oi, -(Ei + Or));
                            if (k != 0) zf[P - k] = cmake(Er + Oi, Ei - Or);
                        }
                        if (lane == 0) zf[P / 2] = cmake(2.0f * xm[gg].x, 2.0f * xm[gg].y);
                    }
                KB_PHASE_END
                KB_SYNC_WARP;
                // ---- phase 2a: strided gather of the packed sequence into registers ----------
                KB_PHASE_BEGIN
                    const int warp = tid >> 5, lane = tid & 31;
                    const int g = lane / Q, q = lane % Q;
                    const int idx = round * FR + warp * FPW + g;
                    const int fi = cl + R_ * idx;
                    const int t = tf0 + fi;
                    if (fi < TFc && t >= 0 && t < p.T) {
                        const cpx* zf = ex_s + warp * EXW + g * ZSTR;
#pragma unroll
                        for (int j = 0; j < 32; ++j) R.v[j] = zf[q + Q * j];
                    }
                KB_PHASE_END
                KB_SYNC_WARP;
                // ---- phase 2b: 32-point DFTs, twiddle, transpose-store ------------------------
                KB_PHASE_BEGIN
                    const int warp = tid >> 5, lane = tid & 31;
                    const int g = lane / Q, q = lane % Q;
                    const int idx = round * FR + warp * FPW + g;
                    const int fi = cl + R_ * idx;
                    const int t = tf0 + fi;
                    if (fi < TFc && t >= 0 && t < p.T) {
                        kb_fft_dif<32>(R.v);
                        cpx* ex = ex_s + warp * EXW + (g * Q + q) * 33;
                        const cpx* tw = twp_s + q * 33;
                        ex[0] = R.v[0];
#pragma unroll
                        for (int k1 = 1; k1 < 32; ++k1) ex[k1] = cmul(R.v[kb_brev<32>(k1)], tw[k1]);
                    }
                KB_PHASE_END
                KB_SYNC_WARP;
                // ---- phase 3: column gather, Q-point DFTs, window, overlap-add ----------------
                KB_PHASE_BEGIN
                    const int warp = tid >> 5, lane = tid & 31;
                    const int g = lane / Q, q = lane % Q;
                    const int idx = round * FR + warp * FPW + g;
                    const int fi = cl + R_ * idx;
                    const int t = tf0 + fi;
                    if (fi < TFc && t >= 0 && t < p.T) {
                        const cpx* ex = ex_s + warp * EXW + (g * Q) * 33;
#pragma unroll
                        for (int i = 0; i < FPW; ++i) {
                            const int k1 = q + Q * i;
#pragma unroll
                            for (int q2 = 0; q2 < Q; ++q2) R.v[i * Q + q2] = ex[q2 * 33 + k1];
                        }
                        float* of = ola_s + fi * H;
                        const bool pair_ok = ((fi * H) & 1) == 0;
#pragma unroll
                        for (int i = 0; i < FPW; ++i) {
                            kb_fft_dif<Q>(R.v + i * Q);
                            const int k1 = q + Q * i;
#pragma unroll
                            for (int k2 = 0; k2 < Q; ++k2) {
                                const int m2 = 2 * (k1 + 32 * k2);
                                const cpx r = R.v[i * Q + kb_brev<Q>(k2)];
                                if (pair_ok && m2 + 1 < win) {      // aligned sample pair: one 8-byte read-modify-write
                                    cpx* o2 = reinterpret_cast<cpx*>(of + m2);
                                    const cpx d2 = *reinterpret_cast<const cpx*>(dual_s + m2);
                                    *o2 = cadd(*o2, cmul_elem(r, d2));
                                } else {
                                    if (m2 < win) of[m2] += r.re * dual_s[m2];
                                    if (m2 + 1 < win) of[m2 + 1] += r.im * dual_s[m2 + 1];
                                }
                            }
                        }
                    }
                KB_PHASE_END
                KB_SYNC_WARP;
            }
            KB_SYNC_CTA;  // the next class overlaps this one's samples
        }

        // ---- copy the tile's completed hops out ------------------------------------------------
        KB_PHASE_BEGIN
            (void)R;
            const long long s_begin = (long long)h0 * H;
            long long s_end = s_begin + (long long)p.hops_out * H;
            if (s_end > p.out_len) s_end = p.out_len;
            float* ysig = p.y + (long long)b * p.y_sb + (long long)c * p.y_sc;
            const int shift = (R_ - 1) * H;
            for (long long s = s_begin + tid; s < s_end; s += kb_nt)
                ysig[s * p.y_sl] = ola_s[(int)(s - s_begin) + shift];
        KB_PHASE_END
        KB_SYNC_CTA;
    }
}


// ------------------------------------------------------------------------------------------------
// Streaming formulation (round 2).  A tile owns `seg` consecutive output hops of one signal and walks
// them in rounds of FR = n_warps * FPW consecutive frames.  Per round every warp inverse-transforms its
// frames exactly as above but leaves the windowed time-domain frame in its OWN exchange region (the
// frame's 2P floats fit the (P + Q) complex slots its spectrum occupied); after one CTA barrier all
// threads gather-sum the <= R frames that cover each output sample, add the carry of the previous round
// (the win - hop samples past the last complete hop), store the FR complete hops and write the new
// carry.  Against the class-ordered overlap-add above: no (TFc * hop + win) accumulation buffer (37 KB
// at n_fft 1024 -- it capped the residency at two 4-warp CTAs per SM), one shared-memory store + <= R
// loads per sample instead of R read-modify-writes, R - 1 halo frames per `seg` hops instead of per 29.
struct KbIstft2Smem {
    int dual, twp, twn, carry, ex, total;
    int carry_len;            // floats per carry buffer (two of them, ping-pong)
};

KB_HD KbIstft2Smem kb_istft2_smem_layout(int Q, int n_fft, int hop, int win, int n_warps) {
    KbIstft2Smem s;
    const int P = 32 * Q;
    int off = 0;
    s.dual = off; off += kb_align16((n_fft + 4) * 4);      // zero beyond win: samples past win_length vanish in the frame
    s.twp = off;  off += kb_align16(Q * 33 * 8);
    s.twn = off;  off += kb_align16((P / 2) * 8);
    s.carry_len = win > hop ? ((win - hop + 3) & ~3) : 4;
    s.carry = off; off += 2 * kb_align16(s.carry_len * 4);
    s.ex = off;   off += n_warps * (32 * 33 * 8);
    s.total = off;
    return s;
}

KB_HD int kb_istft2_tiles(int T, int hop, int win_length, int seg) {
    const long long out_len = (long long)(T - 1) * hop + win_length;
    const long long hops = (out_len + hop - 1) / hop;
    return (int)((hops + seg - 1) / seg);
}

// Spectrum prefetch of the streaming kernel: the 16 bin pairs (X[k], X[P-k]) a lane needs for its warp's frames of the
// round that starts at frame number tfr, into the FFT registers -- those are idle from the end
// of phase 3b to phase 2a of the next round, so the global loads fly during the CTA barrier and the gather phase instead of
// stalling phase 1.  R.v[e] = X[k], R.v[16 + e] = X[P - k] for e = gg * (Q/2) + i, k = lane + 32 i; lane gg's R.aux = X[P/2] of frame gg.
template <int Q>
KB_FN void kb_istft2_prefetch(KbThreadRegs& R, const KbIstftParams& p, const float2* Xsig, int tid, int tfr) {
    constexpr int P = 32 * Q, FPW = 32 / Q, HQ = Q / 2;
    const int warp = tid >> 5, lane = tid & 31;
    // branch-free: frames outside [0, T) (and the ones past the tile's last frame) read a clamped, valid row whose values
    // phase 1 never uses -- 32 independent loads issue back to back (per-pair `if (live)` blocks made each pair wait for
    // the one before: 0.27 -> 0.44 ms at B256 x 5 s)
    const float2* Xf[FPW];
#pragma unroll
    for (int gg = 0; gg < FPW; ++gg) {
        int t = tfr + warp * FPW + gg;
        t = t < 0 ? 0 : (t > p.T - 1 ? p.T - 1 : t);
        Xf[gg] = Xsig + (long long)t * p.x_st;
    }
    if (p.x_sk == 1) {     // contiguous bins: one base per lane, compile-time offsets
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            const int gg = e / HQ, i = e % HQ;
            const float2 a = (Xf[gg] + lane)[32 * i];
            const float2 b = (Xf[gg] + (P - lane))[-32 * i];
            R.v[e] = cmake(a.x, a.y);
            R.v[16 + e] = cmake(b.x, b.y);
        }
    } else {
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            const int gg = e / HQ, i = e % HQ;
            const int k = lane + 32 * i;
            const float2 a = Xf[gg][(long long)k * p.x_sk];
            const float2 b = Xf[gg][(long long)(P - k) * p.x_sk];
            R.v[e] = cmake(a.x, a.y);
            R.v[16 + e] = cmake(b.x, b.y);
        }
    }
    {   // lane gg fetches the middle bin of the warp's frame gg (lanes >= FPW: a harmless duplicate of frame FPW - 1's)
        int t = tfr + warp * FPW + (lane < FPW ? lane : FPW - 1);
        t = t < 0 ? 0 : (t > p.T - 1 ? p.T - 1 : t);
        const float2 m = Xsig[(long long)t * p.x_st + (long long)(P / 2) * p.x_sk];
        R.aux = cmake(m.x, m.y);
    }
}

// ADJ: the STFT adjoint (kapre_stft_backward) -- honours p.y_off and p.edge2; the inverse instantiation ignores both.
template <int Q, bool ADJ = false>
#if defined(KB_HOST_EMU)
inline void kb_istft2_cta(const KbIstftParams& p, char* smem, int cta, int n_cta)
#else
__device__ __forceinline__ void kb_istft2_cta(const KbIstftParams& p, char* smem, int cta, int n_cta)
#endif
{
    constexpr int P = 32 * Q;
    constexpr int FPW = 32 / Q;
    constexpr int ZSTR = P + Q;
    constexpr int EXW = 32 * 33;
    const int NW = p.n_warps;
    const int kb_nt = NW * 32;
    (void)kb_nt;
    const int H = p.hop, win = p.win, Rm1 = p.R - 1, seg = p.seg;
    const KbIstft2Smem L = kb_istft2_smem_layout(Q, p.n_fft, H, win, NW);
    float* dual_s = reinterpret_cast<float*>(smem + L.dual);
    cpx* twp_s = reinterpret_cast<cpx*>(smem + L.twp);
    cpx* twn_s = reinterpret_cast<cpx*>(smem + L.twn);
    float* carry_s = reinterpret_cast<float*>(smem + L.carry);
    const int carry_stride = kb_align16(L.carry_len * 4) / 4;
    cpx* ex_s = reinterpret_cast<cpx*>(smem + L.ex);
    const int FR = NW * FPW;                       // frames per round
    const int clen = win > H ? win - H : 0;        // live carry samples
    const int n_tiles = p.B * p.C * p.n_tiles_t;
    const int n_need = seg + Rm1;                  // frames a tile transforms (incl. the R - 1 halo frames in front)
    const int n_rounds = (n_need + FR - 1) / FR;
    const bool vec4 = (H & 3) == 0 && (win & 3) == 0;
    // phase 4 walks (hop row, float4 in the row) pairs; a thread's next pair is kb_nt further on
    const int n_rows = FR + (clen + H - 1) / H;
    const int step_h = vec4 ? kb_nt / (H >> 2) : 0, step_i = vec4 ? kb_nt - step_h * (H >> 2) : 0;

#if defined(KB_HOST_EMU)
    std::vector<KbThreadRegs> kb_regs(kb_nt);
#else
    KbThreadRegs kb_regs;
#endif

    KB_PHASE_BEGIN
        (void)R;
        for (int i = tid; i < p.n_fft + 4; i += kb_nt) dual_s[i] = i < win ? p.dual[i] : 0.0f;
        for (int i = tid; i < Q * 33; i += kb_nt) { float2 t = p.twp[i]; twp_s[i] = cmake(t.x, t.y); }
        for (int i = tid; i < P / 2; i += kb_nt) { float2 t = p.twn[i]; twn_s[i] = cmake(t.x, t.y); }
    KB_PHASE_END
    KB_SYNC_CTA;

    for (int tile = cta; tile < n_tiles; tile += n_cta) {
        const int sig = tile / p.n_tiles_t;
        const int tt = tile - sig * p.n_tiles_t;
        const int b = sig / p.C, c = sig - b * p.C;
        const int h0 = tt * seg;                 // first output hop of the tile
        const int tf0 = h0 - Rm1;                // first (possibly negative) frame transformed
        const float2* Xsig = p.X + (long long)b * p.x_sb + (long long)c * p.x_sc;
        // (shifted by y_off: sample s is stored at y[s - y_off]; only s >= y_off is stored)
        const int y_off = ADJ ? p.y_off : 0;
        float* ysig = p.y + (long long)b * p.y_sb + (long long)c * p.y_sc - (long long)y_off * p.y_sl;
        long long s_lo = (long long)h0 * H;
        long long s_hi = s_lo + (long long)seg * H;
        if (s_lo < y_off) s_lo = y_off;
        if (s_hi > p.out_len) s_hi = p.out_len;

        KB_PHASE_BEGIN
            for (int i = tid; i < L.carry_len; i += kb_nt) carry_s[i] = 0.0f;
            kb_istft2_prefetch<Q>(R, p, Xsig, tid, tf0);
        KB_PHASE_END
        // (the first read of the carry is behind the round's CTA barrier)

        for (int round = 0; round < n_rounds; ++round) {
            const int f_base = round * FR;       // index of the round's first frame within the tile
            const int tfr = tf0 + f_base;        // its frame number
            // ---- phase 1: X[k], X[P-k] -> conj(2 Z[k]), conj(2 Z[P-k]) in natural order ----
            KB_PHASE_BEGIN
                const int warp = tid >> 5, lane = tid & 31;
                // the lane's 16 bin pairs were prefetched into R.v (kb_istft2_prefetch) one round ahead
                constexpr int HQ = Q / 2;
#pragma unroll
                for (int e = 0; e < 16; ++e) {
                    const int gg = e / HQ, i = e % HQ;
                    const int fl = warp * FPW + gg;
                    const int t = tfr + fl;
                    if (!(f_base + fl < n_need && t >= 0 && t < p.T)) continue;
                    cpx* zf = ex_s + warp * EXW + gg * ZSTR;
                    const int k = lane + 32 * i;
                    cpx a = R.v[e];
                    cpx bq = R.v[16 + e];
                    if (k == 0) {                               // C2R ignores Im of DC / Nyquist
                        a.im = 0.0f; bq.im = 0.0f;
                        if (ADJ && p.edge2) { a.re *= 2.0f; bq.re *= 2.0f; }
                    }
                    const cpx W = twn_s[k];
                    // packed arithmetic: E = a + conj(b), D = a - conj(b), O = conj(W) D;
                    // conj(2 Z[k]) = conj(E + i O), conj(2 Z[P-k]) = E - i O
                    const cpx E = cadd_conj(a, bq);
                    const cpx D = csub_conj(a, bq);
                    const cpx O = cmul(D, cmake(W.re, -W.im));
                    const cpx iO = cmake(-O.im, O.re);
                    const cpx S = cadd(E, iO);
                    zf[k] = cmake(S.re, -S.im);
                    if (k != 0) zf[P - k] = csub(E, iO);
                }
                if (lane < FPW) {
                    const int fl = warp * FPW + lane;
                    const int t = tfr + fl;
                    if (f_base + fl < n_need && t >= 0 && t < p.T)
                        ex_s[warp * EXW + lane * ZSTR + P / 2] = cmake(2.0f * R.aux.re, 2.0f * R.aux.im);
                }
            KB_PHASE_END
            KB_SYNC_WARP;
            // ---- phase 2a: strided gather of the packed sequence into registers ----------
            KB_PHASE_BEGIN
                const int warp = tid >> 5, lane = tid & 31;
                const int g = lane / Q, q = lane % Q;
                const int fl = warp * FPW + g;
                const int t = tfr + fl;
                if (f_base + fl < n_need && t >= 0 && t < p.T) {
                    const cpx* zf = ex_s + warp * EXW + g * ZSTR;
#pragma unroll
                    for (int j = 0; j < 32; ++j) R.v[j] = zf[q + Q * j];
                }
            KB_PHASE_END
            KB_SYNC_WARP;
            // ---- phase 2b: 32-point DFTs, twiddle, transpose-store ------------------------
            KB_PHASE_BEGIN
                const int warp = tid >> 5, lane = tid & 31;
                const int g = lane / Q, q = lane % Q;
                const int fl = warp * FPW + g;
                const int t = tfr + fl;
                if (f_base + fl < n_need && t >= 0 && t < p.T) {
                    kb_fft_dif<32>(R.v);
                    cpx* ex = ex_s + warp * EXW + (g * Q + q) * 33;
                    const cpx* tw = twp_s + q * 33;
                    ex[0] = R.v[0];
#pragma unroll
                    for (int k1 = 1; k1 < 32; ++k1) ex[k1] = cmul(R.v[kb_brev<32>(k1)], tw[k1]);
                }
            KB_PHASE_END
            KB_SYNC_WARP;
            // ---- phase 3a: column gather --------------------------------------------------
            KB_PHASE_BEGIN
                const int warp = tid >> 5, lane = tid & 31;
                const int g = lane / Q, q = lane % Q;
                const int fl = warp * FPW + g;
                const int t = tfr + fl;
                if (f_base + fl < n_need && t >= 0 && t < p.T) {
                    const cpx* ex = ex_s + warp * EXW + (g * Q) * 33;
#pragma unroll
                    for (int i = 0; i < FPW; ++i) {
                        const int k1 = q + Q * i;
#pragma unroll
                        for (int q2 = 0; q2 < Q; ++q2) R.v[i * Q + q2] = ex[q2 * 33 + k1];
                    }
                }
            KB_PHASE_END
            KB_SYNC_WARP;    // every lane has its columns: the frame's slots may now take the time-domain samples
            // ---- phase 3b: Q-point DFTs, dual window, frame left in place (natural sample order) ----
            KB_PHASE_BEGIN
                const int warp = tid >> 5, lane = tid & 31;
                const int g = lane / Q, q = lane % Q;
                const int fl = warp * FPW + g;
                const int t = tfr + fl;
                if (f_base + fl < n_need && t >= 0 && t < p.T) {
                    cpx* fr = ex_s + warp * EXW + g * ZSTR;
                    const cpx* d2 = reinterpret_cast<const cpx*>(dual_s);
#pragma unroll
                    for (int i = 0; i < FPW; ++i) {
                        kb_fft_dif<Q>(R.v + i * Q);
                        const int k1 = q + Q * i;
#pragma unroll
                        for (int k2 = 0; k2 < Q; ++k2) {
                            const int cidx = k1 + 32 * k2;       // samples 2 cidx, 2 cidx + 1
                            fr[cidx] = cmul_elem(R.v[i * Q + kb_brev<Q>(k2)], d2[cidx]);
                        }
                    }
                }
                // the FFT registers are free until phase 2a of the next round: fetch that round's spectra into them now
                if (round + 1 < n_rounds) kb_istft2_prefetch<Q>(R, p, Xsig, tid, tfr + FR);
            KB_PHASE_END
            KB_SYNC_CTA;
            // ---- phase 4: gather-sum the frames over each sample, store FR hops, write the new carry ----
            KB_PHASE_BEGIN
                (void)R;
                const float* cin = carry_s + (round & 1) * carry_stride;
                float* cout = carry_s + ((round & 1) ^ 1) * carry_stride;
                const int E = FR * H + clen;             // samples touched by this round
                // frames of this round that exist
                int fv_lo = -tfr; if (fv_lo < 0) fv_lo = 0;
                int fv_hi = FR - 1;
                if (fv_hi > p.T - 1 - tfr) fv_hi = p.T - 1 - tfr;
                if (fv_hi > n_need - 1 - f_base) fv_hi = n_need - 1 - f_base;
                const long long s0 = (long long)tfr * H; // sample number of u = 0
                const bool yvec = vec4 && p.y_sl == 1 && ((reinterpret_cast<uintptr_t>(ysig) & 15) == 0);
                // range of u this tile stores (complete hops of the round that lie in the tile's segment)
                const int FRH = FR * H;
                const long long lo64 = s_lo - s0, hi64 = s_hi - s0;
                const int u_lo = lo64 < 0 ? 0 : (lo64 > FRH ? FRH : (int)lo64);
                const int u_hi = hi64 < 0 ? 0 : (hi64 > FRH ? FRH : (int)hi64);
                if (vec4) {
                    // (hop row h, float4 i4 within the row), stepped without divisions: u = h H + 4 i4 is covered by the frames
                    // f = h, h - 1, ... at offsets 4 i4, 4 i4 + H, ... (< win).  Frame f's samples start at float 2 ZSTR f
                    // of the exchange area (FPW ZSTR = 32 * 33: the warps' regions continue the stride).
                    const int H4 = H >> 2;
                    const int Rw = (win + H - 1) / H, rem_w = win - (Rw - 1) * H;   // once per round, not per element
                    const float* exf = reinterpret_cast<const float*>(ex_s);
                    const int dstep = H - 2 * ZSTR;      // frame f -> f - 1 at the same output sample
                    float* yrow = ysig + s0;             // only dereferenced inside [u_lo, u_hi)
                    int h = tid / H4, i4 = tid - h * H4;
                    for (; h < n_rows; ) {
                        const int i = i4 * 4, u = h * H + i;
                        if (u < E) {
                            kb_f4 v;
                            if (u < clen) v = *reinterpret_cast<const kb_f4*>(cin + u);
                            else { v.x = 0.0f; v.y = 0.0f; v.z = 0.0f; v.w = 0.0f; }
                            const int f_top = h < fv_hi ? h : fv_hi;
                            int off = (h - f_top) * H + i;
                            const float* fp = exf + f_top * (2 * ZSTR) + off;
                            int cnt = f_top - fv_lo + 1;                 // frames at or below f_top that exist ...
                            // ... and reach sample u: offsets off, off + H, ... below win, i.e. ceil((win - off) / H) of them.  With
                            // off = (h - f_top) H + i and win = (Rw - 1) H + rem that is (i < rem ? Rw : Rw - 1) - (h - f_top): no division
                            int lim = (i < rem_w ? Rw : Rw - 1) - (h - f_top);
                            if (lim < 0) lim = 0;
                            if (cnt > lim) cnt = lim;
                            if (cnt == 4) {                              // the interior case at hop = win / 4: four independent loads
                                const kb_f4 a0 = *reinterpret_cast<const kb_f4*>(fp);
                                const kb_f4 a1 = *reinterpret_cast<const kb_f4*>(fp + dstep);
                                const kb_f4 a2 = *reinterpret_cast<const kb_f4*>(fp + 2 * dstep);
                                const kb_f4 a3 = *reinterpret_cast<const kb_f4*>(fp + 3 * dstep);
                                v.x += a0.x; v.y += a0.y; v.z += a0.z; v.w += a0.w;
                                v.x += a1.x; v.y += a1.y; v.z += a1.z; v.w += a1.w;
                                v.x += a2.x; v.y += a2.y; v.z += a2.z; v.w += a2.w;
                                v.x += a3.x; v.y += a3.y; v.z += a3.z; v.w += a3.w;
                            } else {
                                for (; cnt > 0; --cnt, fp += dstep) {
                                    const kb_f4 a = *reinterpret_cast<const kb_f4*>(fp);
                                    v.x += a.x; v.y += a.y; v.z += a.z; v.w += a.w;
                                }
                            }
                            if (u >= FRH) *reinterpret_cast<kb_f4*>(cout + (u - FRH)) = v;
                            else if (yvec && u >= u_lo && u + 3 < u_hi) *reinterpret_cast<kb_f4*>(yrow + u) = v;
                            else {
                                if (u >= u_lo && u < u_hi) ysig[(s0 + u) * p.y_sl] = v.x;
                                if (u + 1 >= u_lo && u + 1 < u_hi) ysig[(s0 + u + 1) * p.y_sl] = v.y;
                                if (u + 2 >= u_lo && u + 2 < u_hi) ysig[(s0 + u + 2) * p.y_sl] = v.z;
                                if (u + 3 >= u_lo && u + 3 < u_hi) ysig[(s0 + u + 3) * p.y_sl] = v.w;
                            }
                        }
                        h += step_h; i4 += step_i;
                        if (i4 >= H4) { i4 -= H4; ++h; }
                    }
                } else {
                    const float* exf = reinterpret_cast<const float*>(ex_s);
                    for (int u = tid; u < E; u += kb_nt) {
                        float v = u < clen ? cin[u] : 0.0f;
                        int f_hi = u / H; if (f_hi > fv_hi) f_hi = fv_hi;
                        int f_lo = u - win + H; f_lo = f_lo > 0 ? f_lo / H : 0; if (f_lo < fv_lo) f_lo = fv_lo;
                        for (int f = f_lo; f <= f_hi; ++f) v += exf[f * (2 * ZSTR) + (u - f * H)];
                        if (u >= FRH) cout[u - FRH] = v;
                        else if (u >= u_lo && u < u_hi) ysig[(s0 + u) * p.y_sl] = v;
                    }
                }
            KB_PHASE_END
            KB_SYNC_CTA;
        }
        // an odd number of rounds leaves the live carry in buffer 1; the next tile zeroes buffer 0 and starts
        // with round 0 reading buffer 0 -- nothing carries over between tiles
    }
}
