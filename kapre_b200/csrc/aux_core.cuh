// Stand-alone kernel bodies for the layers when they are used one by one
// (kapre/composed.py:5-12 tells users they may decompose `.layers`):
//   * kb_fb_cta    -- ApplyFilterbank.call, kapre/time_frequency.py:535-548
//   * kb_dft_cta   -- STFT for any n_fft that is not 64*{4,8,16,32} (the reference's own tests
//                     use n_fft=1000): direct windowed DFT, same semantics as
//                     kapre/time_frequency.py:169-182
//   * kb_idft_cta  -- InverseSTFT for such n_fft, kapre/time_frequency.py:307-314
// Same phase/emulation conventions as stft_core.cuh.
#pragma once
#include "stft_core.cuh"

// ------------------------------------------------------------------ ApplyFilterbank
struct KbFbParams {
    const float* x;                       // (batch, channel, frame, bin) element strides
    long long x_sb, x_sc, x_st, x_sk;
    int B, C, T, F;
    const KbBand* bands;
    const float* fbw;
    int n_bands;
    float* out;
    long long o_sb, o_sc, o_st, o_sk;
    int n_tiles_t;                        // ceil(T / R)
    int n_warps;
    int R;                                // frames per tile: 32, or 16 / 8 / 4 / 2 / 1 when 32 spectra do not fit shared memory
};

// A tile holds R whole spectra ([bin][frame], row stride R + 1); R shrinks for long spectra (n_fft 4096: 2049 bins
// -> 16 frames) so that every n_freq the STFT kernels produce can be filtered.
struct KbFbSmem { int mag, outs, total, Mp; };
KB_HD KbFbSmem kb_fb_smem_layout(int F, int n_bands, int R = 32) {
    KbFbSmem s;
    s.Mp = n_bands | 1;
    s.mag = 0;
    s.outs = kb_align16((F + 3) * (R + 1) * 4);
    s.total = s.outs + kb_align16(R * s.Mp * 4);
    return s;
}
static inline int kb_fb_pick_r(int F, int n_bands, int smem_limit) {
    for (int R = 32; R >= 1; R >>= 1)
        if (kb_fb_smem_layout(F, n_bands, R).total <= smem_limit) return R;
    return 0;
}

template <int FRT>
#if defined(KB_HOST_EMU)
inline void kb_fb_cta_r(const KbFbParams& p, char* smem, int cta, int n_cta)
#else
__device__ __forceinline__ void kb_fb_cta_r(const KbFbParams& p, char* smem, int cta, int n_cta)
#endif
{
    constexpr int RS = FRT + 1;
    const int NW = p.n_warps;
    const int kb_nt = NW * 32;
    (void)kb_nt;
    const KbFbSmem L = kb_fb_smem_layout(p.F, p.n_bands, FRT);
    float* mag_s = reinterpret_cast<float*>(smem + L.mag);
    float* out_s = reinterpret_cast<float*>(smem + L.outs);
    const int n_tiles = p.B * p.C * p.n_tiles_t;
#if defined(KB_HOST_EMU)
    std::vector<KbThreadRegs> kb_regs(kb_nt);
#else
    KbThreadRegs kb_regs;
#endif
    for (int tile = cta; tile < n_tiles; tile += n_cta) {
        const int sig = tile / p.n_tiles_t;
        const int tt = tile - sig * p.n_tiles_t;
        const int b = sig / p.C, c = sig - b * p.C;
        const int t0 = tt * FRT;
        const float* xs = p.x + (long long)b * p.x_sb + (long long)c * p.x_sc;
        const long long obase = (long long)b * p.o_sb + (long long)c * p.o_sc;
        KB_PHASE_BEGIN
            (void)R;
            const int tot = FRT * p.F;
            for (int idx = tid; idx < 3 * RS; idx += kb_nt) mag_s[p.F * RS + idx] = 0.0f;  // pad rows
            for (int idx = tid; idx < tot; idx += kb_nt) {
                const int r = idx / p.F, k = idx - r * p.F;
                const int t = t0 + r;
                mag_s[k * RS + r] = (t < p.T) ? xs[(long long)t * p.x_st + (long long)k * p.x_sk] : 0.0f;
            }
        KB_PHASE_END
        KB_SYNC_CTA;
        KB_PHASE_BEGIN
            (void)R;
            const int warp = tid >> 5, lane = tid & 31;
            if (lane < FRT) {
                const float* mcol = mag_s + lane;
                for (int m = warp; m < p.n_bands; m += NW) {
                    const KbBand bd = p.bands[m];
                    const float acc = kb_band_dot<RS>(p.fbw + bd.off, mcol + bd.lo * RS, (bd.hi - bd.lo) >> 2);
                    out_s[lane * L.Mp + m] = acc;
                }
            }
        KB_PHASE_END
        KB_SYNC_CTA;
        KB_PHASE_BEGIN
            (void)R;
            const int M = p.n_bands;
            const int tot = FRT * M;
            for (int idx = tid; idx < tot; idx += kb_nt) {
                const int r = idx / M, m = idx - r * M;
                const int t = t0 + r;
                if (t < p.T) p.out[obase + (long long)t * p.o_st + (long long)m * p.o_sk] = out_s[r * L.Mp + m];
            }
        KB_PHASE_END
        KB_SYNC_CTA;
    }
}

#if defined(KB_HOST_EMU)
inline void kb_fb_cta(const KbFbParams& p, char* smem, int cta, int n_cta)
#else
__device__ __forceinline__ void kb_fb_cta(const KbFbParams& p, char* smem, int cta, int n_cta)
#endif
{
    switch (p.R) {
        case 32: kb_fb_cta_r<32>(p, smem, cta, n_cta); break;
        case 16: kb_fb_cta_r<16>(p, smem, cta, n_cta); break;
        case 8: kb_fb_cta_r<8>(p, smem, cta, n_cta); break;
        case 4: kb_fb_cta_r<4>(p, smem, cta, n_cta); break;
        case 2: kb_fb_cta_r<2>(p, smem, cta, n_cta); break;
        default: kb_fb_cta_r<1>(p, smem, cta, n_cta); break;
    }
}

// ------------------------------------------------------------------ generic-N forward DFT
#define KB_DFT_TF 8
struct KbDftParams {
    const float* x;
    long long x_sb, x_sc, x_sl;
    int B, C, L;
    int n_fft, hop, T, pad_left;
    int win_eff;              // min(win_length, n_fft) window samples actually transformed
    const float* w;           // window[0 .. win_eff)
    const float2* tw;         // exp(-2 pi i r / n_fft), r < n_fft
    void* out;
    long long o_sb, o_sc, o_st, o_sk;
    int mode;                 // KB_OUT_COMPLEX or KB_OUT_MAG
    int n_tiles_t;            // ceil(T / KB_DFT_TF)
    int n_warps;
};

struct KbDftSmem { int tw, wx, total; };
KB_HD KbDftSmem kb_dft_smem_layout(int n_fft, int win_eff) {
    KbDftSmem s;
    s.tw = 0;
    s.wx = kb_align16(n_fft * 8);
    s.total = s.wx + kb_align16(KB_DFT_TF * win_eff * 4);
    return s;
}

#if defined(KB_HOST_EMU)
inline void kb_dft_cta(const KbDftParams& p, char* smem, int cta, int n_cta)
#else
__device__ __forceinline__ void kb_dft_cta(const KbDftParams& p, char* smem, int cta, int n_cta)
#endif
{
    const int NW = p.n_warps;
    const int kb_nt = NW * 32;
    (void)kb_nt;
    const int N = p.n_fft, We = p.win_eff, F = N / 2 + 1;
    const KbDftSmem L = kb_dft_smem_layout(N, We);
    cpx* tw_s = reinterpret_cast<cpx*>(smem + L.tw);
    float* wx_s = reinterpret_cast<float*>(smem + L.wx);
    const int n_tiles = p.B * p.C * p.n_tiles_t;
#if defined(KB_HOST_EMU)
    std::vector<KbThreadRegs> kb_regs(kb_nt);
#else
    KbThreadRegs kb_regs;
#endif
    KB_PHASE_BEGIN
        (void)R;
        for (int i = tid; i < N; i += kb_nt) { float2 t = p.tw[i]; tw_s[i] = cmake(t.x, t.y); }
    KB_PHASE_END
    KB_SYNC_CTA;
    for (int tile = cta; tile < n_tiles; tile += n_cta) {
        const int sig = tile / p.n_tiles_t;
        const int tt = tile - sig * p.n_tiles_t;
        const int b = sig / p.C, c = sig - b * p.C;
        const int t0 = tt * KB_DFT_TF;
        const float* xsig = p.x + (long long)b * p.x_sb + (long long)c * p.x_sc;
        const long long obase = (long long)b * p.o_sb + (long long)c * p.o_sc;
        KB_PHASE_BEGIN
            (void)R;
            const int tot = KB_DFT_TF * We;
            for (int idx = tid; idx < tot; idx += kb_nt) {
                const int f = idx / We, n = idx - f * We;
                const long long s = (long long)(t0 + f) * p.hop + n - p.pad_left;
                float v = 0.0f;
                if (s >= 0 && s < p.L && (t0 + f) < p.T) v = xsig[s * p.x_sl] * p.w[n];
                wx_s[idx] = v;
            }
        KB_PHASE_END
        KB_SYNC_CTA;
        KB_PHASE_BEGIN
            (void)R;
            for (int k = tid; k < F; k += kb_nt) {
                float ar[KB_DFT_TF], ai[KB_DFT_TF];
#pragma unroll
                for (int f = 0; f < KB_DFT_TF; ++f) { ar[f] = 0.0f; ai[f] = 0.0f; }
                int r = 0;
                for (int n = 0; n < We; ++n) {
                    const cpx t = tw_s[r];
#pragma unroll
                    for (int f = 0; f < KB_DFT_TF; ++f) {
                        const float v = wx_s[f * We + n];
                        ar[f] += v * t.re;
                        ai[f] += v * t.im;
                    }
                    r += k;
                    if (r >= N) r -= N;
                }
#pragma unroll
                for (int f = 0; f < KB_DFT_TF; ++f) {
                    const int t = t0 + f;
                    if (t < p.T) {
                        const long long o = obase + (long long)t * p.o_st + (long long)k * p.o_sk;
                        if (p.mode == KB_OUT_COMPLEX)
                            reinterpret_cast<float2*>(p.out)[o] = make_float2(ar[f], ai[f]);
                        else
                            reinterpret_cast<float*>(p.out)[o] = kb_sqrt(ar[f] * ar[f] + ai[f] * ai[f]);
                    }
                }
            }
        KB_PHASE_END
        KB_SYNC_CTA;
    }
}

// ------------------------------------------------------------------ generic-N inverse DFT + OLA
// One thread per output sample: y[s] = sum over the frames t covering s of
//   dualn[n] * sum_k c_k Re(X_t[k] e^{+2 pi i k n / N}),  n = s - t*hop < win,
// with c_0 = 1, c_{N/2} = 1 (even N), c_k = 2 otherwise and Im X[0], Im X[N/2] ignored
// (C2R semantics of irfft).  dualn = dual window / n_fft.
struct KbIdftParams {
    const float2* X;
    long long x_sb, x_sc, x_st, x_sk;
    int B, C, T;
    int n_fft, hop, win;      // win = min(win_length, n_fft)
    int out_len;
    const float* dualn;       // dual[n] / n_fft, n < win
    const float2* tw;         // exp(+2 pi i r / n_fft)
    float* y;
    long long y_sb, y_sc, y_sl;
    int n_tiles_s;            // ceil(out_len / (32 * n_warps))
    int n_warps;
    int y_off, edge2;         // STFT adjoint only (see KbIstftParams); zero for the inverse STFT
};

#if defined(KB_HOST_EMU)
inline void kb_idft_cta(const KbIdftParams& p, char* smem, int cta, int n_cta)
#else
__device__ __forceinline__ void kb_idft_cta(const KbIdftParams& p, char* smem, int cta, int n_cta)
#endif
{
    const int NW = p.n_warps;
    const int kb_nt = NW * 32;
    const int N = p.n_fft, F = N / 2 + 1;
    cpx* tw_s = reinterpret_cast<cpx*>(smem);
    const int n_tiles = p.B * p.C * p.n_tiles_s;
#if defined(KB_HOST_EMU)
    std::vector<KbThreadRegs> kb_regs(kb_nt);
#else
    KbThreadRegs kb_regs;
#endif
    KB_PHASE_BEGIN
        (void)R;
        for (int i = tid; i < N; i += kb_nt) { float2 t = p.tw[i]; tw_s[i] = cmake(t.x, t.y); }
    KB_PHASE_END
    KB_SYNC_CTA;
    for (int tile = cta; tile < n_tiles; tile += n_cta) {
        const int sig = tile / p.n_tiles_s;
        const int ts = tile - sig * p.n_tiles_s;
        const int b = sig / p.C, c = sig - b * p.C;
        const float2* Xsig = p.X + (long long)b * p.x_sb + (long long)c * p.x_sc;
        KB_PHASE_BEGIN
            (void)R;
            const int s = ts * kb_nt + tid;
            if (s >= p.y_off && s < p.out_len) {
                float acc = 0.0f;
                int t_hi = s / p.hop;
                if (t_hi > p.T - 1) t_hi = p.T - 1;
                for (int t = t_hi; t >= 0; --t) {
                    const int n = s - t * p.hop;
                    if (n >= p.win) break;
                    const float2* Xf = Xsig + (long long)t * p.x_st;
                    float sum = p.edge2 ? 2.0f * Xf[0].x : Xf[0].x;
                    int r = n % N;
                    const int step = r;
                    for (int k = 1; k < F; ++k) {
                        const float2 xv = Xf[(long long)k * p.x_sk];
                        const cpx w = tw_s[r];
                        const bool nyq = ((N & 1) == 0) && (k == F - 1);
                        if (nyq) sum += (p.edge2 ? 2.0f * xv.x : xv.x) * w.re;
                        else sum += 2.0f * (xv.x * w.re - xv.y * w.im);
                        r += step;
                        if (r >= N) r -= N;
                    }
                    acc += sum * p.dualn[n];
                }
                p.y[(long long)b * p.y_sb + (long long)c * p.y_sc + (long long)(s - p.y_off) * p.y_sl] = acc;
            }
        KB_PHASE_END
    }
}
