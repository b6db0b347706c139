// Backward (vector-Jacobian product) kernel bodies of the magnitude / filterbank / decibel layers.
//
// Written in the barrier-free phase style of stft_core.cuh, so that tests/emu/kb_emu.cpp runs this source on the
// CPU under KB_HOST_EMU.  The rules restate TensorFlow's registered gradients of the ops the reference calls:
//   Magnitude (tf.abs of complex, ComplexAbs):  G = g X / |X|, 0 where |X| = 0 (div_no_nan)
//   ApplyFilterbank (tensordot, MatMul):         g_mag = g_fb fb^T per frame
//   MagnitudeToDecibel (kapre/backend.py:186-192: Log, Maximum, Max):
//       l = 10 log10(max(x, amin)) - c,  m = max_item(l),  thr = m - dynamic_range,  y = max(l, thr)
//       dL/dl_i = g_i [l_i >= thr] + [l_i == m] (sum_j g_j [l_j < thr]) / #{l_j == m}
//       dL/dx_i = dL/dl_i * 10 / (ln 10 max(x_i, amin)) [x_i >= amin]
//
// Which elements the clamp bound is read from the forward output y, not recomputed: every clamped element holds
// exactly the threshold, which is then the item minimum of y.  An item's clamp counts as binding when
// min(y) <= max(y) - dynamic_range + tol, tol = 2^-20 (|max(y)| + dynamic_range) (a few float32 ulps: the forward's
// threshold and max(y) - dynamic_range may round apart), and an element counts as clamped when the clamp binds and
// y_i == min(y).  So an unclamped l_i within float32 rounding of thr is classified as clamped; the rule above leaves
// that case open.  Ties of the maximum are counted on y (== l there), as TF counts them on the float32 l.
#pragma once
#include "stft_core.cuh"

#define KB_DBS_MAX_CHUNKS 64      // CTAs per item of the statistics pass
#define KB_DBS_THREADS 256

// Per-item statistics of the decibel VJP, 4 floats per item: max(y), #ties of max(y), the clamped value (the item
// minimum when the clamp binds, -inf otherwise) and the sum of the upstream gradient over the clamped elements.
struct KbDbStats { float ymax, nmax, yclamp, gsum; };

// The 4-D views below are (item, d1, d2, d3) with element strides; the stand-alone layer passes (n_items, 1, 1, size).
struct KbDbStatParams {
    const float* y;           // forward output
    long long y_s0, y_s1, y_s2, y_s3;
    const float* g;           // upstream gradient (any strides, 0 included)
    long long g_s0, g_s1, g_s2, g_s3;
    int n_items, d1, d2, d3;
    int chunks;               // CTAs per item (<= KB_DBS_MAX_CHUNKS)
    float dyn_range;
    KbDbStats* part;          // n_items * chunks partials
    unsigned int* arrive;     // n_items arrival counters: zero on entry, left zero (the last CTA of an item resets it)
    KbDbStats* stats;         // n_items combined statistics
};

KB_HD void kb_dbs_merge(KbDbStats& a, const KbDbStats& b) {
    if (b.ymax > a.ymax) { a.ymax = b.ymax; a.nmax = b.nmax; }
    else if (b.ymax == a.ymax) a.nmax += b.nmax;
    if (b.yclamp < a.yclamp) { a.yclamp = b.yclamp; a.gsum = b.gsum; }
    else if (b.yclamp == a.yclamp) a.gsum += b.gsum;
}

KB_HD KbDbStats kb_dbs_empty() {
    KbDbStats s;
    s.ymax = -INFINITY; s.nmax = 0.0f; s.yclamp = INFINITY; s.gsum = 0.0f;
    return s;
}

KB_HD long long kb_off4(long long i, int d2, int d3, long long s1, long long s2, long long s3) {
    const long long k = i % d3, r = i / d3;
    return (r / d2) * s1 + (r % d2) * s2 + k * s3;
}

#if defined(KB_HOST_EMU)
static inline unsigned int kb_arrive(unsigned int* c) { return (*c)++; }
static inline void kb_fence() {}
#else
KB_D unsigned int kb_arrive(unsigned int* c) { return atomicAdd(c, 1u); }
KB_D void kb_fence() { __threadfence(); }
#endif

// One CTA per (item, chunk): per-thread partials over a strided walk of the chunk, merged in thread order by thread 0
// (fixed order: the result does not depend on scheduling), stored; the item's last CTA to arrive merges the item's
// partials in chunk order.  Deterministic for a given shape.
#if defined(KB_HOST_EMU)
inline void kb_dbstat_cta(const KbDbStatParams& p, char* smem, int cta, int n_cta)
#else
__device__ __forceinline__ void kb_dbstat_cta(const KbDbStatParams& p, char* smem, int cta, int n_cta)
#endif
{
    (void)n_cta;
    const int kb_nt = KB_DBS_THREADS;
    KbDbStats* ps = reinterpret_cast<KbDbStats*>(smem);
    int* last_s = reinterpret_cast<int*>(smem + kb_nt * sizeof(KbDbStats));
    const int item = cta / p.chunks, chunk = cta - item * p.chunks;
    const long long n = (long long)p.d1 * p.d2 * p.d3;
    const long long per = (n + p.chunks - 1) / p.chunks;
    const long long i0 = chunk * per, i1 = (i0 + per < n) ? i0 + per : n;
    const float* yi = p.y + (long long)item * p.y_s0;
    const float* gi = p.g + (long long)item * p.g_s0;
    const float tol = 9.5367431640625e-07f;   // 2^-20
#if defined(KB_HOST_EMU)
    std::vector<KbThreadRegs> kb_regs(kb_nt);
#else
    KbThreadRegs kb_regs;
#endif
    KB_PHASE_BEGIN
        (void)R;
        KbDbStats s = kb_dbs_empty();
        for (long long i = i0 + tid; i < i1; i += kb_nt) {
            const float y = yi[kb_off4(i, p.d2, p.d3, p.y_s1, p.y_s2, p.y_s3)];
            const float g = gi[kb_off4(i, p.d2, p.d3, p.g_s1, p.g_s2, p.g_s3)];
            if (y > s.ymax) { s.ymax = y; s.nmax = 1.0f; } else if (y == s.ymax) s.nmax += 1.0f;
            if (y < s.yclamp) { s.yclamp = y; s.gsum = g; } else if (y == s.yclamp) s.gsum += g;
        }
        ps[tid] = s;
    KB_PHASE_END
    KB_SYNC_CTA;
    KB_PHASE_BEGIN
        (void)R;
        if (tid == 0) {
            KbDbStats s = ps[0];
            for (int j = 1; j < kb_nt; ++j) kb_dbs_merge(s, ps[j]);
            p.part[(long long)item * p.chunks + chunk] = s;
            kb_fence();
            *last_s = (kb_arrive(p.arrive + item) == (unsigned int)(p.chunks - 1)) ? 1 : 0;
        }
    KB_PHASE_END
    KB_SYNC_CTA;
    KB_PHASE_BEGIN
        (void)R;
        if (tid == 0 && *last_s) {
            kb_fence();
            const volatile KbDbStats* pv = p.part + (long long)item * p.chunks;
            KbDbStats s = kb_dbs_empty();
            for (int j = 0; j < p.chunks; ++j) {
                KbDbStats t;
                t.ymax = pv[j].ymax; t.nmax = pv[j].nmax; t.yclamp = pv[j].yclamp; t.gsum = pv[j].gsum;
                kb_dbs_merge(s, t);
            }
            const float thr = s.ymax - p.dyn_range;
            const bool binds = s.yclamp <= thr + tol * (fabsf(s.ymax) + p.dyn_range);
            if (!binds) { s.yclamp = -INFINITY; s.gsum = 0.0f; }
            p.stats[item] = s;
            p.arrive[item] = 0u;
        }
    KB_PHASE_END
}

// dL/dl of one element from its forward output y and upstream gradient g (rule in the header comment).
KB_HD float kb_db_dl(const KbDbStats& s, float y, float g) {
    float d = (y == s.yclamp) ? 0.0f : g;
    if (y == s.ymax) d += s.gsum / s.nmax;
    return d;
}

// dl/dx factor: 10 / (ln 10 max(x, amin)) for x >= amin, else 0 (tf.maximum sends the gradient to amin).
KB_HD float kb_db_dx(float x, float amin) {
    return x >= amin ? 4.3429448190325175f / x : 0.0f;
}

// ------------------------------------------------------------------------------------------------------------------
// Spectral VJP: complex STFT X + upstream gradient (+ forward output for the decibel modes) -> complex gradient G of
// the STFT, for the fused chains MAG, MAG_DB, FB, FB_DB.  One frame per CTA iteration: the frame's spectrum is staged
// in shared memory before G is written, so G may alias X.
struct KbSpecVjpParams {
    const float2* X;
    long long x_sb, x_sc, x_st, x_sk;
    float2* G;
    long long G_sb, G_sc, G_st, G_sk;
    const float* g;              // (b, c, t, K) upstream gradient, any strides
    long long g_sb, g_sc, g_st, g_sk;
    const float* y;              // (b, c, t, K) forward output (decibel modes)
    long long y_sb, y_sc, y_st, y_sk;
    int B, C, T, F, K;           // K = F, or the band count in the filterbank modes
    int fb, db;
    const KbBand* bands;         // band-major filterbank: band j covers bins [lo, hi) with weights at fbw + off
    const float* fbw;
    const KbBand* bandsT;        // the transposed matrix: bin f covers bands [lo, hi) with weights at fbwT + off
    const float* fbwT;
    float amin;
    const KbDbStats* stats;      // per batch item (decibel modes)
    int n_warps;
};

struct KbSpecVjpSmem { int x, mag, gl, total; };
KB_HD KbSpecVjpSmem kb_specvjp_smem_layout(int F, int K) {
    KbSpecVjpSmem s;
    s.x = 0;
    s.mag = kb_align16(F * 8);
    s.gl = s.mag + kb_align16(F * 4);
    s.total = s.gl + kb_align16(K * 4);
    return s;
}

#if defined(KB_HOST_EMU)
inline void kb_specvjp_cta(const KbSpecVjpParams& p, char* smem, int cta, int n_cta)
#else
__device__ __forceinline__ void kb_specvjp_cta(const KbSpecVjpParams& p, char* smem, int cta, int n_cta)
#endif
{
    const int kb_nt = p.n_warps * 32;
    const KbSpecVjpSmem L = kb_specvjp_smem_layout(p.F, p.K);
    cpx* xs = reinterpret_cast<cpx*>(smem + L.x);
    float* mag = reinterpret_cast<float*>(smem + L.mag);
    float* gl = reinterpret_cast<float*>(smem + L.gl);
    const long long n_frames = (long long)p.B * p.C * p.T;
#if defined(KB_HOST_EMU)
    std::vector<KbThreadRegs> kb_regs(kb_nt);
#else
    KbThreadRegs kb_regs;
#endif
    for (long long fr = cta; fr < n_frames; fr += n_cta) {
        const int t = (int)(fr % p.T);
        const long long bc = fr / p.T;
        const int c = (int)(bc % p.C), b = (int)(bc / p.C);
        const float2* Xf = p.X + b * p.x_sb + c * p.x_sc + t * p.x_st;
        KB_PHASE_BEGIN
            (void)R;
            for (int f = tid; f < p.F; f += kb_nt) {
                const float2 v = Xf[(long long)f * p.x_sk];
                xs[f] = cmake(v.x, v.y);
                mag[f] = kb_sqrt(v.x * v.x + v.y * v.y);
            }
        KB_PHASE_END
        KB_SYNC_CTA;
        KB_PHASE_BEGIN
            (void)R;
            const float* gf = p.g + b * p.g_sb + c * p.g_sc + t * p.g_st;
            const float* yf = p.y + b * p.y_sb + c * p.y_sc + t * p.y_st;
            for (int j = tid; j < p.K; j += kb_nt) {
                float d = gf[(long long)j * p.g_sk];
                if (p.db) {
                    float x;
                    if (p.fb) {
                        const KbBand bd = p.bands[j];
                        const int hi = bd.hi < p.F ? bd.hi : p.F;
                        x = 0.0f;
                        for (int f = bd.lo; f < hi; ++f) x += mag[f] * p.fbw[bd.off + (f - bd.lo)];
                    } else {
                        x = mag[j];
                    }
                    d = kb_db_dl(p.stats[b], yf[(long long)j * p.y_sk], d) * kb_db_dx(x, p.amin);
                }
                gl[j] = d;
            }
        KB_PHASE_END
        KB_SYNC_CTA;
        KB_PHASE_BEGIN
            (void)R;
            float2* Gf = p.G + b * p.G_sb + c * p.G_sc + t * p.G_st;
            for (int f = tid; f < p.F; f += kb_nt) {
                float gm;
                if (p.fb) {
                    const KbBand bd = p.bandsT[f];
                    const int hi = bd.hi < p.K ? bd.hi : p.K;
                    gm = 0.0f;
                    for (int j = bd.lo; j < hi; ++j) gm += gl[j] * p.fbwT[bd.off + (j - bd.lo)];
                } else {
                    gm = gl[f];
                }
                const float m = mag[f];
                const float s = m > 0.0f ? gm / m : 0.0f;
                Gf[(long long)f * p.G_sk] = make_float2(s * xs[f].re, s * xs[f].im);
            }
        KB_PHASE_END
        KB_SYNC_CTA;   // the next frame reuses the staging buffers
    }
}
