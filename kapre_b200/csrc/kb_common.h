// kapre_b200 -- shared host/device definitions for the STFT hot path.
//
// The kernel bodies in stft_core.cuh / istft_core.cuh are written as sequences of
// barrier-free "phases".  Under nvcc each phase runs once per CUDA thread and phases are
// separated by __syncwarp()/__syncthreads(); under a plain host compiler (KB_HOST_EMU, used
// only by tests/emu to validate the index arithmetic without a GPU) each phase is a loop
// over all threads of the CTA, which is a legal serialisation of the same program.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define KB_HD __host__ __device__ __forceinline__
#define KB_D __device__ __forceinline__
#else
#define KB_HD inline
#define KB_D inline
#include <cmath>
#include <cstring>
struct float2 { float x, y; };
static inline float2 make_float2(float a, float b) { float2 r; r.x = a; r.y = b; return r; }
#endif

#define KB_MAX_WARPS 8

struct alignas(16) kb_f4 { float x, y, z, w; };
struct alignas(8) kb_i2 { int x, y; };

// ---- output modes of the fused forward kernel -------------------------------------------
enum KbMode {
    KB_OUT_COMPLEX = 0,  // complex64 STFT            (kapre.STFT)
    KB_OUT_MAG = 1,      // |STFT|                    (STFT -> Magnitude)
    KB_OUT_MAG_DB = 2,   // dB(|STFT|), unclamped     (... -> MagnitudeToDecibel)
    KB_OUT_FB = 3,       // filterbank(|STFT|)        (... -> ApplyFilterbank)
    KB_OUT_FB_DB = 4,    // dB(filterbank(|STFT|))    (get_melspectrogram_layer(return_decibel))
    KB_OUT_MAG_PHASE = 5,  // |STFT| (or its dB) and angle(STFT) side by side   (get_stft_mag_phase)
};

// Filterbank in "banded" form: band m covers bins [lo, hi) with weights w[off + (k - lo)];
// off and hi - lo are multiples of 4 (zero-padded) so the kernels read weights as 16 B vectors.
struct KbBand { int lo, hi, off, pad; };

struct KbStftParams {
    // input waveform, element strides (batch, channel, sample)
    const float* x;
    long long x_sb, x_sc, x_sl;
    int B, C, L;
    // [x_lo, x_hi): byte range of the waveform tensor; the 16 B-rounded TMA bulk copies must
    // stay inside it.  bulk_ok: x_sl == 1 and x is 4 B-aligned (else the fallback loader runs).
    const void* x_lo;
    const void* x_hi;
    long long x_numel;   // elements addressable from x (max element offset + 1)
    unsigned x_align;    // ((uintptr_t)x >> 2) & 3: position of x inside its 16 B line, in floats
    int bulk_ok;
    int dbuf;            // 1: two sample buffers (next tile prefetched during the current one)
    // transform
    int n_fft, hop, T;   // T = number of frames per (batch, channel)
    int pad_left;        // zeros prepended (n_fft - hop if pad_begin)  kapre/time_frequency.py:169-172
    // tables (device): wh = 0.5 * window zero-padded / cropped to n_fft;
    // twp[q*33 + k1] = exp(-2 pi i q k1 / P); twn[k] = exp(-2 pi i k / n_fft), k < P/2 (P = n_fft/2)
    const float* wh;
    const float2* twp;
    const float2* twn;
    const float2* twn2;  // kb_make_twn2: twn for the paired-column pair step (fused filterbank modes)
    // cosine-sum windows (hann, hamming, ... with win_length == n_fft): 0.5*w[n] = cw_a0 - B cos(2 pi n / n_fft)
    // is evaluated in registers instead of loaded: cwq[q] = B * (cos a_e, cos a_o, sin a_e, sin a_o) with
    // a_e = 2 pi (2q) / n_fft, a_o = 2 pi (2q + 1) / n_fft; the other factor exp(2 pi i j / 32) is a constant.
    int cosw;
    float cw_a0;
    const kb_f4* cwq;
    // output, element strides (batch, channel, frame, bin)
    void* out;
    long long o_sb, o_sc, o_st, o_sk;
    int mode;
    // filterbank (modes FB / FB_DB)
    const KbBand* bands;
    const float* fbw;
    int n_bands;
    int n_fbw;           // floats in fbw (bands are padded to multiples of 4 weights)
    // the same filterbank as flat lists of 4-weight chunks, one list per lane group (32 groups):
    // chunk i multiplies bins [cm[i].x, cm[i].x + 4); cm[i].y is the band to store after this
    // chunk (its last one) or -1.  Group g owns chunks [cg[g], cg[g+1]).
    const kb_f4* cw;
    const kb_i2* cm;
    const int* cg;
    int n_chunks;
    // two-level form (kb_make_fb_band_desc): fb_bands = 1 makes the single-channel kernel walk band descriptors
    int fb_bands;
    int variant;         // bit 1: natural-order pair step instead of the paired-column form (A/B alternative)
    const kb_i2* bd;
    const int* bg;
    int n_bd;
    // tensor-core form (kb_make_fb_mma): fb_mma = 1 runs the filterbank phase as a block-banded
    // mma.sync m16n8k8 3xTF32 GEMM; mw is read from global memory (L2-resident), ms / mg are staged.
    int fb_mma;
    const kb_f4* mw;
    const kb_i2* ms;
    const int* mg;
    int n_msteps;
    // decibel (modes *_DB): y = db_mul * log2(max(v, amin)) - db_sub; per-item max of max(v, amin)
    float amin, db_mul, db_sub;
    int db_ftz;              // amin >= FLT_MIN: every clamped value is a normal float, log2 may flush denormals
    int db_on;               // KB_OUT_MAG_PHASE only: 1 = the magnitude half is decibel-scaled
    long long ph_off;        // KB_OUT_MAG_PHASE only: element offset from a magnitude to its phase
    unsigned int* item_max;  // B entries, uint view of non-negative floats, zero-initialised
    // tiling
    int TF;          // frames per tile
    int n_tiles_t;   // ceil(T / TF)
    int n_warps;     // warps per CTA
    // multi-channel tiles (stft_mc_core.cuh): TF = time frames per tile, all C channels each
    int mc_wh;                 // window table needed in shared memory (no in-register window, or odd hop)
    int mc_cl_in;              // input is channel-interleaved (x_sc < x_sl): walk (sample, channel) in memory order
    int mc_out;                // output is channel-interleaved (o_sc == 1): cooperative pair step
    unsigned mc_magic_c, mc_magic_g, mc_magic_fr, mc_magic_last;   // kb_magic() of C, CTA size / C, columns per round (full / last)
};

struct KbIstftParams {
    const float2* X;                     // complex STFT, element strides (batch, channel, frame, bin)
    long long x_sb, x_sc, x_st, x_sk;
    int B, C, T;
    int n_fft, hop, win;                 // win = min(win_length, n_fft) samples kept per frame
    int out_len;                         // (T-1)*hop + win_length
    const float* dual;                   // dual window / P scaling folded in, length win (device)
    const float2* twp;
    const float2* twn;
    float* y;                            // element strides (batch, channel, sample)
    long long y_sb, y_sc, y_sl;
    int TFc;                             // frames computed per tile (incl. halo)
    int R;                               // overlap classes = ceil(win / hop)
    int hops_out;                        // output hops per tile = TFc - (R - 1)
    int n_tiles_t;
    int n_warps;
    int seg;                             // streaming kernel (kb_istft2_cta): output hops per tile
    // STFT adjoint (kapre_stft_backward) only; zero for the inverse STFT.  y_off: output sample s goes to y[s - y_off]
    // and samples below y_off are dropped (the pad_begin prefix); edge2: Re X[0] and Re X[N/2] are doubled at load.
    int y_off;
    int edge2;
};

// Complex number = one aligned register pair.  On sm_100a the arithmetic below compiles to the
// packed fp32x2 instructions (SASS FADD2 / FMUL2 / FFMA2): one instruction per complex add,
// two per complex multiply; ptxas folds the lane swaps / sign patterns into operand modifiers.
struct alignas(8) cpx { float re, im; };
KB_HD cpx cmake(float a, float b) { cpx r; r.re = a; r.im = b; return r; }

#if defined(__CUDA_ARCH__)
typedef unsigned long long kb_u64;
KB_D kb_u64 kb_pk(float lo, float hi) { kb_u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
KB_D cpx kb_up(kb_u64 v) { cpx r; asm("mov.b64 {%0, %1}, %2;" : "=f"(r.re), "=f"(r.im) : "l"(v)); return r; }
KB_D kb_u64 kb_add2(kb_u64 a, kb_u64 b) { kb_u64 r; asm("add.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
KB_D kb_u64 kb_sub2(kb_u64 a, kb_u64 b) { kb_u64 r; asm("sub.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
KB_D kb_u64 kb_mul2(kb_u64 a, kb_u64 b) { kb_u64 r; asm("mul.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
KB_D kb_u64 kb_fma2(kb_u64 a, kb_u64 b, kb_u64 c) { kb_u64 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
#endif

KB_HD cpx cadd(cpx a, cpx b) {
#if defined(__CUDA_ARCH__)
    return kb_up(kb_add2(kb_pk(a.re, a.im), kb_pk(b.re, b.im)));
#else
    return cmake(a.re + b.re, a.im + b.im);
#endif
}
KB_HD cpx csub(cpx a, cpx b) {
#if defined(__CUDA_ARCH__)
    return kb_up(kb_sub2(kb_pk(a.re, a.im), kb_pk(b.re, b.im)));
#else
    return cmake(a.re - b.re, a.im - b.im);
#endif
}
// a + conj(b) and a - conj(b)
KB_HD cpx cadd_conj(cpx a, cpx b) {
#if defined(__CUDA_ARCH__)
    return kb_up(kb_add2(kb_pk(a.re, a.im), kb_pk(b.re, -b.im)));
#else
    return cmake(a.re + b.re, a.im - b.im);
#endif
}
KB_HD cpx csub_conj(cpx a, cpx b) {
#if defined(__CUDA_ARCH__)
    return kb_up(kb_sub2(kb_pk(a.re, a.im), kb_pk(b.re, -b.im)));
#else
    return cmake(a.re - b.re, a.im + b.im);
#endif
}
// complex product a * b = a (.) (b.re, b.re) + swap(a) (.) (-b.im, b.im)
KB_HD cpx cmul(cpx a, cpx b) {
#if defined(__CUDA_ARCH__)
    const kb_u64 t = kb_mul2(kb_pk(a.re, a.im), kb_pk(b.re, b.re));
    return kb_up(kb_fma2(kb_pk(a.im, a.re), kb_pk(-b.im, b.im), t));
#else
    return cmake(a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re);
#endif
}
// element-wise product (a.re * b.re, a.im * b.im): window multiply of two packed samples
KB_HD cpx cmul_elem(cpx a, cpx b) {
#if defined(__CUDA_ARCH__)
    return kb_up(kb_mul2(kb_pk(a.re, a.im), kb_pk(b.re, b.im)));
#else
    return cmake(a.re * b.re, a.im * b.im);
#endif
}
// a * s for a real scalar s
KB_HD cpx cscale(cpx a, float s) {
#if defined(__CUDA_ARCH__)
    return kb_up(kb_mul2(kb_pk(a.re, a.im), kb_pk(s, s)));
#else
    return cmake(a.re * s, a.im * s);
#endif
}
// a * s + c element-wise for a real scalar s (one packed FMA)
KB_HD cpx cfma_s(cpx a, float s, cpx c) {
#if defined(__CUDA_ARCH__)
    return kb_up(kb_fma2(kb_pk(a.re, a.im), kb_pk(s, s), kb_pk(c.re, c.im)));
#else
    return cmake(a.re * s + c.re, a.im * s + c.im);
#endif
}
// d * (c - i sn): twiddle with separately given cosine / sine (compile-time constants at the call sites)
KB_HD cpx cmul_tw(cpx d, float c, float sn) {
#if defined(__CUDA_ARCH__)
    const kb_u64 t = kb_mul2(kb_pk(d.re, d.im), kb_pk(c, c));
    return kb_up(kb_fma2(kb_pk(d.im, d.re), kb_pk(sn, -sn), t));
#else
    return cmake(d.re * c + d.im * sn, d.im * c - d.re * sn);
#endif
}
// |a|^2
KB_HD float cnorm(cpx a) {
#if defined(__CUDA_ARCH__)
    const cpx q = kb_up(kb_mul2(kb_pk(a.re, a.im), kb_pk(a.re, a.im)));
    return q.re + q.im;
#else
    return a.re * a.re + a.im * a.im;
#endif
}

// Decibel epilogues: tf.maximum / tf.reduce_max propagate NaN (kapre/backend.py:186-192), fmaxf does not.
//   kb_floor_keepnan(v, amin) = max(v, amin) that keeps a NaN v;
//   kb_max_keepnan(a, b): both arguments are positive (>= amin) or NaN, so the unsigned order of the bit patterns
//   is the float order with NaN on top -- an integer max (and the per-item atomicMax works on the same view).
KB_HD float kb_floor_keepnan(float v, float amin) { return v < amin ? amin : v; }
KB_HD float kb_max_keepnan(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __uint_as_float(max(__float_as_uint(a), __float_as_uint(b)));
#else
    uint32_t ua, ub;
    std::memcpy(&ua, &a, 4); std::memcpy(&ub, &b, 4);
    return ua > ub ? a : b;
#endif
}

// log2 of a power of two
KB_HD int kb_ilog2(int v) {
#if defined(__CUDA_ARCH__)
    return __ffs(v) - 1;
#else
    int r = 0;
    while ((1 << r) < v) ++r;
    return r;
#endif
}

// shared-memory footprint helpers (bytes), shared by host launch code and kernels
KB_HD int kb_align16(int v) { return (v + 15) & ~15; }
