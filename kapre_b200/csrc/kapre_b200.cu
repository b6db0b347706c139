// kapre_b200 -- CUDA kernels (sm_100a) and the C ABI declared in include/kapre_b200.h.
//
// Kernel bodies live in stft_core.cuh / istft_core.cuh / aux_core.cuh (shared with the CPU
// emulation harness under tests/emu); this file holds the __global__ wrappers, the
// element-wise kernels, launch-configuration logic and the extern "C" entry points.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <string>
#include <vector>

#include "../../include/kapre_b200.h"
#include "kb_tables.h"
#include "stft_core.cuh"
#include "stft_mc_core.cuh"
#include "istft_core.cuh"
#include "aux_core.cuh"
#include "mr_core.cuh"
#include "tc_dft.cuh"
#include "tc_mel.cuh"
#include "grad_core.cuh"

// ------------------------------------------------------------------------------------------
// error handling
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static thread_local std::string g_launch_info;
static std::atomic<uint64_t> g_launches{0};

// optional kernel timing (bench.py roofline): event pairs around the dominant kernels
#include <mutex>
static std::mutex g_prof_mu;
static int g_prof_on = 0;             // 0: off, n: every n-th dominant-kernel launch is bracketed by events
static std::atomic<uint64_t> g_prof_seq{0};
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_prof_events;

struct KbProfScope {
    cudaStream_t st;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    explicit KbProfScope(cudaStream_t s) : st(s) {
        const int every = g_prof_on;
        if (!every) return;
        // sampling: an event record between two kernels serialises them (no programmatic dependent
        // launch across it), so a stride > 1 leaves most launches of a timed loop undisturbed
        if ((g_prof_seq++ % (uint64_t)every) != 0) return;
        if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) { e0 = e1 = nullptr; return; }
        cudaEventRecord(e0, st);
    }
    ~KbProfScope() {
        if (!e0) return;
        cudaEventRecord(e1, st);
        std::lock_guard<std::mutex> lk(g_prof_mu);
        g_prof_events.emplace_back(e0, e1);
    }
};

static int kb_fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define KB_CUDA(expr)                                                                         \
    do {                                                                                      \
        cudaError_t e_ = (expr);                                                              \
        if (e_ != cudaSuccess)                                                                \
            return kb_fail(KAPRE_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                           __FILE__, __LINE__);                                               \
    } while (0)

// ------------------------------------------------------------------------------------------
// __global__ wrappers
// ------------------------------------------------------------------------------------------
template <int Q, int MODE>
__global__ void __launch_bounds__(KB_MAX_WARPS * 32, 2) kb_stft_kernel(const __grid_constant__ KbStftParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_stft_cta<Q, MODE>(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

// variant with the filterbank phase on the tensor pipe (mma.sync 3xTF32), selected by KAPRE_B200_FBMMA=1
template <int Q, int MODE>
__global__ void __launch_bounds__(KB_MAX_WARPS * 32, 2) kb_stft_kernel_mma(const __grid_constant__ KbStftParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_stft_cta<Q, MODE, 1>(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

// the A/B alternative of the pair step (template bit 1: natural-order pair step instead of the paired-column form)
template <int Q, int MODE, int V>
__global__ void __launch_bounds__(KB_MAX_WARPS * 32, 2) kb_stft_kernel_v(const __grid_constant__ KbStftParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_stft_cta<Q, MODE, V>(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

// 16-warp CTAs, one per SM: n_fft = 2048 in the filterbank modes, where an 8-warp CTA already needs more than
// half of the SM's shared memory (8.4 KB of exchange buffer per warp), so two CTAs never fit
template <int Q, int MODE>
__global__ void __launch_bounds__(512, 1) kb_stft_kernel_w16(const __grid_constant__ KbStftParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_stft_cta<Q, MODE>(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

template <int Q, int MODE>
__global__ void __launch_bounds__(KB_MAX_WARPS * 32, 2) kb_stft_mcfb_kernel(const __grid_constant__ KbStftParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_stft_mcfb_cta<Q, MODE>(p, kb_smem, blockIdx.x, gridDim.x);
}

// multi-channel tiles (interleaved tensors): up to 16 warps, one or two CTAs per SM
template <int Q, int MODE>
__global__ void __launch_bounds__(512, 1) kb_stft_mc_kernel(const __grid_constant__ KbStftParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_stft_mc_cta<Q, MODE>(p, kb_smem, blockIdx.x, gridDim.x);
}

// 4 warps per CTA (one FFT round per overlap class), two or three CTAs per SM: the register file is not the
// limit here, so the kernel may use up to 168 registers and keeps the round's global loads in flight.
#define KB_ISTFT_MAX_WARPS 4
template <int Q>
__global__ void __launch_bounds__(KB_ISTFT_MAX_WARPS * 32, 3) kb_istft_kernel(const __grid_constant__ KbIstftParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_istft_cta<Q>(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

__global__ void __launch_bounds__(KB_MAX_WARPS * 32) kb_fb_kernel(const __grid_constant__ KbFbParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_fb_cta(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

__global__ void __launch_bounds__(KB_MAX_WARPS * 32) kb_dft_kernel(const __grid_constant__ KbDftParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_dft_cta(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

__global__ void __launch_bounds__(512) kb_mr_kernel(const __grid_constant__ KbMrParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_mr_cta(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

__global__ void __launch_bounds__(KB_MAX_WARPS * 32) kb_idft_kernel(const __grid_constant__ KbIdftParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_idft_cta(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

// ---- backward kernels (grad_core.cuh) ----
__global__ void __launch_bounds__(KB_DBS_THREADS) kb_dbstat_kernel(const __grid_constant__ KbDbStatParams p) {
    __shared__ __align__(16) char kb_smem[KB_DBS_THREADS * sizeof(KbDbStats) + 16];
    kb_dbstat_cta(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

__global__ void __launch_bounds__(KB_MAX_WARPS * 32) kb_specvjp_kernel(const __grid_constant__ KbSpecVjpParams p) {
    extern __shared__ __align__(16) char kb_smem[];
    kb_specvjp_cta(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

// Stand-alone MagnitudeToDecibel VJP, element-wise on contiguous (n_items, item_size) x / y; g has (item, element) strides.
__global__ void kb_db_backward_kernel(const float* __restrict__ x, const float* __restrict__ y, const float* __restrict__ g,
                                      long long g_si, long long g_se, float* __restrict__ dx, long long item_size, long long n,
                                      const KbDbStats* __restrict__ stats, float amin) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const long long item = i / item_size, e = i - item * item_size;
        dx[i] = kb_db_dl(stats[item], y[i], g[item * g_si + e * g_se]) * kb_db_dx(x[i], amin);
    }
}

// InverseSTFT VJP fix-up: the forward STFT of the upstream gradient carries weight 2/N on every bin; bins 0 and N/2
// (even N) of the irfft count once, so they are halved, and their imaginary parts (which irfft ignores) get 0.
__global__ void kb_istft_grad_edges_kernel(float2* __restrict__ G, long long sb, long long sc, long long st, long long sk,
                                           int C, int T, long long n_frames, int last, int even) {
    for (long long fr = (long long)blockIdx.x * blockDim.x + threadIdx.x; fr < n_frames; fr += (long long)gridDim.x * blockDim.x) {
        const long long t = fr % T, bc = fr / T;
        float2* Gf = G + (bc / C) * sb + (bc % C) * sc + t * st;
        Gf[0] = make_float2(0.5f * Gf[0].x, 0.0f);
        if (even) Gf[(long long)last * sk] = make_float2(0.5f * Gf[(long long)last * sk].x, 0.0f);
    }
}

// Dynamic-range clamp, kapre/backend.py:190-192: y = max(y, max_item(y) - dynamic_range).
// item_max holds max(x, amin) per item (uint view); log is monotone, so the item maximum in
// dB is dB(item_max).  `chunks` CTAs per item (so that one long item is rewritten by many CTAs when the
// clamp binds): each reads the maximum and returns immediately when the clamp cannot bind (threshold <=
// dB(amin)), which is the common case (SURVEY section 7), so no output byte is re-read.  The workspace is
// SELF-CLEANING: words [0, n_items) are the maxima, words [n_items, 2 n_items) count the CTAs of an item that
// have read its maximum; the last one resets both to zero.  A NaN anywhere in an item makes its maximum NaN
// (the producers keep NaN through their max()), and tf.maximum(y, NaN) is NaN for the whole item.
// Launched with programmatic dependent launch: the grid is scheduled while the producer kernel drains.
__global__ void kb_db_clamp_kernel(float* __restrict__ y, long long item_size, long long run, long long period,
                                   unsigned int* __restrict__ item_max, unsigned int n_items, int chunks, float amin,
                                   float db_mul, float db_sub, float dyn_range) {
#if __CUDA_ARCH__ >= 900
    asm volatile("griddepcontrol.launch_dependents;");   // the next fused kernel may start its table prologue
    cudaGridDependencySynchronize();
#endif
    const long long item = blockIdx.x / chunks;
    const int chunk = (int)(blockIdx.x - item * chunks);
    __shared__ unsigned int s_mx;
    if (threadIdx.x == 0) s_mx = item_max[item];
    __syncthreads();
    if (threadIdx.x == 0) {
        // every CTA of the item has its copy of the maximum before the last arrival clears it
        unsigned int* cnt = item_max + n_items + item;
        if (chunks == 1 || atomicAdd(cnt, 1u) == (unsigned int)(chunks - 1)) {
            item_max[item] = 0u;
            if (chunks > 1) *cnt = 0u;
        }
    }
    const float mx = __uint_as_float(s_mx);
    float thr = (db_mul * __log2f(fmaxf(mx, amin)) - db_sub) - dyn_range;
    const float floor_db = db_mul * __log2f(amin) - db_sub;
    const bool nan_item = mx != mx;
    if (!nan_item && !(thr > floor_db)) return;
    if (nan_item) thr = mx;
    float* yi = y + item * item_size;
    const long long step = (long long)chunks * blockDim.x;
    // only elements with (i mod period) < run are decibel values (magnitude half of a mag+phase tensor)
    for (long long i = (long long)chunk * blockDim.x + threadIdx.x; i < item_size; i += step) {
        if (run >= period || i % period < run) yi[i] = nan_item ? thr : fmaxf(yi[i], thr);
    }
}

// Stand-alone MagnitudeToDecibel pass 1: y = db(max(x, amin)), per-item max of max(x, amin).
__global__ void kb_db_kernel(const float* __restrict__ x, float* __restrict__ y, long long item_size,
                             int chunks, unsigned int* __restrict__ item_max, float amin,
                             float db_mul, float db_sub) {
    const long long item = blockIdx.x / chunks;
    const int chunk = blockIdx.x - (int)(item * chunks);
    const float* xi = x + item * item_size;
    float* yi = y + item * item_size;
    unsigned int mxu = 0u;
    for (long long i = (long long)chunk * blockDim.x + threadIdx.x; i < item_size;
         i += (long long)chunks * blockDim.x) {
        const float xv = xi[i];
        const float v = xv < amin ? amin : xv;               // max that keeps NaN (tf.maximum propagates it)
        mxu = max(mxu, __float_as_uint(v));                    // v > 0 or NaN: the uint order is the float order, NaN on top
        yi[i] = db_mul * __log2f(v) - db_sub;
    }
    const unsigned int wm = __reduce_max_sync(0xffffffffu, mxu);
    if ((threadIdx.x & 31) == 0 && wm != 0u) atomicMax(item_max + item, wm);
}

__global__ void kb_magnitude_kernel(const float2* __restrict__ x, float* __restrict__ y, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const float2 v = x[i];
        y[i] = kb_sqrt(v.x * v.x + v.y * v.y);
    }
}

__global__ void kb_phase_kernel(const float2* __restrict__ x, float* __restrict__ y, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        const float2 v = x[i];
        y[i] = atan2f(v.y, v.x);
    }
}

// kapre.ConcatenateFrequencyMap (kapre/time_frequency.py:648-744): out = concat(x, linspace(0, 1, F) broadcast over
// (batch, time)) along the channel axis.  One pass: every output element is either a copy or the map value.
__global__ void kb_concat_freq_map_kernel(const float* __restrict__ x, float* __restrict__ y, long long B, long long C,
                                          long long T, long long F, int channels_last) {
    const long long Co = C + 1;
    const long long total = B * Co * T * F;
    const float step = F > 1 ? 1.0f / (float)(F - 1) : 0.0f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        long long b, c, t, f;
        if (channels_last) { c = i % Co; f = (i / Co) % F; t = (i / (Co * F)) % T; b = i / (Co * F * T); }
        else { f = i % F; t = (i / F) % T; c = (i / (F * T)) % Co; b = i / (F * T * Co); }
        float v;
        if (c == C) v = (f == F - 1 && F > 1) ? 1.0f : (float)f * step;      // tf.linspace: exact end point
        else v = channels_last ? x[((b * T + t) * F + f) * C + c] : x[((b * C + c) * T + t) * F + f];
        y[i] = v;
    }
}

// kapre.SpecAugment (kapre/augmentation.py:116-326): per item, every element whose time index lies in one of the item's time
// masks [start, start + width] or whose frequency index lies in one of its frequency masks is replaced by mask_value
// (tf.where(mask, mask_value, x) after reduce_any over the masks).  The (start, width) pairs are drawn on the host
// (the reference draws them with tf.random.uniform per item and mask); depth is 1, so both data formats are (b, t, f).
__global__ void kb_spec_augment_kernel(const float* __restrict__ x, float* __restrict__ y, long long B, long long T, long long F,
                                       const int* __restrict__ tmask, int n_t, const int* __restrict__ fmask, int n_f,
                                       float mask_value) {
    const long long total = B * T * F;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long f = i % F, t = (i / F) % T, b = i / (F * T);
        bool m = false;
        for (int j = 0; j < n_t; ++j) {
            const int s0 = tmask[(b * n_t + j) * 2], w = tmask[(b * n_t + j) * 2 + 1];
            m = m || (t >= s0 && t <= s0 + w);
        }
        for (int j = 0; j < n_f; ++j) {
            const int s0 = fmask[(b * n_f + j) * 2], w = fmask[(b * n_f + j) * 2 + 1];
            m = m || (f >= s0 && f <= s0 + w);
        }
        y[i] = m ? mask_value : x[i];
    }
}

// ---- adjacent layers: Delta / Frame / Energy (element-wise or small-window kernels, HBM-bound) ----
__device__ __forceinline__ long long kb_pad_index(long long t, long long T, int mode) {
    // index into [0, T) for an out-of-range t under tf.pad's SYMMETRIC (0) / REFLECT (1); -1 = zero (CONSTANT)
    if (t >= 0 && t < T) return t;
    if (mode == 2) return -1;
    if (t < 0) t = (mode == 0) ? (-t - 1) : (-t);
    else t = (mode == 0) ? (2 * T - 1 - t) : (2 * T - 2 - t);
    return (t >= 0 && t < T) ? t : -1;
}

__global__ void kb_delta_kernel(const float* __restrict__ x, float* __restrict__ y, long long outer, long long T,
                                long long inner, int n, float inv_denom, int mode) {
    const long long total = outer * T * inner;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long in = i % inner;
        const long long t = (i / inner) % T;
        const long long o = i / (inner * T);
        const float* base = x + o * T * inner + in;
        float acc = 0.0f;
        for (int m = 1; m <= n; ++m) {
            const long long tp = kb_pad_index(t + m, T, mode), tm = kb_pad_index(t - m, T, mode);
            const float a = tp >= 0 ? base[tp * inner] : 0.0f;
            const float b = tm >= 0 ? base[tm * inner] : 0.0f;
            acc += (float)m * (a - b);
        }
        y[i] = acc * inv_denom;
    }
}

__global__ void kb_frame_kernel(const float* __restrict__ x, long long x_sb, long long x_sc, long long x_sl, int B, int C,
                                int L, int fl, int hop, int T, float pad_value, float* __restrict__ out, long long o_sb,
                                long long o_sc, long long o_st, long long o_sk) {
    const long long total = (long long)B * C * T * fl;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int n = (int)(i % fl);
        const long long r = i / fl;
        const int t = (int)(r % T);
        const long long bc = r / T;
        const int c = (int)(bc % C), b = (int)(bc / C);
        const long long s = (long long)t * hop + n;
        const float v = s < L ? x[b * x_sb + c * x_sc + s * x_sl] : pad_value;
        out[b * o_sb + c * o_sc + t * o_st + n * o_sk] = v;
    }
}

__global__ void kb_energy_kernel(const float* __restrict__ x, long long x_sb, long long x_sc, long long x_sl, int B, int C,
                                 int L, int fl, int hop, int T, float pad_value, float scale, float* __restrict__ out,
                                 long long o_sb, long long o_sc, long long o_st) {
    const long long n_frames = (long long)B * C * T;
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long n_warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long f = warp0; f < n_frames; f += n_warps) {
        const int t = (int)(f % T);
        const long long bc = f / T;
        const int c = (int)(bc % C), b = (int)(bc / C);
        const float* xs = x + b * x_sb + c * x_sc;
        float acc = 0.0f;
        for (int n = lane; n < fl; n += 32) {
            const long long s = (long long)t * hop + n;
            const float v = s < L ? xs[s * x_sl] : pad_value;
            acc += v * v;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) out[b * o_sb + c * o_sc + t * o_st] = scale * acc;
    }
}

// ------------------------------------------------------------------------------------------
// plans
// ------------------------------------------------------------------------------------------
struct DevInfo {
    int device = -1;
    int sm_count = 0;
    int smem_optin = 0;
};

static int kb_dev_info(DevInfo* d) {
    KB_CUDA(cudaGetDevice(&d->device));
    KB_CUDA(cudaDeviceGetAttribute(&d->sm_count, cudaDevAttrMultiProcessorCount, d->device));
    KB_CUDA(cudaDeviceGetAttribute(&d->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, d->device));
    return 0;
}

template <typename T>
static int kb_upload(const std::vector<T>& h, T** d) {
    KB_CUDA(cudaMalloc((void**)d, h.size() * sizeof(T)));
    KB_CUDA(cudaMemcpy(*d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return 0;
}

struct kapre_stft_plan {
    int n_fft, win_length, hop, Q;
    DevInfo dev;
    float* wh = nullptr;      // fused path: 0.5 * window padded to n_fft
    kb_f4* cwq = nullptr;     // cosine-sum window factors (cosw), see KbStftParams
    int cosw = 0;
    float cw_a0 = 0.0f;
    float2* twp = nullptr;
    float2* twn = nullptr;
    float2* twn2 = nullptr;   // kb_make_twn2 (paired-column pair step)
    float* w = nullptr;       // generic path: window[0, win_eff)
    float2* tw = nullptr;     // generic path: exp(-2 pi i r / n_fft)
    int win_eff;
    // STFT adjoint (kapre_stft_backward): the inverse kernels with the window n_fft/2 * w in place of the dual window
    float* adj = nullptr;     // streaming body: kb_make_dual(n_fft/2 * window)
    float* adj_dn = nullptr;  // direct body: (n_fft/2 * window) / n_fft = window / 2
    float2* adj_tw = nullptr; // direct body: exp(+2 pi i r / n_fft)
    // tensor-core path (tc_mel.cuh; n_fft = win_length = 1024, cosine-sum window a - b cos): constant operands
    double win_a = 0.0, win_b = 0.0;
    float* tc_f1 = nullptr;   // stage-1 matrix hi/lo
    float* tc_cs = nullptr;   // stage-2 C / S matrices hi/lo
    unsigned short* tc_csb = nullptr;   // the same matrices in bf16 (lo-part products)
    float2* tc_tw = nullptr;  // a e^{-2 pi i n2 k1 / 1024}
    float2* tc_w32 = nullptr; // e^{-2 pi i j / 32}
};

// (K = 32 rows, N = 32 columns) matrix -> the K-major interleaved (8 kchunk, 32 col, 4) layout of the UMMA B operand
static void kb_tc_pack_b(const double* M, float* hi, float* lo) {
    for (int kc = 0; kc < 8; ++kc)
        for (int c = 0; c < 32; ++c)
            for (int e = 0; e < 4; ++e) {
                const float w = (float)M[(4 * kc + e) * 32 + c], h = kb_tf32_rn(w);
                hi[(kc * 32 + c) * 4 + e] = h;
                lo[(kc * 32 + c) * 4 + e] = w - h;
            }
}

static int kb_tc_tables(kapre_stft_plan* p) {
    std::vector<double> M(1024);
    std::vector<float> f1(2048), cs(4096);
    for (int n1 = 0; n1 < 32; ++n1)
        for (int c = 0; c < 32; ++c) {
            const int k1 = c >> 1;
            const double a = -2.0 * M_PI * (double)((n1 * k1) % 32) / 32.0;
            M[n1 * 32 + c] = (c == 1) ? ((n1 & 1) ? -1.0 : 1.0) : ((c & 1) ? sin(a) : cos(a));
        }
    kb_tc_pack_b(M.data(), f1.data(), f1.data() + 1024);
    for (int n2 = 0; n2 < 32; ++n2)
        for (int k2 = 0; k2 < 32; ++k2) M[n2 * 32 + k2] = cos(2.0 * M_PI * (double)((n2 * k2) % 32) / 32.0);
    kb_tc_pack_b(M.data(), cs.data(), cs.data() + 1024);
    for (int n2 = 0; n2 < 32; ++n2)
        for (int k2 = 0; k2 < 32; ++k2) M[n2 * 32 + k2] = sin(2.0 * M_PI * (double)((n2 * k2) % 32) / 32.0);
    kb_tc_pack_b(M.data(), cs.data() + 2048, cs.data() + 3072);
    // bf16 copies of C and S, K-major interleaved (4 kchunk, 32 col, 8)
    std::vector<unsigned short> csb(2048);
    for (int which = 0; which < 2; ++which)
        for (int kc = 0; kc < 4; ++kc)
            for (int c = 0; c < 32; ++c)
                for (int e = 0; e < 8; ++e) {
                    const int n2 = 8 * kc + e;
                    const double a = 2.0 * M_PI * (double)((n2 * c) % 32) / 32.0;
                    const float w = (float)(which ? sin(a) : cos(a));
                    uint32_t u;
                    memcpy(&u, &w, 4);
                    u += 0x7fffu + ((u >> 16) & 1u);                 // round to nearest even
                    csb[(size_t)which * 1024 + (kc * 32 + c) * 8 + e] = (unsigned short)(u >> 16);
                }
    std::vector<float2> tw(18 * 32), w32(16);
    for (int k1 = 0; k1 < 18; ++k1)
        for (int n2 = 0; n2 < 32; ++n2) {
            const double a = -2.0 * M_PI * (double)(n2 * k1) / 1024.0;
            tw[k1 * 32 + n2] = make_float2((float)(p->win_a * cos(a)), (float)(p->win_a * sin(a)));
        }
    for (int j = 0; j < 16; ++j) {
        const double a = -2.0 * M_PI * (double)j / 32.0;
        w32[j] = make_float2((float)cos(a), (float)sin(a));
    }
    int rc;
    if ((rc = kb_upload(f1, &p->tc_f1)) || (rc = kb_upload(cs, &p->tc_cs)) || (rc = kb_upload(csb, &p->tc_csb)) || (rc = kb_upload(tw, &p->tc_tw)) ||
        (rc = kb_upload(w32, &p->tc_w32)))
        return rc;
    return 0;
}

struct kapre_istft_plan {
    int n_fft, win_length, hop, Q, win;
    DevInfo dev;
    float* dual = nullptr;    // fused path (kb_make_dual)
    float2* twp = nullptr;
    float2* twn = nullptr;
    float* dualn = nullptr;   // generic path: dual / n_fft
    float2* tw = nullptr;     // generic path: exp(+2 pi i r / n_fft)
    kapre_stft_plan* grad = nullptr;   // VJP (kapre_istft_backward): forward STFT with the window 2/n_fft * dual
};

struct kapre_filterbank {
    int n_freq, n_bands, n_w;
    DevInfo dev;
    KbBand* bands = nullptr;   // band-major form (stand-alone ApplyFilterbank kernel)
    float* w = nullptr;
    KbBand* bandsT = nullptr;  // the same form of the transposed matrix (per bin: the bands it feeds), spectral VJP
    float* wT = nullptr;
    int Q = 0;                 // chunk-list form for the fused kernel (n_freq == 32*Q + 1), else 0
    int n_chunks = 0;
    kb_f4* cw = nullptr;
    kb_i2* cm = nullptr;
    int* cg = nullptr;
    int n_bd = 0;              // band descriptors of the two-level walk (kb_make_fb_band_desc)
    kb_i2* bd = nullptr;
    int* bg = nullptr;
    int n_msteps = 0;          // tensor-core form (kb_make_fb_mma) for the fused kernel
    kb_f4* mw = nullptr;
    kb_i2* ms = nullptr;
    int* mg = nullptr;
};

static float2* g_tc_dbg = nullptr;   // experimental: complex-spectrum dump of the next tensor-core launch (kapre_tc_set_debug)

static int kb_env_int(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

// ------------------------------------------------------------------------------------------
// launch configuration of the fused forward kernel
// ------------------------------------------------------------------------------------------
struct FwdCfg { int TF, NW, smem, bps; };
#ifndef KB_PAIRED_DEFAULT
#define KB_PAIRED_DEFAULT 1
#endif
#ifndef KB_FBMMA_DEFAULT
#define KB_FBMMA_DEFAULT 0
#endif
#ifndef KB_TC_DEFAULT
#define KB_TC_DEFAULT 0
#endif

// Tile shape of the fused forward kernel.  Measured on B200 (profiles/): the kernel is
// latency-bound, so resident warps per SM (up to the 16 the 128-register kernel allows) matter
// most, then larger tiles (less re-staging of the hop overlap).  Filterbank modes keep the
// tile's magnitudes in the warps' exchange regions, which needs TF == frames per round.
// `n_sig` signals of `T` frames each: small batches (BASELINE cfg1 is 244 frames) that cannot fill the machine are
// latency-bound and get their own choice (see below); everything else maximises resident warps.
static bool kb_pick_fwd_cfg(const DevInfo& dev, int Q, int n_fft, int hop, int mode, int n_bands, int n_chunks,
                            int fbmma, long long n_sig, int T, FwdCfg* out) {
    const int FPW = 32 / Q;
    const bool fb = (mode == KB_OUT_FB || mode == KB_OUT_FB_DB);
    const int force_tf = kb_env_int("KAPRE_B200_TF", 0);
    const int force_nw = kb_env_int("KAPRE_B200_NW", 0);
    const int sm_smem = 228 * 1024;
    bool found = false;
    FwdCfg best{};
    double best_score = -1.0;
    const int nws[5] = {1, 2, 4, 8, 16};
    for (int a = 0; a < 5; ++a) {
        const int NW = nws[a];
        if (force_nw && NW != force_nw) continue;
        if (NW == 16 && !(Q == 32 && fb && !fbmma)) continue;      // only kb_stft_kernel_w16's instantiations
        const int FR = NW * FPW;
        if (FR > 32) continue;
        for (int TF = 32; TF >= 1; TF >>= 1) {
            if (fb ? (TF != FR) : (TF % FR != 0)) continue;
            if (!fb && force_tf && TF != force_tf) continue;
            const KbStftSmem L = kb_stft_smem_layout(Q, n_fft, hop, TF, NW, mode, n_bands, n_chunks, fbmma);
            if (L.total > dev.smem_optin) continue;
            int bps = sm_smem / (L.total + 1024);
            if (bps > 16 / NW) bps = 16 / NW;                 // 128 registers per thread: 16 warps per SM
            if (bps < 1) continue;
            const int warps = bps * NW;
            // throughput score (large problems): resident warps first, then longer tiles (less re-staging of the overlap)
            double score = (double)warps * 1000.0 + TF * 10.0 + NW;
            if (n_sig > 0 && T > 0) {
                const double tiles = (double)n_sig * (double)((T + TF - 1) / TF);
                const double slots = (double)dev.sm_count * bps;
                if (tiles < slots) {
                    // latency regime: all tiles run at once and the call costs one tile (~10 us: table prologue, one FFT round,
                    // filterbank, copy-out).  Measured on cfg1 (244 frames, profiles/r2_small_batch_latency.txt): 4-warp CTAs 10.3 us,
                    // 8-, 2- and 1-warp CTAs 12.3 us -- so prefer 4 warps, then one round per tile, then more tiles.
                    const double rounds = (double)((TF + FR - 1) / FR);
                    score = 1.0e6 - (NW == 4 ? 0.0 : 500.0) - rounds * 200.0 - (double)TF;
                } else {
                    score += 2.0e6;                               // any shape that fills the machine beats one that does not
                }
            }
            if (score > best_score) {
                best_score = score;
                best = FwdCfg{TF, NW, L.total, bps};
                found = true;
            }
        }
    }
    *out = best;
    return found;
}

template <typename K>
static int kb_set_smem(K kernel, int smem) {
    if (smem > 48 * 1024)
        KB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    return 0;
}

// Launch of a kernel whose body starts with griddepcontrol.wait (kb_stft_cta): programmatic dependent
// launch lets its table prologue overlap the tail of the previous kernel in the stream (the clamp of the
// previous call).  Only kernels that contain the wait may be launched this way.
template <typename Kern>
static int kb_launch_pdl(Kern kernel, int grid, int block, int smem, cudaStream_t st, const KbStftParams& p) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = (size_t)smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = kb_env_int("KAPRE_B200_PDL_FWD", 1) ? 1 : 0;
    KB_CUDA(cudaLaunchKernelEx(&cfg, kernel, p));
    return 0;
}

template <int Q, int MODE>
static int kb_launch_stft_qm(const KbStftParams& p, int grid, int smem, cudaStream_t st) {
    if (p.n_warps > KB_MAX_WARPS) {
        if constexpr (Q == 32 && (MODE == KB_OUT_FB || MODE == KB_OUT_FB_DB)) {
            int rc = kb_set_smem(kb_stft_kernel_w16<Q, MODE>, smem);
            if (rc) return rc;
            KbProfScope prof(st);
            if ((rc = kb_launch_pdl(kb_stft_kernel_w16<Q, MODE>, grid, p.n_warps * 32, smem, st, p))) return rc;
            g_launches++;
            return 0;
        } else {
            return kb_fail(KAPRE_E_UNSUPPORTED, "no 16-warp instantiation for Q=%d mode=%d", Q, MODE);
        }
    }
    if constexpr (Q == 16) {
        if (p.variant & 2) {   // the other form of the pair step (KAPRE_B200_PAIRED=0): the A/B alternative, n_fft 1024 only
            int rc = kb_set_smem(kb_stft_kernel_v<Q, MODE, 2>, smem);
            if (rc) return rc;
            KbProfScope prof(st);
            if ((rc = kb_launch_pdl(kb_stft_kernel_v<Q, MODE, 2>, grid, p.n_warps * 32, smem, st, p))) return rc;
            g_launches++;
            return 0;
        }
    }
    if constexpr (MODE == KB_OUT_FB || MODE == KB_OUT_FB_DB) {
        if (p.fb_mma) {
            int rc = kb_set_smem(kb_stft_kernel_mma<Q, MODE>, smem);
            if (rc) return rc;
            KbProfScope prof(st);
            if ((rc = kb_launch_pdl(kb_stft_kernel_mma<Q, MODE>, grid, p.n_warps * 32, smem, st, p))) return rc;
            g_launches++;
            return 0;
        }
    }
    int rc = kb_set_smem(kb_stft_kernel<Q, MODE>, smem);
    if (rc) return rc;
    KbProfScope prof(st);
    if ((rc = kb_launch_pdl(kb_stft_kernel<Q, MODE>, grid, p.n_warps * 32, smem, st, p))) return rc;
    g_launches++;
    return 0;
}

template <int Q>
static int kb_launch_stft(const KbStftParams& p, int grid, int smem, cudaStream_t st) {
    switch (p.mode) {
        case KB_OUT_COMPLEX: return kb_launch_stft_qm<Q, KB_OUT_COMPLEX>(p, grid, smem, st);
        case KB_OUT_MAG: return kb_launch_stft_qm<Q, KB_OUT_MAG>(p, grid, smem, st);
        case KB_OUT_MAG_DB: return kb_launch_stft_qm<Q, KB_OUT_MAG_DB>(p, grid, smem, st);
        case KB_OUT_FB: return kb_launch_stft_qm<Q, KB_OUT_FB>(p, grid, smem, st);
        case KB_OUT_FB_DB: return kb_launch_stft_qm<Q, KB_OUT_FB_DB>(p, grid, smem, st);
        case KB_OUT_MAG_PHASE: return kb_launch_stft_qm<Q, KB_OUT_MAG_PHASE>(p, grid, smem, st);
    }
    return kb_fail(KAPRE_E_INVALID, "bad mode");
}

template <int Q, bool ADJ>
__global__ void __launch_bounds__(KB_ISTFT_MAX_WARPS * 32, 4) kb_istft2_kernel(const __grid_constant__ KbIstftParams p) {
    extern __shared__ __align__(128) char kb_smem[];
    kb_istft2_cta<Q, ADJ>(p, kb_smem, (int)blockIdx.x, (int)gridDim.x);
}

template <int Q, bool ADJ = false>
static int kb_launch_istft2(const KbIstftParams& p, int grid, int smem, cudaStream_t st) {
    int rc = kb_set_smem(kb_istft2_kernel<Q, ADJ>, smem);
    if (rc) return rc;
    KbProfScope prof(st);
    kb_istft2_kernel<Q, ADJ><<<grid, p.n_warps * 32, smem, st>>>(p);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

template <int Q>
static int kb_launch_istft(const KbIstftParams& p, int grid, int smem, cudaStream_t st) {
    int rc = kb_set_smem(kb_istft_kernel<Q>, smem);
    if (rc) return rc;
    KbProfScope prof(st);
    kb_istft_kernel<Q><<<grid, p.n_warps * 32, smem, st>>>(p);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}


// Launch configuration of the streaming inverse kernel (kb_istft2_cta) for `out_len` output samples: tiles of
// seg = m * FR - (R - 1) output hops, m rounds of FR = NW * FPW frames each.  m is the round count that minimises
// (waves of tiles over the resident CTAs) x (rounds per tile).  Fills the shape fields of *p; returns 1 when the tile
// does not fit shared memory (the caller falls back), 0 on success, < 0 on error.
static int kb_istft2_cfg(const DevInfo& dev, int Q, int n_fft, int hop, int win, int batch, int channels, int frames,
                         long long out_len, KbIstftParams* pp, int* grid_out) {
    const int FPW = 32 / Q;
    const int R = (win + hop - 1) / hop;
    const int NW = KB_ISTFT_MAX_WARPS, FR = NW * FPW;
    const KbIstft2Smem L2 = kb_istft2_smem_layout(Q, n_fft, hop, win, NW);
    if (L2.total > dev.smem_optin) return 1;
    int bps = (228 * 1024) / (L2.total + 1024);
    if (bps > 4) bps = 4;              // __launch_bounds__(128, 4)
    if (bps < 1) bps = 1;
    const long long slots = (long long)dev.sm_count * bps;
    const long long hops = (out_len + hop - 1) / hop;
    // rounds per tile: the most (<= 6: R - 1 halo frames per tile cost <= 6 %) that still leave about one tile per
    // resident CTA.  Measured (profiles/r2_istft_streaming.md): at B256 x 5 s tiles of 6 rounds beat one wave of 28-round
    // tiles by 6 % (the static tile walk balances per SM, not per CTA); at B128 x 1 s tiles of 3 rounds (512 tiles on
    // 592 slots) beat 2 and 4.
    // Floor: tiles long enough that the halo stays under ~20 % of the frames (hop << win: R is large).
    int m_lo = (5 * (R - 1) + FR - 1) / FR;
    if (m_lo < 1) m_lo = 1;
    const int m_hi = m_lo > 6 ? m_lo : 6;
    int best_m = m_lo, best_seg = m_lo * FR - (R - 1);
    for (int m = m_hi; m >= m_lo; --m) {
        const int seg = m * FR - (R - 1);
        const long long nt = (long long)batch * channels * ((hops + seg - 1) / seg);
        best_m = m; best_seg = seg;
        if (nt * 100 >= slots * 85) break;
    }
    const int m_env = kb_env_int("KAPRE_B200_ISTFT2_M", 0);
    if (m_env > 0 && m_env * FR - (R - 1) >= 1) { best_m = m_env; best_seg = m_env * FR - (R - 1); }
    KbIstftParams& p = *pp;
    p.B = batch; p.C = channels; p.T = frames; p.n_fft = n_fft; p.hop = hop; p.win = win;
    p.out_len = (int)out_len;
    p.R = R; p.seg = best_seg; p.n_warps = NW;
    p.n_tiles_t = (int)((hops + best_seg - 1) / best_seg);
    const long long tiles = (long long)batch * channels * p.n_tiles_t;
    if (tiles > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "too many tiles");
    const int grid = (int)(tiles < slots ? tiles : slots);
    {
        char buf[160];
        snprintf(buf, sizeof(buf), "ISTFT2 Q%d NW%d seg%d rounds%d tiles%lld grid%d smem%d bps%d", Q, NW, best_seg, best_m, tiles, grid, L2.total, bps);
        g_launch_info = buf;
    }
    *grid_out = grid;
    return 0;
}

template <bool ADJ>
static int kb_launch_istft2_q(int Q, const KbIstftParams& p, int grid, cudaStream_t st) {
    const int smem = kb_istft2_smem_layout(Q, p.n_fft, p.hop, p.win, p.n_warps).total;
    switch (Q) {
        case 4: return kb_launch_istft2<4, ADJ>(p, grid, smem, st);
        case 8: return kb_launch_istft2<8, ADJ>(p, grid, smem, st);
        case 16: return kb_launch_istft2<16, ADJ>(p, grid, smem, st);
        case 32: return kb_launch_istft2<32, ADJ>(p, grid, smem, st);
        default: return kb_fail(KAPRE_E_UNSUPPORTED, "bad Q");
    }
}


// Tile shape of the multi-channel kernel: TF time frames x C channels = columns, FR = NW * FPW of
// them per round.  Prefer many resident warps, full rounds, two CTAs per SM (their barriers
// overlap), then longer tiles (less re-staging of the frame overlap).
static bool kb_pick_mc_cfg(const DevInfo& dev, int Q, int n_fft, int hop, int C, int with_wh, FwdCfg* out) {
    const int FPW = 32 / Q;
    const int sm_smem = 228 * 1024;
    const int force_tf = kb_env_int("KAPRE_B200_MC_TF", 0);
    const int force_nw = kb_env_int("KAPRE_B200_MC_NW", 0);
    bool found = false;
    FwdCfg best{};
    double best_score = -1.0;
    for (int NW = 1; NW <= 16; ++NW) {
        if (force_nw && NW != force_nw) continue;
        const int FR = NW * FPW;
        if (FR > 32) continue;
        for (int TF = 1; TF <= 32; ++TF) {
            if (force_tf && TF != force_tf) continue;
            const int ncol = TF * C;
            const int rounds = (ncol + FR - 1) / FR;
            if (rounds > 8) break;
            const KbStftMcSmem L = kb_stft_mc_smem_layout(Q, n_fft, hop, TF, C, NW, with_wh);
            if (L.total > dev.smem_optin) break;
            if (NW * 32 < C) continue;                                // the loader gives every channel >= 1 thread
            int bps = sm_smem / (L.total + 1024);
            if (bps > 16 / NW) bps = 16 / NW;                         // 128 registers per thread
            if (bps < 1) continue;
            int warps = bps * NW;
            const double eff = (double)ncol / (double)(rounds * FR);
            const double score = warps * eff * 1000.0 + (bps >= 2 ? 400.0 : 0.0) + TF * 5.0 - rounds * 20.0;
            if (score > best_score) {
                best_score = score;
                best = FwdCfg{TF, NW, L.total, bps};
                found = true;
            }
        }
    }
    *out = best;
    return found;
}

// Filterbank modes on all-channel tiles: one round per tile, TF = floor(NW * FPW / C) time frames.
static bool kb_pick_mcfb_cfg(const DevInfo& dev, int Q, int n_fft, int hop, int C, int with_wh, int n_bands,
                             int n_chunks, FwdCfg* out) {
    const int FPW = 32 / Q;
    const int sm_smem = 228 * 1024;
    bool found = false;
    FwdCfg best{};
    double best_score = -1.0;
    const int nws[3] = {2, 4, 8};
    for (int a = 0; a < 3; ++a) {
        const int NW = nws[a];
        const int FR = NW * FPW;
        if (FR > 32 || FR < C || NW * 32 < C) continue;
        const int TF = FR / C;
        const KbStftMcFbSmem L = kb_stft_mcfb_smem_layout(Q, n_fft, hop, TF, C, NW, with_wh, n_bands, n_chunks);
        if (L.total > dev.smem_optin) continue;
        int bps = sm_smem / (L.total + 1024);
        if (bps > 16 / NW) bps = 16 / NW;
        if (bps < 1) continue;
        const double eff = (double)(TF * C) / (double)FR;
        const double score = bps * NW * eff * 1000.0 + TF * 10.0 + NW;
        if (score > best_score) { best_score = score; best = FwdCfg{TF, NW, L.total, bps}; found = true; }
    }
    *out = best;
    return found;
}

template <int Q, int MODE>
static int kb_launch_stft_mcfb_qm(const KbStftParams& p, int grid, int smem, cudaStream_t st) {
    int rc = kb_set_smem(kb_stft_mcfb_kernel<Q, MODE>, smem);
    if (rc) return rc;
    KbProfScope prof(st);
    kb_stft_mcfb_kernel<Q, MODE><<<grid, p.n_warps * 32, smem, st>>>(p);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

template <int Q>
static int kb_launch_stft_mcfb(const KbStftParams& p, int grid, int smem, cudaStream_t st) {
    if (p.mode == KB_OUT_FB) return kb_launch_stft_mcfb_qm<Q, KB_OUT_FB>(p, grid, smem, st);
    if (p.mode == KB_OUT_FB_DB) return kb_launch_stft_mcfb_qm<Q, KB_OUT_FB_DB>(p, grid, smem, st);
    return kb_fail(KAPRE_E_INVALID, "bad mode for the multi-channel filterbank kernel");
}

template <int Q, int MODE>
static int kb_launch_stft_mc_qm(const KbStftParams& p, int grid, int smem, cudaStream_t st) {
    int rc = kb_set_smem(kb_stft_mc_kernel<Q, MODE>, smem);
    if (rc) return rc;
    KbProfScope prof(st);
    kb_stft_mc_kernel<Q, MODE><<<grid, p.n_warps * 32, smem, st>>>(p);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

template <int Q>
static int kb_launch_stft_mc(const KbStftParams& p, int grid, int smem, cudaStream_t st) {
    switch (p.mode) {
        case KB_OUT_COMPLEX: return kb_launch_stft_mc_qm<Q, KB_OUT_COMPLEX>(p, grid, smem, st);
        case KB_OUT_MAG: return kb_launch_stft_mc_qm<Q, KB_OUT_MAG>(p, grid, smem, st);
        case KB_OUT_MAG_DB: return kb_launch_stft_mc_qm<Q, KB_OUT_MAG_DB>(p, grid, smem, st);
        case KB_OUT_MAG_PHASE: return kb_launch_stft_mc_qm<Q, KB_OUT_MAG_PHASE>(p, grid, smem, st);
    }
    return kb_fail(KAPRE_E_INVALID, "bad mode for the multi-channel kernel");
}

static int kb_check_device(const DevInfo& d) {
    int cur = -1;
    KB_CUDA(cudaGetDevice(&cur));
    if (cur != d.device)
        return kb_fail(KAPRE_E_INVALID, "plan was created on device %d but device %d is current", d.device, cur);
    return 0;
}

static int kb_launch_clamp(float* y, long long n_items, long long item_size, unsigned int* item_max,
                           float amin, float db_mul, float db_sub, float dr, cudaStream_t st,
                           long long run = 1, long long period = 1) {
    if (n_items <= 0 || item_size <= 0) return 0;
    // one CTA per 32 Ki elements of an item (at most 64): a binding clamp on a long item is rewritten in parallel
    long long chunks = (item_size + 32767) / 32768;
    if (chunks > 64) chunks = 64;
    if (chunks < 1) chunks = 1;
    if (n_items * chunks > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "too many items for the clamp kernel");
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(n_items * chunks));
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = kb_env_int("KAPRE_B200_PDL", 1) ? 1 : 0;
    KB_CUDA(cudaLaunchKernelEx(&cfg, kb_db_clamp_kernel, y, item_size, run, period, item_max, (unsigned int)n_items,
                               (int)chunks, amin, db_mul, db_sub, dr));
    g_launches++;
    return 0;
}

static void kb_db_consts(const kapre_db_cfg* db, float* db_mul, float* db_sub) {
    // 10*log10(v) = (10*log10(2)) * log2(v);  kapre/backend.py:187-188
    *db_mul = (float)(10.0 * log10(2.0));
    const double m = db->amin > db->ref_value ? db->amin : db->ref_value;
    *db_sub = (float)(10.0 * log10(m));
}

static int kb_check_db(const kapre_db_cfg* db) {
    if (!db) return kb_fail(KAPRE_E_INVALID, "decibel configuration required");
    // kapre/backend.py:168-173
    if (!(db->ref_value > 0)) return kb_fail(KAPRE_E_INVALID, "ref_value must be positive, got: %g", db->ref_value);
    if (!(db->amin > 0)) return kb_fail(KAPRE_E_INVALID, "amin must be positive, got: %g", db->amin);
    if (!(db->dynamic_range > 0)) return kb_fail(KAPRE_E_INVALID, "dynamic_range must be positive, got: %g", db->dynamic_range);
    return 0;
}

// ------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------
extern "C" {

const char* kapre_last_error(void) { return g_err.c_str(); }
int kapre_version(void) { return KAPRE_B200_VERSION; }
uint64_t kapre_launch_count(void) { return g_launches.load(); }
const char* kapre_last_launch_info(void) { return g_launch_info.c_str(); }

int kapre_profile_enable(int enable) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_on = enable > 0 ? enable : 0;
    g_prof_seq = 0;
    return 0;
}

int kapre_profile_read(double* total_ms, uint64_t* launches) {
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> evs;
    {
        std::lock_guard<std::mutex> lk(g_prof_mu);
        evs.swap(g_prof_events);
    }
    double tot = 0.0;
    uint64_t n = 0;
    for (auto& pr : evs) {
        float ms = 0.0f;
        if (cudaEventSynchronize(pr.second) == cudaSuccess && cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
            tot += ms;
            ++n;
        }
        cudaEventDestroy(pr.first);
        cudaEventDestroy(pr.second);
    }
    if (total_ms) *total_ms = tot;
    if (launches) *launches = n;
    return 0;
}

int kapre_stft_plan_create(int n_fft, int win_length, int hop_length, const float* window_host,
                           kapre_stft_plan** out) {
    if (!out || !window_host) return kb_fail(KAPRE_E_INVALID, "null argument");
    if (n_fft < 2 || win_length < 1 || hop_length < 1)
        return kb_fail(KAPRE_E_INVALID, "n_fft=%d win_length=%d hop_length=%d out of range", n_fft, win_length, hop_length);
    if (n_fft > 16384) return kb_fail(KAPRE_E_UNSUPPORTED, "n_fft=%d > 16384 is not supported", n_fft);
    kapre_stft_plan* p = new kapre_stft_plan();
    p->n_fft = n_fft; p->win_length = win_length; p->hop = hop_length;
    p->Q = kb_q_for_nfft(n_fft);
    p->win_eff = win_length < n_fft ? win_length : n_fft;
    int rc = kb_dev_info(&p->dev);
    if (rc) { delete p; return rc; }
    if (p->Q) {
        std::vector<float> wh; std::vector<float2> twp, twn, twn2;
        kb_make_wh(window_host, win_length, n_fft, wh);
        kb_make_twp(p->Q, twp);
        kb_make_twn(n_fft, twn);
        kb_make_twn2(n_fft, twn2);
        if ((rc = kb_upload(wh, &p->wh)) || (rc = kb_upload(twp, &p->twp)) || (rc = kb_upload(twn, &p->twn)) ||
            (rc = kb_upload(twn2, &p->twn2))) {
            kapre_stft_plan_destroy(p); return rc;
        }
        double ca = 0.0, cb = 0.0;
        if (kb_fit_cosine_window(window_host, win_length, n_fft, &ca, &cb) && kb_env_int("KAPRE_B200_NOCOSW", 0) == 0) {
            std::vector<kb_f4> cwq;
            kb_make_cwq(p->Q, n_fft, cb, cwq);
            if ((rc = kb_upload(cwq, &p->cwq))) { kapre_stft_plan_destroy(p); return rc; }
            p->cosw = 1;
            p->cw_a0 = (float)(0.5 * ca);
        }
        if (n_fft == 1024 && win_length == 1024 && kb_fit_cosine_window(window_host, win_length, n_fft, &ca, &cb) && ca > 0.0) {
            p->win_a = ca; p->win_b = cb;
            if ((rc = kb_tc_tables(p))) { kapre_stft_plan_destroy(p); return rc; }
        }
    }
    {   // generic tables are always built: they also serve sizes the fused kernel cannot take
        std::vector<float> w(window_host, window_host + p->win_eff);
        std::vector<float2> tw(n_fft);
        for (int r = 0; r < n_fft; ++r) {
            const double a = -2.0 * M_PI * (double)r / (double)n_fft;
            tw[r] = make_float2((float)cos(a), (float)sin(a));
        }
        if ((rc = kb_upload(w, &p->w)) || (rc = kb_upload(tw, &p->tw))) { kapre_stft_plan_destroy(p); return rc; }
    }
    {   // adjoint tables
        std::vector<float> wa(p->win_eff), dn(p->win_eff);
        for (int m = 0; m < p->win_eff; ++m) {
            wa[m] = (float)(0.5 * (double)n_fft * (double)window_host[m]);
            dn[m] = (float)(0.5 * (double)window_host[m]);
        }
        std::vector<float2> tw(n_fft);
        for (int r = 0; r < n_fft; ++r) {
            const double a = 2.0 * M_PI * (double)r / (double)n_fft;
            tw[r] = make_float2((float)cos(a), (float)sin(a));
        }
        if ((rc = kb_upload(dn, &p->adj_dn)) || (rc = kb_upload(tw, &p->adj_tw))) { kapre_stft_plan_destroy(p); return rc; }
        if (p->Q) {
            std::vector<float> adj;
            kb_make_dual(wa.data(), p->win_eff, n_fft, adj);
            if ((rc = kb_upload(adj, &p->adj))) { kapre_stft_plan_destroy(p); return rc; }
        }
    }
    *out = p;
    return 0;
}

void kapre_stft_plan_destroy(kapre_stft_plan* p) {
    if (!p) return;
    cudaFree(p->adj); cudaFree(p->adj_dn); cudaFree(p->adj_tw);
    cudaFree(p->wh); cudaFree(p->cwq); cudaFree(p->twp); cudaFree(p->twn); cudaFree(p->twn2); cudaFree(p->w); cudaFree(p->tw);
    cudaFree(p->tc_f1); cudaFree(p->tc_cs); cudaFree(p->tc_csb); cudaFree(p->tc_tw); cudaFree(p->tc_w32);
    delete p;
}

int kapre_stft_num_frames(const kapre_stft_plan* p, int length, int pad_begin, int pad_end) {
    if (!p || length < 0) return kb_fail(KAPRE_E_INVALID, "bad argument");
    const long long Lp = (long long)length + (pad_begin ? (p->n_fft - p->hop) : 0);
    if (pad_end) return (int)((Lp + p->hop - 1) / p->hop);
    if (Lp < p->win_length) return 0;
    return (int)(1 + (Lp - p->win_length) / p->hop);
}

int kapre_stft_supports_mode(const kapre_stft_plan* p, int mode) {
    if (!p) return 0;
    if (mode < KAPRE_OUT_COMPLEX || mode > KAPRE_OUT_MAG_PHASE) return 0;
    if (p->Q) return 1;
    if (mode == KAPRE_OUT_COMPLEX || mode == KAPRE_OUT_MAG) return 1;
    if (mode == KAPRE_OUT_MAG_PHASE) return 0;
    // fused filterbank / decibel tail of the mixed-radix kernel: 5-smooth transform length whose buffers fit
    int radix[KB_MR_MAX_PASS];
    const int P = (p->n_fft & 1) ? p->n_fft : p->n_fft / 2;
    if (kb_mr_factor(P, radix) < 0 || kb_env_int("KAPRE_B200_NOMR", 0)) return 0;
    int nw, g, b;
    if (mode == KAPRE_OUT_MAG_DB) return kb_mr_pick(P, p->dev.smem_optin, 228 * 1024, 32, &nw, &g, &b) > 0 ? 1 : 0;
    // 128 bands as the sizing assumption for the filterbank tile (the launch re-picks with the real count and fails loudly)
    return kb_mr_pick(P, p->dev.smem_optin, 228 * 1024, 32, &nw, &g, &b, p->n_fft / 2 + 1, 128, 8) > 0 ? 1 : 0;
}

int kapre_stft_forward(const kapre_stft_plan* plan, const float* x_dev, const kapre_wave_desc* xd,
                       int pad_begin, int pad_end, int mode, void* out_dev, const kapre_spec_desc* od,
                       const kapre_filterbank* fb, const kapre_db_cfg* db, void* workspace_dev, void* stream) {
    if (!plan || !xd || !od) return kb_fail(KAPRE_E_INVALID, "null argument");
    if (mode < KAPRE_OUT_COMPLEX || mode > KAPRE_OUT_MAG_PHASE) return kb_fail(KAPRE_E_INVALID, "bad mode %d", mode);
    int rc = kb_check_device(plan->dev);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const int B = xd->batch, C = xd->channels, Ln = xd->length;
    if (B < 0 || C < 0 || Ln < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    if (pad_begin && plan->hop > plan->n_fft)
        return kb_fail(KAPRE_E_INVALID, "pad_begin needs hop_length <= n_fft (the padding is n_fft - hop_length = %d)",
                       plan->n_fft - plan->hop);
    const int T = kapre_stft_num_frames(plan, Ln, pad_begin, pad_end);
    if (B == 0 || C == 0 || T <= 0) return 0;
    if (!x_dev || !out_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    if ((long long)T * plan->hop + plan->n_fft > 0x7fffffffLL)
        return kb_fail(KAPRE_E_UNSUPPORTED, "signal too long");
    const bool fbmode = (mode == KAPRE_OUT_FB || mode == KAPRE_OUT_FB_DB);
    const bool dbmode = (mode == KAPRE_OUT_MAG_DB || mode == KAPRE_OUT_FB_DB || (mode == KAPRE_OUT_MAG_PHASE && db != nullptr));
    if (fbmode) {
        if (!fb) return kb_fail(KAPRE_E_INVALID, "filterbank required for mode %d", mode);
        if (fb->n_freq != plan->n_fft / 2 + 1)
            return kb_fail(KAPRE_E_INVALID, "filterbank has %d rows but n_fft/2+1 = %d", fb->n_freq, plan->n_fft / 2 + 1);
        if (fb->dev.device != plan->dev.device) return kb_fail(KAPRE_E_INVALID, "filterbank lives on another device");
        if (plan->Q && fb->Q != plan->Q) return kb_fail(KAPRE_E_INVALID, "filterbank was not prepared for n_fft=%d", plan->n_fft);
    }
    float db_mul = 0, db_sub = 0;
    long long db_item_size = 0, db_run = 1, db_period = 1;
    if (dbmode) {
        if ((rc = kb_check_db(db))) return rc;
        if (!workspace_dev) return kb_fail(KAPRE_E_INVALID, "workspace required for decibel modes");
        kb_db_consts(db, &db_mul, &db_sub);
        // Output layout of the clamp pass, checked BEFORE anything is launched (a late failure would leave
        // per-item maxima in the self-cleaning workspace).  Items are contiguous blocks of stride_b elements
        // in both data formats.
        const long long K = fbmode ? fb->n_bands : (plan->n_fft / 2 + 1);
        const long long chans = (mode == KAPRE_OUT_MAG_PHASE) ? 2LL * C : C;
        db_item_size = chans * T * K;
        if (od->stride_b != db_item_size)
            return kb_fail(KAPRE_E_UNSUPPORTED, "decibel modes need a batch-contiguous output (stride_b=%lld, item=%lld)",
                           (long long)od->stride_b, db_item_size);
        if (mode == KAPRE_OUT_MAG_PHASE) {   // clamp only the magnitude channels [0, C) of the 2C-channel item
            if (od->stride_c == 1 && od->stride_f == chans && od->stride_t == K * chans) { db_run = C; db_period = chans; }
            else if (od->stride_f == 1 && od->stride_t == K && od->stride_c == (long long)T * K) { db_run = (long long)C * T * K; db_period = db_item_size; }
            else return kb_fail(KAPRE_E_UNSUPPORTED, "mag+phase decibel output must be a contiguous channels_first or channels_last tensor");
        }
    }
    const int pad_left = pad_begin ? (plan->n_fft - plan->hop) : 0;

    if (!plan->Q) {
        if (mode == KAPRE_OUT_MAG_PHASE)
            return kb_fail(KAPRE_E_UNSUPPORTED, "n_fft=%d has no fused magnitude+phase path; chain the stand-alone ops", plan->n_fft);
        KbDftParams p{};
        p.x = x_dev; p.x_sb = xd->stride_b; p.x_sc = xd->stride_c; p.x_sl = xd->stride_l;
        p.B = B; p.C = C; p.L = Ln; p.n_fft = plan->n_fft; p.hop = plan->hop; p.T = T; p.pad_left = pad_left;
        p.win_eff = plan->win_eff; p.w = plan->w; p.tw = plan->tw;
        p.out = out_dev; p.o_sb = od->stride_b; p.o_sc = od->stride_c; p.o_st = od->stride_t; p.o_sk = od->stride_f;
        p.mode = mode; p.n_tiles_t = (T + KB_DFT_TF - 1) / KB_DFT_TF; p.n_warps = 8;
        {   // mixed-radix Stockham FFT when n_fft/2 (even) or n_fft (odd) is 5-smooth and the buffers fit
            KbMrParams q{};
            q.half = (plan->n_fft & 1) ? 0 : 1;
            q.P = q.half ? plan->n_fft / 2 : plan->n_fft;
            q.n_pass = kb_mr_factor(q.P, q.radix);
            int NW = 8, G = 1, bps = 1, FRT = 0, fit = 0;
            const int want = kb_env_int("KAPRE_B200_MR_WARPS", 32);
            const int F = plan->n_fft / 2 + 1, nb = fbmode ? fb->n_bands : 0;
            if (q.n_pass >= 0 && kb_env_int("KAPRE_B200_NOMR", 0) == 0) {
                if (!fbmode) fit = kb_mr_pick(q.P, plan->dev.smem_optin, 228 * 1024, want, &NW, &G, &bps);
                else {
                    // filterbank tile of 32 frames unless a smaller one keeps clearly more warps resident
                    for (int frt = 32; frt >= 8; frt >>= 1) {
                        int nw = 8, g = 1, b2 = 1;
                        const int f2 = kb_mr_pick(q.P, plan->dev.smem_optin, 228 * 1024, want, &nw, &g, &b2, F, nb, frt);
                        if (f2 > fit + fit / 2) { fit = f2; NW = nw; G = g; bps = b2; FRT = frt; }
                    }
                }
            }
            if (fit > 0) {
                const int smem = kb_mr_smem_layout(q.P, NW / G, F, nb, FRT).total;
                q.d = p; q.d.n_warps = NW;
                q.G = G;
                q.pad1 = (q.n_pass > 0 && q.radix[0] % 2 == 0) ? 1 : 0;
                q.FRT = FRT;
                if (fbmode) { q.bands = fb->bands; q.fbw = fb->w; q.n_bands = fb->n_bands; }
                kb_mr_finish(q);
                // frames per group and tile: 16 amortises the per-tile bookkeeping (two divisions, 64-bit bases) unless the
                // batch is small -- keep at least ~8 tiles per resident CTA for the tail
                int fpg = 16;
                while (fpg > 4 && (long long)B * C * ((T + fpg * (NW / G) - 1) / (fpg * (NW / G))) < 8LL * plan->dev.sm_count * bps)
                    fpg >>= 1;
                q.TF = FRT > 0 ? FRT : fpg * (NW / G);
                if (dbmode) {
                    q.amin = db->amin; q.db_mul = db_mul; q.db_sub = db_sub; q.item_max = (unsigned int*)workspace_dev;
                    q.db_ftz = (db->amin >= 1.17549435e-38f) ? 1 : 0;
                }
                if ((rc = kb_set_smem(kb_mr_kernel, smem))) return rc;
                const long long tiles = (long long)B * C * ((T + q.TF - 1) / q.TF);
                const long long gmax = (long long)plan->dev.sm_count * bps;
                const int grid = (int)(tiles < gmax ? tiles : gmax);
                {
                    KbProfScope prof(st);
                    kb_mr_kernel<<<grid, NW * 32, smem, st>>>(q);
                    KB_CUDA(cudaGetLastError());
                    g_launches++;
                }
                char buf[160];
                snprintf(buf, sizeof(buf), "MR P%d passes%d NW%d G%d grid%d smem%d bps%d frt%d", q.P, q.n_pass, NW, G, grid, smem, bps, FRT);
                g_launch_info = buf;
                if (dbmode)
                    rc = kb_launch_clamp((float*)out_dev, B, db_item_size, (unsigned int*)workspace_dev, db->amin, db_mul, db_sub,
                                         db->dynamic_range, st, db_run, db_period);
                return rc;
            }
        }
        if (!(mode == KAPRE_OUT_COMPLEX || mode == KAPRE_OUT_MAG))
            return kb_fail(KAPRE_E_UNSUPPORTED, "n_fft=%d (prime factor above 5) has no fused filterbank/decibel path; chain the stand-alone ops", plan->n_fft);
        const KbDftSmem L = kb_dft_smem_layout(plan->n_fft, plan->win_eff);
        if (L.total > plan->dev.smem_optin) return kb_fail(KAPRE_E_UNSUPPORTED, "n_fft=%d has a prime factor above 5 and is too large for the direct-DFT kernel (%d B of shared memory needed)", plan->n_fft, L.total);
        if ((rc = kb_set_smem(kb_dft_kernel, L.total))) return rc;
        long long tiles = (long long)B * C * p.n_tiles_t;
        int grid = (int)(tiles < plan->dev.sm_count * 4LL ? tiles : plan->dev.sm_count * 4LL);
        kb_dft_kernel<<<grid, 256, L.total, st>>>(p);
        KB_CUDA(cudaGetLastError());
        g_launches++;
        {
            char buf[96];
            snprintf(buf, sizeof(buf), "DFT n_fft%d grid%d smem%d (direct O(N^2): prime factor > 5)", plan->n_fft, grid, L.total);
            g_launch_info = buf;
        }
        return 0;
    }

    // address range of the waveform tensor (non-negative strides): the rounded bulk copies stay inside
    const long long max_off = (long long)(B - 1) * xd->stride_b + (long long)(C - 1) * xd->stride_c +
                              (long long)(Ln - 1) * xd->stride_l;
    const bool bulk = (xd->stride_l == 1) && (((uintptr_t)x_dev & 3) == 0) && xd->stride_b >= 0 && xd->stride_c >= 0 &&
                      kb_env_int("KAPRE_B200_NOBULK", 0) == 0;
    // ---- tensor-core FFT path (tc_mel.cuh): n_fft = win_length = 1024, cosine-sum window, hop 128 / 256, planar signals ----
    if (fbmode && plan->tc_f1 && (plan->hop == 256 || plan->hop == 128) && xd->stride_l == 1 && fb->n_bands <= 128 &&
        fb->cw && kb_env_int("KAPRE_B200_TC", KB_TC_DEFAULT)) {
        const KbTcMelSmem TL = kb_tcm_smem_layout(fb->n_chunks);
        if (TL.total <= plan->dev.smem_optin) {
            KbTcMelParams q{};
            q.x = x_dev; q.x_sb = xd->stride_b; q.x_sc = xd->stride_c;
            q.B = B; q.C = C; q.L = Ln; q.T = T; q.hop = plan->hop; q.pad_left = pad_left;
            q.wc = (float)(plan->win_b / (2.0 * plan->win_a));
            q.f1 = plan->tc_f1; q.cs = plan->tc_cs; q.csb = plan->tc_csb; q.tw = plan->tc_tw; q.w32 = plan->tc_w32;
            q.cw = fb->cw; q.cm = fb->cm; q.cg = fb->cg; q.n_chunks = fb->n_chunks; q.n_bands = fb->n_bands;
            q.out = (float*)out_dev; q.o_sb = od->stride_b; q.o_sc = od->stride_c; q.o_st = od->stride_t; q.o_sk = od->stride_f;
            q.db = dbmode ? 1 : 0;
            if (dbmode) { q.amin = db->amin; q.db_mul = db_mul; q.db_sub = db_sub; q.item_max = (unsigned int*)workspace_dev; }
            q.dbg = g_tc_dbg; g_tc_dbg = nullptr;
            q.n_tiles_t = (T + TCM_TF - 1) / TCM_TF;
            q.ablate = kb_env_int("KAPRE_B200_TC_ABLATE", 0);
            const long long tiles = (long long)B * C * q.n_tiles_t;
            if (tiles > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "too many tiles");
            const int grid = (int)(tiles < plan->dev.sm_count ? tiles : plan->dev.sm_count);
            if ((rc = kb_set_smem(kb_tc_mel_kernel, TL.total))) return rc;
            {
                KbProfScope prof(st);
                cudaLaunchConfig_t lc{};
                lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3(TCM_THREADS); lc.dynamicSmemBytes = (size_t)TL.total; lc.stream = st;
                cudaLaunchAttribute attr[1];
                attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
                attr[0].val.programmaticStreamSerializationAllowed = 1;
                lc.attrs = attr; lc.numAttrs = kb_env_int("KAPRE_B200_PDL_FWD", 1) ? 1 : 0;
                KB_CUDA(cudaLaunchKernelEx(&lc, kb_tc_mel_kernel, q));
                g_launches++;
            }
            char buf[160];
            snprintf(buf, sizeof(buf), "TC tcgen05 n_fft1024 hop%d grid%d smem%d tiles%lld", plan->hop, grid, TL.total, tiles);
            g_launch_info = buf;
            if (dbmode)
                rc = kb_launch_clamp((float*)out_dev, B, db_item_size, (unsigned int*)workspace_dev, db->amin, db_mul, db_sub,
                                     db->dynamic_range, st, db_run, db_period);
            return rc;
        }
    }
    FwdCfg cfg;
    // filterbank phase on the tensor pipe (mma.sync 3xTF32) or on the CUDA cores (chunk lists)
    const int fbmma = (fbmode && fb->mw && kb_env_int("KAPRE_B200_FBMMA", KB_FBMMA_DEFAULT)) ? 1 : 0;
    // Pair step of the register kernel: kb_stft_cta picks the paired-column or the natural-order form per (n_fft, mode) from
    // the measurements in profiles/r2_small_experiments.md; KAPRE_B200_PAIRED=0 runs the other form (variant bit 1,
    // instantiated for n_fft 1024 only: the A/B alternative).
    const int variant = (!fbmma && plan->Q == 16 && kb_env_int("KAPRE_B200_PAIRED", KB_PAIRED_DEFAULT) == 0) ? 2 : 0;
    if (!kb_pick_fwd_cfg(plan->dev, plan->Q, plan->n_fft, plan->hop, mode, fbmode ? fb->n_bands : 0,
                         fbmode ? (fbmma ? fb->n_msteps : fb->n_chunks) : 0, fbmma, (long long)B * C, T, &cfg))
        return kb_fail(KAPRE_E_UNSUPPORTED, "no launch configuration fits shared memory (n_fft=%d hop=%d bands=%d)",
                       plan->n_fft, plan->hop, fbmode ? fb->n_bands : 0);
    KbStftParams p{};
    p.x = x_dev; p.x_sb = xd->stride_b; p.x_sc = xd->stride_c; p.x_sl = xd->stride_l;
    p.B = B; p.C = C; p.L = Ln; p.n_fft = plan->n_fft; p.hop = plan->hop; p.T = T; p.pad_left = pad_left;
    p.x_lo = x_dev; p.x_hi = x_dev + max_off + 1; p.x_numel = max_off + 1;
    p.x_align = (unsigned)(((uintptr_t)x_dev >> 2) & 3); p.bulk_ok = bulk ? 1 : 0; p.dbuf = 0;
    p.wh = plan->wh; p.twp = plan->twp; p.twn = plan->twn; p.twn2 = plan->twn2;
    p.cosw = plan->cosw; p.cw_a0 = plan->cw_a0; p.cwq = plan->cwq;
    p.out = out_dev; p.o_sb = od->stride_b; p.o_sc = od->stride_c; p.o_st = od->stride_t; p.o_sk = od->stride_f;
    p.mode = mode;
    if (fbmode) {
        p.bands = fb->bands; p.fbw = fb->w; p.n_bands = fb->n_bands; p.n_fbw = fb->n_w;
        p.cw = fb->cw; p.cm = fb->cm; p.cg = fb->cg; p.n_chunks = fb->n_chunks;
        p.mw = fb->mw; p.ms = fb->ms; p.mg = fb->mg; p.n_msteps = fb->n_msteps;
        p.bd = fb->bd; p.bg = fb->bg; p.n_bd = fb->n_bd;
        // measured slower than the flat predicated chunk list (0.184 vs 0.1765 ms on cfg2, profiles/r2_small_experiments.md):
        // the groups of a warp walk bands of different lengths, the flat list is balanced per group.  Off by default.
        p.fb_bands = (fb->bd && kb_env_int("KAPRE_B200_FBBANDS", 0)) ? 1 : 0;
    }
    if (dbmode) {
        p.amin = db->amin; p.db_mul = db_mul; p.db_sub = db_sub; p.item_max = (unsigned int*)workspace_dev;
        p.db_ftz = (db->amin >= 1.17549435e-38f) ? 1 : 0;
    }
    if (mode == KAPRE_OUT_MAG_PHASE) { p.db_on = dbmode ? 1 : 0; p.ph_off = (long long)C * od->stride_c; }
    // interleaved (channels_last) tensors with several channels: tiles that hold all channels
    const bool strided_in = xd->stride_l != 1, strided_out = od->stride_f != 1;
    const bool mc_ok = C > 1 && C <= 32 && (strided_in || strided_out) && xd->stride_b >= 0 &&
                       xd->stride_c >= 0 && xd->stride_l >= 0 && kb_env_int("KAPRE_B200_NOMC", 0) == 0;
    FwdCfg mcfg{};
    const int mc_wh = (!plan->cosw || (plan->hop & 1)) ? 1 : 0;
    const bool use_mc = mc_ok && (fbmode ? kb_pick_mcfb_cfg(plan->dev, plan->Q, plan->n_fft, plan->hop, C, mc_wh,
                                                            fb->n_bands, fb->n_chunks, &mcfg)
                                         : kb_pick_mc_cfg(plan->dev, plan->Q, plan->n_fft, plan->hop, C, mc_wh, &mcfg));
    long long tiles;
    int grid;
    if (use_mc) {
        cfg = mcfg;
        p.TF = cfg.TF; p.n_tiles_t = (T + cfg.TF - 1) / cfg.TF; p.n_warps = cfg.NW;
        p.mc_wh = mc_wh;
        p.mc_cl_in = (xd->stride_c < xd->stride_l) ? 1 : 0;
        p.mc_out = (od->stride_c == 1) ? 1 : 0;
        const int FR = cfg.NW * (32 / plan->Q), ncol = cfg.TF * C;
        const int last = ncol - ((ncol - 1) / FR) * FR;
        p.mc_magic_c = kb_magic((unsigned)C);
        p.mc_magic_g = kb_magic((unsigned)((cfg.NW * 32) / C));
        p.mc_magic_fr = kb_magic((unsigned)(FR < ncol ? FR : ncol));
        p.mc_magic_last = kb_magic((unsigned)last);
        tiles = (long long)B * p.n_tiles_t;
        if (tiles > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "too many tiles");
        const long long gmax = (long long)plan->dev.sm_count * cfg.bps;
        grid = (int)(tiles < gmax ? tiles : gmax);
        if (fbmode) {
            switch (plan->Q) {
                case 4: rc = kb_launch_stft_mcfb<4>(p, grid, cfg.smem, st); break;
                case 8: rc = kb_launch_stft_mcfb<8>(p, grid, cfg.smem, st); break;
                case 16: rc = kb_launch_stft_mcfb<16>(p, grid, cfg.smem, st); break;
                case 32: rc = kb_launch_stft_mcfb<32>(p, grid, cfg.smem, st); break;
                default: rc = kb_fail(KAPRE_E_UNSUPPORTED, "bad Q");
            }
        } else {
            switch (plan->Q) {
                case 4: rc = kb_launch_stft_mc<4>(p, grid, cfg.smem, st); break;
                case 8: rc = kb_launch_stft_mc<8>(p, grid, cfg.smem, st); break;
                case 16: rc = kb_launch_stft_mc<16>(p, grid, cfg.smem, st); break;
                case 32: rc = kb_launch_stft_mc<32>(p, grid, cfg.smem, st); break;
                default: rc = kb_fail(KAPRE_E_UNSUPPORTED, "bad Q");
            }
        }
    } else {
        p.TF = cfg.TF; p.n_tiles_t = (T + cfg.TF - 1) / cfg.TF; p.n_warps = cfg.NW;
        p.fb_mma = fbmma;
        p.variant = variant;

        tiles = (long long)B * C * p.n_tiles_t;
        if (tiles > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "too many tiles");
        const long long gmax = (long long)plan->dev.sm_count * cfg.bps;
        grid = (int)(tiles < gmax ? tiles : gmax);
        switch (plan->Q) {
            case 4: rc = kb_launch_stft<4>(p, grid, cfg.smem, st); break;
            case 8: rc = kb_launch_stft<8>(p, grid, cfg.smem, st); break;
            case 16: rc = kb_launch_stft<16>(p, grid, cfg.smem, st); break;
            case 32: rc = kb_launch_stft<32>(p, grid, cfg.smem, st); break;
            default: rc = kb_fail(KAPRE_E_UNSUPPORTED, "bad Q");
        }
    }
    if (rc) return rc;
    {
        char buf[160];
        snprintf(buf, sizeof(buf), "%sQ%d TF%d NW%d bulk%d grid%d smem%d bps%d tiles%lld fbmma%d v%d", use_mc ? "MC " : "", plan->Q,
                 cfg.TF, cfg.NW, use_mc ? 0 : (int)bulk, grid, cfg.smem, cfg.bps, tiles, use_mc ? 0 : fbmma,
                 use_mc ? 0 : p.variant);
        g_launch_info = buf;
    }
    if (dbmode)
        rc = kb_launch_clamp((float*)out_dev, B, db_item_size, (unsigned int*)workspace_dev, db->amin, db_mul, db_sub,
                             db->dynamic_range, st, db_run, db_period);
    return rc;
}

int kapre_istft_plan_create(int n_fft, int win_length, int hop_length, const float* dual_window_host,
                            kapre_istft_plan** out) {
    if (!out || !dual_window_host) return kb_fail(KAPRE_E_INVALID, "null argument");
    if (n_fft < 2 || win_length < 1 || hop_length < 1)
        return kb_fail(KAPRE_E_INVALID, "n_fft=%d win_length=%d hop_length=%d out of range", n_fft, win_length, hop_length);
    if (n_fft > 16384) return kb_fail(KAPRE_E_UNSUPPORTED, "n_fft=%d > 16384 is not supported", n_fft);
    kapre_istft_plan* p = new kapre_istft_plan();
    p->n_fft = n_fft; p->win_length = win_length; p->hop = hop_length;
    p->Q = kb_q_for_nfft(n_fft);
    p->win = win_length < n_fft ? win_length : n_fft;
    int rc = kb_dev_info(&p->dev);
    if (rc) { delete p; return rc; }
    if (p->Q) {
        std::vector<float> dual; std::vector<float2> twp, twn;
        kb_make_dual(dual_window_host, p->win, n_fft, dual);
        kb_make_twp(p->Q, twp);
        kb_make_twn(n_fft, twn);
        if ((rc = kb_upload(dual, &p->dual)) || (rc = kb_upload(twp, &p->twp)) || (rc = kb_upload(twn, &p->twn))) {
            kapre_istft_plan_destroy(p); return rc;
        }
    }
    {
        std::vector<float> dn(p->win);
        for (int m = 0; m < p->win; ++m) dn[m] = (float)((double)dual_window_host[m] / (double)n_fft);
        std::vector<float2> tw(n_fft);
        for (int r = 0; r < n_fft; ++r) {
            const double a = 2.0 * M_PI * (double)r / (double)n_fft;
            tw[r] = make_float2((float)cos(a), (float)sin(a));
        }
        if ((rc = kb_upload(dn, &p->dualn)) || (rc = kb_upload(tw, &p->tw))) { kapre_istft_plan_destroy(p); return rc; }
    }
    {   // VJP: the forward STFT of the upstream gradient with the window 2/n_fft * dual (kapre_istft_backward)
        std::vector<float> w2(win_length);
        for (int m = 0; m < win_length; ++m) w2[m] = (float)(2.0 * (double)dual_window_host[m] / (double)n_fft);
        if ((rc = kapre_stft_plan_create(n_fft, win_length, hop_length, w2.data(), &p->grad))) { kapre_istft_plan_destroy(p); return rc; }
    }
    *out = p;
    return 0;
}

void kapre_istft_plan_destroy(kapre_istft_plan* p) {
    if (!p) return;
    cudaFree(p->dual); cudaFree(p->twp); cudaFree(p->twn); cudaFree(p->dualn); cudaFree(p->tw);
    kapre_stft_plan_destroy(p->grad);
    delete p;
}

int kapre_istft_inverse(const kapre_istft_plan* plan, const void* stft_dev, int batch, int channels, int frames,
                        const kapre_spec_desc* sd, float* y_dev, const kapre_wave_desc* yd, void* stream) {
    if (!plan || !sd || !yd) return kb_fail(KAPRE_E_INVALID, "null argument");
    int rc = kb_check_device(plan->dev);
    if (rc) return rc;
    if (batch < 0 || channels < 0 || frames < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    if (batch == 0 || channels == 0 || frames == 0) return 0;
    if (!stft_dev || !y_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const long long out_len = (long long)(frames - 1) * plan->hop + plan->win_length;
    if (out_len > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "signal too long");
    if (yd->length != (int)out_len)
        return kb_fail(KAPRE_E_INVALID, "output length must be (frames-1)*hop+win_length = %lld, got %d", out_len, yd->length);

    if (!plan->Q) {
        KbIdftParams p{};
        p.X = (const float2*)stft_dev; p.x_sb = sd->stride_b; p.x_sc = sd->stride_c; p.x_st = sd->stride_t; p.x_sk = sd->stride_f;
        p.B = batch; p.C = channels; p.T = frames; p.n_fft = plan->n_fft; p.hop = plan->hop; p.win = plan->win;
        p.out_len = (int)out_len; p.dualn = plan->dualn; p.tw = plan->tw;
        p.y = y_dev; p.y_sb = yd->stride_b; p.y_sc = yd->stride_c; p.y_sl = yd->stride_l;
        p.n_warps = 8; p.n_tiles_s = (int)((out_len + 255) / 256);
        const int smem = plan->n_fft * 8;
        if (smem > plan->dev.smem_optin) return kb_fail(KAPRE_E_UNSUPPORTED, "n_fft too large");
        if ((rc = kb_set_smem(kb_idft_kernel, smem))) return rc;
        long long tiles = (long long)batch * channels * p.n_tiles_s;
        int grid = (int)(tiles < plan->dev.sm_count * 8LL ? tiles : plan->dev.sm_count * 8LL);
        kb_idft_kernel<<<grid, 256, smem, st>>>(p);
        KB_CUDA(cudaGetLastError());
        g_launches++;
        return 0;
    }

    const int Q = plan->Q, FPW = 32 / Q;
    const int R = (plan->win + plan->hop - 1) / plan->hop;
    if (kb_env_int("KAPRE_B200_ISTFT2", 1)) {
        KbIstftParams p{};
        int grid = 0;
        if ((rc = kb_istft2_cfg(plan->dev, Q, plan->n_fft, plan->hop, plan->win, batch, channels, frames, out_len, &p, &grid)) < 0)
            return rc;
        if (rc == 0) {
            p.X = (const float2*)stft_dev; p.x_sb = sd->stride_b; p.x_sc = sd->stride_c; p.x_st = sd->stride_t; p.x_sk = sd->stride_f;
            p.dual = plan->dual; p.twp = plan->twp; p.twn = plan->twn;
            p.y = y_dev; p.y_sb = yd->stride_b; p.y_sc = yd->stride_c; p.y_sl = yd->stride_l;
            return kb_launch_istft2_q<false>(Q, p, grid, st);
        }
    }
    // one FFT round per overlap class: TFc = R * NW * FPW frames per tile
    int NW = kb_env_int("KAPRE_B200_INW", KB_ISTFT_MAX_WARPS), TFc = 0, smem = 0, bps = 0;
    if (NW > KB_ISTFT_MAX_WARPS || NW < 1) NW = KB_ISTFT_MAX_WARPS;
    for (;; NW >>= 1) {
        if (NW < 1) return kb_fail(KAPRE_E_UNSUPPORTED, "inverse STFT tile does not fit shared memory (n_fft=%d hop=%d)", plan->n_fft, plan->hop);
        TFc = R * NW * FPW;
        if (TFc < R) TFc = R;
        const KbIstftSmem L = kb_istft_smem_layout(Q, plan->n_fft, plan->hop, plan->win, TFc, NW);
        smem = L.total;
        if (smem <= plan->dev.smem_optin) break;
    }
    bps = (228 * 1024) / (smem + 1024);
    if (bps > 3) bps = 3;              // __launch_bounds__(128, 3): 168 registers per thread
    if (bps < 1) bps = 1;
    KbIstftParams p{};
    p.X = (const float2*)stft_dev; p.x_sb = sd->stride_b; p.x_sc = sd->stride_c; p.x_st = sd->stride_t; p.x_sk = sd->stride_f;
    p.B = batch; p.C = channels; p.T = frames; p.n_fft = plan->n_fft; p.hop = plan->hop; p.win = plan->win;
    p.out_len = (int)out_len; p.dual = plan->dual; p.twp = plan->twp; p.twn = plan->twn;
    p.y = y_dev; p.y_sb = yd->stride_b; p.y_sc = yd->stride_c; p.y_sl = yd->stride_l;
    p.TFc = TFc; p.R = R; p.hops_out = TFc - (R - 1);
    p.n_tiles_t = kb_istft_tiles(frames, plan->hop, plan->win_length, p.hops_out);
    p.n_warps = NW;
    const long long tiles = (long long)batch * channels * p.n_tiles_t;
    if (tiles > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "too many tiles");
    const long long gmax = (long long)plan->dev.sm_count * bps;
    const int grid = (int)(tiles < gmax ? tiles : gmax);
    switch (Q) {
        case 4: rc = kb_launch_istft<4>(p, grid, smem, st); break;
        case 8: rc = kb_launch_istft<8>(p, grid, smem, st); break;
        case 16: rc = kb_launch_istft<16>(p, grid, smem, st); break;
        case 32: rc = kb_launch_istft<32>(p, grid, smem, st); break;
        default: rc = kb_fail(KAPRE_E_UNSUPPORTED, "bad Q");
    }
    return rc;
}

int kapre_filterbank_create(const float* fb_host, int n_freq, int n_bands, kapre_filterbank** out) {
    if (!out || !fb_host) return kb_fail(KAPRE_E_INVALID, "null argument");
    if (n_freq < 1 || n_bands < 1) return kb_fail(KAPRE_E_INVALID, "empty filterbank");
    kapre_filterbank* f = new kapre_filterbank();
    f->n_freq = n_freq; f->n_bands = n_bands;
    int rc = kb_dev_info(&f->dev);
    if (rc) { delete f; return rc; }
    std::vector<KbBand> bands; std::vector<float> w;
    kb_make_bands(fb_host, n_freq, n_bands, bands, w);
    f->n_w = (int)w.size();
    if ((rc = kb_upload(bands, &f->bands)) || (rc = kb_upload(w, &f->w))) { kapre_filterbank_destroy(f); return rc; }
    {   // transposed form for the spectral VJP (g_mag = g_fb fb^T)
        std::vector<float> fbT((size_t)n_freq * n_bands);
        for (int k = 0; k < n_freq; ++k)
            for (int m = 0; m < n_bands; ++m) fbT[(size_t)m * n_freq + k] = fb_host[(size_t)k * n_bands + m];
        std::vector<KbBand> bT; std::vector<float> wT;
        kb_make_bands(fbT.data(), n_bands, n_freq, bT, wT);
        if ((rc = kb_upload(bT, &f->bandsT)) || (rc = kb_upload(wT, &f->wT))) { kapre_filterbank_destroy(f); return rc; }
    }
    f->Q = kb_q_for_nfft((n_freq - 1) * 2);
    if (f->Q) {
        std::vector<kb_f4> cw; std::vector<kb_i2> cm; std::vector<int> cg;
        kb_make_fb_chunks(fb_host, n_freq, n_bands, 32, cw, cm, cg);
        f->n_chunks = (int)cw.size();
        if ((rc = kb_upload(cw, &f->cw)) || (rc = kb_upload(cm, &f->cm)) || (rc = kb_upload(cg, &f->cg))) {
            kapre_filterbank_destroy(f); return rc;
        }
        std::vector<kb_i2> bd; std::vector<int> bg;
        kb_make_fb_band_desc(cm, cg, 32, bd, bg);
        f->n_bd = (int)bd.size();
        if ((rc = kb_upload(bd, &f->bd)) || (rc = kb_upload(bg, &f->bg))) { kapre_filterbank_destroy(f); return rc; }
        std::vector<kb_f4> mw; std::vector<kb_i2> ms; std::vector<int> mg;
        kb_make_fb_mma(fb_host, n_freq, n_bands, mw, ms, mg);
        f->n_msteps = (int)ms.size();
        if ((rc = kb_upload(mw, &f->mw)) || (rc = kb_upload(ms, &f->ms)) || (rc = kb_upload(mg, &f->mg))) {
            kapre_filterbank_destroy(f); return rc;
        }
    }
    *out = f;
    return 0;
}

void kapre_filterbank_destroy(kapre_filterbank* f) {
    if (!f) return;
    cudaFree(f->bands); cudaFree(f->w); cudaFree(f->bandsT); cudaFree(f->wT); cudaFree(f->cw); cudaFree(f->cm); cudaFree(f->cg);
    cudaFree(f->mw); cudaFree(f->ms); cudaFree(f->mg); cudaFree(f->bd); cudaFree(f->bg);
    delete f;
}

int kapre_apply_filterbank(const kapre_filterbank* fb, const float* x_dev, int batch, int channels, int frames,
                           const kapre_spec_desc* xd, float* out_dev, const kapre_spec_desc* od, void* stream) {
    if (!fb || !xd || !od) return kb_fail(KAPRE_E_INVALID, "null argument");
    int rc = kb_check_device(fb->dev);
    if (rc) return rc;
    if (batch < 0 || channels < 0 || frames < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    if (batch == 0 || channels == 0 || frames == 0) return 0;
    if (!x_dev || !out_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    KbFbParams p{};
    p.x = x_dev; p.x_sb = xd->stride_b; p.x_sc = xd->stride_c; p.x_st = xd->stride_t; p.x_sk = xd->stride_f;
    p.B = batch; p.C = channels; p.T = frames; p.F = fb->n_freq;
    p.bands = fb->bands; p.fbw = fb->w; p.n_bands = fb->n_bands;
    p.out = out_dev; p.o_sb = od->stride_b; p.o_sc = od->stride_c; p.o_st = od->stride_t; p.o_sk = od->stride_f;
    p.R = kb_fb_pick_r(fb->n_freq, fb->n_bands, fb->dev.smem_optin);
    if (p.R == 0)
        return kb_fail(KAPRE_E_UNSUPPORTED, "filterbank %dx%d does not fit shared memory", fb->n_freq, fb->n_bands);
    p.n_tiles_t = (frames + p.R - 1) / p.R; p.n_warps = 8;
    const KbFbSmem L = kb_fb_smem_layout(fb->n_freq, fb->n_bands, p.R);
    if ((rc = kb_set_smem(kb_fb_kernel, L.total))) return rc;
    int bps = (228 * 1024) / (L.total + 1024);
    if (bps > 8) bps = 8;
    if (bps < 1) bps = 1;
    const long long tiles = (long long)batch * channels * p.n_tiles_t;
    const long long gmax = (long long)fb->dev.sm_count * bps;
    const int grid = (int)(tiles < gmax ? tiles : gmax);
    kb_fb_kernel<<<grid, 256, L.total, (cudaStream_t)stream>>>(p);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

static int kb_ew_grid(int64_t n, int* grid) {
    int dev = 0, sms = 0;
    KB_CUDA(cudaGetDevice(&dev));
    KB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    long long g = (n + 255) / 256;
    const long long cap = (long long)sms * 16;
    *grid = (int)(g < cap ? g : cap);
    if (*grid < 1) *grid = 1;
    return 0;
}

int kapre_magnitude(const void* x_complex_dev, float* out_dev, int64_t n, void* stream) {
    if (n < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    if (n == 0) return 0;
    if (!x_complex_dev || !out_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    int grid, rc;
    if ((rc = kb_ew_grid(n, &grid))) return rc;
    kb_magnitude_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float2*)x_complex_dev, out_dev, n);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

int kapre_phase(const void* x_complex_dev, float* out_dev, int64_t n, void* stream) {
    if (n < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    if (n == 0) return 0;
    if (!x_complex_dev || !out_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    int grid, rc;
    if ((rc = kb_ew_grid(n, &grid))) return rc;
    kb_phase_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const float2*)x_complex_dev, out_dev, n);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

int kapre_concat_frequency_map(const float* x_dev, float* out_dev, int64_t batch, int64_t channels, int64_t frames,
                               int64_t n_freq, int channels_last, void* stream) {
    if (batch < 0 || channels < 0 || frames < 0 || n_freq < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    const long long total = (long long)batch * (channels + 1) * frames * n_freq;
    if (total == 0) return 0;
    if (!out_dev || (!x_dev && channels > 0)) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    int grid, rc;
    if ((rc = kb_ew_grid(total, &grid))) return rc;
    kb_concat_freq_map_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x_dev, out_dev, batch, channels, frames, n_freq, channels_last ? 1 : 0);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

int kapre_spec_augment(const float* x_dev, float* out_dev, int64_t batch, int64_t frames, int64_t n_freq,
                       const int* time_masks_dev, int n_time_masks, const int* freq_masks_dev, int n_freq_masks,
                       float mask_value, void* stream) {
    if (batch < 0 || frames < 0 || n_freq < 0 || n_time_masks < 0 || n_freq_masks < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    const long long total = (long long)batch * frames * n_freq;
    if (total == 0) return 0;
    if (!x_dev || !out_dev || (n_time_masks && !time_masks_dev) || (n_freq_masks && !freq_masks_dev))
        return kb_fail(KAPRE_E_INVALID, "null data pointer");
    int grid, rc;
    if ((rc = kb_ew_grid(total, &grid))) return rc;
    kb_spec_augment_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x_dev, out_dev, batch, frames, n_freq, time_masks_dev,
                                                                 n_time_masks, freq_masks_dev, n_freq_masks, mask_value);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

static int kb_frames_for(int L, int fl, int hop, int pad_end) {
    if (pad_end) return (L + hop - 1) / hop;
    return L < fl ? 0 : 1 + (L - fl) / hop;
}

int kapre_delta(const float* x_dev, float* out_dev, int64_t outer, int64_t frames, int64_t inner, int win_length,
                int pad_mode, void* stream) {
    if (win_length < 3 || (win_length & 1) == 0) return kb_fail(KAPRE_E_INVALID, "win_length must be odd and >= 3, got %d", win_length);
    if (pad_mode < 0 || pad_mode > 2) return kb_fail(KAPRE_E_INVALID, "bad pad_mode %d", pad_mode);
    if (outer < 0 || frames < 0 || inner < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    const long long total = (long long)outer * frames * inner;
    if (total == 0) return 0;
    if (!x_dev || !out_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    if (x_dev == out_dev) return kb_fail(KAPRE_E_INVALID, "delta cannot run in place");
    const int n = (win_length - 1) / 2;
    double denom = 0;
    for (int m = 1; m <= n; ++m) denom += 2.0 * m * m;
    int grid, rc;
    if ((rc = kb_ew_grid(total, &grid))) return rc;
    kb_delta_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x_dev, out_dev, outer, frames, inner, n, (float)(1.0 / denom), pad_mode);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

int kapre_frame(const float* x_dev, const kapre_wave_desc* xd, int frame_length, int hop_length, int pad_end, float pad_value,
                float* out_dev, const kapre_spec_desc* od, void* stream) {
    if (!xd || !od) return kb_fail(KAPRE_E_INVALID, "null argument");
    if (frame_length <= 0 || hop_length <= 0) return kb_fail(KAPRE_E_INVALID, "frame_length and hop_length must be positive");
    const int T = kb_frames_for(xd->length, frame_length, hop_length, pad_end);
    const long long total = (long long)xd->batch * xd->channels * T * frame_length;
    if (total <= 0) return 0;
    if (!x_dev || !out_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    int grid, rc;
    if ((rc = kb_ew_grid(total, &grid))) return rc;
    kb_frame_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x_dev, xd->stride_b, xd->stride_c, xd->stride_l, xd->batch,
                                                          xd->channels, xd->length, frame_length, hop_length, T, pad_value,
                                                          out_dev, od->stride_b, od->stride_c, od->stride_t, od->stride_f);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

int kapre_energy(const float* x_dev, const kapre_wave_desc* xd, int frame_length, int hop_length, int pad_end, float pad_value,
                 float scale, float* out_dev, const kapre_wave_desc* od, void* stream) {
    if (!xd || !od) return kb_fail(KAPRE_E_INVALID, "null argument");
    if (frame_length <= 0 || hop_length <= 0) return kb_fail(KAPRE_E_INVALID, "frame_length and hop_length must be positive");
    const int T = kb_frames_for(xd->length, frame_length, hop_length, pad_end);
    const long long n_frames = (long long)xd->batch * xd->channels * T;
    if (n_frames <= 0) return 0;
    if (!x_dev || !out_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    if (od->length != T) return kb_fail(KAPRE_E_INVALID, "output must have %d frames, got %d", T, od->length);
    int grid, rc;
    if ((rc = kb_ew_grid(n_frames * 32, &grid))) return rc;
    kb_energy_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x_dev, xd->stride_b, xd->stride_c, xd->stride_l, xd->batch,
                                                           xd->channels, xd->length, frame_length, hop_length, T, pad_value,
                                                           scale, out_dev, od->stride_b, od->stride_c, od->stride_l);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

int kapre_magnitude_to_decibel(const float* x_dev, float* out_dev, int64_t n_items, int64_t item_size,
                               const kapre_db_cfg* db, void* workspace_dev, void* stream) {
    int rc = kb_check_db(db);
    if (rc) return rc;
    if (n_items < 0 || item_size < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    if (n_items == 0 || item_size == 0) return 0;
    if (!x_dev || !out_dev || !workspace_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    cudaStream_t st = (cudaStream_t)stream;
    float db_mul, db_sub;
    kb_db_consts(db, &db_mul, &db_sub);
    long long chunks = (item_size + 256 * 8 - 1) / (256 * 8);
    if (chunks > 64) chunks = 64;
    if (chunks < 1) chunks = 1;
    const long long grid = n_items * chunks;
    if (grid > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "too many items");
    kb_db_kernel<<<(unsigned)grid, 256, 0, st>>>(x_dev, out_dev, item_size, (int)chunks, (unsigned int*)workspace_dev,
                                                 db->amin, db_mul, db_sub);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return kb_launch_clamp(out_dev, n_items, item_size, (unsigned int*)workspace_dev, db->amin, db_mul, db_sub,
                           db->dynamic_range, st);
}

// Experimental: the next tensor-core log-mel launch also dumps its complex spectrum (signals, T, 513) float2 to dbg_dev.
int kapre_tc_set_debug(void* dbg_dev) { g_tc_dbg = (float2*)dbg_dev; return 0; }

// ---- experimental: tensor-core (tcgen05) DFT stage, see tc_dft.cuh -----------------------------------
// Stage 1 of the 32 x 32 factorisation of the n_fft = 1024 / hop = 256 real FFT over `n_items` waveforms of
// `length` samples (`item_stride` floats apart).  store != 0: out = (items, T, 32, 32) floats with
// out[i, f, n2, 2 k1 + {0,1}] = Re / Im of sum_n1 x[256 f + 32 n1 + n2] exp(-2 pi i n1 k1 / 32), k1 = 0..15, except
// column 1 (Im of k1 = 0, identically zero), which carries the real k1 = 16 sum.  store == 0 (timing): out must
// hold grid * 256 floats of checksums; *grid_out receives the grid size.  T = 1 + (length - 1024) / 256.
int kapre_tc_dft_stage1(const float* x_dev, int n_items, long long item_stride, int length, float* out_dev, int store,
                        int* grid_out, const float* fmat_override_dev, void* stream) {
    if (!x_dev || !out_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    if (n_items < 1 || length < KB_TC_NFFT) return kb_fail(KAPRE_E_INVALID, "need n_items >= 1 and length >= 1024");
    DevInfo dev;
    int rc = kb_dev_info(&dev);
    if (rc) return rc;
    static float* d_fmat[64] = {nullptr};
    if (dev.device < 0 || dev.device >= 64) return kb_fail(KAPRE_E_UNSUPPORTED, "device index");
    if (!d_fmat[dev.device]) {
        std::vector<float> f(2048);
        for (int kc = 0; kc < 8; ++kc)
            for (int c = 0; c < 32; ++c)
                for (int e = 0; e < 4; ++e) {
                    const int n1 = 4 * kc + e, k1 = c >> 1;
                    double v;
                    if (c == 1) v = (n1 & 1) ? -1.0 : 1.0;                       // k1 = 16: (-1)^n1
                    else {
                        const double a = -2.0 * M_PI * (double)((n1 * k1) % 32) / 32.0;
                        v = (c & 1) ? sin(a) : cos(a);
                    }
                    const float w = (float)v, hi = kb_tf32_hi(w);
                    f[(size_t)(kc * 32 + c) * 4 + e] = hi;
                    f[1024 + (size_t)(kc * 32 + c) * 4 + e] = w - hi;
                }
        if ((rc = kb_upload(f, &d_fmat[dev.device]))) return rc;
    }
    KbTcParams p{};
    p.x = x_dev; p.item_stride = item_stride; p.n_items = n_items; p.length = length;
    p.T = 1 + (length - KB_TC_NFFT) / KB_TC_HOP;
    p.out = out_dev; p.store = store;
    p.fmat = fmat_override_dev ? fmat_override_dev : d_fmat[dev.device];   // override: layout debugging (2048 floats)
    p.n_tiles_t = (p.T + KB_TC_TILE_F - 1) / KB_TC_TILE_F;
    const long long tiles = (long long)n_items * p.n_tiles_t;
    const long long gmax = (long long)dev.sm_count * 2;
    const int grid = (int)(tiles < gmax ? tiles : gmax);
    if (grid_out) *grid_out = grid;
    if ((rc = kb_set_smem(kb_tc_dft_stage1_kernel, KB_TC_SMEM))) return rc;
    KbProfScope prof((cudaStream_t)stream);
    kb_tc_dft_stage1_kernel<<<grid, KB_TC_THREADS, KB_TC_SMEM, (cudaStream_t)stream>>>(p);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

// ---- backward (vector-Jacobian products), grad_core.cuh -----------------------------------------------------------
// Workspace of the decibel statistics: [arrival counters, n_items words | pad to 16 B][stats, 16 B per item]
// [partials, KB_DBS_MAX_CHUNKS * 16 B per item]
static void kb_dbs_ws(void* ws, long long n_items, unsigned int** arrive, KbDbStats** stats, KbDbStats** part) {
    char* base = (char*)ws;
    const long long a = (n_items * 4 + 15) & ~15LL;
    *arrive = (unsigned int*)base;
    *stats = (KbDbStats*)(base + a);
    *part = (KbDbStats*)(base + a + n_items * (long long)sizeof(KbDbStats));
}

// Statistics pass over a (n_items, d1, d2, d3) view of y and g; leaves the combined KbDbStats per item in the workspace.
static int kb_launch_dbstat(KbDbStatParams& q, void* ws, float dyn_range, cudaStream_t st, KbDbStats** stats_out) {
    const long long item = (long long)q.d1 * q.d2 * q.d3;
    long long chunks = (item + 32767) / 32768;
    if (chunks > KB_DBS_MAX_CHUNKS) chunks = KB_DBS_MAX_CHUNKS;
    if (chunks < 1) chunks = 1;
    if ((long long)q.n_items * chunks > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "too many items");
    q.chunks = (int)chunks;
    q.dyn_range = dyn_range;
    KbDbStats* part;
    kb_dbs_ws(ws, q.n_items, &q.arrive, &q.stats, &part);
    q.part = part;
    kb_dbstat_kernel<<<(unsigned)(q.n_items * chunks), KB_DBS_THREADS, 0, st>>>(q);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    *stats_out = q.stats;
    return 0;
}

int kapre_stft_backward(const kapre_stft_plan* plan, const void* grad_spec_dev, int batch, int channels, int frames,
                        const kapre_spec_desc* gsd, int pad_begin, int pad_end, float* grad_x_dev,
                        const kapre_wave_desc* gxd, void* stream) {
    if (!plan || !gsd || !gxd) return kb_fail(KAPRE_E_INVALID, "null argument");
    int rc = kb_check_device(plan->dev);
    if (rc) return rc;
    if (batch < 0 || channels < 0 || frames < 0 || gxd->length < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    if (gxd->batch != batch || gxd->channels != channels)
        return kb_fail(KAPRE_E_INVALID, "gradient is (%d, %d) signals, the spectrum (%d, %d)", gxd->batch, gxd->channels, batch, channels);
    if (pad_begin && plan->hop > plan->n_fft)
        return kb_fail(KAPRE_E_INVALID, "pad_begin needs hop_length <= n_fft (the padding is n_fft - hop_length = %d)",
                       plan->n_fft - plan->hop);
    const int L = gxd->length;
    const int T = kapre_stft_num_frames(plan, L, pad_begin, pad_end);
    if (T != frames) return kb_fail(KAPRE_E_INVALID, "%d samples give %d frames, the spectrum has %d", L, T, frames);
    if (batch == 0 || channels == 0 || L == 0) return 0;
    if (!grad_x_dev || (frames > 0 && !grad_spec_dev)) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    const int pad_left = pad_begin ? (plan->n_fft - plan->hop) : 0;
    const long long out_len = (long long)pad_left + L;      // padded coordinates; [0, pad_left) is dropped
    if (out_len + plan->n_fft > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "signal too long");
    cudaStream_t st = (cudaStream_t)stream;
    if (plan->Q && frames > 0 && kb_env_int("KAPRE_B200_ISTFT2", 1)) {
        KbIstftParams p{};
        int grid = 0;
        if ((rc = kb_istft2_cfg(plan->dev, plan->Q, plan->n_fft, plan->hop, plan->win_eff, batch, channels, frames, out_len,
                                &p, &grid)) < 0)
            return rc;
        if (rc == 0) {
            p.X = (const float2*)grad_spec_dev; p.x_sb = gsd->stride_b; p.x_sc = gsd->stride_c; p.x_st = gsd->stride_t;
            p.x_sk = gsd->stride_f;
            p.dual = plan->adj; p.twp = plan->twp; p.twn = plan->twn;
            p.y = grad_x_dev; p.y_sb = gxd->stride_b; p.y_sc = gxd->stride_c; p.y_sl = gxd->stride_l;
            p.y_off = pad_left; p.edge2 = 1;
            return kb_launch_istft2_q<true>(plan->Q, p, grid, st);
        }
    }
    // direct body: every n_fft, O(n_fft) work per output sample and frame (also zero-fills when there are no frames)
    KbIdftParams p{};
    p.X = (const float2*)grad_spec_dev; p.x_sb = gsd->stride_b; p.x_sc = gsd->stride_c; p.x_st = gsd->stride_t; p.x_sk = gsd->stride_f;
    p.B = batch; p.C = channels; p.T = frames; p.n_fft = plan->n_fft; p.hop = plan->hop; p.win = plan->win_eff;
    p.out_len = (int)out_len; p.dualn = plan->adj_dn; p.tw = plan->adj_tw;
    p.y = grad_x_dev; p.y_sb = gxd->stride_b; p.y_sc = gxd->stride_c; p.y_sl = gxd->stride_l;
    p.y_off = pad_left; p.edge2 = 1;
    p.n_warps = 8; p.n_tiles_s = (int)((out_len + 255) / 256);
    const int smem = plan->n_fft * 8;
    if (smem > plan->dev.smem_optin) return kb_fail(KAPRE_E_UNSUPPORTED, "n_fft too large");
    if ((rc = kb_set_smem(kb_idft_kernel, smem))) return rc;
    const long long tiles = (long long)batch * channels * p.n_tiles_s;
    if (tiles > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "too many tiles");
    const int grid = (int)(tiles < plan->dev.sm_count * 8LL ? tiles : plan->dev.sm_count * 8LL);
    kb_idft_kernel<<<grid, 256, smem, st>>>(p);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

int kapre_istft_backward(const kapre_istft_plan* plan, const float* grad_y_dev, const kapre_wave_desc* gyd,
                         void* grad_spec_dev, int frames, const kapre_spec_desc* gsd, void* stream) {
    if (!plan || !gyd || !gsd) return kb_fail(KAPRE_E_INVALID, "null argument");
    int rc = kb_check_device(plan->dev);
    if (rc) return rc;
    if (gyd->batch < 0 || gyd->channels < 0 || frames < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    if (gyd->batch == 0 || gyd->channels == 0 || frames == 0) return 0;
    const long long out_len = (long long)(frames - 1) * plan->hop + plan->win_length;
    if (gyd->length != out_len)
        return kb_fail(KAPRE_E_INVALID, "gradient length must be (frames-1)*hop+win_length = %lld, got %d", out_len, gyd->length);
    if (!grad_y_dev || !grad_spec_dev) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    if ((rc = kapre_stft_forward(plan->grad, grad_y_dev, gyd, 0, 0, KAPRE_OUT_COMPLEX, grad_spec_dev, gsd, nullptr, nullptr,
                                 nullptr, stream)))
        return rc;
    const long long n_frames = (long long)gyd->batch * gyd->channels * frames;
    int grid = 0;
    if ((rc = kb_ew_grid(n_frames, &grid))) return rc;
    kb_istft_grad_edges_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((float2*)grad_spec_dev, gsd->stride_b, gsd->stride_c,
                                                                       gsd->stride_t, gsd->stride_f, gyd->channels, frames,
                                                                       n_frames, plan->n_fft / 2, (plan->n_fft & 1) == 0);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

int kapre_spectral_backward(const kapre_filterbank* fb, int mode, const void* x_dev, int batch, int channels, int frames,
                            int n_freq, const kapre_spec_desc* xd, const float* grad_dev, const kapre_spec_desc* gd,
                            const float* y_dev, const kapre_spec_desc* yd, const kapre_db_cfg* db, void* workspace_dev,
                            void* grad_x_dev, const kapre_spec_desc* gxd, void* stream) {
    if (!xd || !gd || !gxd) return kb_fail(KAPRE_E_INVALID, "null argument");
    if (mode != KAPRE_OUT_MAG && mode != KAPRE_OUT_MAG_DB && mode != KAPRE_OUT_FB && mode != KAPRE_OUT_FB_DB)
        return kb_fail(KAPRE_E_INVALID, "bad mode %d for the spectral VJP", mode);
    if (batch < 0 || channels < 0 || frames < 0 || n_freq < 1) return kb_fail(KAPRE_E_INVALID, "bad size");
    const bool fbm = mode == KAPRE_OUT_FB || mode == KAPRE_OUT_FB_DB;
    const bool dbm = mode == KAPRE_OUT_MAG_DB || mode == KAPRE_OUT_FB_DB;
    int rc = 0;
    if (fbm) {
        if (!fb) return kb_fail(KAPRE_E_INVALID, "filterbank required for mode %d", mode);
        if (fb->n_freq != n_freq) return kb_fail(KAPRE_E_INVALID, "filterbank has %d rows, the spectrum %d bins", fb->n_freq, n_freq);
        if ((rc = kb_check_device(fb->dev))) return rc;
    }
    if (dbm) {
        if ((rc = kb_check_db(db))) return rc;
        if (!yd) return kb_fail(KAPRE_E_INVALID, "forward output required for decibel modes");
        if (!workspace_dev) return kb_fail(KAPRE_E_INVALID, "workspace required for decibel modes");
    }
    if (batch == 0 || channels == 0 || frames == 0) return 0;
    if (!x_dev || !grad_dev || !grad_x_dev || (dbm && !y_dev)) return kb_fail(KAPRE_E_INVALID, "null data pointer");
    const int K = fbm ? fb->n_bands : n_freq;
    cudaStream_t st = (cudaStream_t)stream;
    DevInfo dev;
    if ((rc = kb_dev_info(&dev))) return rc;
    KbSpecVjpParams p{};
    if (dbm) {
        KbDbStatParams q{};
        q.y = y_dev; q.y_s0 = yd->stride_b; q.y_s1 = yd->stride_c; q.y_s2 = yd->stride_t; q.y_s3 = yd->stride_f;
        q.g = grad_dev; q.g_s0 = gd->stride_b; q.g_s1 = gd->stride_c; q.g_s2 = gd->stride_t; q.g_s3 = gd->stride_f;
        q.n_items = batch; q.d1 = channels; q.d2 = frames; q.d3 = K;
        KbDbStats* stats = nullptr;
        if ((rc = kb_launch_dbstat(q, workspace_dev, db->dynamic_range, st, &stats))) return rc;
        p.stats = stats;
        p.amin = db->amin;
        p.y = y_dev; p.y_sb = yd->stride_b; p.y_sc = yd->stride_c; p.y_st = yd->stride_t; p.y_sk = yd->stride_f;
    }
    p.X = (const float2*)x_dev; p.x_sb = xd->stride_b; p.x_sc = xd->stride_c; p.x_st = xd->stride_t; p.x_sk = xd->stride_f;
    p.G = (float2*)grad_x_dev; p.G_sb = gxd->stride_b; p.G_sc = gxd->stride_c; p.G_st = gxd->stride_t; p.G_sk = gxd->stride_f;
    p.g = grad_dev; p.g_sb = gd->stride_b; p.g_sc = gd->stride_c; p.g_st = gd->stride_t; p.g_sk = gd->stride_f;
    p.B = batch; p.C = channels; p.T = frames; p.F = n_freq; p.K = K;
    p.fb = fbm; p.db = dbm;
    if (fbm) { p.bands = fb->bands; p.fbw = fb->w; p.bandsT = fb->bandsT; p.fbwT = fb->wT; }
    p.n_warps = 4;
    const int smem = kb_specvjp_smem_layout(n_freq, K).total;
    if (smem > dev.smem_optin) return kb_fail(KAPRE_E_UNSUPPORTED, "spectrum of %d bins does not fit shared memory", n_freq);
    if ((rc = kb_set_smem(kb_specvjp_kernel, smem))) return rc;
    int bps = (228 * 1024) / (smem + 1024);
    if (bps > 16) bps = 16;
    if (bps < 1) bps = 1;
    const long long n_frames = (long long)batch * channels * frames;
    const long long gmax = (long long)dev.sm_count * bps;
    const int grid = (int)(n_frames < gmax ? n_frames : gmax);
    kb_specvjp_kernel<<<grid, p.n_warps * 32, smem, st>>>(p);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

int kapre_magnitude_to_decibel_backward(const float* x_dev, const float* y_dev, const float* grad_dev,
                                        int64_t grad_item_stride, int64_t grad_elem_stride, float* grad_x_dev,
                                        int64_t n_items, int64_t item_size, const kapre_db_cfg* db, void* workspace_dev,
                                        void* stream) {
    int rc = kb_check_db(db);
    if (rc) return rc;
    if (n_items < 0 || item_size < 0) return kb_fail(KAPRE_E_INVALID, "negative size");
    if (n_items == 0 || item_size == 0) return 0;
    if (!x_dev || !y_dev || !grad_dev || !grad_x_dev || !workspace_dev) return kb_fail(KAPRE_E_INVALID, "null pointer");
    if (n_items > 0x7fffffffLL || item_size > 0x7fffffffLL) return kb_fail(KAPRE_E_UNSUPPORTED, "tensor too large");
    cudaStream_t st = (cudaStream_t)stream;
    KbDbStatParams q{};
    q.y = y_dev; q.y_s0 = item_size; q.y_s1 = 0; q.y_s2 = 0; q.y_s3 = 1;
    q.g = grad_dev; q.g_s0 = grad_item_stride; q.g_s1 = 0; q.g_s2 = 0; q.g_s3 = grad_elem_stride;
    q.n_items = (int)n_items; q.d1 = 1; q.d2 = 1; q.d3 = (int)item_size;
    KbDbStats* stats = nullptr;
    if ((rc = kb_launch_dbstat(q, workspace_dev, db->dynamic_range, st, &stats))) return rc;
    const long long n = n_items * item_size;
    int grid = 0;
    if ((rc = kb_ew_grid(n, &grid))) return rc;
    kb_db_backward_kernel<<<grid, 256, 0, st>>>(x_dev, y_dev, grad_dev, grad_item_stride, grad_elem_stride, grad_x_dev,
                                                item_size, n, stats, db->amin);
    KB_CUDA(cudaGetLastError());
    g_launches++;
    return 0;
}

}  // extern "C"

