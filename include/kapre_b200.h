/*
 * kapre_b200 -- C ABI of the B200-native STFT -> |.| -> filterbank -> dB hot path (+ inverse STFT).
 *
 * This is the drop-in boundary of the repo: everything the reference computes inside
 * TensorFlow for the five hot-path layers is reachable through these entry points, with
 * plain pointers and sizes only (no torch / CUDA types in the signatures).  The Python
 * layer classes in kapre_b200/ (mirrors of kapre.STFT / InverseSTFT / Magnitude /
 * ApplyFilterbank / MagnitudeToDecibel) bind them with ctypes; INTEGRATION.md shows the
 * stub a kapre maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative KAPRE_E_* code; the message is
 *     available from kapre_last_error() (thread-local).  Nothing throws across the ABI.
 *   - `*_dev` pointers are device pointers on the CUDA device that was current when the plan
 *     was created; the caller owns every data buffer.  The library allocates only the small
 *     constant tables held by plans (window, twiddles, banded filterbank).
 *   - every call only enqueues work on `stream` (a cudaStream_t passed as void*; NULL = the
 *     legacy default stream) and returns; nothing synchronises.
 *   - tensors are described by element strides, so both of kapre's data formats
 *     ('channels_first' (B,C,T,F) / 'channels_last' (B,T,F,C); waveforms (B,C,L) / (B,L,C))
 *     are served without transposes (replaces kapre/time_frequency.py:164-167,184-185,
 *     304-305,316-317,546-547).
 */
#ifndef KAPRE_B200_H_
#define KAPRE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KAPRE_B200_VERSION 200

enum {
    KAPRE_OK = 0,
    KAPRE_E_INVALID = -1,      /* bad argument */
    KAPRE_E_UNSUPPORTED = -2,  /* valid in the reference but not implemented here */
    KAPRE_E_CUDA = -3,         /* CUDA runtime error (see kapre_last_error) */
    KAPRE_E_NOMEM = -4
};

/* What kapre_stft_forward writes.  One launch replaces the layer chain named on the right. */
enum {
    KAPRE_OUT_COMPLEX = 0, /* complex64   kapre.STFT                         time_frequency.py:146-187 */
    KAPRE_OUT_MAG = 1,     /* float32     STFT -> Magnitude                  time_frequency.py:351-359 */
    KAPRE_OUT_MAG_DB = 2,  /* float32     STFT -> Magnitude -> MagnitudeToDecibel      composed.py:32-135 */
    KAPRE_OUT_FB = 3,      /* float32     STFT -> Magnitude -> ApplyFilterbank         composed.py:138-261 */
    KAPRE_OUT_FB_DB = 4,   /* float32     ... -> ApplyFilterbank -> MagnitudeToDecibel composed.py:254-261 */
    KAPRE_OUT_MAG_PHASE = 5 /* float32    get_stft_mag_phase (composed.py:420-511): the output tensor has 2*channels
                             *             channels, magnitudes (dB-scaled if `db` is given) in channels [0, C) and
                             *             tf.math.angle phases in channels [C, 2C) */
};

/* Waveform tensor: element strides of (batch, channel, sample). */
typedef struct {
    int32_t batch, channels, length;
    int64_t stride_b, stride_c, stride_l;
} kapre_wave_desc;

/* Spectrogram tensor: element strides of (batch, channel, frame, bin).  Elements are
 * float32, or complex64 (one element = 8 bytes) for complex STFTs. */
typedef struct {
    int64_t stride_b, stride_c, stride_t, stride_f;
} kapre_spec_desc;

/* kapre.MagnitudeToDecibel(ref_value, amin, dynamic_range), kapre/backend.py:126-194. */
typedef struct {
    float ref_value, amin, dynamic_range;
} kapre_db_cfg;

typedef struct kapre_stft_plan kapre_stft_plan;
typedef struct kapre_istft_plan kapre_istft_plan;
typedef struct kapre_filterbank kapre_filterbank;

/* ---- forward STFT (kapre.STFT.__init__/call, kapre/time_frequency.py:101-187) -------------
 * `window_host`: win_length analysis-window samples (host memory), i.e. what
 * backend.get_window_fn(window_name)(win_length) returns (kapre/backend.py:58-100).
 * n_fft in {256,512,1024,2048} runs the fused FFT kernel; any other n_fft >= 2 runs the
 * direct-DFT kernel (same results, slower). */
int kapre_stft_plan_create(int n_fft, int win_length, int hop_length, const float* window_host,
                           kapre_stft_plan** out);
void kapre_stft_plan_destroy(kapre_stft_plan* plan);

/* Frames produced for `length` samples: tf.signal.frame semantics after kapre's pad_begin
 * (n_fft - hop zeros in front, kapre/time_frequency.py:169-172). */
int kapre_stft_num_frames(const kapre_stft_plan* plan, int length, int pad_begin, int pad_end);

/* 1 if kapre_stft_forward can produce `mode` in one fused launch for this plan. */
int kapre_stft_supports_mode(const kapre_stft_plan* plan, int mode);

/* Enqueue the transform.  `fb` is required for KAPRE_OUT_FB / _FB_DB, `db` for *_DB.
 * `workspace_dev`: at least 8 * batch bytes, needed for *_DB (per-item maxima for the
 * dynamic-range clamp of kapre/backend.py:190-192 + per-item arrival counters of the clamp pass, which
 * runs several CTAs per long item); may be NULL otherwise.  The workspace is
 * SELF-CLEANING: it must be all-zero when first passed in (cudaMemset once after allocation)
 * and every call leaves it all-zero again, so it can be reused by later calls on the same
 * stream without further memsets. */
int kapre_stft_forward(const kapre_stft_plan* plan, const float* x_dev, const kapre_wave_desc* x_desc,
                       int pad_begin, int pad_end, int mode, void* out_dev,
                       const kapre_spec_desc* out_desc, const kapre_filterbank* fb,
                       const kapre_db_cfg* db, void* workspace_dev, void* stream);

/* ---- inverse STFT (kapre.InverseSTFT, kapre/time_frequency.py:246-319) ---------------------
 * `dual_window_host`: win_length samples of tf.signal.inverse_stft_window_fn(hop, forward
 * window) (kapre/time_frequency.py:278-280).  Output length is (frames-1)*hop + win_length. */
int kapre_istft_plan_create(int n_fft, int win_length, int hop_length, const float* dual_window_host,
                            kapre_istft_plan** out);
void kapre_istft_plan_destroy(kapre_istft_plan* plan);
int kapre_istft_inverse(const kapre_istft_plan* plan, const void* stft_dev, int batch, int channels,
                        int frames, const kapre_spec_desc* stft_desc, float* y_dev,
                        const kapre_wave_desc* y_desc, void* stream);

/* ---- filterbank (kapre.ApplyFilterbank, kapre/time_frequency.py:501-548) --------------------
 * `fb_host`: row-major (n_freq, n_bands) float32 matrix, e.g. backend.filterbank_mel(...)
 * (kapre/backend.py:197-231) or backend.filterbank_log(...) (kapre/backend.py:234-299). */
int kapre_filterbank_create(const float* fb_host, int n_freq, int n_bands, kapre_filterbank** out);
void kapre_filterbank_destroy(kapre_filterbank* fb);
int kapre_apply_filterbank(const kapre_filterbank* fb, const float* x_dev, int batch, int channels,
                           int frames, const kapre_spec_desc* x_desc, float* out_dev,
                           const kapre_spec_desc* out_desc, void* stream);

/* ---- element-wise layers ------------------------------------------------------------------- */
/* kapre.Magnitude (tf.abs of complex64), kapre/time_frequency.py:351-359; n complex elements. */
int kapre_magnitude(const void* x_complex_dev, float* out_dev, int64_t n, void* stream);
/* kapre.Phase (tf.math.angle), kapre/time_frequency.py:391-402; n complex elements. */
int kapre_phase(const void* x_complex_dev, float* out_dev, int64_t n, void* stream);
/* backend.magnitude_to_decibel on a contiguous (n_items, item_size) tensor: the maximum for the
 * dynamic-range clamp is taken per item (kapre/backend.py:178-192); pass n_items = 1 for a
 * 1-D input (global maximum).  workspace_dev: >= 8 * n_items bytes, zero on entry, left zero
 * (self-cleaning, see kapre_stft_forward).  In-place is allowed. */
int kapre_magnitude_to_decibel(const float* x_dev, float* out_dev, int64_t n_items, int64_t item_size,
                               const kapre_db_cfg* db, void* workspace_dev, void* stream);

/* kapre.ConcatenateFrequencyMap (kapre/time_frequency.py:648-744): contiguous (b, t, f, ch) [channels_last != 0] or
 * (b, ch, t, f) float32 input -> the same with one more channel holding linspace(0, 1, n_freq) along the frequency axis. */
int kapre_concat_frequency_map(const float* x_dev, float* out_dev, int64_t batch, int64_t channels, int64_t frames,
                               int64_t n_freq, int channels_last, void* stream);

/* kapre.SpecAugment (kapre/augmentation.py:116-326) on a contiguous (batch, frames, n_freq) float32 tensor (depth 1: both data
 * formats have this memory layout).  `time_masks_dev` / `freq_masks_dev`: (batch, n_masks, 2) int32 (start, width) pairs; an element
 * whose time (frequency) index lies in [start, start + width] of any mask of its item becomes mask_value.  The pairs are drawn by the
 * caller (width ~ U{0..param-1}, start ~ U{0..limit-width-1}, as the reference does per item and mask). */
int kapre_spec_augment(const float* x_dev, float* out_dev, int64_t batch, int64_t frames, int64_t n_freq,
                       const int* time_masks_dev, int n_time_masks, const int* freq_masks_dev, int n_freq_masks,
                       float mask_value, void* stream);

/* ---- adjacent layers (SURVEY 8f "next" rows) ------------------------------------------------ */
/* kapre.Delta (kapre/time_frequency.py:563-644): y[t] = sum_{m=-n..n} m * x[t+m] / (2 sum m^2) along the
 * time axis of a contiguous tensor viewed as (outer, frames, inner); x is extended beyond its ends by
 * `pad_mode` (0 = symmetric, 1 = reflect, 2 = constant zero -- tf.pad's modes).  win_length = 2n+1. */
int kapre_delta(const float* x_dev, float* out_dev, int64_t outer, int64_t frames, int64_t inner,
                int win_length, int pad_mode, void* stream);
/* kapre.Frame (kapre/signal.py:22-119, tf.signal.frame): out[b, c, t, n] = x[b, c, t*hop + n], or
 * pad_value beyond the signal when pad_end.  out_desc strides are (batch, channel, frame, sample-in-frame). */
int kapre_frame(const float* x_dev, const kapre_wave_desc* x_desc, int frame_length, int hop_length, int pad_end,
                float pad_value, float* out_dev, const kapre_spec_desc* out_desc, void* stream);
/* kapre.Energy (kapre/signal.py:123-233): scale * sum_n frame[n]^2 per frame; out_desc.length = frames. */
int kapre_energy(const float* x_dev, const kapre_wave_desc* x_desc, int frame_length, int hop_length, int pad_end,
                 float pad_value, float scale, float* out_dev, const kapre_wave_desc* out_desc, void* stream);

/* ---- backward: vector-Jacobian products of the hot-path layers -------------------------------------------------
 * The rules restate TensorFlow's registered gradients of the ops the reference calls (RFFT / IRFFT, ComplexAbs,
 * MatMul, Log, Maximum, Max, tf.signal.frame's scatter-add, tf.pad's slice).  A complex gradient G is
 * dL/dRe + i dL/dIm.  Windows, filterbanks and dual windows are constants.  Every input is described by element
 * strides; any stride may be 0 (the gradient of a sum arrives as an expanded tensor).  Results are deterministic:
 * the same inputs give the same bits on every run. */

/* VJP of kapre_stft_forward(KAPRE_OUT_COMPLEX): complex64 gradient of the (batch, channels, frames, n_fft/2+1)
 * spectrum -> float32 gradient of the waveform, `grad_x_desc->length` samples (frames must equal
 * kapre_stft_num_frames(plan, length, pad_begin, pad_end)).  Frame t contributes
 * w[n] * sum_{k <= n_fft/2} Re(G_t[k] e^{+2 pi i k n / n_fft}) at padded sample t*hop + n, n < min(win_length, n_fft);
 * the pad_begin prefix is dropped and samples no frame covers get 0.  n_fft in {256,512,1024,2048}: the streaming
 * inverse-FFT kernel of kapre_istft_inverse with the window n_fft/2 * w; any other n_fft: a direct O(n_fft) sum per
 * sample and frame.  No workspace.  grad_spec and grad_x must not overlap. */
int kapre_stft_backward(const kapre_stft_plan* plan, const void* grad_spec_dev, int batch, int channels, int frames,
                        const kapre_spec_desc* grad_spec_desc, int pad_begin, int pad_end, float* grad_x_dev,
                        const kapre_wave_desc* grad_x_desc, void* stream);

/* VJP of kapre_istft_inverse: float32 gradient of the (batch, channels, (frames-1)*hop+win_length) waveform ->
 * complex64 gradient of the spectrum, G_t[k] = (c_k / n_fft) sum_{n < min(win_length, n_fft)} dual[n] g[t*hop + n]
 * e^{-2 pi i k n / n_fft} with c_0 = c_{n_fft/2} = 1 (n_fft/2 for even n_fft only), c_k = 2 otherwise; Im G[0] and
 * Im G[n_fft/2] are 0.  Runs kapre_stft_forward(KAPRE_OUT_COMPLEX) with a forward plan the inverse plan holds
 * (window 2/n_fft * dual), then halves the edge bins: every n_fft is served.  No workspace; no overlap. */
int kapre_istft_backward(const kapre_istft_plan* plan, const float* grad_y_dev, const kapre_wave_desc* grad_y_desc,
                         void* grad_spec_dev, int frames, const kapre_spec_desc* grad_spec_desc, void* stream);

/* VJP of the chain |X| [-> filterbank] [-> dB] at the complex64 STFT X (batch, channels, frames, n_freq), `mode` one
 * of KAPRE_OUT_MAG, _MAG_DB, _FB, _FB_DB (KAPRE_OUT_MAG alone is kapre.Magnitude's VJP).  grad: float32 upstream
 * gradient of the chain's (batch, channels, frames, K) output, K = n_freq or fb's band count; y (decibel modes):
 * that forward output.  Writes the complex64 gradient of X: G = g_mag X / |X| (0 where |X| = 0) with
 * g_mag = g_fb fb^T and the decibel rule of kapre_magnitude_to_decibel_backward per batch item.
 * workspace_dev (decibel modes): >= 1056 * batch + 16 bytes, zero on entry, left zero (self-cleaning).
 * grad_x may alias x exactly (same pointer and strides: in place); no other overlap. */
int kapre_spectral_backward(const kapre_filterbank* fb, int mode, const void* x_dev, int batch, int channels, int frames,
                            int n_freq, const kapre_spec_desc* x_desc, const float* grad_dev,
                            const kapre_spec_desc* grad_desc, const float* y_dev, const kapre_spec_desc* y_desc,
                            const kapre_db_cfg* db, void* workspace_dev, void* grad_x_dev,
                            const kapre_spec_desc* grad_x_desc, void* stream);

/* VJP of kapre_magnitude_to_decibel on contiguous (n_items, item_size) x (its input) and y (its output); the upstream
 * gradient has element strides (grad_item_stride, grad_elem_stride).  With l = 10 log10(max(x, amin)) - c,
 * m = max_item(l), thr = m - dynamic_range:
 *   dL/dl_i = g_i [l_i >= thr] + [l_i == m] sum_j g_j [l_j < thr] / #{l_j == m}   (the clamp's gradient goes to the
 *   item maximum, ties split it equally),  dL/dx_i = dL/dl_i 10 / (ln 10 max(x_i, amin)) [x_i >= amin].
 * Clamped elements are read from y: an item's clamp binds when min(y) <= max(y) - dynamic_range within a few float32
 * ulps, and then exactly the elements with y_i == min(y) are clamped (an unclamped l_i within float32 rounding of thr
 * counts as clamped).  Two launches: per-item statistics in fixed order (last-CTA combine), then the element rule.
 * workspace_dev: >= 1056 * n_items + 16 bytes, zero on entry, left zero.  grad_x may alias grad when both are
 * contiguous; no other overlap. */
int kapre_magnitude_to_decibel_backward(const float* x_dev, const float* y_dev, const float* grad_dev,
                                        int64_t grad_item_stride, int64_t grad_elem_stride, float* grad_x_dev,
                                        int64_t n_items, int64_t item_size, const kapre_db_cfg* db, void* workspace_dev,
                                        void* stream);

/* ---- misc ---------------------------------------------------------------------------------- */
const char* kapre_last_error(void);
int kapre_version(void);
/* Number of kernels this library has launched in this process (for bench.py's gpu_launches). */
uint64_t kapre_launch_count(void);
/* Name of the last fused-forward launch configuration, e.g. "Q16 TF16 NW4 grid296 smem98304". */
const char* kapre_last_launch_info(void);
/* Kernel timing for bench.py's roofline: enable = n > 0 brackets every n-th fused forward / inverse
 * kernel launch by CUDA events on its own stream (n = 1: every launch; a stride leaves the other
 * launches free to overlap their predecessor through programmatic dependent launch); 0 = off.  kapre_profile_read synchronises with
 * the recorded events, adds their durations to *total_ms / *launches and clears the list. */
int kapre_profile_enable(int enable);
int kapre_profile_read(double* total_ms, uint64_t* launches);

/* Experimental (measured prototype, not on the product path): stage 1 of the 32 x 32 factorisation of the
 * n_fft = 1024 / hop = 256 real FFT as a tcgen05 (5th-gen tensor core) GEMM with TMEM accumulators, fp32-grade via
 * the 3xTF32 split.  Layout of `out_dev` and the meaning of `store` are documented at the definition
 * (kapre_b200/csrc/kapre_b200.cu) and in DESIGN.md. */
/* Experimental: the next tensor-core (KAPRE_B200_TC=1) fused launch also writes its complex spectrum, (signals, frames, 513)
 * complex64, to dbg_dev -- used by the parity tests of the tcgen05 FFT stages. */
int kapre_tc_set_debug(void* dbg_dev);
int kapre_tc_dft_stage1(const float* x_dev, int n_items, long long item_stride, int length, float* out_dev, int store,
                        int* grid_out, const float* fmat_override_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KAPRE_B200_H_ */
