/*
 * b200aa.h -- C ABI of libb200aa.so, the B200 (sm_100a) short-term / mid-term audio
 * feature extractor that replaces pyAudioAnalysis' NumPy hot path.
 *
 * Boundary rules: extern "C", plain pointers and sizes, no C++ / torch types, no
 * exceptions.  Every function returns 0 (B200AA_OK) or a negative b200aa_status.
 * Pointers named d_* are device pointers of the current CUDA device, h_* are host
 * pointers; the caller owns every buffer.  `stream` is a cudaStream_t passed as
 * void* (NULL = default stream); device-pointer entry points are asynchronous on it.
 *
 * The reference has no FFI of its own: its boundary is four Python functions.  Each
 * entry point below names the reference code it replaces (paths relative to
 * pyAudioAnalysis/ in the reference tree).  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 */
#ifndef B200AA_H_
#define B200AA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200AA_ABI_VERSION 1

typedef enum b200aa_status {
    B200AA_OK = 0,
    B200AA_ERR_INVALID = -1,      /* bad argument (NULL pointer, window < 2, step < 1, ...)              */
    B200AA_ERR_TOO_SHORT = -2,    /* clip shorter than one window: the reference raises ValueError
                                     ("need at least one array to concatenate", ShortTermFeatures.py:684) */
    B200AA_ERR_CHROMA = -3,       /* semitone index >= num_fft: the reference's chroma else-branch
                                     (ShortTermFeatures.py:290-294) raises ValueError                     */
    B200AA_ERR_MEL_RANGE = -4,    /* mel filter edge beyond num_fft: the reference raises IndexError
                                     (ShortTermFeatures.py:230-231)                                       */
    B200AA_ERR_CUDA = -5,         /* a CUDA call failed; see b200aa_last_cuda_error()                     */
    B200AA_ERR_UNSUPPORTED = -6,  /* window too large for the on-chip transform buffers                  */
    B200AA_ERR_NO_DEVICE = -7     /* no CUDA device / not an sm_100 device                                */
} b200aa_status;

/* sample formats of the clip buffer */
#define B200AA_DTYPE_I16 0        /* int16 PCM as scipy.io.wavfile.read returns it (audioBasicIO.py:99) */
#define B200AA_DTYPE_F32 1        /* float32 samples (any scale; the path is scale invariant)           */

#define B200AA_N_BASE 34          /* ShortTermFeatures.py:580-585 */
#define B200AA_N_MEL 40           /* ShortTermFeatures.py:191-192 */
#define B200AA_N_MFCC 13

/* Per-clip affine normalisation y = a*(x - m) + bp that reproduces `/2**15` + dc_normalize()
 * (ShortTermFeatures.py:567-570, :14-19), plus exact thresholds for sign(x - mean).  32 bytes. */
typedef struct b200aa_clip_norm {
    float a;        /* 1 / (max|x - mean| + 2^15 * 1e-10)                      */
    float bp;       /* a * (m - mean)                                          */
    float m;        /* value nearest to the clip mean that is exact in float   */
    float lo;       /* largest representable sample value <= mean, minus m    */
    float hi;       /* smallest representable sample value >= mean, minus m   */
    float rsv[3];   /* scratch used while the statistics are accumulated       */
} b200aa_clip_norm;

typedef struct b200aa_plan b200aa_plan;   /* opaque: constant tables of one (fs, window, step) on one device */

/* ------------------------------------------------------------------ library ---------- */
int         b200aa_abi_version(void);
const char *b200aa_status_string(int status);
const char *b200aa_last_cuda_error(void);        /* thread-local text of the last CUDA failure */
int         b200aa_device_ok(void);              /* B200AA_OK iff the current device is sm_100 */

/* ------------------------------------------------------------------ host tables -------
 * Pure host code, usable without a GPU (the CPU test-suite checks them against the oracle).
 *   which = 0: mel filterbank, dense [40 x K] doubles           (mfcc_filter_banks, ShortTermFeatures.py:191-233)
 *   which = 1: chroma operator, dense [12 x K] doubles           (chroma_features_init + scatter, :257-302)
 *   which = 2: DCT-II ortho rows 0..12, dense [13 x 40] doubles  (scipy dct call at :253)
 * K = window / 2.  Returns B200AA_ERR_CHROMA / B200AA_ERR_MEL_RANGE where the reference raises. */
int b200aa_host_table(int fs, int window, int which, double *h_out);

/* frame / row counts of the three reference entry points */
int64_t b200aa_num_frames(int64_t n_samples, int window, int step);            /* ShortTermFeatures.py:608 */
int64_t b200aa_spectrogram_rows(int64_t n_samples, int window, int step);      /* :413 */
int64_t b200aa_chromagram_rows(int64_t n_samples, int window, int step);       /* :347 */
int64_t b200aa_mid_windows(int64_t n_frames, int step_ratio);                  /* MidTermFeatures.py:116-124 */

/* ------------------------------------------------------------------ plan --------------- */
int  b200aa_plan_create(b200aa_plan **out, int fs, int window, int step);
void b200aa_plan_destroy(b200aa_plan *plan);
/* kernel that feature launches of this plan use: 0 = generic mixed-radix kernel (any window), 1 = register-tiled
 * CTA kernel (windows 320/400/480/600/640/800/882), 2 = warp-autonomous pair kernel (windows 32*R: 320/480/512/640/
 * 800/960/1024), 3 = warp-autonomous per-frame kernel (windows 882/400/600, also their spectrogram / chromagram rows) */
int  b200aa_plan_kernel_kind(const b200aa_plan *plan);
/* restrict the plan to one kernel (testing / A-B runs): -1 = automatic (default), 0..3 as above; a kind that
 * does not exist for the plan's window falls through to the next one */
int  b200aa_plan_prefer_kernel(b200aa_plan *plan, int kind);
/* force the generic kernel (testing): returns the previous setting */
int  b200aa_plan_force_generic(b200aa_plan *plan, int on);

/* frees the device workspaces the host entry points keep between calls (grown to the largest call seen) */
int  b200aa_plan_trim(b200aa_plan *plan);

/* ------------------------------------------------------------------ device entry points */

/* Kernel 0: per-clip statistics -> normalisation records.
 * d_sig: [n_clips] clips, clip b starts at element b*clip_stride; d_len (nullable, int64[n_clips])
 * gives ragged lengths (<= n_samples); d_norm: [n_clips] records.
 * Replaces: `signal / 2**15` + dc_normalize (ShortTermFeatures.py:567-570, :14-19). */
int b200aa_clip_stats(const void *d_sig, int dtype, int64_t n_clips, int64_t n_samples,
                      int64_t clip_stride, const int64_t *d_len,
                      b200aa_clip_norm *d_norm, void *stream);

/* Kernel 1: fused short-term features.  d_out: float32 [n_clips, F, t_stride] with
 * F = 34 (deltas == 0) or 68, frame t of clip b, feature f at d_out[(b*F + f)*t_stride + t];
 * t_stride >= frames of the longest clip.  Columns >= the clip's own frame count are not written.
 * Replaces: the frame loop of ShortTermFeatures.feature_extraction (:608-685). */
int b200aa_st_features(const b200aa_plan *plan, const void *d_sig, int dtype, int64_t n_clips,
                       int64_t n_samples, int64_t clip_stride, const int64_t *d_len,
                       const b200aa_clip_norm *d_norm, int deltas,
                       float *d_out, int64_t t_stride, void *stream);

/* Spectrogram rows: d_out float32 [n_clips, R, K], R = b200aa_spectrogram_rows(n_samples),
 * trailing rows zero exactly as the reference leaves them (ShortTermFeatures.py:413-422). */
int b200aa_spectrogram(const b200aa_plan *plan, const void *d_sig, int dtype, int64_t n_clips,
                       int64_t n_samples, int64_t clip_stride,
                       const b200aa_clip_norm *d_norm, float *d_out, void *stream);

/* Chromagram rows: d_out float32 [n_clips, R, 12], R = b200aa_chromagram_rows(n_samples)
 * (ShortTermFeatures.py:347-359), including the zero last row / clipped last frame cases. */
int b200aa_chromagram(const b200aa_plan *plan, const void *d_sig, int dtype, int64_t n_clips,
                      int64_t n_samples, int64_t clip_stride,
                      const b200aa_clip_norm *d_norm, float *d_out, void *stream);

/* Kernel 2: mid-term pooling.  d_st float32 [n_clips, F, t_stride] (n_frames valid columns),
 * d_mid float32 [n_clips, 2F, M], M = b200aa_mid_windows(n_frames, step_ratio): rows 0..F-1 means,
 * F..2F-1 population standard deviations of st[f][c : min(c+ratio, T)], c = j*step_ratio.
 * Replaces: MidTermFeatures.mid_feature_extraction's pooling loops (:110-126). */
int b200aa_mid_pool(const float *d_st, int64_t n_clips, int n_feats, int64_t n_frames,
                    int64_t t_stride, int ratio, int step_ratio, float *d_mid, void *stream);

/* Long-term average (SURVEY 8f rank 1): d_out float32 [n_clips, n_rows], the mean of every row of
 * d_mid [n_clips, n_rows, n_windows] over the windows.
 * Replaces: `mid_features.mean(axis=0)` in directory_feature_extraction (MidTermFeatures.py:200-201). */
int b200aa_long_term_mean(const float *d_mid, int64_t n_clips, int n_rows, int64_t n_windows,
                          float *d_out, void *stream);

/* Feature vectors for the classifiers that consume the mid-term matrix (SURVEY 8f rank 4): d_out float32
 * [n_clips, n_windows, n_rows], vector j of clip b = (d_mid[b, :, j] - mean) / std -- the transpose the per-window loops
 * build one column at a time.  d_mean / d_std: float32 [n_rows] on the device.  Any number of clips; more than
 * 65 535 * 32 rows returns B200AA_ERR_UNSUPPORTED.
 * Replaces: `feature_vector = (mt_feats[:, col_index] - mean) / std` per window (audioSegmentation.py:581-584,
 * audioTrainTest.py:1091) and per short-term frame (audioSegmentation.py:744-748, with d_mid = the [68 x T] matrix). */
int b200aa_normalize_windows(const float *d_mid, int64_t n_clips, int n_rows, int64_t n_windows,
                             const float *d_mean, const float *d_std, float *d_out, void *stream);

/* ------------------------------------------------------------------ host entry points --
 * Same operations on HOST buffers: pinned or pageable input is copied to the device, the
 * kernels run, the result is copied back and the call returns after the stream drained.
 * These are what a ctypes / cffi binding of the reference would call (INTEGRATION.md). */
int b200aa_st_features_host(const b200aa_plan *plan, const void *h_sig, int dtype, int64_t n_clips,
                            int64_t n_samples, int deltas, float *h_out /* [n_clips, F, T] */);
int b200aa_spectrogram_host(const b200aa_plan *plan, const void *h_sig, int dtype,
                            int64_t n_samples, float *h_out /* [R, K] */);
int b200aa_chromagram_host(const b200aa_plan *plan, const void *h_sig, int dtype,
                           int64_t n_samples, float *h_out /* [R, 12] */);
int b200aa_mid_features_host(const b200aa_plan *plan, const void *h_sig, int dtype, int64_t n_samples,
                             int ratio, int step_ratio,
                             float *h_mid /* [136, M] */, float *h_st /* [68, T], nullable */);

/* Pinned (page-locked) host buffers for the host entry points: with them the chunked pipeline inside
 * b200aa_st_features_host overlaps the PCIe copies of neighbouring chunks with the kernels.  Pages are placed by
 * the calling thread's NUMA policy -- bind the thread to the GPU's node first (pyaudioanalysis_b200/numa.py).
 * Replaces nothing in the reference (its arrays are pageable NumPy buffers, audioBasicIO.py:86-110); SURVEY 8f rank 2. */
int b200aa_host_alloc(void **h_out, size_t bytes);
int b200aa_host_free(void *h_ptr);

/* Peer-mapped gather target (SURVEY 8e, BASELINE configs[4]): the root rank creates one device buffer for the
 * features of ALL clips and exports a 64-byte handle; every other rank of the box opens it (CUDA IPC, NVLink peer
 * mapping).  A rank then either pushes its finished block with b200aa_peer_copy (copy engines, asynchronous on a
 * stream of its own so the transfer rides under the next batch's kernels; no collective kernel, no SM on either
 * side) or passes `peer_ptr + its slice offset` straight as d_out of b200aa_st_features (the tile stores land in
 * the root's HBM: free at 2 GPUs, but 32-byte remote stores from 7 GPUs into one collapse to ~220 GB/s at 8).
 * Handles travel between the processes by any byte channel (the Python host side uses torch.distributed). */
#define B200AA_IPC_HANDLE_BYTES 64
int b200aa_peer_buffer_create(size_t bytes, void **d_out, unsigned char *handle_out /* [64] */);
int b200aa_peer_buffer_open(const unsigned char *handle /* [64] */, void **d_out);
int b200aa_peer_copy(void *d_dst /* peer-mapped or local */, const void *d_src, size_t bytes, void *stream);
int b200aa_peer_buffer_close(void *d_ptr, int owner /* 1: the creating rank (frees), 0: a mapping rank (unmaps) */);

/* debugging: when set (device pointer, float32 [n_clips, t_stride, K]) the pair kernel also dumps its |X| rows */
int b200aa_debug_set_dump(float *d_rows);

/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t b200aa_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B200AA_H_ */
