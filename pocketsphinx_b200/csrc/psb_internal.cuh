// psb_internal.cuh -- shared declarations of libpsb200.so (not part of the ABI).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>
#include <string>
#include <vector>

#include "../../include/psb200.h"

#define PSB_SENSCR_SHIFT 10      // hmm.h:72
#define PSB_MAX_NEG_ASCR 96      // tied_mgau_common.h:91
#define PSB_TMAT_WORST (-255)    // hmm.h:89
#define PSB_BAD_SSID 0xffff
#define PSB_LOGADD8_N 512        // 8-bit add table: 256 entries (logmath.c:116-120) continued with zeros

void psb_set_error(const char *fmt, ...);
extern std::atomic<long long> g_psb_launches;

#define PSB_CUDA(call)                                                                   \
    do {                                                                                 \
        cudaError_t e__ = (call);                                                        \
        if (e__ != cudaSuccess) {                                                        \
            psb_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call,                  \
                          cudaGetErrorString(e__));                                      \
            return PSB_ERR_CUDA;                                                         \
        }                                                                                \
    } while (0)

#define PSB_LAUNCH_CHECK()                                                               \
    do {                                                                                 \
        g_psb_launches.fetch_add(1, std::memory_order_relaxed);                          \
        cudaError_t e__ = cudaGetLastError();                                            \
        if (e__ != cudaSuccess) {                                                        \
            psb_set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__,              \
                          cudaGetErrorString(e__));                                      \
            return PSB_ERR_CUDA;                                                         \
        }                                                                                \
    } while (0)

#define PSB_REQUIRE(cond, ...)                                                           \
    do {                                                                                 \
        if (!(cond)) {                                                                   \
            psb_set_error(__VA_ARGS__);                                                  \
            return PSB_ERR_ARG;                                                          \
        }                                                                                \
    } while (0)

static inline int roundup(int x, int m) { return (x + m - 1) / m * m; }

// Gaussian record of one codeword in HBM/SMEM: {det, mean0, var0, mean1, var1, ...} padded
// with zeros to a multiple of 4 floats so that a warp-uniform LDS.128 stream feeds the
// distance loop.
static inline int rec_floats(int featlen) { return roundup(1 + 2 * featlen, 4); }

struct psb_model_s {
    int device;
    int kind, n_sen, n_mgau, n_feat, n_density, topn, ds_ratio, aw;
    int featlen[PSB_MAX_FEAT], featoff[PSB_MAX_FEAT], sumlen;
    int K;                        // n_mgau * n_feat (codebook, stream) pairs
    bool mixw_4bit;
    bool fixed_point;             // FIXED_POINT build arithmetic: mean/var/det/features are int32 (Q12) bit patterns
    int mixw_row;                 // bytes per (feat, codeword) row as given by the host
    int mixw_stride;              // padded row pitch on the device (multiple of 128)
    int logadd_ms_size, logadd_ms_zero;
    // device buffers
    float *d_rec;                 // records; (cb, f) block at rec_off[cb * n_feat + f]
    std::vector<size_t> rec_off;  // float offsets, host copy
    size_t *d_rec_off;
    float *d_rec2;                // pair-interleaved, negated records for the packed-FP32 kernels
    size_t *d_rec2_off;
    uint8_t *d_mixw;              // [n_feat][n_density][mixw_stride] (ptm/semi) or raw pdf (ms)
    uint8_t *d_mixw_cb;           // 16 bytes or null
    uint16_t *d_sen2cb;           // [n_sen] (ptm)
    int32_t *d_sen2cb32;          // [n_sen] (ms)
    bool sen_is_cb;               // ms: senone s uses codebook s (continuous models): distances and mixtures in one kernel
    int16_t *d_quadcb;            // [ceil(n_sen/4)] codebook of a uniform senone quad, else -1
    int32_t *d_bsen;              // senones of the non-uniform quads
    int n_bsen;
    int logadd8_max;              // largest entry of the 8-bit add table (bias bound of the 16x2 senone kernel)
    uint8_t *d_logadd8;           // [PSB_LOGADD8_N]: the 256-entry table continued with zeros
    uint32_t *d_logadd_ms;
    float *d_msT, *d_msdetT;      // ms back-end: codebook-minor Gaussians (see psb_ms.cu)
    int32_t *d_featlen, *d_featoff;
    uint8_t topn_beam[PSB_MAX_FEAT];
    int32_t *d_topn_beam;         // [PSB_MAX_FEAT]
    bool has_topn_beam;
    // tensor-core filter path (psb_ptm_tc.cu): W in the tcgen05 operand layout, centres, error-bound coefficients
    bool tc_ok;
    float *d_tc_wumma, *d_tc_cen, *d_tc_bnd;
};

struct psb_batch_s {
    psb_model_t *m;
    cudaStream_t stream;
    int max_utts;
    long long max_frames;
    // device
    float *d_feats;               // [max_frames][sumlen] staging for the _host path
    int16_t *d_senscr;            // [max_frames][n_sen]
    float *d_featT;               // transposed groups
    size_t featT_cap;             // floats
    int4 *d_topn;                 // [max_frames][K]
    int32_t *d_tab;               // per-call lane/group tables
    size_t tab_cap;
    int32_t *h_tab;               // pinned
    // pinned host staging for the _host path
    float *h_feats;
    int16_t *h_senscr;
    cudaEvent_t ev[4];
    cudaEvent_t tev[2];           // user stopwatch (psb_batch_event_record)
    bool have_ev;
    long long last_frames;
    float2 *d_semi_dist; size_t semi_cap;      // semi-continuous split path: {d, partial} per (stream, frame, codeword)
    int32_t *d_uttoff; size_t uttoff_cap;
    bool force_scan;              // PSB_TOPN_VARIANT=5: the scan kernels even where the tensor-core filter applies
                                  // (6, the default: the model's shape decides)
    unsigned *d_tc_flags; size_t tc_flag_cap, tc_flag_words;   // [K][words]: frames the tie fix-up redoes
    float *d_tc_check;            // debug (PSB_TC_CHECK=1): max |a - d| / eps, max candidates
    uint4 *d_tc_items; unsigned *d_tc_nitems; unsigned tc_item_cap;   // rows the filter left in doubt (ptm_tc_exact_kernel)
    // phone-loop outputs for psb_decode_batch_host
    int32_t *d_best, *d_pen;
    int32_t *h_best, *h_pen;
    size_t pen_cap;
    int32_t *d_off;               // utt_off on the device for the phone loop
    void *d_msdist;               // ms back-end: per-chunk top-N distance lists
    int32_t *d_msbest;
    size_t ms_cap;
    size_t off_cap;
    // pipelined decode: sub-batches on their own streams sharing this batch's big buffers
    std::vector<psb_batch_t *> kids;
    cudaEvent_t fork_ev, join_ev;
    int n_pipe;                   // PSB_PIPELINE: 0 = auto (default), 1 = everything on `stream`, n = n ranges
    bool is_kid;
    bool last_pipelined;
    int last_kids;                // sub-batches used by the last decode call
    int32_t *h_off;               // pinned copy of a sub-batch's utterance offsets
};

// ---- launchers implemented in the .cu files ----
cudaStream_t psb_batch_stream(psb_batch_t *b);
int psb_phoneloop_launch(psb_phoneloop_t *p, const int16_t *d_senscr, const int32_t *d_utt_off, int32_t n_utt,
                         int32_t *d_best, int32_t *d_pen, psb_hmm_t *d_final, psb_hmm_t *d_trace, cudaStream_t st);
int psb_phoneloop_n_phones(const psb_phoneloop_t *p);
int psb_launch_ptm_batch(psb_batch_t *b, const float *d_feats, const int32_t *utt_off,
                         int32_t n_utt, int16_t *d_senscr);
int psb_tc_prepare(psb_model_t *m, const float *hm, const float *hv, const float *hd);
bool psb_tc_usable(const psb_batch_t *b);
int psb_launch_ptm_tc(psb_batch_t *b, const float *d_feats, const int32_t *utt_off, int32_t n_utt, const int32_t *d_klist,
                      const int32_t *d_featoff);
int psb_ms_score_one(psb_model_t *m, cudaStream_t st, const float *d_feat, void *d_dist, int32_t *d_best,
                     int16_t *d_senscr, const int32_t *d_list, int n_items);
size_t psb_ms_dist_bytes(const psb_model_t *m);
int psb_launch_ms_batch(psb_batch_t *b, const float *d_feats, const int32_t *utt_off, int32_t n_utt, int16_t *d_senscr);
