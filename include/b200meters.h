/* b200meters.h — C ABI of the B200-native batched audio-metering engine.
 *
 * One "bank" = N independent instances of one reference DSP class, all processed by one CUDA
 * kernel launch per process() call.  Entry points mirror, one for one, the methods an LV2 host
 * reaches through x42/meters.lv2's run() callbacks; each declaration cites the reference
 * interface it replaces (paths relative to the reference tree).
 *
 * Conventions
 *  - plain C, no CUDA/torch types: device pointers and streams travel as void*.
 *  - every function returns 0 on success or a negative B200M_E_* code; nothing throws.
 *  - audio is planar float32, exactly what an LV2 host connects to an audio port
 *    (src/meters.cc:257-296): channel k (k = inst*nchan + c) of a process call starts at
 *    in + k*stride and holds nfram samples.  `*_process_device` takes a device pointer and is
 *    asynchronous on `stream` (a cudaStream_t, NULL = legacy default stream);
 *    `*_process_host` takes a host pointer (pinned memory recommended: b200m_host_alloc),
 *    performs the host->device copy itself and is asynchronous on the bank's own stream.
 *  - `*_read_device` mirrors the reference's read()/getter step on the device (including its
 *    reset-latch side effects) and stores the values in a device result block;
 *    `*_results` copies that block to the host (synchronises the stream it was given).
 *  - there is NO CPU fallback: a bank cannot be created without a CUDA device, and every
 *    sample is processed by the sm_100a kernels in meters.lv2_b200/csrc/.
 */
#ifndef B200METERS_H
#define B200METERS_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)   /* the library is built with -fvisibility=hidden */
#endif

#define B200M_ABI_VERSION 1

enum {
    B200M_OK            =  0,
    B200M_E_INVAL       = -1,   /* bad argument (NULL handle, n out of range, bad stride ...) */
    B200M_E_NOMEM       = -2,   /* host or device allocation failed */
    B200M_E_CUDA        = -3,   /* CUDA runtime error: see b200m_last_error() */
    B200M_E_UNSUPPORTED = -4,   /* valid in the reference, not provided by this engine */
    B200M_E_NODEVICE    = -5    /* no CUDA device: the engine has no CPU path */
};

#define B200M_MAX_BLOCK 8192u     /* TruePeakdsp::process asserts n <= 8192 (jmeters/truepeakdsp.cc:43-44);
                                     robtk/jackwrap.c:35 MAXPERIOD 8192 */
#define B200M_HIST_LEN  751       /* Ebu_r128_hist bins, -70.0 .. +5.0 dB (ebumeter/ebu_r128_proc.cc:34) */

int         b200m_abi_version (void);
const char* b200m_last_error (void);            /* thread-local text of the last failure */
int         b200m_device_count (void);
/* pinned host memory for process_host()/results(): cudaHostAlloc / cudaFreeHost */
int         b200m_host_alloc (void** p, size_t bytes);
int         b200m_host_free (void* p);
/* number of kernel launches issued by this library since load (bench.py's gpu_launches) */
uint64_t    b200m_launch_count (void);

/* ALU ceilings measured on the device (the driver's MEASURED_PEAKS.json has only HBM and bf16 GEMM):
 * kind 0 = fp32 unfused FMUL+FADD issue rate, kind 1 = fp64 DMUL+DADD, kind 2 = packed fp32x2 FMUL2+FADD2;
 * result in 1e9 lane-operations/s. */
int         b200m_peak_probe (int device, int kind, double* gops);

/* Self-test hook: log10f of the `count` floats whose bit patterns are first_bits, first_bits + 1, ... written to the DEVICE
 * array d_out, evaluated by the device function every loudness / dB value of the engine goes through (a restatement of
 * glibc's log10f: the reference bins log10f results into integer histograms, ebumeter/ebu_r128_proc.cc:66-79,116-141,259).
 * tests/test_log10f_sweep_gpu.py sweeps all 2^31 non-negative floats against the host libm with it. */
int         b200m_selftest_log10f (int device, uint32_t first_bits, uint32_t count, float* d_out, void* stream);

/* Host-side coefficient design, callable without a GPU (pure functions of the sample rate, computed with
 * the host libm in the reference's expression types so that every value is bitwise the reference's):
 *   ebu : detect_init (ebumeter/ebu_r128_proc.cc:263-293)           -> a0 a1 a2 b1 b2 c3 c4
 *   tpk : TruePeakdsp::init (jmeters/truepeakdsp.cc:148-157), zita table (zita-resampler/resampler-table.cc:
 *         52-75; hl=24 np=4 fr=1), Kmeterdsp::init (jmeters/kmeterdsp.cc:47-54) -> w1 w2 w3 g | ctab | omega hold
 *   cor : Stcorrdsp::init (jmeters/stcorrdsp.cc:85-93)              -> w1 w2
 *   spec: spectrum_instantiate band table + bandpass_setup (src/spectrumlv2.c:100-118, src/spectr.c:89-206)
 *         -> W[30][6][6] = a0 a1 a2 b0 b1 b2 per section */
int b200m_design_ebu (float fsamp, float out7[7]);
int b200m_design_tpk (float fsamp, float w[4], float ctab[120], float km[2]);
int b200m_design_cor (int fsamp, float flp, float tcf, float w[2]);
int b200m_design_spec (double rate, double* W1080);

/* ======================================================================================
 * EBU R128 loudness bank — replaces LV2M::Ebu_r128_proc (ebumeter/ebu_r128_proc.h:66-125)
 * as driven by ebur128_run (src/ebulv2.cc:341-358).
 * ====================================================================================== */
typedef struct b200m_ebu b200m_ebu;

typedef struct b200m_ebu_result {          /* getters, ebumeter/ebu_r128_proc.h:81-89 */
    float loudness_M, maxloudn_M, loudness_S, maxloudn_S;
    float integrated, integ_thr, range_min, range_max, range_thr;
    int32_t hist_M_count, hist_S_count;    /* :93-94 */
    float   frag_power;                    /* last completed 50 ms fragment power (_power[_wrind-1]) */
} b200m_ebu_result;

/* Ebu_r128_proc() + init(nchan, fsamp) (:166-173) for n_inst instances.  nchan 1..5 (the EBUr128 plugin uses 2, src/ebulv2.cc:190;
 * 3..5: surround layouts with the channel gains 1 1 1 1.41 1.41 of ebu_r128_proc.cc:29). */
int b200m_ebu_create (b200m_ebu** out, int device, uint32_t n_inst, uint32_t nchan, float fsamp);
int b200m_ebu_destroy (b200m_ebu* h);
/* Ebu_r128_proc::reset (:176-190).  All instances share the 50 ms fragment clock, so only
 * inst = -1 (every instance) is accepted. */
int b200m_ebu_reset (b200m_ebu* h, int32_t inst, void* stream);
/* integr_start / integr_pause (ebu_r128_proc.h:77-78) / integr_reset (.cc:193-204); inst = -1: all */
/* one instance back to its state after init(): integration off, filters, ring, loudness values and histograms cleared; the bank's
 * shared fragment clock keeps running (slot reuse in shared banks) */
int b200m_ebu_clear (b200m_ebu* h, int32_t inst, void* stream);
int b200m_ebu_integr_start (b200m_ebu* h, int32_t inst, void* stream);
int b200m_ebu_integr_pause (b200m_ebu* h, int32_t inst, void* stream);
int b200m_ebu_integr_reset (b200m_ebu* h, int32_t inst, void* stream);
/* Ebu_r128_proc::process(nfram, input[]) (:207-248) for every instance. 0 < nfram <= 8192. */
int b200m_ebu_process_device (b200m_ebu* h, const float* d_in, size_t stride, uint32_t nfram, void* stream);
int b200m_ebu_process_host (b200m_ebu* h, const float* in, size_t stride, uint32_t nfram);
/* getters -> host array of n_inst results.  stream = the stream last used for processing
 * (ignored after process_host, which uses the bank's stream). */
int b200m_ebu_results (b200m_ebu* h, b200m_ebu_result* out, void* stream);
/* histogram_M()/histogram_S() (:91-92) of one instance: 751 + 751 int32 */
int b200m_ebu_histogram (b200m_ebu* h, uint32_t inst, int32_t* hist_M, int32_t* hist_S, void* stream);
/* K-weighting coefficients as designed on the host (detect_init, :263-293): a0 a1 a2 b1 b2 c3 c4 */
size_t b200m_ebu_snapshot_size (b200m_ebu* h);                          /* see b200m_r128_snapshot */
int b200m_ebu_snapshot (b200m_ebu* h, void* buf, size_t bytes, void* stream);
int b200m_ebu_restore (b200m_ebu* h, const void* buf, size_t bytes, void* stream);
int b200m_ebu_coeffs (const b200m_ebu* h, float out7[7]);
/* internal state of one instance for differential tests: z[nchan][4], power ring[64], frpwr,
 * counters {frcnt, wrind, div1, div2} */
int b200m_ebu_state (b200m_ebu* h, uint32_t inst, float* z, float* power64, float* frpwr, int32_t counters4[4], void* stream);
/* Whole-mix gated loudness (an extension; the reference has no cross-instance quantity):
 * sums hist_M/hist_S/counts of all instances on the device into d_out[2*752+...]; the caller
 * may all-reduce that int32 vector across GPUs (NCCL) and hand it to b200m_ebu_mix_finish. */
#define B200M_MIX_WORDS 1508      /* histM[752] histS[752] cntM cntS errM errS */
int b200m_ebu_mix_reduce (b200m_ebu* h, int32_t* d_out, void* stream);
/* calc_integ + calc_range (:105-150) on a summed histogram vector (device pointer);
 * out5 (host) = integrated, integ_thr, range_min, range_max, range_thr */
int b200m_ebu_mix_finish (b200m_ebu* h, const int32_t* d_mix, float out5[5], void* stream);

/* ======================================================================================
 * True-peak + K-meter bank — replaces LV2M::TruePeakdsp (jmeters/truepeakdsp.h:28-61) and
 * LV2M::Kmeterdsp (jmeters/kmeterdsp.h:27-62), one mono meter of each kind per channel, as
 * driven by dr14_run in TPnRMS mode (src/dr14.c:391-394,425-450), dbtp_run / kmeter_run
 * (src/meters.cc:333-508) and ebur128_run's dBTP option (src/ebulv2.cc:344-347,360-367).
 * ====================================================================================== */
typedef struct b200m_tpk b200m_tpk;

#define B200M_TPK_TRUEPEAK 1u     /* run TruePeakdsp per channel */
#define B200M_TPK_KMETER   2u     /* run Kmeterdsp per channel   */
#define B200M_TP_MODE_PROCESS 0u  /* TruePeakdsp::process      (:41-99)  */
#define B200M_TP_MODE_MAX     1u  /* TruePeakdsp::process_max  (:101-124) */

typedef struct b200m_tpk_result {
    float tp_m, tp_p;             /* TruePeakdsp::read(m,p) (:133-138) — linear */
    float km_rms, km_peak;        /* Kmeterdsp::read(rms,peak) (kmeterdsp.cc:150-155) — linear */
} b200m_tpk_result;

int b200m_tpk_create (b200m_tpk** out, int device, uint32_t n_chan, float fsamp, uint32_t flags);
int b200m_tpk_destroy (b200m_tpk* h);
/* process() of every enabled meter over one block; tp_mode selects process / process_max */
int b200m_tpk_process_device (b200m_tpk* h, const float* d_in, size_t stride, uint32_t nfram, uint32_t tp_mode, void* stream);
int b200m_tpk_process_host (b200m_tpk* h, const float* in, size_t stride, uint32_t nfram, uint32_t tp_mode);
/* Arithmetic of the 4x polyphase FIR (zita-resampler/resampler.cc:213-230).
 *   B200M_PREC_EXACT (default): the reference's operation order, unfused -- every float bit-identical to the reference build.
 *   B200M_PREC_FMA: fused multiply-add accumulation using the table's symmetry, phase 0 taken as the pure delay it is to
 *     7.7e-16: 2.4x fewer instructions; true-peak / dBTP readings stay within +-1e-4 dB of the reference (measured <= 2e-5 dB),
 *     the K-meter and every integer result are unaffected.  Default can be preset with B200M_TPK_PRECISION=fma. */
enum { B200M_PREC_EXACT = 0, B200M_PREC_FMA = 1 };
int b200m_tpk_set_precision (b200m_tpk* h, int mode);
int b200m_tpk_precision (const b200m_tpk* h);
/* read() of every enabled meter (sets TruePeakdsp::_res / Kmeterdsp::_flag) */
int b200m_tpk_read_device (b200m_tpk* h, void* stream);
int b200m_tpk_results (b200m_tpk* h, b200m_tpk_result* out, void* stream);
/* TruePeakdsp::reset (:140-145) / Kmeterdsp::reset (kmeterdsp.cc:157-162); chan = -1: all */
int b200m_tpk_reset (b200m_tpk* h, int32_t chan, void* stream);
/* reset() plus zero ballistics filters and oversampler history: the channel as a newly constructed meter leaves init(); chan = -1: all */
int b200m_tpk_clear (b200m_tpk* h, int32_t chan, void* stream);
/* Kmeterdsp::reset of every channel only (reset_peaks of the TPnRMS / DR14 plugin, src/dr14.c:241-258) */
int b200m_tpk_reset_kmeter (b200m_tpk* h, void* stream);
/* host-designed constants: w[4] = w1 w2 w3 g (truepeakdsp.cc:153-157); ctab[120] = zita table
 * (zita-resampler/resampler-table.cc:52-75, hl=24 np=4 fr=1); km[2] = omega, (float)hold */
size_t b200m_tpk_snapshot_size (b200m_tpk* h);                          /* see b200m_r128_snapshot */
int b200m_tpk_snapshot (b200m_tpk* h, void* buf, size_t bytes, void* stream);
int b200m_tpk_restore (b200m_tpk* h, const void* buf, size_t bytes, void* stream);
int b200m_tpk_coeffs (const b200m_tpk* h, float w[4], float ctab[120], float km[2]);
/* internal state for differential tests, arrays of n_chan: tp {m,p,z1,z2,res}, km [n][8] as
 * z1 z2 rms peak fall cnt fpp flag */
int b200m_tpk_state (b200m_tpk* h, float* tp_m, float* tp_p, float* tp_z1, float* tp_z2, int32_t* tp_res, float* km8, void* stream);
/* the raw 4x oversampled stream of the LAST processed block of one channel (4*nfram floats),
 * only kept when enabled with b200m_tpk_debug_capture(h,1): FIR bit-exactness tests */
int b200m_tpk_debug_capture (b200m_tpk* h, int enable);
int b200m_tpk_debug_upsampled (b200m_tpk* h, uint32_t chan, float* out, uint32_t n_out, void* stream);
/* launch timeline of the opt-in slab pipeline (B200M_TPK_SPLIT=2 with B200M_TPK_TIMELINE=1): up to n slots of
 * {first CTA start, last CTA end} in %globaltimer ns, two slots (filter, ballistics) per slab; returns the count, -1 = off */
int b200m_tpk_debug_timeline (b200m_tpk* h, unsigned long long* out, int n);

/* ======================================================================================
 * EBUr128 plugin cycle — the audio part of ebur128_run (src/ebulv2.cc:341-367) for N stereo
 * instances: Ebu_r128_proc::process + (if dbtp_enable) TruePeakdsp::process_max on both channels,
 * the getters, and the dBTP hold  tp_max = max (tp_max, coef_to_db (max (tp0, tp1)))  (:227-230,360-367).
 * One host->device copy per block feeds both meters.  Atom/radar/GUI messaging is out of scope.
 * ====================================================================================== */
typedef struct b200m_r128 b200m_r128;
enum { B200M_R128_START = 1, B200M_R128_PAUSE = 2, B200M_R128_RESET = 3, B200M_R128_CLEAR_TPMAX = 4, B200M_R128_CLEAR = 5 };   /* CLEAR: one slot back to a freshly created instance (inst >= 0) */   /* CTL_START/PAUSE/RESET, src/uris.h:187-203; RESET = ebu_reset
                                                                                * (src/ebulv2.cc:45-61): integr_reset + tp_max hold cleared;
                                                                                * CLEAR_TPMAX: the hold alone (a dBTP-disabled cycle, :365-366) */
int b200m_r128_create (b200m_r128** out, int device, uint32_t n_inst, float fsamp, int dbtp_enable);
int b200m_r128_destroy (b200m_r128* h);
int b200m_r128_control (b200m_r128* h, int32_t inst, int cmd, void* stream);      /* inst = -1: all */
int b200m_r128_run_device (b200m_r128* h, const float* d_in, size_t stride, uint32_t nfram, void* stream);
int b200m_r128_run_host (b200m_r128* h, const float* in, size_t stride, uint32_t nfram);
/* PCM input: the cycle above on the sample format a decoder, capture card or file reader already holds, converted on the GPU.
 * fmt = sample type | layout; all types little-endian.  Value handed to the meters (the float32 a host would have passed to
 * b200m_r128_run_*):
 *   B200M_PCM_F32  float32                  the bits unchanged (NaN payloads, -0, denormals, +-inf pass through)
 *   B200M_PCM_S16  int16                    (float)x * 0x1p-15f                                         (exact)
 *   B200M_PCM_S24  packed 3-byte signed     sign-extended to int32, then (float)x * 0x1p-23f            (exact)
 *   B200M_PCM_S32  int32                    __int2float_rn (x) * 0x1p-31f: round to nearest even, as the host's (float)x under
 *                                           the default MXCSR and numpy's astype (np.float32)
 * Layouts, `stride` counted in elements of the sample type:
 *   B200M_PCM_PLANAR       channel k = inst*nchan + c starts at element k*stride (the float convention above)
 *   B200M_PCM_INTERLEAVED  instance inst's frames start at element inst*stride*nchan, sample (f, c) at + f*nchan + c;
 *                          stride is in frames
 * Only the alignment of the sample type is assumed (1 byte for S24, 2 for S16, 4 otherwise).  stride >= nfram, 0 < nfram <= 8192.
 * F32 | PLANAR is b200m_r128_run_device / _run_host itself.  run_device_pcm converts the block on `stream` into a float buffer of
 * the bank, then runs the cycle on it; run_host_pcm copies the raw PCM bytes (1/2 of the float32 bytes for S16, 3/4 for S24) in
 * the same instance slices as run_host, and converts each slice on a stream of its own as soon as its copy has landed. */
enum { B200M_PCM_F32 = 0, B200M_PCM_S16 = 1, B200M_PCM_S24 = 2, B200M_PCM_S32 = 3,
       B200M_PCM_PLANAR = 0, B200M_PCM_INTERLEAVED = 16 };
int b200m_r128_run_device_pcm (b200m_r128* h, const void* d_in, uint32_t fmt, size_t stride, uint32_t nfram, void* stream);
int b200m_r128_run_host_pcm (b200m_r128* h, const void* in, uint32_t fmt, size_t stride, uint32_t nfram);
/* any bank's device path: a PCM block of n_inst x nchan channels (nchan 1..8; same formats and layouts as above, src_stride in
 * elements) -> planar float32 rows, row k = inst*nchan + c at d_dst + k*dst_stride (d_dst 16-byte aligned, dst_stride a multiple
 * of 4 and >= nfram).  Asynchronous on `stream`; the rows then go to any b200m_*_process_device / _run_device. */
int b200m_pcm_convert (int device, const void* d_src, uint32_t fmt, uint32_t nchan, uint32_t n_inst, size_t src_stride,
                       uint32_t nfram, float* d_dst, size_t dst_stride, void* stream);
/* ebu_out: n_inst getter blocks (may be NULL); tp_max_db: n_inst floats, -inf when dBTP is disabled (may be NULL) */
int b200m_r128_results (b200m_r128* h, b200m_ebu_result* ebu_out, float* tp_max_db, void* stream);
/* self->dbtp_enable (CTL_UISETTINGS bit 64, src/ebulv2.cc:316-317): the true-peak meters only run while enabled; while
 * disabled tp_max is -inf every cycle (:365-366).  Takes effect with the next run. */
int b200m_r128_set_dbtp (b200m_r128* h, int enable);
/* precision of the true-peak FIR (b200m_tpk_set_precision); Ebu_r128_proc's arithmetic is always exact */
int b200m_r128_set_precision (b200m_r128* h, int mode);
/* histogram_M() / histogram_S() of one instance (src/ebulv2.cc:425-429), ordered after the bank's last run */
int b200m_r128_histogram (b200m_r128* h, uint32_t inst, int32_t* hist_M, int32_t* hist_S, void* stream);
/* Checkpoint / resume (new: the reference saves only UI settings, never DSP state -- src/ebulv2.cc:513-548): the complete
 * state of the bank (filters, 64-fragment rings, both histograms of every instance, gating clocks, true-peak histories and
 * holds) as one host blob.  restore() needs a bank created with the same n_inst / fsamp; processing then continues
 * bit-identically to the bank the snapshot was taken from.  Also available per bank: b200m_ebu_* / b200m_tpk_*. */
size_t b200m_r128_snapshot_size (b200m_r128* h);
int b200m_r128_snapshot (b200m_r128* h, void* buf, size_t bytes, void* stream);
int b200m_r128_restore (b200m_r128* h, const void* buf, size_t bytes, void* stream);
b200m_ebu* b200m_r128_ebu (b200m_r128* h);     /* the underlying banks (histograms, state, coefficients) */
b200m_tpk* b200m_r128_tpk (b200m_r128* h);

/* ======================================================================================
 * DR-14 / TPnRMS bank (SURVEY §8f rank 2) — replaces dr14_run (src/dr14.c:354-482) for n_inst instances of
 * n_channels (1 or 2): Kmeterdsp::process + TruePeakdsp::process + read() per channel and, with dr_mode, the 3 s
 * window statistics of dr14_calc_rms_score (:285-352).  The result block mirrors the plugin's output ports
 * (DRPortIndex :27-43): all values in dB as the reference writes them.  Every instance shares the 3 s window clock, so
 * reset_peaks (:241-258) is bank-wide.  dr_mode needs rate >= 2731 Hz (a window longer than the largest block).
 * ====================================================================================== */
typedef struct b200m_dr14 b200m_dr14;
typedef struct b200m_dr14_result {
    float v_rms[2], v_peak[2];       /* *p_v_rms = coeff_to_db (km rms), *p_v_peak = coeff_to_db (true-peak ballistic m) (:430-431) */
    float m_peak[2], m_rms[2];       /* coeff_to_db (max true peak) (:432); DR mode: top-20 % RMS score, else coeff_to_db (km peak) (:444-446) */
    float dr[2], dr_total;           /* DR mode: per channel and averaged, clamped to 1..20; 21 = not yet valid (:436-458) */
    float block_count;               /* 3.0 * num_fragments (:460) */
} b200m_dr14_result;
int b200m_dr14_create (b200m_dr14** out, int device, uint32_t n_inst, uint32_t n_channels, double rate, int dr_mode);
int b200m_dr14_destroy (b200m_dr14* h);
int b200m_dr14_run_device (b200m_dr14* h, const float* d_in, size_t stride, uint32_t nfram, void* stream);   /* rows: inst * n_channels + c */
int b200m_dr14_run_host (b200m_dr14* h, const float* in, size_t stride, uint32_t nfram);
int b200m_dr14_reset (b200m_dr14* h, void* stream);                                       /* reset_peaks, every instance */
int b200m_dr14_results (b200m_dr14* h, b200m_dr14_result* out, void* stream);
int b200m_dr14_histogram (b200m_dr14* h, uint32_t inst, uint32_t chan, uint32_t* hist8000, void* stream);   /* hist[c] (:46,309-311) */

/* ======================================================================================
 * Stereo correlation bank — replaces LV2M::Stcorrdsp (jmeters/stcorrdsp.h:27-55) as driven by
 * cor_run (src/meters.cc:511-536) and xfer_run (src/xfer.c:248-251).
 * ====================================================================================== */
typedef struct b200m_cor b200m_cor;
int b200m_cor_create (b200m_cor** out, int device, uint32_t n_inst, int fsamp, float flp, float tcf);
int b200m_cor_destroy (b200m_cor* h);
int b200m_cor_process_device (b200m_cor* h, const float* d_in, size_t stride, uint32_t nfram, void* stream);
int b200m_cor_process_host (b200m_cor* h, const float* in, size_t stride, uint32_t nfram);
int b200m_cor_results (b200m_cor* h, float* out, void* stream);           /* Stcorrdsp::read (:79-82) */
/* B200M_PREC_EXACT (default): the five recurrences run serially in time, one lane per pair, bit-identical to the reference.
 * B200M_PREC_FMA: time-parallel evaluation -- the recurrences are linear one-pole filters, so a warp owns ONE pair, its lanes take
 * consecutive time segments and an affine warp scan stitches them: 32x more parallelism for small banks (2048 pairs are 64 warps
 * in exact mode); the correlation stays within 1e-5 of the reference (measured ~1e-7). */
int b200m_cor_set_precision (b200m_cor* h, int mode);
int b200m_cor_state (b200m_cor* h, float* state5, void* stream);          /* [n][5] zl zr zlr zll zrr */
int b200m_cor_coeffs (const b200m_cor* h, float w[2]);

/* ======================================================================================
 * Needle-meter ballistics bank (SURVEY §8f rank 3) — replaces LV2M::Vumeterdsp (jmeters/vumeterdsp.cc:45-93),
 * Iec1ppmdsp / Iec2ppmdsp (jmeters/iec1ppmdsp.cc, iec2ppmdsp.cc :47-99) and Msppmdsp (jmeters/msppmdsp.cc:50-143)
 * as driven by run() and bbcm_run() (src/meters.cc:298-331,552-589).
 * kind VU / IEC1 / IEC2: n_units mono meters (row i = meter i).  kind MS: n_units stereo pairs (rows 2i, 2i+1),
 * two meters per pair, M = processM at index 2i, S = processS at index 2i+1.
 * ====================================================================================== */
typedef struct b200m_ppm b200m_ppm;
enum { B200M_PPM_VU = 0, B200M_PPM_IEC1 = 1, B200M_PPM_IEC2 = 2, B200M_PPM_MS = 3 };
int b200m_ppm_create (b200m_ppm** out, int device, uint32_t n_units, float fsamp, int kind);
int b200m_ppm_destroy (b200m_ppm* h);
int b200m_ppm_set_gain (b200m_ppm* h, float db_m, float db_s);       /* Msppmdsp::set_gain of the M and S meters (default -6, -6) */
int b200m_ppm_process_device (b200m_ppm* h, const float* d_in, size_t stride, uint32_t nfram, void* stream);
int b200m_ppm_process_host (b200m_ppm* h, const float* in, size_t stride, uint32_t nfram);
int b200m_ppm_read_device (b200m_ppm* h, void* stream);                /* read(): _res = true, value = _g * _m */
int b200m_ppm_results (b200m_ppm* h, float* out, void* stream);        /* one float per meter */
int b200m_ppm_state (b200m_ppm* h, float* state4, void* stream);       /* per meter: z1 z2 m res */
int b200m_design_ppm (int kind, float fsamp, float w[4]);              /* w1 w2 w3 g (VU: w 0 0 g) */

/* ======================================================================================
 * Bit-meter and signal-distribution-histogram banks (SURVEY §8f rank 1), N mono instances each.
 * bit-meter: float_stats + the acquisition / ~5 fps window logic of bim_run (src/bitmeter.c:63-105,248-327);
 *   results = int32 histS[584] (layout src/uris.h:52-60), counters {zero,pos,nan,inf,den}, {min,max}, integration time.
 * SigDistHist: the sample loop of sdh_run (src/sigdistlv2.c:287-327): int32 histS[361], {max count, peak bin},
 *   {sum, running mean, running variance accumulator} in double, integration time.
 * Controls mirror the plugins' CTL_* messages (src/uris.h:187-203).
 * ====================================================================================== */
typedef struct b200m_bim b200m_bim;
typedef struct b200m_sdh b200m_sdh;
enum { B200M_CTL_START = 1, B200M_CTL_PAUSE = 2, B200M_CTL_RESET = 3, B200M_CTL_AVERAGE = 4, B200M_CTL_WINDOWED = 5 };
int b200m_bim_create (b200m_bim** out, int device, uint32_t n_inst, double rate);
int b200m_bim_destroy (b200m_bim* h);
int b200m_bim_control (b200m_bim* h, int cmd, void* stream);
int b200m_bim_run_device (b200m_bim* h, const float* d_in, size_t stride, uint32_t nfram, void* stream);
int b200m_bim_run_host (b200m_bim* h, const float* in, size_t stride, uint32_t nfram);
int b200m_bim_results (b200m_bim* h, uint32_t inst, int32_t* hist584, int32_t* cnt5, float* minmax2, int64_t* integration_time, void* stream);
/* 1 if the last run closed a ~5 fps window (self->radar_resync >= fps_limit, src/bitmeter.c:264-267,293); the statistics
 * as they stood at that moment -- what bim_run publishes in its bim_stats message before the windowed-mode bim_clear
 * (:269-291,323-325) -- stay readable through b200m_bim_published until the next window closes */
int b200m_bim_window_closed (const b200m_bim* h);
int b200m_bim_published (b200m_bim* h, uint32_t inst, int32_t* hist584, int32_t* cnt5, float* minmax2, int64_t* integration_time, void* stream);
int b200m_sdh_create (b200m_sdh** out, int device, uint32_t n_inst, double rate);
int b200m_sdh_destroy (b200m_sdh* h);
int b200m_sdh_control (b200m_sdh* h, int cmd, void* stream);
int b200m_sdh_run_device (b200m_sdh* h, const float* d_in, size_t stride, uint32_t nfram, void* stream);
int b200m_sdh_run_host (b200m_sdh* h, const float* in, size_t stride, uint32_t nfram);
int b200m_sdh_results (b200m_sdh* h, uint32_t inst, int32_t* hist361, int32_t* max_peak2, double* avg_tmp_var3, int64_t* integration_time, void* stream);

/* ======================================================================================
 * 30-band 1/3-octave spectrum bank — replaces spectrum_instantiate / spectrum_run
 * (src/spectrumlv2.c:73-121,159-257) over bandpass_setup / bandpass_process (src/spectr.c:68-206).
 * ====================================================================================== */
typedef struct b200m_spec b200m_spec;
int b200m_spec_create (b200m_spec** out, int device, uint32_t n_inst, uint32_t nchan, double rate);
int b200m_spec_destroy (b200m_spec* h);
/* one spectrum_run(): speed = *port 60, reset = *port 61 (same value for every instance) */
int b200m_spec_process_device (b200m_spec* h, const float* d_in, size_t stride, uint32_t nfram, float speed, float reset, void* stream);
int b200m_spec_process_host (b200m_spec* h, const float* in, size_t stride, uint32_t nfram, float speed, float reset);
/* B200M_PREC_EXACT (default): the reference's fp64 rounding sequence, ports bit-identical.  B200M_PREC_FMA: fused multiply-adds in the
 * biquad cascade (25 instead of 39 fp64 instructions per frame and band); band levels within +-1e-4 dB (measured ~1e-12 dB). */
int b200m_spec_set_precision (b200m_spec* h, int mode);
/* ports 0..59 of every instance: 30 band levels (dB), 30 band maxima (dB) */
int b200m_spec_results (b200m_spec* h, float* out60, void* stream);
int b200m_spec_state (b200m_spec* h, uint32_t inst, double* z360, float* val30, float* max30, void* stream);
int b200m_spec_coeffs (const b200m_spec* h, double* W1080);              /* [30][6][6] a0 a1 a2 b0 b1 b2 */

/* ======================================================================================
 * Phasewheel FFT analysis bank — replaces fftx_init / fftx_run / ft_analyze (gui/fft.c:208-361)
 * for both channels plus process_audio (gui/phasewheel.c:1307-1342).
 * ====================================================================================== */
typedef struct b200m_pw b200m_pw;
/* fft_bins: the GUI's selector values (gui/phasewheel.c:1108-1116): 64, 128, ... 8192 and 6144 (window = 2 * fft_bins) */
int b200m_pw_create (b200m_pw** out, int device, uint32_t n_inst, uint32_t fft_bins, double rate);
int b200m_pw_destroy (b200m_pw* h);
/* which GUI's process_audio follows the FFTs: PHASEWHEEL (default; phase difference, level, peak: gui/phasewheel.c:1307-1342)
 * or STEREOSCOPE (gui/stereoscope.c:705-741: smoothed lr[] returned in `phase`, smoothed level[]; db_thresh fixed at 1e-20,
 * no peak; the reference GUI defaults to fft_bins 512).  Re-initialises the outputs like the GUI's reinitialize_fft. */
enum { B200M_PW_PHASEWHEEL = 0, B200M_PW_STEREOSCOPE = 1 };
int b200m_pw_set_mode (b200m_pw* h, int mode);
/* returns (via *fired) whether this call completed an analysis (fftx_run()==0) */
int b200m_pw_process_device (b200m_pw* h, const float* d_in, size_t stride, uint32_t nfram, float db_thresh, int* fired, void* stream);
int b200m_pw_process_host (b200m_pw* h, const float* in, size_t stride, uint32_t nfram, float db_thresh, int* fired);
/* phase[n_inst][fft_bins], level[n_inst][fft_bins], peak[n_inst] (ui->phase/level/peak) */
int b200m_pw_results (b200m_pw* h, float* phase, float* level, float* peak, void* stream);
/* ft->power / ft->phase of both channels of the last analysis (gui/fft.c:163-180), kept only while b200m_pw_debug_capture is on */
int b200m_pw_debug_capture (b200m_pw* h, int enable);
int b200m_pw_raw (b200m_pw* h, uint32_t inst, float* powL, float* powR, float* phL, float* phR, void* stream);
/* Fused feed: with a correlation bank of n_inst pairs attached, b200m_pw_process_* also runs Stcorrdsp::process of that bank on the
 * same block (what xfer_run does per cycle, src/xfer.c:248-251) in ONE kernel that reads the input once: the block is staged in
 * shared memory for the correlation recurrences and appended to the FFT ring from there.  Read the correlation with
 * b200m_cor_results; do not call b200m_cor_process_* on an attached bank.  cor = NULL detaches. */
int b200m_pw_attach_cor (b200m_pw* h, b200m_cor* cor);
/* device pointers of the result planes, for callers that keep the spectra on the GPU */
int b200m_pw_device_results (b200m_pw* h, const float** d_phase, const float** d_level, const float** d_peak);

/* ======================================================================================
 * LV2 facade: the library also exports `lv2_descriptor (index)` (the one symbol of the reference's meters.so,
 * src/meters.cc:739-792) serving all 38 plugin URIs.  b200m_lv2_gon_layout lists, for tests, the offsets of the goniometer
 * instance struct that the reference GUI reads through instance-access (src/goniometer.h:113-169): rb, ui_active,
 * rb_overrun, s_sfact, s_linewidth, input, rate, ntfy, msg_thread_lock, map, sizeof; returns how many there are.
 * ====================================================================================== */
int b200m_lv2_gon_layout (size_t* out, int n);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* B200METERS_H */
