// r128.cu — the EBUr128 plugin's audio cycle for N stereo instances: EBU R128 loudness + optional dBTP.
//
// Mirrors what ebur128_run does between its atom parsing and atom forging (src/ebulv2.cc:341-367):
//   ebu->process (n, {inL, inR});  if (dbtp_enable) { mtr[0]->process_max (inL); mtr[1]->process_max (inR); }
//   lm/mm/ls/ms/il/rn/rx getters;  tp = coef_to_db (max (mtr[0]->read (), mtr[1]->read ()));  tp_max = max (tp_max, tp)
// It composes the EBU bank (ebu.cu) and the true-peak bank (tpk.cu) over ONE host->device copy of the block.
#include <math.h>
#include <stdlib.h>
#include "common.cuh"

namespace b200m {

// coef_to_db (src/ebulv2.cc:227-230) and the tp_max hold (:360-367) run in the epilogue of tpk_kernel<TPMAX> (tpk.cu)
__global__ void r128_fill_kernel (int n, float* p, float v) { const int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }

}  // namespace b200m

// sliced process entry points of the two banks (ebu.cu, tpk.cu)
extern "C" int ebu_process_sliced (b200m_ebu* h, const float* d_in, size_t stride, uint32_t nfram, cudaStream_t st, int nsl, const uint32_t* bounds, cudaEvent_t* ready,
                                   int (*after_k1) (void*), void* after_arg);
int tpk_process_sliced (b200m_tpk* h, const float* d_in, size_t stride, uint32_t nfram, uint32_t tp_mode, cudaStream_t st, int nsl, const uint32_t* bounds, cudaEvent_t* ready,
                        float* r128_tpmax, bool pdl, const void* dr);
namespace b200m {                     // PCM ingest (pcm.cu)
int pcm_check_fmt (uint32_t fmt);
int pcm_sample_bytes (uint32_t fmt);
int pcm_convert_launch (const void* d_src, uint32_t fmt, uint32_t nchan, uint32_t n_inst, size_t src_stride, uint32_t nfram,
                        float* d_dst, size_t dst_stride, cudaStream_t st);
}

using namespace b200m;

constexpr int R128_SLICES = 8;        // maximum; default 4 (B200M_R128_SLICES)

struct b200m_r128 {
    int device; uint32_t n_inst; int dbtp;
    b200m_ebu* ebu = nullptr; b200m_tpk* tpk = nullptr;
    float* d_tpmax = nullptr;
    // own: EBU kernels + joins (host path);  side: true-peak kernels (run concurrently with the latency-bound EBU
    // kernel);  copy: host->device slices, so that the copy of slice s+1 overlaps the kernels of slice s
    cudaStream_t own = nullptr, side = nullptr, copy = nullptr;
    cudaEvent_t ev_tp = nullptr, ev_done = nullptr, ev_ready[R128_SLICES] = {nullptr};
    HostStage stage; bool last_host = false; int concurrent = 1, slices = R128_SLICES;
    // PCM host path: raw bytes of the block as copied, and the stream that converts slice s once ev_copied[s] has fired,
    // so that no conversion queues in front of a copy or of an earlier slice's kernels (created on first use)
    uint8_t* d_raw = nullptr; size_t raw_bytes = 0;
    cudaStream_t cvt = nullptr;
    cudaEvent_t ev_copied[R128_SLICES] = {nullptr};
};

static int env_int (const char* name, int dflt) { const char* v = getenv (name); return v ? atoi (v) : dflt; }

struct R128Step { b200m_r128* h; const float* d_in; size_t stride; uint32_t nfram; cudaStream_t st; const uint32_t* bc; };

// device path: the true-peak kernel goes onto the caller's stream right behind the first K-weighting launch, with
// programmatic dependent launch, so that the two kernels share the SMs (see r128_run)
static int r128_tp_behind_k1 (void* p)
{
    R128Step* a = (R128Step*)p;
    return tpk_process_sliced (a->h->tpk, a->d_in, a->stride, a->nfram, B200M_TP_MODE_MAX, a->st, 1, a->bc, nullptr, a->h->d_tpmax, true, nullptr);
}

static int r128_run (b200m_r128* h, const float* d_in, size_t stride, uint32_t nfram, cudaStream_t st, int nsl, cudaEvent_t* ready)
{
    uint32_t bi[R128_SLICES + 1], bc[R128_SLICES + 1];
    for (int s = 0; s <= nsl; ++s) { bi[s] = (uint32_t)((uint64_t)h->n_inst * s / nsl); bc[s] = 2 * bi[s]; }
    // The K-weighting kernel is latency bound on 4 warps per SM and the true-peak kernel issue bound: run together they
    // cost little more than the true-peak kernel alone, PROVIDED the K-weighting CTAs are resident first (104 KB of shared
    // memory each: they do not fit once the true-peak CTAs fill an SM).
    //  * device path (B200M_R128_CONCURRENT >= 2): same stream; the K-weighting kernel triggers programmatic launch
    //    completion at its start and the true-peak kernel is launched behind it with the programmatic-serialization
    //    attribute -> deterministic order, no events.  The true-peak kernel's epilogue does read() x 2 + coef_to_db + the
    //    tp_max hold per instance and ends with griddepcontrol.wait, so everything queued behind it is ordered after both.
    //  * sliced host path (>= 1): true-peak kernels on the side stream, each slice behind its copy event.
    // B200M_R128_CONCURRENT=0 serialises everything on one stream.
    const bool pdl = h->dbtp && h->concurrent >= 2 && !ready;
    const bool conc = h->dbtp && h->concurrent >= 1 && ready;
    R128Step step = {h, d_in, stride, nfram, st, bc};
    if (int rc = ebu_process_sliced (h->ebu, d_in, stride, nfram, st, nsl, bi, ready, pdl ? r128_tp_behind_k1 : nullptr, &step)) return rc;
    if (h->dbtp) {
        if (!pdl) {
            if (int rc = tpk_process_sliced (h->tpk, d_in, stride, nfram, B200M_TP_MODE_MAX, conc ? h->side : st, nsl, bc, conc ? ready : nullptr, h->d_tpmax, false, nullptr)) return rc;
            if (conc) { B200M_CUDA (cudaEventRecord (h->ev_tp, h->side)); B200M_CUDA (cudaStreamWaitEvent (st, h->ev_tp, 0)); }
        }
    } else {
        r128_fill_kernel<<<(h->n_inst + 255) / 256, 256, 0, st>>> ((int)h->n_inst, h->d_tpmax, -INFINITY);   // :365-366
        B200M_LAUNCHED (1);
    }
    B200M_CUDA (cudaGetLastError ());
    return 0;
}

extern "C" {

int b200m_r128_create (b200m_r128** out, int device, uint32_t n_inst, float fsamp, int dbtp_enable)
{
    if (!out) return set_err (B200M_E_INVAL, "NULL out pointer");
    *out = nullptr;
    b200m_r128* h = new (std::nothrow) b200m_r128;
    if (!h) return set_err (B200M_E_NOMEM, "host allocation failed");
    h->device = device; h->n_inst = n_inst; h->dbtp = dbtp_enable ? 1 : 0;
    h->concurrent = env_int ("B200M_R128_CONCURRENT", 2);      // 0: serial, 1: sliced host path only, 2: device path too
    h->slices = env_int ("B200M_R128_SLICES", 4);
    if (h->slices < 1) h->slices = 1;
    if (h->slices > R128_SLICES) h->slices = R128_SLICES;
    int rc = b200m_ebu_create (&h->ebu, device, n_inst, 2, fsamp);                 // ebu->init (2, rate), src/ebulv2.cc:190
    if (!rc) rc = b200m_tpk_create (&h->tpk, device, 2 * n_inst, fsamp, B200M_TPK_TRUEPEAK);   // 2 x TruePeakdsp, :192-196
    if (!rc) {
        DeviceGuard g (device);
        cudaError_t e = cudaMalloc ((void**)&h->d_tpmax, n_inst * sizeof (float));
        for (cudaStream_t* sp : {&h->own, &h->side, &h->copy}) if (e == cudaSuccess) e = cudaStreamCreateWithFlags (sp, cudaStreamNonBlocking);
        for (cudaEvent_t* ep : {&h->ev_tp, &h->ev_done}) if (e == cudaSuccess) e = cudaEventCreateWithFlags (ep, cudaEventDisableTiming);
        for (int s = 0; s < R128_SLICES; ++s) if (e == cudaSuccess) e = cudaEventCreateWithFlags (&h->ev_ready[s], cudaEventDisableTiming);
        if (e == cudaSuccess) {
            r128_fill_kernel<<<(n_inst + 255) / 256, 256>>> ((int)n_inst, h->d_tpmax, -INFINITY);
            B200M_LAUNCHED (1);
            e = cudaDeviceSynchronize ();
        }
        if (e != cudaSuccess) rc = cuda_fail (e, "r128_create", __FILE__, __LINE__);
    }
    if (rc) { b200m_r128_destroy (h); return rc; }
    *out = h;
    return 0;
}

int b200m_r128_destroy (b200m_r128* h)
{
    if (!h) return 0;
    b200m_ebu_destroy (h->ebu); b200m_tpk_destroy (h->tpk);
    DeviceGuard g (h->device);
    cudaDeviceSynchronize ();
    cudaFree (h->d_tpmax); h->stage.release ();
    if (h->d_raw) cudaFree (h->d_raw);
    for (cudaStream_t sp : {h->own, h->side, h->copy, h->cvt}) if (sp) cudaStreamDestroy (sp);
    for (cudaEvent_t ep : {h->ev_tp, h->ev_done}) if (ep) cudaEventDestroy (ep);
    for (int s = 0; s < R128_SLICES; ++s) {
        if (h->ev_ready[s]) cudaEventDestroy (h->ev_ready[s]);
        if (h->ev_copied[s]) cudaEventDestroy (h->ev_copied[s]);
    }
    delete h;
    return 0;
}

int b200m_r128_control (b200m_r128* h, int32_t inst, int cmd, void* stream)
{
    if (!h) return set_err (B200M_E_INVAL, "NULL handle");
    void* st = h->last_host ? (void*)h->own : stream;
    switch (cmd) {
    case B200M_R128_START: return b200m_ebu_integr_start (h->ebu, inst, st);
    case B200M_R128_PAUSE: return b200m_ebu_integr_pause (h->ebu, inst, st);
    case B200M_R128_RESET:                                  // ebu_reset (src/ebulv2.cc:45-61): integr_reset + tp_max = -inf
    case B200M_R128_CLEAR_TPMAX: {                          // tp_max = -inf alone: what a cycle with dBTP disabled leaves behind (:365-366)
        if (inst >= (int32_t)h->n_inst) return set_err (B200M_E_INVAL, "bad instance %d", inst);
        DeviceGuard g (h->device);
        const int first = inst < 0 ? 0 : inst, cnt = inst < 0 ? (int)h->n_inst : 1;
        r128_fill_kernel<<<(cnt + 255) / 256, 256, 0, (cudaStream_t)st>>> (cnt, h->d_tpmax + first, -INFINITY);
        B200M_LAUNCHED (1);
        B200M_CUDA (cudaGetLastError ());
        return cmd == B200M_R128_RESET ? b200m_ebu_integr_reset (h->ebu, inst, st) : 0;
    }
    case B200M_R128_CLEAR: {                                // a fresh instance in this slot (shared banks: a plugin left, another may join)
        if (inst < 0 || inst >= (int32_t)h->n_inst) return set_err (B200M_E_INVAL, "bad instance %d", inst);
        DeviceGuard g (h->device);
        r128_fill_kernel<<<1, 32, 0, (cudaStream_t)st>>> (1, h->d_tpmax + inst, -INFINITY);
        B200M_LAUNCHED (1);
        B200M_CUDA (cudaGetLastError ());
        if (int rc = b200m_ebu_clear (h->ebu, inst, st)) return rc;
        if (int rc = b200m_tpk_clear (h->tpk, 2 * inst, st)) return rc;
        return b200m_tpk_clear (h->tpk, 2 * inst + 1, st);
    }
    default: return set_err (B200M_E_INVAL, "unknown control %d", cmd);
    }
}

int b200m_r128_run_device (b200m_r128* h, const float* d_in, size_t stride, uint32_t nfram, void* stream)
{
    if (int rc = check_block_args (h, d_in, stride, nfram)) return rc;
    DeviceGuard g (h->device);
    h->last_host = false;
    return r128_run (h, d_in, stride, nfram, (cudaStream_t)stream, 1, nullptr);
}

int b200m_r128_run_host (b200m_r128* h, const float* in, size_t stride, uint32_t nfram)
{
    if (int rc = check_block_args (h, in, stride, nfram)) return rc;
    DeviceGuard g (h->device);
    B200M_ENTER_HOST_PATH (h);
    const size_t nch = (size_t)2 * h->n_inst;
    if (h->stage.ensure (nch, nfram)) return set_err (B200M_E_NOMEM, "staging buffer allocation failed");
    // the staging buffer is single: the next copy may only start when the previous cycle's kernels have read it
    if (h->last_host) B200M_CUDA (cudaStreamWaitEvent (h->copy, h->ev_done, 0));
    const int nsl = h->n_inst >= 64 ? h->slices : 1;
    for (int s = 0; s < nsl; ++s) {
        const size_t r0 = 2 * ((uint64_t)h->n_inst * s / nsl), r1 = 2 * ((uint64_t)h->n_inst * (s + 1) / nsl);
        if (stride == nfram && h->stage.cap == nfram)          // both sides dense: one contiguous DMA per slice (faster than 4 KB rows)
            B200M_CUDA (cudaMemcpyAsync (h->stage.d + r0 * h->stage.cap, in + r0 * stride, (r1 - r0) * (size_t)nfram * sizeof (float), cudaMemcpyHostToDevice, h->copy));
        else
            B200M_CUDA (cudaMemcpy2DAsync (h->stage.d + r0 * h->stage.cap, h->stage.cap * sizeof (float), in + r0 * stride, stride * sizeof (float),
                                           (size_t)nfram * sizeof (float), r1 - r0, cudaMemcpyHostToDevice, h->copy));
        B200M_CUDA (cudaEventRecord (h->ev_ready[s], h->copy));
    }
    h->last_host = true;
    if (int rc = r128_run (h, h->stage.d, h->stage.cap, nfram, h->own, nsl, h->ev_ready)) return rc;
    B200M_CUDA (cudaEventRecord (h->ev_done, h->own));
    return 0;
}

static int check_pcm_args (b200m_r128* h, const void* in, uint32_t fmt, size_t stride, uint32_t nfram)
{
    if (int rc = pcm_check_fmt (fmt)) return rc;
    if (int rc = check_block_args (h, in, stride, nfram)) return rc;
    const int bps = pcm_sample_bytes (fmt);
    if ((uintptr_t)in % (bps == 3 ? 1 : bps)) return set_err (B200M_E_INVAL, "input not aligned to its sample type");
    return 0;
}

int b200m_r128_run_device_pcm (b200m_r128* h, const void* d_in, uint32_t fmt, size_t stride, uint32_t nfram, void* stream)
{
    if (int rc = check_pcm_args (h, d_in, fmt, stride, nfram)) return rc;
    if (fmt == (B200M_PCM_F32 | B200M_PCM_PLANAR)) return b200m_r128_run_device (h, (const float*)d_in, stride, nfram, stream);
    DeviceGuard g (h->device);
    const cudaStream_t st = (cudaStream_t)stream;
    if (h->stage.ensure ((size_t)2 * h->n_inst, nfram)) return set_err (B200M_E_NOMEM, "conversion buffer allocation failed");
    // the float rows reuse the host path's staging buffer: after a host-path cycle, the conversion waits for its kernels
    if (h->last_host) B200M_CUDA (cudaStreamWaitEvent (st, h->ev_done, 0));
    h->last_host = false;
    if (int rc = pcm_convert_launch (d_in, fmt, 2, h->n_inst, stride, nfram, h->stage.d, h->stage.cap, st)) return rc;
    return r128_run (h, h->stage.d, h->stage.cap, nfram, st, 1, nullptr);
}

int b200m_r128_run_host_pcm (b200m_r128* h, const void* in, uint32_t fmt, size_t stride, uint32_t nfram)
{
    if (int rc = check_pcm_args (h, in, fmt, stride, nfram)) return rc;
    if (fmt == (B200M_PCM_F32 | B200M_PCM_PLANAR)) return b200m_r128_run_host (h, (const float*)in, stride, nfram);
    DeviceGuard g (h->device);
    B200M_ENTER_HOST_PATH (h);
    const size_t nch = (size_t)2 * h->n_inst;
    if (h->stage.ensure (nch, nfram)) return set_err (B200M_E_NOMEM, "staging buffer allocation failed");
    if (!h->cvt) {
        B200M_CUDA (cudaStreamCreateWithFlags (&h->cvt, cudaStreamNonBlocking));
        for (int s = 0; s < R128_SLICES; ++s) B200M_CUDA (cudaEventCreateWithFlags (&h->ev_copied[s], cudaEventDisableTiming));
    }
    // one segment = a channel row (planar) or the frames of one instance (interleaved); on the device the segments are dense
    const bool il = (fmt & B200M_PCM_INTERLEAVED) != 0;
    const size_t bps = (size_t)pcm_sample_bytes (fmt), spi = il ? 1 : 2;          // segments per instance
    const size_t seg_bytes = (size_t)nfram * bps * (il ? 2 : 1), src_pitch = stride * bps * (il ? 2 : 1);
    const size_t need = seg_bytes * h->n_inst * spi;
    if (need > h->raw_bytes) {                                  // grown on demand, never shrunk
        if (h->d_raw) { B200M_CUDA (cudaStreamSynchronize (h->own)); cudaFree (h->d_raw); h->d_raw = nullptr; h->raw_bytes = 0; }
        B200M_CUDA (cudaMalloc (&h->d_raw, need));
        h->raw_bytes = need;
    }
    // single buffers, raw and float: the next copy may only start when the previous cycle's conversions and kernels have
    // read them (ev_done follows both: the kernels of every slice waited for its conversion)
    if (h->last_host) B200M_CUDA (cudaStreamWaitEvent (h->copy, h->ev_done, 0));
    const int nsl = h->n_inst >= 64 ? h->slices : 1;
    for (int s = 0; s < nsl; ++s) {
        const size_t i0 = (uint64_t)h->n_inst * s / nsl, i1 = (uint64_t)h->n_inst * (s + 1) / nsl;
        const size_t g0 = i0 * spi, ng = (i1 - i0) * spi;
        if (stride == nfram)                                    // the host rows are contiguous: one DMA per slice
            B200M_CUDA (cudaMemcpyAsync (h->d_raw + g0 * seg_bytes, (const uint8_t*)in + g0 * src_pitch, ng * seg_bytes, cudaMemcpyHostToDevice, h->copy));
        else
            B200M_CUDA (cudaMemcpy2DAsync (h->d_raw + g0 * seg_bytes, seg_bytes, (const uint8_t*)in + g0 * src_pitch, src_pitch,
                                           seg_bytes, ng, cudaMemcpyHostToDevice, h->copy));
        B200M_CUDA (cudaEventRecord (h->ev_copied[s], h->copy));
        B200M_CUDA (cudaStreamWaitEvent (h->cvt, h->ev_copied[s], 0));
        if (int rc = pcm_convert_launch (h->d_raw + g0 * seg_bytes, fmt, 2, (uint32_t)(i1 - i0), nfram, nfram,
                                         h->stage.d + 2 * i0 * h->stage.cap, h->stage.cap, h->cvt)) return rc;
        B200M_CUDA (cudaEventRecord (h->ev_ready[s], h->cvt));
    }
    h->last_host = true;
    if (int rc = r128_run (h, h->stage.d, h->stage.cap, nfram, h->own, nsl, h->ev_ready)) return rc;
    B200M_CUDA (cudaEventRecord (h->ev_done, h->own));
    return 0;
}

int b200m_r128_results (b200m_r128* h, b200m_ebu_result* ebu_out, float* tp_max_db, void* stream)
{
    if (!h) return set_err (B200M_E_INVAL, "NULL handle");
    DeviceGuard g (h->device);
    cudaStream_t st = h->last_host ? h->own : (cudaStream_t)stream;
    if (tp_max_db) B200M_CUDA (cudaMemcpyAsync (tp_max_db, h->d_tpmax, h->n_inst * sizeof (float), cudaMemcpyDeviceToHost, st));
    if (ebu_out) return b200m_ebu_results (h->ebu, ebu_out, st);
    B200M_CUDA (cudaStreamSynchronize (st));
    return 0;
}

int b200m_r128_set_dbtp (b200m_r128* h, int enable)
{
    if (!h) return set_err (B200M_E_INVAL, "NULL handle");
    h->dbtp = enable ? 1 : 0;                              // takes effect with the next run: self->dbtp_enable (src/ebulv2.cc:316-317,344-347)
    return 0;
}

int b200m_r128_set_precision (b200m_r128* h, int mode)
{
    if (!h) return set_err (B200M_E_INVAL, "NULL handle");
    return b200m_tpk_set_precision (h->tpk, mode);         // the EBU R128 part is always exact: it feeds the integer histograms
}

int b200m_r128_histogram (b200m_r128* h, uint32_t inst, int32_t* hist_M, int32_t* hist_S, void* stream)
{
    if (!h) return set_err (B200M_E_INVAL, "NULL handle");
    return b200m_ebu_histogram (h->ebu, inst, hist_M, hist_S, h->last_host ? (void*)h->own : stream);
}

// snapshot = [u64 ebu bytes][u64 tpk bytes][ebu blob][tpk blob][tp_max floats][dbtp flag]
size_t b200m_r128_snapshot_size (b200m_r128* h)
{
    if (!h) return 0;
    return 16 + b200m_ebu_snapshot_size (h->ebu) + b200m_tpk_snapshot_size (h->tpk) + (((size_t)h->n_inst * 4 + 15) & ~size_t (15)) + 16;
}

int b200m_r128_snapshot (b200m_r128* h, void* buf, size_t bytes, void* stream)
{
    if (!h || !buf || bytes < b200m_r128_snapshot_size (h)) return set_err (B200M_E_INVAL, "bad argument / buffer too small");
    DeviceGuard g (h->device);
    void* st = h->last_host ? (void*)h->own : stream;
    const uint64_t eb = b200m_ebu_snapshot_size (h->ebu), tb = b200m_tpk_snapshot_size (h->tpk);
    uint8_t* o = (uint8_t*)buf;
    memcpy (o, &eb, 8); memcpy (o + 8, &tb, 8); o += 16;
    if (int rc = b200m_ebu_snapshot (h->ebu, o, eb, st)) return rc;
    o += eb;
    if (int rc = b200m_tpk_snapshot (h->tpk, o, tb, st)) return rc;
    o += tb;
    B200M_CUDA (cudaMemcpyAsync (o, h->d_tpmax, (size_t)h->n_inst * 4, cudaMemcpyDeviceToHost, (cudaStream_t)st));
    B200M_CUDA (cudaStreamSynchronize ((cudaStream_t)st));
    o += ((size_t)h->n_inst * 4 + 15) & ~size_t (15);
    const int32_t fl[4] = {h->dbtp, 0, 0, 0};
    memcpy (o, fl, 16);
    return 0;
}

int b200m_r128_restore (b200m_r128* h, const void* buf, size_t bytes, void* stream)
{
    if (!h || !buf || bytes < b200m_r128_snapshot_size (h)) return set_err (B200M_E_INVAL, "bad argument / buffer too small");
    DeviceGuard g (h->device);
    void* st = h->last_host ? (void*)h->own : stream;
    uint64_t eb, tb;
    const uint8_t* o = (const uint8_t*)buf;
    memcpy (&eb, o, 8); memcpy (&tb, o + 8, 8); o += 16;
    if (eb != b200m_ebu_snapshot_size (h->ebu) || tb != b200m_tpk_snapshot_size (h->tpk)) return set_err (B200M_E_INVAL, "snapshot does not match this bank");
    if (int rc = b200m_ebu_restore (h->ebu, o, eb, st)) return rc;
    o += eb;
    if (int rc = b200m_tpk_restore (h->tpk, o, tb, st)) return rc;
    o += tb;
    B200M_CUDA (cudaMemcpyAsync (h->d_tpmax, o, (size_t)h->n_inst * 4, cudaMemcpyHostToDevice, (cudaStream_t)st));
    B200M_CUDA (cudaStreamSynchronize ((cudaStream_t)st));
    o += ((size_t)h->n_inst * 4 + 15) & ~size_t (15);
    int32_t fl[4]; memcpy (fl, o, 16);
    h->dbtp = fl[0] ? 1 : 0;
    return 0;
}

b200m_ebu* b200m_r128_ebu (b200m_r128* h) { return h ? h->ebu : nullptr; }
b200m_tpk* b200m_r128_tpk (b200m_r128* h) { return h ? h->tpk : nullptr; }

}  // extern "C"
