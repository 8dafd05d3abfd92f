// pcm.cu — PCM ingest: interleaved or planar int16 / packed int24 / int32 / float32 blocks -> the dense planar float32
// rows every bank reads.  Decoders, capture cards and file readers hand out interleaved integer PCM; converting it here
// instead of on the host saves the host a pass over the block and, for 16- and 24-bit input, PCIe bytes.
//
// Value handed to the meters (include/b200meters.h):  F32 the bits unchanged;  S16 (float)x * 2^-15;  S24 sign-extended,
// then (float)x * 2^-23 (both exact);  S32 __int2float_rn (x) * 2^-31 (round to nearest even, as the host's (float)x).
#include "common.cuh"

namespace b200m {

constexpr int PCM_THREADS = 256;
constexpr int PCM_TILE_FLOATS = 4096;    // planar floats one CTA emits at most: frames per tile = 4096 / nchan

__host__ __device__ constexpr int pcm_bytes (uint32_t type) { return type == B200M_PCM_S16 ? 2 : type == B200M_PCM_S24 ? 3 : 4; }

// frames per tile (a multiple of 4, so that every tile starts on a float4 of the destination row) and the padded row
// length of the planar tile in shared memory: rows 32/nchan words apart spread one warp's stores over the banks
static inline int pcm_tile_frames (int nchan) { return (PCM_TILE_FLOATS / nchan) & ~3; }
__host__ __device__ inline int pcm_row_pitch (int tf, int nchan) { return tf + 4 * ((8 + nchan - 1) / nchan); }

template <typename T> struct PcmSample;
template <> struct PcmSample<float>   { static B200M_DEV float get (const uint8_t* p) { return __uint_as_float (*(const uint32_t*)p); } };
template <> struct PcmSample<int16_t> { static B200M_DEV float get (const uint8_t* p) { return __fmul_rn (__int2float_rn (*(const int16_t*)p), 0x1p-15f); } };
template <> struct PcmSample<int32_t> { static B200M_DEV float get (const uint8_t* p) { return __fmul_rn (__int2float_rn (*(const int32_t*)p), 0x1p-31f); } };
struct s24_t { uint8_t b[3]; };                  // packed little-endian 24-bit sample (alignment 1)
template <> struct PcmSample<s24_t> {
    static B200M_DEV float get (const uint8_t* p) {
        const int32_t v = (int32_t)(((uint32_t)p[0] << 8) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 24)) >> 8;
        return __fmul_rn (__int2float_rn (v), 0x1p-23f);
    }
};

// One CTA = one tile of `tf` frames of one segment: a planar row (nchan = 1) or the interleaved frames of one instance.
//  1. the tile's contiguous source bytes -> shared memory, 16-byte loads for the aligned interior, byte loads for the
//     (at most 15-byte) head and tail; byte j of the tile lands at raw[mis + j], mis = the source's address mod 16, so
//     that the 16-byte chunks land aligned;
//  2. sample e = f * nchan + c of the tile is converted by thread e % 256 and stored to the planar tile pl[c][f];
//  3. each thread emits float4s of one channel row to global memory (scalar stores for a row's last < 4 frames).
// Reads: bytes_per_sample, writes: 4 bytes per sample; both coalesced.
template <typename T, bool INTERLEAVED>
__global__ void __launch_bounds__ (PCM_THREADS) pcm_to_planar_kernel (const uint8_t* __restrict__ src, size_t seg_pitch, int nchan_rt, int nfram, int tf,
                                                                       uint32_t div_magic, float* __restrict__ dst, size_t dst_stride)
{
    extern __shared__ __align__ (16) uint8_t smem[];
    constexpr int BPS = (int)sizeof (T);
    const int nchan = INTERLEAVED ? nchan_rt : 1;
    const int f0 = blockIdx.y * tf;
    const int nf = min (tf, nfram - f0);
    const int ne = nf * nchan;
    const int nbytes = ne * BPS;
    const int pitch = pcm_row_pitch (tf, nchan);
    float* pl = (float*)smem;                                                     // [nchan][pitch]
    uint8_t* raw = smem + (size_t)nchan * pitch * 4;                              // 16-byte aligned: pitch % 4 == 0
    const uint8_t* g = src + (size_t)blockIdx.x * seg_pitch + (size_t)f0 * nchan * BPS;

    const int mis = (int)((uintptr_t)g & 15);
    const int head = min ((16 - mis) & 15, nbytes);
    const int nvec = (nbytes - head) >> 4;
    const int tail = head + nvec * 16;
    for (int i = threadIdx.x; i < nvec; i += PCM_THREADS)
        *(int4*)(raw + mis + head + 16 * i) = __ldcs ((const int4*)(g + head) + i);
    if (threadIdx.x < head) raw[mis + threadIdx.x] = g[threadIdx.x];
    if (threadIdx.x < nbytes - tail) raw[mis + tail + threadIdx.x] = g[tail + threadIdx.x];
    __syncthreads ();

    for (int e = threadIdx.x; e < ne; e += PCM_THREADS) {
        int f = e, c = 0;
        if (INTERLEAVED && nchan > 1) { f = (int)__umulhi ((uint32_t)e, div_magic); c = e - f * nchan; }
        pl[c * pitch + f] = PcmSample<T>::get (raw + mis + e * BPS);
    }
    __syncthreads ();

    const int nq = nf >> 2;
    float* out = dst + (size_t)blockIdx.x * nchan * dst_stride + f0;
    for (int c = 0; c < nchan; ++c) {
        float* o = out + (size_t)c * dst_stride;
        const float* p = pl + c * pitch;
        for (int q = threadIdx.x; q < nq; q += PCM_THREADS) ((float4*)o)[q] = ((const float4*)p)[q];
        const int f = 4 * nq + (int)threadIdx.x;
        if (f < nf) o[f] = p[f];
    }
}

int pcm_check_fmt (uint32_t fmt)
{
    const uint32_t type = fmt & 15u, layout = fmt & ~15u;
    if (type > B200M_PCM_S32 || (layout != B200M_PCM_PLANAR && layout != B200M_PCM_INTERLEAVED))
        return set_err (B200M_E_INVAL, "bad PCM format code 0x%x", fmt);
    return 0;
}

int pcm_sample_bytes (uint32_t fmt) { return pcm_bytes (fmt & 15u); }

// Launches the conversion of n_inst x nchan channels; arguments checked by the caller.  dst must be 16-byte aligned with
// dst_stride % 4 == 0.
int pcm_convert_launch (const void* d_src, uint32_t fmt, uint32_t nchan, uint32_t n_inst, size_t src_stride, uint32_t nfram,
                        float* d_dst, size_t dst_stride, cudaStream_t st)
{
    const bool il = (fmt & B200M_PCM_INTERLEAVED) != 0;
    const int nc = il ? (int)nchan : 1;                             // planar: every channel row is a segment of its own
    const size_t nseg = il ? n_inst : (size_t)n_inst * nchan;
    const int bps = pcm_sample_bytes (fmt);
    const size_t seg_pitch = src_stride * nc * bps;
    const int tf = min (pcm_tile_frames (nc), (int)(nfram + 3) & ~3);
    const size_t smem = (size_t)nc * pcm_row_pitch (tf, nc) * 4 + ((size_t)tf * nc * bps + 16 + 15) / 16 * 16;
    const uint32_t magic = (uint32_t)((0x100000000ull + nc - 1) / nc);   // e / nc == umulhi (e, magic) for e < 2^32 / nc (nc > 1)
    if (nseg > 0x7fffffffu) return set_err (B200M_E_INVAL, "too many channels");
    dim3 grid ((unsigned)nseg, (nfram + tf - 1) / tf);
    const uint8_t* s = (const uint8_t*)d_src;
#define PCM_LAUNCH(T, IL) pcm_to_planar_kernel<T, IL><<<grid, PCM_THREADS, smem, st>>> (s, seg_pitch, nc, (int)nfram, tf, magic, d_dst, dst_stride)
    switch ((fmt & 15u) * 2 + (il ? 1 : 0)) {
    case 0: PCM_LAUNCH (float, false); break;    case 1: PCM_LAUNCH (float, true); break;
    case 2: PCM_LAUNCH (int16_t, false); break;  case 3: PCM_LAUNCH (int16_t, true); break;
    case 4: PCM_LAUNCH (s24_t, false); break;    case 5: PCM_LAUNCH (s24_t, true); break;
    case 6: PCM_LAUNCH (int32_t, false); break;  case 7: PCM_LAUNCH (int32_t, true); break;
    default: return set_err (B200M_E_INVAL, "bad PCM format code 0x%x", fmt);
    }
#undef PCM_LAUNCH
    B200M_LAUNCHED (1);
    B200M_CUDA (cudaGetLastError ());
    return 0;
}

}  // namespace b200m

using namespace b200m;

extern "C" int b200m_pcm_convert (int device, const void* d_src, uint32_t fmt, uint32_t nchan, uint32_t n_inst, size_t src_stride,
                                  uint32_t nfram, float* d_dst, size_t dst_stride, void* stream)
{
    if (int rc = pcm_check_fmt (fmt)) return rc;
    if (!d_src || !d_dst) return set_err (B200M_E_INVAL, "NULL source or destination");
    if (nchan < 1 || nchan > 8) return set_err (B200M_E_INVAL, "nchan %u outside 1..8", nchan);
    if (n_inst == 0) return set_err (B200M_E_INVAL, "n_inst = 0");
    if (nfram == 0 || nfram > B200M_MAX_BLOCK) return set_err (B200M_E_INVAL, "nfram %u outside 1..%u", nfram, B200M_MAX_BLOCK);
    if (src_stride < nfram || dst_stride < nfram) return set_err (B200M_E_INVAL, "stride < nfram %u", nfram);
    const int bps = pcm_sample_bytes (fmt);
    if ((uintptr_t)d_src % (bps == 3 ? 1 : bps)) return set_err (B200M_E_INVAL, "source not aligned to its sample type");
    if ((uintptr_t)d_dst % 16 || dst_stride % 4) return set_err (B200M_E_INVAL, "destination rows must be 16-byte aligned");
    if (b200m_device_count () <= 0) return set_err (B200M_E_NODEVICE, "no CUDA device: b200meters has no CPU path");
    DeviceGuard g (device);
    if (!g.ok) return set_err (B200M_E_INVAL, "bad device %d", device);
    return pcm_convert_launch (d_src, fmt, nchan, n_inst, src_stride, nfram, d_dst, dst_stride, (cudaStream_t)stream);
}
