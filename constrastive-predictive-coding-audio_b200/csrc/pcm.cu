// Batch assembly from raw PCM WAV bytes: the decode of read_wav (audio_dataset.py) for every segment of a batch in one
// launch.  The host stages whole interleaved frames as they lie in the files; each thread turns one frame's first-channel
// sample into fp32 and stores it at its place in the (B, L) batch.  Memory-bound (a few MB per batch): byte loads, since
// 24-bit samples and odd block alignments have no aligned word; plain stores, every output element has one writer.
#include "common.cuh"

namespace cpc {

static_assert(sizeof(cpc_pcm_segment) == 32, "cpc_pcm_segment layout");

constexpr int PCM_THREADS = 256;
constexpr int PCM_FRAMES_PER_THREAD = 4;
constexpr int PCM_CHUNK = PCM_THREADS * PCM_FRAMES_PER_THREAD;   // frames per (segment, chunk) block
constexpr int PCM_MAX_GRID_Y = 65535;

// The conversions of read_wav, exact: every divisor is a power of two, and int32 -> fp32 rounds to nearest even as
// numpy's astype(np.float32) does.
__device__ __forceinline__ float pcm_decode(const unsigned char* __restrict__ s, int width) {
    switch (width) {
        case 1: return ((float)__ldg(s) - 128.f) / 128.f;
        case 2: {
            const int v = (int)(short)((unsigned)__ldg(s) | ((unsigned)__ldg(s + 1) << 8));
            return (float)v / 32768.f;
        }
        case 3: {
            int v = (int)((unsigned)__ldg(s) | ((unsigned)__ldg(s + 1) << 8) | ((unsigned)__ldg(s + 2) << 16));
            v -= (v & 0x800000) << 1;
            return (float)v / 8388608.f;
        }
        default: {
            const int v = (int)((unsigned)__ldg(s) | ((unsigned)__ldg(s + 1) << 8) | ((unsigned)__ldg(s + 2) << 16) |
                                ((unsigned)__ldg(s + 3) << 24));
            return __int2float_rn(v) / 2147483648.f;
        }
    }
}

// grid (segments, chunks of PCM_CHUNK frames; a grid-stride loop when a segment has more than 65535 chunks)
__global__ void __launch_bounds__(PCM_THREADS) pcm_assemble_kernel(const cpc_pcm_segment* __restrict__ segments,
                                                                    const unsigned char* __restrict__ raw,
                                                                    float* __restrict__ out, int64_t row_stride) {
    const cpc_pcm_segment seg = segments[blockIdx.x];
    const unsigned char* src = raw + seg.src_byte_offset;
    float* dst = out + (int64_t)seg.dst_item * row_stride + seg.dst_offset;
    for (int64_t c0 = (int64_t)blockIdx.y * PCM_CHUNK; c0 < seg.frames; c0 += (int64_t)gridDim.y * PCM_CHUNK) {
#pragma unroll
        for (int u = 0; u < PCM_FRAMES_PER_THREAD; ++u) {
            const int64_t f = c0 + u * PCM_THREADS + threadIdx.x;
            if (f < seg.frames) dst[f] = pcm_decode(src + f * seg.block_align, seg.sample_width);
        }
    }
}

// One pass over the host table: field ranges, and the tiling of every item's [0, item_length) in table order.
static int pcm_validate(const cpc_pcm_params* p, const cpc_pcm_segment* t, int& max_frames) {
    if (p->batch < 1 || p->item_length < 1 || p->n_segments < 1 || p->out_row_stride < p->item_length)
        return CPC_ERR_BAD_SHAPE;
    int item = 0;
    int64_t filled = 0;                                     // columns of `item` covered so far
    max_frames = 0;
    for (int i = 0; i < p->n_segments; ++i) {
        const cpc_pcm_segment& s = t[i];
        if (s.sample_width < 1 || s.sample_width > 4 || s.block_align < s.sample_width) return CPC_ERR_BAD_SHAPE;
        if (s.frames < 0 || s.src_byte_offset < 0 || s.dst_offset < 0) return CPC_ERR_BAD_SHAPE;
        if (s.dst_item < 0 || s.dst_item >= p->batch) return CPC_ERR_BAD_SHAPE;
        if ((int64_t)s.dst_offset + s.frames > p->item_length) return CPC_ERR_BAD_SHAPE;
        if (s.dst_item != item) {                           // the previous item must be complete, the next one starts
            if (filled != p->item_length || s.dst_item != item + 1) return CPC_ERR_BAD_SHAPE;
            item = s.dst_item;
            filled = 0;
        }
        if (s.dst_offset != filled) return CPC_ERR_BAD_SHAPE;   // gap or overlap
        filled += s.frames;
        if (s.frames > max_frames) max_frames = s.frames;
    }
    return (item == p->batch - 1 && filled == p->item_length) ? CPC_OK : CPC_ERR_BAD_SHAPE;
}

}  // namespace cpc

using namespace cpc;

extern "C" int cpc_pcm_assemble(const cpc_pcm_params* p, const cpc_pcm_segment* segments_host,
                                const cpc_pcm_segment* segments_dev, const void* raw_dev, float* out, void* stream) {
    if (!p || !segments_host) return CPC_ERR_NULL;
    int max_frames = 0;
    int st = pcm_validate(p, segments_host, max_frames);
    if (st != CPC_OK) return st;
    if (!segments_dev || !raw_dev || !out) return CPC_ERR_NULL;
    if ((reinterpret_cast<uintptr_t>(segments_dev) & 7) || (reinterpret_cast<uintptr_t>(out) & 3)) return CPC_ERR_ALIGNMENT;
    if ((st = check_device()) != CPC_OK) return st;
    const int chunks = max_frames > 0 ? min(ceil_div(max_frames, PCM_CHUNK), PCM_MAX_GRID_Y) : 1;
    pcm_assemble_kernel<<<dim3(p->n_segments, chunks), PCM_THREADS, 0, (cudaStream_t)stream>>>(
        segments_dev, static_cast<const unsigned char*>(raw_dev), out, p->out_row_stride);
    CPC_LAUNCH_CHECK();
    count_launch();
    return CPC_OK;
}
