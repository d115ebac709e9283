// (2c) VBZ decoding on the device: the StreamVByte + zig-zag delta stage of the VBZ HDF5 filter
// (nanoporetech/vbz_compression), applied to chunk bodies the host has already taken through zstd.
// Bit-exact with warpstr_b200/fast5.py:vbz_decompress, its format errors reported as per-chunk status.
//
// One CTA per chunk (grid-stride over the chunk table).  A chunk is streamed in tiles of NT * SPT
// samples: every thread takes SPT consecutive samples, reads their 2-bit (v0) or 1-bit (v1) length codes,
// a CTA-wide exclusive scan of the per-thread byte counts places each thread in the tile's data bytes
// (fetched into shared memory in whole 16-byte words), a second scan of the per-thread delta sums plus
// the carry of the earlier tiles gives the samples, and the tile leaves through shared memory in 16-byte
// stores aligned to the destination.
#include <limits.h>
#include <stdint.h>

#include "wstr_internal.h"

namespace {

constexpr int NT = 256;              // threads per CTA
constexpr int SPT = 16;              // samples per thread and tile
constexpr int TILE = NT * SPT;       // samples per tile
constexpr int MAX_TILE_BYTES = 4 * TILE;
constexpr int DATA_WORDS = MAX_TILE_BYTES / 16 + 2;   // + the partial words at both ends

struct VbzChunk {
    int64_t in_off, out_off;         // payload byte offset (multiple of 16), output sample offset
    int32_t in_bytes, n;             // payload bytes, samples coded in the body
    int32_t n_out, format;           // samples written (<= n), kind | zigzag << 8
};

struct VbzSmem {
    uint4 data[DATA_WORDS];
    uint4 out[TILE / 8 + 1];         // int16 samples shifted by the destination's misalignment
    uint32_t scan[17];
};

// exclusive prefix over the CTA; *total receives the sum.  Two barriers, and every caller passes
// both: warp 0 overwrites scan[8..16] only after every thread has read the previous call's values.
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *total, uint32_t *scan) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) scan[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = lane < NT / 32 ? scan[lane] : 0u;
        uint32_t s = w;
#pragma unroll
        for (int d = 1; d < NT / 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, s, d);
            if (lane >= d) s += y;
        }
        if (lane < NT / 32) scan[8 + lane] = s - w;
        if (lane == NT / 32 - 1) scan[16] = s;
    }
    __syncthreads();
    *total = scan[16];
    return scan[8 + warp] + x - v;
}

// tile samples [0, cnt) -> dst[0, cnt): 16-byte stores wherever a destination word is whole
__device__ __forceinline__ void store_tile(VbzSmem &sm, int16_t *__restrict__ dst, int cnt) {
    const int shift = (int)((reinterpret_cast<uintptr_t>(dst) >> 1) & 7);
    int16_t *__restrict__ base = dst - shift;
    const int16_t *so = reinterpret_cast<const int16_t *>(sm.out);
    const int nwords = (shift + cnt + 7) >> 3;
    for (int w = threadIdx.x; w < nwords; w += NT) {
        const int a = w * 8, b = a + 8;
        if (a >= shift && b <= shift + cnt) {
            *reinterpret_cast<uint4 *>(base + a) = sm.out[w];
        } else {
            for (int j = a; j < b; ++j)
                if (j >= shift && j < shift + cnt) base[j] = so[j];
        }
    }
}

template <int V>   // 0: 32-bit StreamVByte, 2-bit codes; 1: the 16-bit variant, 1-bit keys
__device__ int decode_chunk(const uint8_t *__restrict__ in, const VbzChunk &c, int16_t *__restrict__ raw, VbzSmem &sm) {
    const int64_t n = c.n;
    const int64_t n_ctrl = V == 0 ? (n + 3) / 4 : (n + 7) / 8;
    if (c.in_bytes < n_ctrl) return WSTR_VBZ_TRUNCATED_CONTROL;
    const bool zigzag = (c.format >> 8) & 1;
    const uint8_t *ctrl = in + c.in_off;
    const int64_t data0 = c.in_off + n_ctrl, span_end = c.in_off + c.in_bytes;
    int64_t carry_bytes = 0;
    uint32_t carry = 0;
    for (int64_t tb = 0; tb < n; tb += TILE) {
        const int64_t t0 = tb + (int64_t)threadIdx.x * SPT;
        uint32_t len[SPT];
        {
            // this thread's codes: SPT/4 control bytes (v0) or SPT/8 key bytes (v1), whole when t0 < n
            uint32_t bits = 0;
            if (t0 < n) {
                if (V == 0) bits = *reinterpret_cast<const uint32_t *>(ctrl + t0 / 4);
                else bits = *reinterpret_cast<const uint16_t *>(ctrl + t0 / 8);
            }
#pragma unroll
            for (int k = 0; k < SPT; ++k) {
                const uint32_t code = V == 0 ? ((bits >> (2 * k)) & 3u) + 1u : ((bits >> k) & 1u) + 1u;
                len[k] = t0 + k < n ? code : 0u;
            }
        }
        uint32_t mine = 0;
#pragma unroll
        for (int k = 0; k < SPT; ++k) mine += len[k];
        uint32_t tile_bytes;
        const uint32_t at = block_excl_scan(mine, &tile_bytes, sm.scan);
        // the tile's data bytes, in whole 16-byte words, never past the chunk's own (16-byte padded) span
        const int64_t a0 = data0 + carry_bytes;
        const int64_t a1 = a0 + tile_bytes < span_end ? a0 + tile_bytes : span_end;
        const int64_t w0 = a0 & ~(int64_t)15;
        const int nw = a1 > a0 ? (int)(((a1 + 15) & ~(int64_t)15) - w0) / 16 : 0;
        const uint4 *src = reinterpret_cast<const uint4 *>(in + w0);
        for (int i = threadIdx.x; i < nw; i += NT) sm.data[i] = src[i];
        __syncthreads();
        const uint8_t *bytes = reinterpret_cast<const uint8_t *>(sm.data) + (a0 - w0) + at;
        uint32_t val[SPT];
        uint32_t p = 0;
#pragma unroll
        for (int k = 0; k < SPT; ++k) {
            uint32_t v = 0;
            for (uint32_t b = 0; b < len[k]; ++b) v |= (uint32_t)bytes[p + b] << (8 * b);
            p += len[k];
            val[k] = v;
        }
        if (zigzag) {
            uint32_t run = 0;
#pragma unroll
            for (int k = 0; k < SPT; ++k) {
                const uint32_t u = val[k];
                // the signed delta; a 16-bit one (v1) sign-extends, which leaves the low 16 bits of every sum alone
                uint32_t d = (u >> 1) ^ (0u - (u & 1u));
                if (V == 1) d = (uint32_t)(int32_t)(int16_t)(uint16_t)d;
                run += d;
                val[k] = run;
            }
            uint32_t tile_sum;
            const uint32_t before = carry + block_excl_scan(run, &tile_sum, sm.scan);
#pragma unroll
            for (int k = 0; k < SPT; ++k) val[k] += before;
            carry += tile_sum;
        }
        const int64_t keep = (int64_t)c.n_out - tb;
        if (keep > 0) {
            const int cnt = keep < TILE ? (int)keep : TILE;
            const int shift = (int)(((uintptr_t)(raw + c.out_off + tb) >> 1) & 7);
            int16_t *so = reinterpret_cast<int16_t *>(sm.out) + shift + threadIdx.x * SPT;
#pragma unroll
            for (int k = 0; k < SPT; ++k) so[k] = (int16_t)(uint16_t)val[k];
            __syncthreads();
            store_tile(sm, raw + c.out_off + tb, cnt);
        }
        carry_bytes += tile_bytes;
    }
    if (n == 0) return WSTR_VBZ_OK;
    const int64_t data_len = c.in_bytes - n_ctrl;
    if (V == 0 && carry_bytes > data_len) return WSTR_VBZ_SHORT_DATA;
    if (V == 1 && carry_bytes != data_len) return WSTR_VBZ_LENGTH_MISMATCH;
    return WSTR_VBZ_OK;
}

__global__ void __launch_bounds__(NT, 4) vbz_decode_kernel(const uint8_t *__restrict__ in, const VbzChunk *__restrict__ chunks,
                                                        int n_chunks, int16_t *__restrict__ raw, int32_t *__restrict__ status) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    VbzSmem &sm = *reinterpret_cast<VbzSmem *>(smem_raw);
    for (int ci = blockIdx.x; ci < n_chunks; ci += gridDim.x) {
        const VbzChunk c = chunks[ci];
        const int kind = c.format & 0xff;
        int st = WSTR_VBZ_OK;
        if (kind == WSTR_VBZ_KIND_V0) {
            st = decode_chunk<0>(in, c, raw, sm);
        } else if (kind == WSTR_VBZ_KIND_V1) {
            st = decode_chunk<1>(in, c, raw, sm);
        } else {   // verbatim little-endian int16
            const int16_t *src = reinterpret_cast<const int16_t *>(in + c.in_off);
            int16_t *dst = raw + c.out_off;
            for (int t = threadIdx.x; t < c.n_out; t += NT) dst[t] = src[t];
        }
        if (threadIdx.x == 0) status[ci] = st;
        __syncthreads();   // shared memory of this chunk's last tile is free again
    }
}

}  // namespace

extern "C" int64_t wstr_vbz_workspace_bytes(int32_t n_chunks) {
    if (n_chunks < 0) return WSTR_ERR_INVALID_ARGUMENT;
    return (int64_t)sizeof(VbzChunk) * n_chunks + 256;
}

extern "C" int wstr_vbz_decode_batch(const uint8_t *d_payload, const int64_t *in_off, const int64_t *in_bytes,
                                     const int32_t *n_samples, const int32_t *n_out, const int32_t *kind,
                                     const int32_t *zigzag, const int64_t *out_off, int32_t n_chunks, int16_t *d_raw,
                                     int32_t *d_status, void *d_workspace, int64_t workspace_bytes, void *stream) {
    if (!in_off || !in_bytes || !n_samples || !n_out || !kind || !zigzag || !out_off || !d_status || !d_workspace ||
        n_chunks < 0)
        return WSTR_ERR_INVALID_ARGUMENT;
    if (n_chunks == 0) return WSTR_OK;
    if (!d_payload || !d_raw || (reinterpret_cast<uintptr_t>(d_payload) & 15) ||
        (reinterpret_cast<uintptr_t>(d_raw) & 1))
        return WSTR_ERR_INVALID_ARGUMENT;
    if (workspace_bytes < wstr_vbz_workspace_bytes(n_chunks)) return WSTR_ERR_WORKSPACE_TOO_SMALL;
    for (int c = 0; c < n_chunks; ++c) {
        const int k = kind[c];
        const bool ok = in_off[c] >= 0 && (in_off[c] & 15) == 0 && in_bytes[c] >= 0 && in_bytes[c] <= INT32_MAX &&
                        out_off[c] >= 0 && n_out[c] >= 0 && (zigzag[c] == 0 || zigzag[c] == 1) &&
                        (k == WSTR_VBZ_KIND_RAW ? 2 * (int64_t)n_out[c] <= in_bytes[c]
                                                : (k == WSTR_VBZ_KIND_V0 || k == WSTR_VBZ_KIND_V1) &&
                                                      n_out[c] <= n_samples[c]);
        if (!ok) return WSTR_ERR_INVALID_ARGUMENT;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const size_t bytes = sizeof(VbzChunk) * (size_t)n_chunks;
    void *h = nullptr, *token = nullptr;
    int rc = wstr_stage_begin(bytes, &h, &token);
    if (rc != WSTR_OK) return rc;
    VbzChunk *hc = static_cast<VbzChunk *>(h);
    for (int c = 0; c < n_chunks; ++c) {
        const int k = kind[c];
        hc[c].in_off = in_off[c];
        hc[c].out_off = out_off[c];
        hc[c].in_bytes = (int32_t)in_bytes[c];
        hc[c].n = k == WSTR_VBZ_KIND_RAW ? n_out[c] : n_samples[c];
        hc[c].n_out = n_out[c];
        hc[c].format = k | (zigzag[c] << 8);
    }
    rc = wstr_stage_commit(token, d_workspace, bytes, s);
    if (rc != WSTR_OK) return rc;
    static unsigned long long attr_done = 0ull;      // devices the function attribute is set on
    int dev = 0;
    WSTR_CUDA(cudaGetDevice(&dev));
    if (!((attr_done >> (dev & 63)) & 1ull)) {
        WSTR_CUDA(cudaFuncSetAttribute(vbz_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(VbzSmem)));
        attr_done |= 1ull << (dev & 63);
    }
    const int grid = n_chunks < 148 * 8 ? n_chunks : 148 * 8;
    vbz_decode_kernel<<<grid, NT, sizeof(VbzSmem), s>>>(d_payload, static_cast<const VbzChunk *>(d_workspace), n_chunks,
                                                        d_raw, d_status);
    WSTR_CUDA(cudaGetLastError());
    return WSTR_OK;
}
