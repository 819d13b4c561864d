// wdx_vbz.cu — C-ABI entry points of the pod5 VBZ decoder (include/wdx_b200.h: wdx_zstd_decompress,
// wdx_vbz_decode_rows): one warp per zstd frame, one CTA per read for the streamvbyte-16 rows.  No CPU compute path.
#include "vbz_kernel.cuh"
#include "wdx_internal.cuh"

using namespace wdx;

namespace {
constexpr int ZSTD_WARPS = 4;        // frames per CTA (4 x ~10 KB of decode tables in shared memory)
constexpr int ROW_THREADS = 256;     // one CTA per read, 8 samples (one key byte) per thread per tile
constexpr int64_t REGION_HDR = 16;   // row decoder scratch region: int64 bytes produced, int32 zstd status, pad

// Frame f of the batch.  ROWS: the frame is chunk f of the reads in read_chunks; its region of the scratch starts with
// a 16-byte header (bytes produced, status) and receives only the prefix the row of `stride` samples needs.
template <bool ROWS>
__global__ void __launch_bounds__(ZSTD_WARPS * 32) zstd_kernel(const uint8_t* __restrict__ src, const int64_t* __restrict__ chunk_off, int64_t m,
                                                               const int64_t* __restrict__ limit, uint8_t* __restrict__ scratch,
                                                               const int64_t* __restrict__ scratch_off, int64_t* __restrict__ produced,
                                                               int32_t* __restrict__ status, const int32_t* __restrict__ samples,
                                                               const int64_t* __restrict__ read_chunks, int64_t n, int64_t stride) {
    __shared__ vbz::Tables tabs[ZSTD_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t f = (int64_t)blockIdx.x * ZSTD_WARPS + warp;
    if (f >= m) return;
    const int64_t in0 = chunk_off[f], nin = chunk_off[f + 1] - in0;
    uint8_t* out;
    int64_t cap, lim, content_max = INT64_MAX;
    int64_t* prod_out;
    int32_t* st_out;
    if (ROWS) {
        if (f < read_chunks[0] || f >= read_chunks[n]) return;
        int64_t lo = 0, hi = n;   // read r: read_chunks[r] <= f < read_chunks[r + 1]
        while (hi - lo > 1) {
            const int64_t mid = (lo + hi) >> 1;
            if (read_chunks[mid] <= f) lo = mid;
            else hi = mid;
        }
        int64_t soff = 0;
        for (int64_t c = read_chunks[lo] + lane; c < f; c += 32) soff += samples[c];
        for (int o = 16; o; o >>= 1) soff += __shfl_xor_sync(0xffffffffu, soff, o);
        if (soff >= stride) return;   // the row is full before this chunk
        const int64_t s = samples[f], t = min(s, stride - soff), nk = (s + 7) / 8;
        const int64_t r0 = scratch_off[f], rlen = scratch_off[f + 1] - r0;
        if ((r0 & 15) || rlen < REGION_HDR + nk + 2 * t || s < 0) return;   // reported by the row kernel
        prod_out = (int64_t*)(scratch + r0);
        st_out = (int32_t*)(scratch + r0 + 8);
        out = scratch + r0 + REGION_HDR;
        content_max = nk + 2 * s;   // svb16 bound
        if (t == s) {               // the whole chunk: decode all of it (its length is checked against `samples`)
            cap = content_max;
            lim = INT64_MAX;
        } else {                    // the keys and at most 2 bytes per sample the row takes
            cap = lim = nk + 2 * t;
        }
    } else {
        out = scratch + scratch_off[f];
        cap = scratch_off[f + 1] - scratch_off[f];
        lim = limit[f];
        prod_out = produced + f;
        st_out = status + f;
    }
    int64_t prod = 0;
    int st;
    if (nin < 0 || cap < 0 || lim < 0) st = vbz::ST_CORRUPT;
    else st = vbz::decode_frame(src + in0, nin, out, cap, lim, content_max, &prod, tabs[warp], lane, 32);
    if (lane == 0) {
        *prod_out = st ? 0 : prod;
        *st_out = st;
    }
}

// exclusive prefix sum over the CTA; *total = the sum of all v
__device__ __forceinline__ uint32_t block_scan(uint32_t v, uint32_t* total, uint32_t* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = v;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) sh[warp] = x;
    __syncthreads();
    uint32_t before = 0, all = 0;
    for (int w = 0; w < ROW_THREADS / 32; w++) {
        const uint32_t sw = sh[w];
        before += w < warp ? sw : 0;
        all += sw;
    }
    __syncthreads();
    *total = all;
    return before + x - v;
}

__global__ void __launch_bounds__(ROW_THREADS) svb16_rows_kernel(const int64_t* __restrict__ read_chunks, const int32_t* __restrict__ samples,
                                                                 const uint8_t* __restrict__ scratch, const int64_t* __restrict__ scratch_off,
                                                                 int64_t stride, int16_t* __restrict__ rows, int32_t* __restrict__ n_valid,
                                                                 int32_t* __restrict__ status) {
    __shared__ uint32_t sh[ROW_THREADS / 32];
    const int64_t r = blockIdx.x;
    const int64_t c0 = read_chunks[r], c1 = read_chunks[r + 1];
    int16_t* row = rows + r * stride;
    int64_t soff = 0, total = 0;
    int st = 0;
    for (int64_t c = c0; c < c1; c++) {
        const int64_t s = samples[c];
        if (s < 0) st = st ? st : vbz::ST_SAMPLES;
        total += s;
        if (st || soff >= stride) continue;
        const int64_t t = min(s, stride - soff), nk = (s + 7) / 8;
        const int64_t r0 = scratch_off[c], rlen = scratch_off[c + 1] - r0;
        if ((r0 & 15) || rlen < REGION_HDR + nk + 2 * t) {
            st = vbz::ST_SCRATCH;
            continue;
        }
        const int64_t produced = *(const int64_t*)(scratch + r0);
        const int zst = *(const int32_t*)(scratch + r0 + 8);
        if (zst) {
            st = zst;
            continue;
        }
        const uint8_t* keys = scratch + r0 + REGION_HDR;
        const uint8_t* data = keys + nk;
        const int64_t avail = produced - nk;
        if (avail < 0) {
            st = vbz::ST_SAMPLES;
            continue;
        }
        int64_t dpos = 0;
        uint16_t carry = 0;
        for (int64_t tile = 0; tile < t; tile += 8 * ROW_THREADS) {
            const int64_t first = tile + 8 * (int64_t)threadIdx.x;
            const int ns = (int)max((int64_t)0, min((int64_t)8, t - first));
            const uint8_t kb = ns > 0 ? keys[first >> 3] : 0;
            const uint32_t w = (uint32_t)vbz::svb16_key_width(kb, ns);
            uint32_t tile_bytes, tile_sum;
            const uint32_t off = block_scan(w, &tile_bytes, sh);
            const bool ok = dpos + off + w <= avail;
            const uint16_t ls = (ok && ns) ? vbz::svb16_delta_sum8(data + dpos + off, kb, ns) : 0;
            const uint32_t pre = block_scan(ls, &tile_sum, sh);
            if (ok && ns) {
                int16_t v[8];
                vbz::svb16_decode8(data + dpos + off, kb, ns, (uint16_t)(carry + pre), v);
                for (int i = 0; i < ns; i++) row[soff + first + i] = v[i];
            }
            if (__syncthreads_or(!ok)) {
                st = vbz::ST_SAMPLES;
                break;
            }
            dpos += tile_bytes;
            carry = (uint16_t)(carry + tile_sum);
        }
        if (!st && t == s && nk + dpos != produced) st = vbz::ST_SAMPLES;
        soff += t;
    }
    const int64_t nv = st ? 0 : min(total, stride);
    for (int64_t i = nv + threadIdx.x; i < stride; i += ROW_THREADS) row[i] = 0;
    if (threadIdx.x == 0) {
        n_valid[r] = (int32_t)nv;
        status[r] = st;
    }
}

bool all_device(std::initializer_list<const void*> ps) {
    for (const void* p : ps)
        if (mem_kind(p) != 2) return false;
    return true;
}
}  // namespace

extern "C" {

int wdx_zstd_decompress(const uint8_t* src, const int64_t* chunk_off, int64_t m, const int64_t* limit, uint8_t* scratch,
                        const int64_t* scratch_off, int64_t* produced, int32_t* status, int device, void* stream) {
    if (m < 0) return fail(WDX_ERR_INVALID, "m=%lld", (long long)m);
    if (m == 0) return WDX_OK;
    if (!src || !chunk_off || !limit || !scratch || !scratch_off || !produced || !status) return fail(WDX_ERR_INVALID, "NULL argument");
    if (!all_device({src, chunk_off, limit, scratch, scratch_off, produced, status}))
        return fail(WDX_ERR_INVALID, "wdx_zstd_decompress takes device pointers");
    CUDA_TRY(cudaSetDevice(device));
    const unsigned grid = (unsigned)((m + ZSTD_WARPS - 1) / ZSTD_WARPS);
    zstd_kernel<false><<<grid, ZSTD_WARPS * 32, 0, (cudaStream_t)stream>>>(src, chunk_off, m, limit, scratch, scratch_off, produced,
                                                                          status, nullptr, nullptr, 0, 0);
    CUDA_TRY(cudaGetLastError());
    g_launches++;
    return WDX_OK;
}

int wdx_vbz_decode_rows(const uint8_t* src, const int64_t* chunk_off, const int32_t* samples, int64_t m, const int64_t* read_chunks,
                        int64_t n, uint8_t* scratch, const int64_t* scratch_off, int16_t* rows, int64_t stride, int32_t* n_valid,
                        int32_t* status, int device, void* stream) {
    if (m < 0 || n < 0 || stride < 1) return fail(WDX_ERR_INVALID, "m=%lld n=%lld stride=%lld", (long long)m, (long long)n, (long long)stride);
    if (n == 0) return WDX_OK;
    if (!read_chunks || !rows || !n_valid || !status) return fail(WDX_ERR_INVALID, "NULL argument");
    if (!all_device({read_chunks, rows, n_valid, status})) return fail(WDX_ERR_INVALID, "wdx_vbz_decode_rows takes device pointers");
    if (m > 0) {
        if (!src || !chunk_off || !samples || !scratch || !scratch_off) return fail(WDX_ERR_INVALID, "NULL argument");
        if (!all_device({src, chunk_off, samples, scratch, scratch_off})) return fail(WDX_ERR_INVALID, "wdx_vbz_decode_rows takes device pointers");
    }
    CUDA_TRY(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    if (m > 0) {
        const unsigned grid = (unsigned)((m + ZSTD_WARPS - 1) / ZSTD_WARPS);
        zstd_kernel<true><<<grid, ZSTD_WARPS * 32, 0, st>>>(src, chunk_off, m, nullptr, scratch, scratch_off, nullptr, nullptr, samples,
                                                           read_chunks, n, stride);
        CUDA_TRY(cudaGetLastError());
        g_launches++;
    }
    svb16_rows_kernel<<<(unsigned)n, ROW_THREADS, 0, st>>>(read_chunks, samples, scratch, scratch_off, stride, rows, n_valid, status);
    CUDA_TRY(cudaGetLastError());
    g_launches++;
    return WDX_OK;
}

}  // extern "C"
