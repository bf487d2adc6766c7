/* mz_cuda_api.cu -- the thin extern "C" shim between the C host side and the sm_100a kernels.
 * Declares nothing new: every entry point is documented in include/mz_cuda_batch.h. */
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "../../include/mz_cuda_batch.h"
#include "concat_kernel.cuh"
#include "crc32_kernel.cuh"
#include "deflate_kernel.cuh"
#include <cstdlib>
#include <cstdio>
#include "inflate_kernel.cuh"
#include "inflate_spec_kernel.cuh"
#include "pkcrypt_kernel.cuh"
#include "sha256_kernel.cuh"
#include "wzaes_kernel.cuh"

#define MZ_OK 0
#define MZ_MEM_ERROR (-4)
#define MZ_PARAM_ERROR (-102)
#define MZ_INTERNAL_ERROR (-104)
#define MZ_SUPPORT_ERROR (-109)

using namespace mzc;

static_assert(sizeof(mz_cuda_inflate_job) == sizeof(InflateJob), "job layout");
static_assert(sizeof(mz_cuda_inflate_state) == sizeof(InflateState), "state layout");
static_assert(sizeof(mz_cuda_spec_summary) == sizeof(SpecSummary), "summary layout");

namespace {

struct DeviceCtx {
    bool ready = false;
    int sm_count = 0;
    CrcConsts *d_consts = nullptr;
    uint32_t *d_crc_scratch = nullptr; /* residues for mz_cuda_crc32_device */
    uint32_t *d_work = nullptr;        /* ring of work-counter pairs for dynamically scheduled launches */
    uint32_t *d_aes = nullptr;         /* K8 tables: 256 words of T-table, then the S-box (256 bytes); made on first use */
    unsigned work_next = 0;
    size_t crc_scratch_n = 0;
};

constexpr int kMaxDev = 16;
/* work-counter pairs for dynamically scheduled launches. A launch takes the next pair of the ring; the kernel's last CTA
 * leaves it zeroed, so a pair is only ever shared if more than kWorkRing launches are in flight on one device at once
 * (the driver's launch queue is far shorter). */
constexpr unsigned kWorkRing = 4096;
DeviceCtx g_dev[kMaxDev];
std::mutex g_mu;
std::mutex g_crc_mu;
CrcConsts g_consts;
bool g_consts_ready = false;
thread_local char g_err[256] = "";

int32_t fail(cudaError_t e, const char *what) {
    snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? MZ_MEM_ERROR : MZ_INTERNAL_ERROR;
}
#define CK(call)                                       \
    do {                                               \
        cudaError_t e_ = (call);                       \
        if (e_ != cudaSuccess) return fail(e_, #call); \
    } while (0)

int32_t get_ctx(DeviceCtx **out) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        snprintf(g_err, sizeof(g_err), "no CUDA device: %s", cudaGetErrorString(e));
        return MZ_SUPPORT_ERROR;
    }
    if (dev < 0 || dev >= kMaxDev) return MZ_PARAM_ERROR;
    DeviceCtx &c = g_dev[dev];
    if (!c.ready) {
        std::lock_guard<std::mutex> lk(g_mu);
        if (!c.ready) {
            if (!g_consts_ready) {
                crc_consts_init(g_consts);
                g_consts_ready = true;
            }
            cudaDeviceProp prop;
            CK(cudaGetDeviceProperties(&prop, dev));
            if (prop.major < 10) {
                snprintf(g_err, sizeof(g_err), "device %d is sm_%d%d; this library is built for sm_100a only", dev, prop.major, prop.minor);
                return MZ_SUPPORT_ERROR;
            }
            c.sm_count = prop.multiProcessorCount;
            CK(cudaMalloc(&c.d_consts, sizeof(CrcConsts)));
            CK(cudaMemcpy(c.d_consts, &g_consts, sizeof(CrcConsts), cudaMemcpyHostToDevice));
            CK(cudaFuncSetAttribute(deflate_chunks_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DF_SMEM_BYTES));
            CK(cudaFuncSetAttribute(deflate_chunks_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, DF_SMEM_BYTES));
            CK(cudaFuncSetAttribute(deflate_chunks_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DF_SMEM_BYTES));
            CK(cudaFuncSetAttribute(deflate_chunks_kernel<1, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, DFH_SMEM_BYTES));
            CK(cudaFuncSetAttribute(crc32_segments_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CRC_SMEM_BYTES));
            CK(cudaFuncSetAttribute(inflate_streams_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, INF_SMEM_BYTES));
            CK(cudaFuncSetAttribute(inflate_spec_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SPEC_RESOLVE_SMEM));
            CK(cudaFuncSetAttribute(inflate_spec_compose_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SPEC_COMPOSE_SMEM));
            CK(cudaFuncSetAttribute(inflate_spec_link_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
            CK(cudaFuncSetAttribute(inflate_spec_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SPEC_MAX_SEGMENTS * 16));
            CK(cudaMalloc(&c.d_work, kWorkRing * 2 * sizeof(uint32_t)));
            CK(cudaMemset(c.d_work, 0, kWorkRing * 2 * sizeof(uint32_t)));
            c.ready = true;
        }
    }
    *out = &c;
    return MZ_OK;
}

uint64_t pick_crc_seg(uint64_t len, int sm_count) {
    /* aim for >= 4 segments per resident warp, segments between 4 KiB and 64 KiB */
    uint64_t warps = (uint64_t)sm_count * (CRC_THREADS / 32);
    uint64_t seg = 65536;
    while (seg > 4096 && len / seg < warps * 2) seg >>= 1;
    return seg;
}

} // namespace

extern "C" {

const char *mz_cuda_last_error(void) { return g_err; }

int32_t mz_cuda_init(void) {
    DeviceCtx *c;
    return get_ctx(&c);
}

int32_t mz_cuda_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int32_t mz_cuda_set_device(int32_t ordinal) {
    CK(cudaSetDevice(ordinal));
    return MZ_OK;
}

int32_t mz_cuda_get_device(void) {
    int d = -1;
    if (cudaGetDevice(&d) != cudaSuccess) return -1;
    return d;
}

int32_t mz_cuda_sm_count(void) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    return err ? err : c->sm_count;
}

void *mz_cuda_malloc(size_t bytes) {
    void *p = nullptr;
    if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void mz_cuda_free(void *p) {
    if (p) cudaFree(p);
}
void *mz_cuda_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 16, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void mz_cuda_host_free(void *p) {
    if (p) cudaFreeHost(p);
}
int32_t mz_cuda_memcpy_h2d(void *d, const void *h, size_t n, void *stream) {
    CK(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return MZ_OK;
}
int32_t mz_cuda_memcpy_d2h(void *h, const void *d, size_t n, void *stream) {
    CK(cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return MZ_OK;
}
int32_t mz_cuda_memcpy_d2d(void *d, const void *s, size_t n, void *stream) {
    CK(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return MZ_OK;
}
int32_t mz_cuda_host_is_pinned(const void *h) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, h) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return a.type == cudaMemoryTypeHost ? 1 : 0;
}
int32_t mz_cuda_memset(void *d, int v, size_t n, void *stream) {
    CK(cudaMemsetAsync(d, v, n, (cudaStream_t)stream));
    return MZ_OK;
}
int32_t mz_cuda_stream_sync(void *stream) {
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    return MZ_OK;
}
void *mz_cuda_stream_create(void) {
    cudaStream_t s = nullptr;
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    return s;
}
void mz_cuda_stream_destroy(void *s) {
    if (s) cudaStreamDestroy((cudaStream_t)s);
}
void *mz_cuda_event_create(void) {
    cudaEvent_t e = nullptr;
    if (cudaEventCreate(&e) != cudaSuccess) return nullptr;
    return e;
}
void mz_cuda_event_destroy(void *e) {
    if (e) cudaEventDestroy((cudaEvent_t)e);
}
int32_t mz_cuda_event_record(void *e, void *stream) {
    CK(cudaEventRecord((cudaEvent_t)e, (cudaStream_t)stream));
    return MZ_OK;
}
int32_t mz_cuda_event_sync(void *e) {
    CK(cudaEventSynchronize((cudaEvent_t)e));
    return MZ_OK;
}
int32_t mz_cuda_event_query(void *e) { /* 1 = everything recorded before it has finished, 0 = not yet, < 0 = error */
    const cudaError_t r = cudaEventQuery((cudaEvent_t)e);
    if (r == cudaSuccess) return 1;
    if (r == cudaErrorNotReady) {
        cudaGetLastError();
        return 0;
    }
    return fail(r, "cudaEventQuery");
}
float mz_cuda_event_elapsed_ms(void *a, void *b) {
    float ms = -1.f;
    if (cudaEventSynchronize((cudaEvent_t)b) != cudaSuccess) return -1.f;
    if (cudaEventElapsedTime(&ms, (cudaEvent_t)a, (cudaEvent_t)b) != cudaSuccess) return -1.f;
    return ms;
}

/* ---- CRC ------------------------------------------------------------------------------------------ */
int32_t mz_cuda_crc32_segments(const void *d_in, uint64_t total_len, uint64_t seg_size, const uint64_t *d_off, const uint32_t *d_len,
                               uint32_t nseg, uint32_t *d_residue, uint32_t *d_crc, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (nseg == 0) return MZ_OK;
    if (!d_residue || (!d_off && seg_size == 0) || (d_off && !d_len)) return MZ_PARAM_ERROR;
    CrcParams P;
    P.in = (const uint8_t *)d_in;
    P.in_off = d_off;
    P.in_len = d_len;
    P.total_len = total_len;
    P.seg_size = seg_size;
    P.nseg = nseg;
    P.consts = c->d_consts;
    P.out_residue = d_residue;
    P.out_crc = d_crc;
    uint32_t warps_per_cta = CRC_THREADS / 32;
    uint32_t grid = (nseg + warps_per_cta - 1) / warps_per_cta;
    if (grid > (uint32_t)c->sm_count) grid = (uint32_t)c->sm_count;
    MZ_LAUNCH(crc32_segments_kernel, dim3(grid), dim3(CRC_THREADS), CRC_SMEM_BYTES, (cudaStream_t)stream, P);
    CK(cudaGetLastError());
    return MZ_OK;
}

int32_t mz_cuda_crc32_fold(const uint32_t *d_residue, uint32_t nseg, uint64_t seg_size, uint64_t total_len, uint32_t *d_out2, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    MZ_LAUNCH(crc32_fold_kernel, dim3(1), dim3(CRCF_THREADS), 0, (cudaStream_t)stream, d_residue, nseg, seg_size, total_len, c->d_consts, d_out2);
    CK(cudaGetLastError());
    return MZ_OK;
}

int32_t mz_cuda_crc32_device(const void *d_in, uint64_t len, uint32_t value, uint32_t *crc) {
    return mz_cuda_crc32_device_stream(d_in, len, value, crc, nullptr);
}

int32_t mz_cuda_crc32_device_stream(const void *d_in, uint64_t len, uint32_t value, uint32_t *crc, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (len == 0) {
        *crc = value;
        return MZ_OK;
    }
    uint64_t seg = pick_crc_seg(len, c->sm_count);
    uint64_t nseg64 = (len + seg - 1) / seg;
    while (nseg64 > 0x7fffffffull) {
        seg <<= 1;
        nseg64 = (len + seg - 1) / seg;
    }
    uint32_t nseg = (uint32_t)nseg64;
    /* the residue scratch is per device: threads sharing a device take turns for the whole operation */
    std::lock_guard<std::mutex> crc_turn(g_crc_mu);
    {
        std::lock_guard<std::mutex> lk(g_mu);
        if (c->crc_scratch_n < (size_t)nseg + 2) {
            if (c->d_crc_scratch) cudaFree(c->d_crc_scratch);
            c->d_crc_scratch = nullptr;
            c->crc_scratch_n = 0;
            CK(cudaMalloc(&c->d_crc_scratch, ((size_t)nseg + 2) * 4));
            c->crc_scratch_n = (size_t)nseg + 2;
        }
    }
    uint32_t *d_res = c->d_crc_scratch, *d_out2 = c->d_crc_scratch + nseg;
    err = mz_cuda_crc32_segments(d_in, len, seg, nullptr, nullptr, nseg, d_res, nullptr, stream);
    if (err) return err;
    err = mz_cuda_crc32_fold(d_res, nseg, seg, len, d_out2, stream);
    if (err) return err;
    uint32_t h[2];
    CK(cudaMemcpyAsync(h, d_out2, 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    CK(cudaStreamSynchronize((cudaStream_t)stream));
    /* chain the running value: crc(v, D) = ~((~v) x^(8|D|) + R(D)) */
    *crc = ~(gf2_mulmod(~value, gf2_xpow(g_consts.x2n, 8ull * len)) ^ h[0]);
    return MZ_OK;
}

uint32_t mz_cuda_crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b) {
    if (!g_consts_ready) {
        std::lock_guard<std::mutex> lk(g_mu);
        if (!g_consts_ready) {
            crc_consts_init(g_consts);
            g_consts_ready = true;
        }
    }
    if (len_b == 0) return crc_a; /* zlib's crc32_combine convention for the degenerate case */
    /* crc(A||B) = crc(A) x^(8|B|) + crc(B): the init/xorout terms cancel (both sides carry them once) */
    return gf2_mulmod(crc_a, gf2_xpow(g_consts.x2n, 8ull * len_b)) ^ crc_b;
}

/* ---- DEFLATE ---------------------------------------------------------------------------------------- */
uint64_t mz_cuda_deflate_slot_bound(uint32_t chunk_size) { return deflate_slot_bound(chunk_size); }

int32_t mz_cuda_deflate_chunks(const void *d_in, uint64_t total_len, uint32_t chunk_size, const uint64_t *d_off, const uint32_t *d_len,
                               const uint8_t *d_flags, uint32_t nchunks, uint32_t last_flags, int32_t level, void *d_slots,
                               uint64_t slot_stride, uint32_t *d_out_len, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (nchunks == 0) return MZ_OK;
    if (level < 0 || level > 9 || !d_slots || !d_out_len || (slot_stride & 15) || ((uintptr_t)d_slots & 15)) return MZ_PARAM_ERROR;
    if (!d_off) {
        if (chunk_size == 0 || chunk_size > MZ_CUDA_CHUNK_MAX || slot_stride < deflate_slot_bound(chunk_size)) return MZ_PARAM_ERROR;
        uint64_t need = total_len == 0 ? 1 : (total_len + chunk_size - 1) / chunk_size;
        if (need != nchunks) return MZ_PARAM_ERROR;
    } else if (!d_len) {
        return MZ_PARAM_ERROR;
    }
    DeflateParams P;
    P.in = (const uint8_t *)d_in;
    P.in_off = d_off;
    P.in_len = d_len;
    P.flags = d_flags;
    P.total_len = total_len;
    P.chunk_size = chunk_size;
    P.nchunks = nchunks;
    P.last_flags = last_flags;
    P.level = level;
    P.out = (uint8_t *)d_slots;
    P.slot_stride = slot_stride;
    P.out_len = d_out_len;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        P.work_counter = c->d_work + 2 * (c->work_next++ % kWorkRing);
    }
    const uint32_t resident = (uint32_t)c->sm_count * 2u; /* two 512-thread CTAs of 111 KB shared memory per SM */
    uint32_t grid = nchunks < resident ? nchunks : resident;
    if (deflate_stride_for_level(level) == 2)
        MZ_LAUNCH((deflate_chunks_kernel<2, false>), dim3(grid), dim3(DF_THREADS), DF_SMEM_BYTES, (cudaStream_t)stream, P);
    else if (!deflate_lazy_for_level(level))
        MZ_LAUNCH((deflate_chunks_kernel<1, false>), dim3(grid), dim3(DF_THREADS), DF_SMEM_BYTES, (cudaStream_t)stream, P);
    else if (!deflate_hist_for_level(level))
        MZ_LAUNCH((deflate_chunks_kernel<1, true>), dim3(grid), dim3(DF_THREADS), DF_SMEM_BYTES, (cudaStream_t)stream, P);
    else { /* the history variant: 208 KiB of shared memory, one CTA per SM */
        const uint32_t grid1 = nchunks < (uint32_t)c->sm_count ? nchunks : (uint32_t)c->sm_count;
        MZ_LAUNCH((deflate_chunks_kernel<1, true, true>), dim3(grid1), dim3(DF_THREADS), DFH_SMEM_BYTES, (cudaStream_t)stream, P);
    }
    CK(cudaGetLastError());
    return MZ_OK;
}

int32_t mz_cuda_concat(const void *d_slots, uint64_t slot_stride, const uint32_t *d_out_len, uint32_t nchunks, uint64_t *d_offsets,
                       void *d_dst, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    MZ_LAUNCH(scan_lengths_kernel, dim3(1), dim3(SCAN_THREADS), 0, (cudaStream_t)stream, d_out_len, nchunks, (uint64_t)0, d_offsets);
    if (nchunks) {
        uint32_t grid = nchunks < (uint32_t)c->sm_count * 16u ? nchunks : (uint32_t)c->sm_count * 16u;
        MZ_LAUNCH(gather_slots_kernel, dim3(grid), dim3(GATHER_THREADS), 0, (cudaStream_t)stream, (const uint8_t *)d_slots, slot_stride,
                  d_out_len, (const uint64_t *)d_offsets, nchunks, (uint8_t *)d_dst);
    }
    CK(cudaGetLastError());
    return MZ_OK;
}

int32_t mz_cuda_gather(const void *d_slots, uint64_t slot_stride, const uint32_t *d_out_len, uint32_t nchunks, const uint64_t *d_offsets, void *d_dst,
                       void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (nchunks == 0) return MZ_OK;
    uint32_t grid = nchunks < (uint32_t)c->sm_count * 16u ? nchunks : (uint32_t)c->sm_count * 16u;
    MZ_LAUNCH(gather_slots_kernel, dim3(grid), dim3(GATHER_THREADS), 0, (cudaStream_t)stream, (const uint8_t *)d_slots, slot_stride, d_out_len, d_offsets,
              nchunks, (uint8_t *)d_dst);
    CK(cudaGetLastError());
    return MZ_OK;
}

int32_t mz_cuda_scatter_blobs(const void *d_blob, const uint32_t *d_blob_off, const uint64_t *d_dst_off, uint32_t n, void *d_dst, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (n == 0) return MZ_OK;
    uint32_t grid = (n + 7) / 8;
    if (grid > (uint32_t)c->sm_count * 8u) grid = (uint32_t)c->sm_count * 8u;
    MZ_LAUNCH(scatter_blobs_kernel, dim3(grid), dim3(256), 0, (cudaStream_t)stream, (const uint8_t *)d_blob, d_blob_off, d_dst_off, n, (uint8_t *)d_dst);
    CK(cudaGetLastError());
    return MZ_OK;
}

int32_t mz_cuda_inflate_streams(const mz_cuda_inflate_job *d_jobs, mz_cuda_inflate_state *d_states, uint32_t nstreams, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (nstreams == 0) return MZ_OK;
    uint32_t maxgrid = (uint32_t)c->sm_count * 32u; /* 32 single-warp CTAs (6.4 KB of tables each) per SM */
    uint32_t grid = nstreams < maxgrid ? nstreams : maxgrid;
    uint32_t *counter;
    {
        std::lock_guard<std::mutex> lk(g_mu);
        counter = c->d_work + 2 * (c->work_next++ % kWorkRing);
    }
    MZ_LAUNCH(inflate_streams_kernel, dim3(grid), dim3(INF_THREADS), INF_SMEM_BYTES, (cudaStream_t)stream, (const InflateJob *)d_jobs,
              (InflateState *)d_states, nstreams, counter);
    CK(cudaGetLastError());
    return MZ_OK;
}

/* workspace carving for K6 (all pieces 256-byte aligned) */
static inline uint64_t al256(uint64_t v) { return (v + 255) & ~255ull; }
uint64_t mz_cuda_inflate_spec_workspace_bytes(uint32_t max_segments) {
    const uint64_t m = max_segments;
    return al256(m * sizeof(SpecSeg)) + al256(m * sizeof(InflateState)) + al256(m * 8) + al256(m * SPEC_RING * 2) + al256(m * 32768) + al256((uint64_t)SPEC_GROUPS * 65536) +
           al256((uint64_t)SPEC_GROUPS * 32768) + 256 + 256;
}

int32_t mz_cuda_inflate_spec_round(const void *d_in, uint64_t in_base, uint64_t in_avail, uint32_t in_final, uint64_t start_bit,
                                   uint64_t seg_bytes, uint32_t nseg, void *d_out, uint64_t out_base, uint64_t out_pos,
                                   uint64_t out_end, void *d_workspace, uint32_t max_segments, mz_cuda_spec_summary *d_summary,
                                   void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (nseg == 0 || nseg > max_segments || max_segments > SPEC_MAX_SEGMENTS || seg_bytes < 64 || ((uintptr_t)d_in & 3) || !d_workspace || !d_summary) return MZ_PARAM_ERROR;
    SpecParams P;
    P.in = (const uint8_t *)d_in;
    P.in_base = in_base;
    P.in_avail = in_avail;
    P.start_bit = start_bit;
    P.seg_bits = seg_bytes * 8;
    P.out = (uint8_t *)d_out;
    P.out_base = out_base;
    P.out_pos = out_pos;
    P.out_end = out_end;
    P.in_final = in_final;
    P.nseg = nseg;
    uint8_t *w = (uint8_t *)(((uintptr_t)d_workspace + 255) & ~(uintptr_t)255);
    const uint64_t m = max_segments;
    P.seg = (SpecSeg *)w;            w += al256(m * sizeof(SpecSeg));
    P.states = (InflateState *)w;    w += al256(m * sizeof(InflateState));
    P.chain = (uint32_t *)w;         w += al256(m * 8);
    P.rings = (uint16_t *)w;         w += al256(m * SPEC_RING * 2);
    P.wins = w;                      w += al256(m * 32768);
    P.gmaps = (uint16_t *)w;         w += al256((uint64_t)SPEC_GROUPS * 65536);
    P.gwins = w;                     w += al256((uint64_t)SPEC_GROUPS * 32768);
    P.work = (uint32_t *)w;
    P.summary = (SpecSummary *)d_summary;
    cudaStream_t s = (cudaStream_t)stream;
    const uint32_t maxgrid = (uint32_t)c->sm_count * 32u;
    const uint32_t grid = nseg < maxgrid ? nseg : maxgrid;
    CK(cudaMemsetAsync(P.work, 0, 16, s));
    const bool trace = getenv("MZ_CUDA_TRACE") != nullptr; /* per-kernel times of the round on stderr (debug aid, serialises) */
    cudaEvent_t ev[6];
    if (trace)
        for (int i = 0; i < 6; i++) CK(cudaEventCreate(&ev[i]));
    if (trace) CK(cudaEventRecord(ev[0], s));
    MZ_LAUNCH(inflate_spec_find_kernel, dim3(grid), dim3(INF_THREADS), SPEC_FIND_SMEM, s, P);
    if (trace) CK(cudaEventRecord(ev[1], s));
    MZ_LAUNCH(inflate_spec_scan_kernel, dim3(grid), dim3(INF_THREADS), INF_SMEM_BYTES, s, P);
    if (trace) CK(cudaEventRecord(ev[2], s));
    MZ_LAUNCH(inflate_spec_chain_kernel, dim3(1), dim3(SPEC_CHAIN_THREADS), (size_t)nseg * 16, s, P);
    if (trace) CK(cudaEventRecord(ev[3], s));
    MZ_LAUNCH(inflate_spec_compose_kernel, dim3(SPEC_GROUPS), dim3(SPEC_RESOLVE_THREADS), SPEC_COMPOSE_SMEM, s, P);
    MZ_LAUNCH(inflate_spec_link_kernel, dim3(1), dim3(SPEC_RESOLVE_THREADS), 65536, s, P);
    MZ_LAUNCH(inflate_spec_resolve_kernel, dim3(SPEC_GROUPS), dim3(SPEC_RESOLVE_THREADS), SPEC_RESOLVE_SMEM, s, P);
    if (trace) CK(cudaEventRecord(ev[4], s));
    MZ_LAUNCH(inflate_spec_emit_kernel, dim3(grid), dim3(INF_THREADS), INF_SMEM_BYTES, s, P);
    if (trace) CK(cudaEventRecord(ev[5], s));
    CK(cudaGetLastError());
    if (trace) {
        CK(cudaEventSynchronize(ev[5]));
        float t[5];
        for (int i = 0; i < 5; i++) CK(cudaEventElapsedTime(&t[i], ev[i], ev[i + 1]));
        fprintf(stderr, "mz_cuda: K6 kernels ms: find %.3f scan %.3f chain %.3f compose+link+resolve %.3f emit %.3f (%u segments)\n", t[0], t[1], t[2], t[3], t[4], nseg);
        for (int i = 0; i < 6; i++) cudaEventDestroy(ev[i]);
    }
    return MZ_OK;
}

int32_t mz_cuda_sha256_batch(const void *d_in, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, void *d_digest, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (n == 0) return MZ_OK;
    if (!d_in || !d_off || !d_len || !d_digest || ((uintptr_t)d_digest & 3)) return MZ_PARAM_ERROR;
    Sha256Params P;
    P.in = (const uint8_t *)d_in;
    P.off = d_off;
    P.len = d_len;
    P.n = n;
    P.digest = (uint8_t *)d_digest;
    uint32_t blocks = (n + SHA_THREADS - 1) / SHA_THREADS;
    const uint32_t cap = (uint32_t)c->sm_count * 16u;
    if (blocks > cap) blocks = cap;
    MZ_LAUNCH(sha256_batch_kernel, dim3(blocks), dim3(SHA_THREADS), 0, (cudaStream_t)stream, P);
    CK(cudaGetLastError());
    return MZ_OK;
}

/* ---- K8: WinZip AES for a batch of entries ------------------------------------------------------------------- */
namespace {
/* FIPS 197 4.2 / 5.1.1: S[x] = affine(inverse of x in GF(2^8) mod x^8 + x^4 + x^3 + x + 1); T[x] = (2 S, S, S, 3 S) */
int32_t aes_tables(DeviceCtx *c) {
    if (c->d_aes) return MZ_OK;
    std::lock_guard<std::mutex> lk(g_mu);
    if (c->d_aes) return MZ_OK;
    uint32_t h[256 + 64];
    uint8_t sbox[256];
    uint8_t p = 1, q = 1;
    do { /* p runs over the multiplicative group (generator 3), q over the inverses */
        p = (uint8_t)(p ^ (p << 1) ^ ((p & 0x80) ? 0x1b : 0));
        q ^= (uint8_t)(q << 1);
        q ^= (uint8_t)(q << 2);
        q ^= (uint8_t)(q << 4);
        if (q & 0x80) q ^= 0x09;
        const uint8_t x = (uint8_t)(q ^ (uint8_t)((q << 1) | (q >> 7)) ^ (uint8_t)((q << 2) | (q >> 6)) ^ (uint8_t)((q << 3) | (q >> 5)) ^ (uint8_t)((q << 4) | (q >> 4)));
        sbox[p] = (uint8_t)(x ^ 0x63);
    } while (p != 1);
    sbox[0] = 0x63;
    for (int i = 0; i < 256; i++) {
        const uint32_t s1 = sbox[i], s2 = ((s1 << 1) ^ ((s1 & 0x80) ? 0x11b : 0)) & 0xff, s3 = s2 ^ s1;
        h[i] = (s2 << 24) | (s1 << 16) | (s1 << 8) | s3;
    }
    memcpy(h + 256, sbox, 256);
    uint32_t *d = nullptr;
    CK(cudaMalloc(&d, sizeof(h)));
    CK(cudaMemcpy(d, h, sizeof(h), cudaMemcpyHostToDevice));
    c->d_aes = d;
    return MZ_OK;
}
bool wz_strength(uint32_t strength, uint32_t *key_len, uint32_t *salt_len) {
    if (strength < 1 || strength > 3) return false;
    *key_len = 8 * strength + 8;   /* MZ_AES_KEY_LENGTH, mz_strm_wzaes.c:19 */
    *salt_len = 4 * strength + 4;  /* MZ_AES_SALT_LENGTH, :21 */
    return true;
}
} // namespace

int32_t mz_cuda_wzaes_derive(const void *d_password, uint32_t pw_len, const void *d_salts, uint32_t n, uint32_t strength, void *d_keys, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    WzDeriveParams P;
    if (!wz_strength(strength, &P.key_len, &P.salt_len) || pw_len > 128) return MZ_PARAM_ERROR;
    if (n == 0) return MZ_OK;
    if (!d_password || !d_salts || !d_keys) return MZ_PARAM_ERROR;
    P.password = (const uint8_t *)d_password;
    P.pw_len = pw_len;
    P.salts = (const uint8_t *)d_salts;
    P.iterations = 1000; /* MZ_AES_KEYING_ITERATIONS, mz_strm_wzaes.c:20 */
    P.n = n;
    P.keys = (uint8_t *)d_keys;
    const uint32_t threads = n * ((2 * P.key_len + 2 + 19) / 20);
    uint32_t blocks = (threads + 127) / 128;
    const uint32_t cap = (uint32_t)c->sm_count * 16u;
    if (blocks > cap) blocks = cap;
    MZ_LAUNCH(wzaes_derive_kernel, dim3(blocks), dim3(128), 0, (cudaStream_t)stream, P);
    CK(cudaGetLastError());
    return MZ_OK;
}

int32_t mz_cuda_wzaes_ctr(void *d_data, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, uint64_t max_len, const void *d_keys, uint32_t strength,
                          void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    WzCtrParams P;
    uint32_t salt_len;
    if (!wz_strength(strength, &P.key_len, &salt_len)) return MZ_PARAM_ERROR;
    if (n == 0 || max_len == 0) return MZ_OK;
    if (!d_data || !d_off || !d_len || !d_keys) return MZ_PARAM_ERROR;
    err = aes_tables(c);
    if (err) return err;
    P.data = (uint8_t *)d_data;
    P.off = d_off;
    P.len = d_len;
    P.n = n;
    P.parts = (uint32_t)((max_len + WZ_CTR_PART - 1) / WZ_CTR_PART);
    if (P.parts > 65535) return MZ_PARAM_ERROR; /* entries up to 4 GiB */
    P.keys = (const uint8_t *)d_keys;
    P.te0 = c->d_aes;
    P.sbox = (const uint8_t *)(c->d_aes + 256);
    const uint32_t gx = n < (uint32_t)c->sm_count * 64u ? n : (uint32_t)c->sm_count * 64u;
    MZ_LAUNCH(wzaes_ctr_kernel, dim3(gx, P.parts), dim3(WZ_CTR_THREADS), 0, (cudaStream_t)stream, P);
    CK(cudaGetLastError());
    return MZ_OK;
}

int32_t mz_cuda_wzaes_hmac(const void *d_data, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, const void *d_keys, uint32_t strength, void *d_mac,
                           void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    WzHmacParams P;
    uint32_t salt_len;
    if (!wz_strength(strength, &P.key_len, &salt_len)) return MZ_PARAM_ERROR;
    if (n == 0) return MZ_OK;
    if (!d_data || !d_off || !d_len || !d_keys || !d_mac) return MZ_PARAM_ERROR;
    P.data = (const uint8_t *)d_data;
    P.off = d_off;
    P.len = d_len;
    P.n = n;
    P.keys = (const uint8_t *)d_keys;
    P.mac = (uint8_t *)d_mac;
    uint32_t blocks = (n + 127) / 128;
    const uint32_t cap = (uint32_t)c->sm_count * 16u;
    if (blocks > cap) blocks = cap;
    MZ_LAUNCH(wzaes_hmac_kernel, dim3(blocks), dim3(128), 0, (cudaStream_t)stream, P);
    CK(cudaGetLastError());
    return MZ_OK;
}

/* ---- K9: PKWARE traditional encryption for a batch of entries ------------------------------------------------ */
namespace {
/* segment size: PK_SEG, or MZ_CUDA_PKCRYPT_SEG (a power of two, 256 .. 65536) for tuning */
uint32_t pk_seg_size() {
    const char *v = getenv("MZ_CUDA_PKCRYPT_SEG");
    if (v) {
        const long s = atol(v);
        if (s >= 256 && s <= 65536 && (s & (s - 1)) == 0) return (uint32_t)s;
    }
    return PK_SEG;
}
/* workspace layout (all pieces 256-byte aligned): per entry the segment counts and their scan, per segment its entry, the
 * three in-tile scans and two key starts, per tile the three aggregates, their flags and the three carries */
uint64_t pk_layout(PkParams *P, uint8_t *w, uint64_t nseg, uint32_t n) {
    const uint64_t tiles = (nseg + PK_THREADS - 1) / PK_THREADS;
    uint64_t o = 0;
    auto take = [&](uint64_t bytes) { uint8_t *p = w ? w + o : nullptr; o += al256(bytes); return p; };
    uint8_t *seg_count = take((uint64_t)n * 4), *seg_base = take(((uint64_t)n + 1) * 8), *seg_entry = take(nseg * 4);
    uint8_t *ks0 = take(nseg * 4), *ks1 = take(nseg * 4);
    uint8_t *incl[3], *agg[3], *aggf[3], *pre[3];
    for (int i = 0; i < 3; i++) {
        incl[i] = take(nseg * 8);
        agg[i] = take(tiles * 8);
        aggf[i] = take(tiles * 4);
        pre[i] = take(tiles * 8);
    }
    if (P) {
        P->seg_count = (uint32_t *)seg_count;
        P->seg_base = (const uint64_t *)seg_base;
        P->seg_entry = (uint32_t *)seg_entry;
        P->ks0 = (uint32_t *)ks0;
        P->ks1 = (uint32_t *)ks1;
        for (int i = 0; i < 3; i++) {
            P->incl[i] = (uint2 *)incl[i];
            P->agg[i] = (uint2 *)agg[i];
            P->aggf[i] = (uint32_t *)aggf[i];
            P->pre[i] = (uint2 *)pre[i];
        }
    }
    return o;
}
} // namespace

uint64_t mz_cuda_pkcrypt_workspace_bytes(uint64_t total_len, uint32_t n) {
    return pk_layout(nullptr, nullptr, total_len / pk_seg_size() + n, n) + 256;
}

int32_t mz_cuda_pkcrypt_encrypt(void *d_data, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, const char *password, void *d_workspace,
                                uint64_t workspace_bytes, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (!password) return MZ_PARAM_ERROR;
    if (n == 0) return MZ_OK;
    if (!d_data || !d_off || !d_len || !d_workspace) return MZ_PARAM_ERROR;
    cudaStream_t s = (cudaStream_t)stream;
    PkParams P;
    memset(&P, 0, sizeof(P));
    P.data = (uint8_t *)d_data;
    P.off = d_off;
    P.len = d_len;
    P.n = n;
    P.seg = pk_seg_size();
    uint32_t keys[3];
    pk_host_keys(password, keys);
    P.key0 = keys[0];
    P.key1 = keys[1];
    P.key2 = keys[2];
    uint8_t *w = (uint8_t *)(((uintptr_t)d_workspace + 255) & ~(uintptr_t)255);
    const uint64_t usable = workspace_bytes > (uint64_t)(w - (uint8_t *)d_workspace) ? workspace_bytes - (uint64_t)(w - (uint8_t *)d_workspace) : 0;
    if (pk_layout(&P, w, 0, n) > usable) return MZ_PARAM_ERROR;
    /* segments per entry and where each entry's segments begin; the total decides the grids and the rest of the layout */
    const uint32_t ge = (n + 255) / 256 < (uint32_t)c->sm_count * 8u ? (n + 255) / 256 : (uint32_t)c->sm_count * 8u;
    MZ_LAUNCH(pk_count_kernel, dim3(ge), dim3(256), 0, s, P);
    MZ_LAUNCH(scan_lengths_kernel, dim3(1), dim3(SCAN_THREADS), 0, s, (const uint32_t *)P.seg_count, n, (uint64_t)0, (uint64_t *)P.seg_base);
    uint64_t nseg = 0;
    CK(cudaMemcpyAsync(&nseg, P.seg_base + n, 8, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (nseg == 0) return MZ_OK;
    if (nseg > 0xffffffffull - PK_THREADS || pk_layout(&P, w, nseg, n) > usable) return MZ_PARAM_ERROR; /* smaller than mz_cuda_pkcrypt_workspace_bytes */
    P.nseg = (uint32_t)nseg;
    P.ntiles = (uint32_t)((nseg + PK_THREADS - 1) / PK_THREADS);
    P.xseg = gf2_xpow(g_consts.x2n, 8ull * P.seg);
    P.aseg = 1;
    for (uint32_t i = 0; i < P.seg; i++) P.aseg *= PK_MUL;
    const uint32_t gt = P.ntiles < (uint32_t)c->sm_count * 6u ? P.ntiles : (uint32_t)c->sm_count * 6u;
    MZ_LAUNCH(pk_pass1_kernel, dim3(gt), dim3(PK_THREADS), 0, s, P);
    MZ_LAUNCH((pk_tile_scan_kernel<0, 0>), dim3(1), dim3(PK_TILE_SCAN_THREADS), 0, s, P);
    MZ_LAUNCH(pk_pass2_kernel, dim3(gt), dim3(PK_THREADS), 0, s, P);
    MZ_LAUNCH((pk_tile_scan_kernel<1, 1>), dim3(1), dim3(PK_TILE_SCAN_THREADS), 0, s, P);
    MZ_LAUNCH(pk_pass3_kernel, dim3(gt), dim3(PK_THREADS), 0, s, P);
    MZ_LAUNCH((pk_tile_scan_kernel<0, 2>), dim3(1), dim3(PK_TILE_SCAN_THREADS), 0, s, P);
    MZ_LAUNCH(pk_pass4_kernel, dim3(gt), dim3(PK_THREADS), 0, s, P);
    CK(cudaGetLastError());
    return MZ_OK;
}

int32_t mz_cuda_pkcrypt_decrypt(void *d_data, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, const char *password, void *stream) {
    DeviceCtx *c;
    int32_t err = get_ctx(&c);
    if (err) return err;
    if (!password) return MZ_PARAM_ERROR;
    if (n == 0) return MZ_OK;
    if (!d_data || !d_off || !d_len) return MZ_PARAM_ERROR;
    PkDecParams P;
    P.data = (uint8_t *)d_data;
    P.off = d_off;
    P.len = d_len;
    P.n = n;
    uint32_t keys[3];
    pk_host_keys(password, keys);
    P.key0 = keys[0];
    P.key1 = keys[1];
    P.key2 = keys[2];
    uint32_t blocks = (n + PKD_THREADS - 1) / PKD_THREADS;
    const uint32_t cap = (uint32_t)c->sm_count * 64u;
    if (blocks > cap) blocks = cap;
    MZ_LAUNCH(pk_decrypt_kernel, dim3(blocks), dim3(PKD_THREADS), 0, (cudaStream_t)stream, P);
    CK(cudaGetLastError());
    return MZ_OK;
}

/* ---- multi-GPU --------------------------------------------------------------------------------------------- */
int32_t mz_cuda_ipc_export(const void *dptr, void *handle64) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    CK(cudaIpcGetMemHandle((cudaIpcMemHandle_t *)handle64, (void *)dptr));
    return MZ_OK;
}
int32_t mz_cuda_ipc_open(const void *handle64, void **dptr) {
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    CK(cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
    return MZ_OK;
}
int32_t mz_cuda_ipc_close(void *dptr) {
    CK(cudaIpcCloseMemHandle(dptr));
    return MZ_OK;
}
int32_t mz_cuda_memcpy_peer(void *dst, const void *src, size_t bytes, void *stream) {
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream)); /* UVA: the driver routes it over NVLink on a copy engine */
    return MZ_OK;
}
int32_t mz_cuda_stream_wait_event(void *stream, void *event) {
    CK(cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)event, 0));
    return MZ_OK;
}

uint64_t mz_cuda_gather_region_bound(uint64_t shard_len) {
    const uint64_t nch = shard_len == 0 ? 1 : (shard_len + MZ_CUDA_CHUNK_MAX - 1) / MZ_CUDA_CHUNK_MAX;
    return (nch * deflate_slot_bound(MZ_CUDA_CHUNK_MAX) + 255) & ~255ull;
}

namespace {
struct ShardCtx { /* per shard slot (= per device in real use), grown on demand, kept for the life of the process */
    int device = -1;
    cudaStream_t compute = nullptr, copy = nullptr;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    uint8_t *d_slots = nullptr;
    uint32_t *d_out_len = nullptr, *d_residue = nullptr, *d_chunk_crc = nullptr, *d_crc2 = nullptr, *d_rows = nullptr;
    uint64_t *d_offsets = nullptr;
    uint64_t *h_total = nullptr; /* pinned: [2] joined bytes of the piece in flight */
    uint32_t *h_crc = nullptr;   /* pinned: [2][2] */
    uint32_t cap_chunks = 0;
};
ShardCtx g_shard[kMaxDev];
std::mutex g_shard_mu;
}

int32_t mz_cuda_deflate_sharded(const mz_cuda_shard *sh, int32_t ndev, int32_t level, int32_t pieces, uint64_t *region_off, uint64_t *stream_len,
                                uint32_t *crc32) {
    if (!sh || ndev < 1 || ndev > kMaxDev || level < 0 || level > 9 || !region_off || !stream_len) return MZ_PARAM_ERROR;
    if (pieces < 1) pieces = 1;
    std::lock_guard<std::mutex> lk(g_shard_mu);
    int prev_dev = 0;
    cudaGetDevice(&prev_dev);
    const uint64_t stride = deflate_slot_bound(MZ_CUDA_CHUNK_MAX);
    std::vector<uint32_t> nch(ndev), chunk_base(ndev);
    uint64_t roff = 0;
    uint32_t cb = 0;
    for (int i = 0; i < ndev; i++) {
        if (sh[i].device < 0 || sh[i].device >= kMaxDev || !sh[i].d_gathered || ((uintptr_t)sh[i].d_in & 15) || ((uintptr_t)sh[i].d_gathered & 15)) return MZ_PARAM_ERROR;
        if (i + 1 < ndev && (sh[i].len == 0 || sh[i].len % MZ_CUDA_CHUNK_MAX)) return MZ_PARAM_ERROR;
        nch[i] = (uint32_t)(sh[i].len == 0 ? 1 : (sh[i].len + MZ_CUDA_CHUNK_MAX - 1) / MZ_CUDA_CHUNK_MAX);
        region_off[i] = roff;
        roff += mz_cuda_gather_region_bound(sh[i].len);
        chunk_base[i] = cb;
        cb += nch[i];
    }
    for (int i = 0; i < ndev; i++)
        if (sh[i].gathered_cap < roff) return MZ_PARAM_ERROR;
    /* contexts, scratch, peer access */
    for (int i = 0; i < ndev; i++) {
        CK(cudaSetDevice(sh[i].device));
        DeviceCtx *c;
        int32_t err = get_ctx(&c);
        if (err) return err;
        ShardCtx &x = g_shard[i];
        if (x.compute && x.device != sh[i].device) return MZ_PARAM_ERROR; /* slot i stays with the device it was first used with */
        if (!x.compute) {
            x.device = sh[i].device;
            CK(cudaStreamCreateWithFlags(&x.compute, cudaStreamNonBlocking));
            CK(cudaStreamCreateWithFlags(&x.copy, cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&x.ev[0], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&x.ev[1], cudaEventDisableTiming));
            CK(cudaHostAlloc((void **)&x.h_total, 16, cudaHostAllocDefault));
            CK(cudaHostAlloc((void **)&x.h_crc, 16, cudaHostAllocDefault));
            CK(cudaMalloc(&x.d_crc2, 16));
        }
        const uint32_t need = (nch[i] + (uint32_t)pieces - 1) / (uint32_t)pieces + 1; /* chunks of the largest piece */
        if (x.cap_chunks < need || !x.d_rows) {
            cudaFree(x.d_slots); cudaFree(x.d_out_len); cudaFree(x.d_residue); cudaFree(x.d_chunk_crc); cudaFree(x.d_offsets); cudaFree(x.d_rows);
            x.cap_chunks = 0;
            CK(cudaMalloc(&x.d_slots, (size_t)need * stride));
            CK(cudaMalloc(&x.d_out_len, (size_t)need * 4));
            CK(cudaMalloc(&x.d_residue, (size_t)need * 4));
            CK(cudaMalloc(&x.d_chunk_crc, (size_t)need * 4));
            CK(cudaMalloc(&x.d_offsets, ((size_t)need + 1) * 8));
            CK(cudaMalloc(&x.d_rows, (size_t)need * 12));
            x.cap_chunks = need;
        }
        for (int j = 0; j < ndev; j++)
            if (j != i && sh[j].device != sh[i].device) {
                cudaError_t e = cudaDeviceEnablePeerAccess(sh[j].device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(e, "cudaDeviceEnablePeerAccess");
                cudaGetLastError();
            }
    }
    std::vector<uint64_t> base(ndev, 0);            /* bytes of device i's stream produced so far */
    std::vector<uint32_t> crc_dev(ndev, 0);
    std::vector<uint64_t> done_len(ndev, 0);        /* input bytes folded into crc_dev */
    auto piece_range = [&](int i, int k, uint32_t &c0, uint32_t &c1) {
        c0 = (uint32_t)((uint64_t)nch[i] * k / pieces);
        c1 = (uint32_t)((uint64_t)nch[i] * (k + 1) / pieces);
    };
    /* finish piece k of device i: learn its size, send it (and its rows) to every other device on the copy stream */
    auto finish = [&](int i, int k) -> int32_t {
        ShardCtx &x = g_shard[i];
        CK(cudaSetDevice(sh[i].device));
        CK(cudaEventSynchronize(x.ev[k & 1]));
        uint32_t c0, c1;
        piece_range(i, k, c0, c1);
        const uint64_t L = x.h_total[k & 1];
        const uint64_t in0 = (uint64_t)c0 * MZ_CUDA_CHUNK_MAX;
        const uint64_t inl = ((uint64_t)c1 * MZ_CUDA_CHUNK_MAX < sh[i].len ? (uint64_t)c1 * MZ_CUDA_CHUNK_MAX : sh[i].len) - (in0 < sh[i].len ? in0 : sh[i].len);
        const uint32_t pc = x.h_crc[(k & 1) * 2 + 1];
        if (inl) {
            crc_dev[i] = done_len[i] == 0 ? pc : mz_cuda_crc32_combine(crc_dev[i], pc, inl);
            done_len[i] += inl;
        }
        if (c1 > c0) {
            const uint8_t *src = (const uint8_t *)sh[i].d_gathered + region_off[i] + base[i];
            for (int j = 0; j < ndev; j++) {
                if (j == i) continue;
                CK(cudaMemcpyPeerAsync((uint8_t *)sh[j].d_gathered + region_off[i] + base[i], sh[j].device, src, sh[i].device, (size_t)L, x.copy));
                if (sh[j].d_rows && sh[i].d_rows)
                    CK(cudaMemcpyPeerAsync(sh[j].d_rows + 3ull * (chunk_base[i] + c0), sh[j].device, sh[i].d_rows + 3ull * (chunk_base[i] + c0), sh[i].device,
                                           (size_t)(c1 - c0) * 12, x.copy));
            }
        }
        base[i] += L;
        return MZ_OK;
    };
    for (int k = 0; k <= pieces; k++) {
        if (k < pieces) {
            for (int i = 0; i < ndev; i++) { /* compression of piece k: does not depend on where the piece will land */
                ShardCtx &x = g_shard[i];
                CK(cudaSetDevice(sh[i].device));
                uint32_t c0, c1;
                piece_range(i, k, c0, c1);
                if (c1 == c0) continue;
                const uint64_t in0 = (uint64_t)c0 * MZ_CUDA_CHUNK_MAX;
                const uint64_t inl = ((uint64_t)c1 * MZ_CUDA_CHUNK_MAX < sh[i].len ? (uint64_t)c1 * MZ_CUDA_CHUNK_MAX : sh[i].len) - in0;
                const uint32_t lastf = (i == ndev - 1 && k == pieces - 1) ? MZ_CUDA_FLAG_FINAL : 0u;
                int32_t err = mz_cuda_deflate_chunks((const uint8_t *)sh[i].d_in + in0, inl, MZ_CUDA_CHUNK_MAX, nullptr, nullptr, nullptr, c1 - c0, lastf, level,
                                                     x.d_slots, stride, x.d_out_len, x.compute);
                if (!err) err = mz_cuda_crc32_segments((const uint8_t *)sh[i].d_in + in0, inl, MZ_CUDA_CHUNK_MAX, nullptr, nullptr, c1 - c0, x.d_residue, x.d_chunk_crc, x.compute);
                if (!err) err = mz_cuda_crc32_fold(x.d_residue, c1 - c0, MZ_CUDA_CHUNK_MAX, inl, x.d_crc2, x.compute);
                if (err) return err;
            }
        }
        if (k > 0)
            for (int i = 0; i < ndev; i++) {
                int32_t err = finish(i, k - 1);
                if (err) return err;
            }
        if (k < pieces) {
            for (int i = 0; i < ndev; i++) { /* join piece k straight into the device's own region of its gathered buffer */
                ShardCtx &x = g_shard[i];
                CK(cudaSetDevice(sh[i].device));
                uint32_t c0, c1;
                piece_range(i, k, c0, c1);
                x.h_total[k & 1] = 0;
                if (c1 > c0) {
                    uint8_t *dst = (uint8_t *)sh[i].d_gathered + region_off[i] + base[i];
                    const uint64_t in0 = (uint64_t)c0 * MZ_CUDA_CHUNK_MAX;
                    const uint64_t inl = ((uint64_t)c1 * MZ_CUDA_CHUNK_MAX < sh[i].len ? (uint64_t)c1 * MZ_CUDA_CHUNK_MAX : sh[i].len) - in0;
                    int32_t err = mz_cuda_concat(x.d_slots, stride, x.d_out_len, c1 - c0, x.d_offsets, dst, x.compute);
                    if (err) return err;
                    if (sh[i].d_rows) {
                        MZ_LAUNCH(pack_rows_kernel, dim3((c1 - c0 + 255) / 256), dim3(256), 0, x.compute, (const uint32_t *)x.d_chunk_crc, (const uint32_t *)x.d_out_len,
                                  c1 - c0, inl, (uint32_t)MZ_CUDA_CHUNK_MAX, sh[i].d_rows + 3ull * (chunk_base[i] + c0));
                        CK(cudaGetLastError());
                    }
                    CK(cudaMemcpyAsync(&x.h_total[k & 1], x.d_offsets + (c1 - c0), 8, cudaMemcpyDeviceToHost, x.compute));
                    CK(cudaMemcpyAsync(&x.h_crc[(k & 1) * 2], x.d_crc2, 8, cudaMemcpyDeviceToHost, x.compute));
                }
                CK(cudaEventRecord(x.ev[k & 1], x.compute));
                CK(cudaStreamWaitEvent(x.copy, x.ev[k & 1], 0)); /* the copies of this piece (issued later) follow its join */
            }
        }
    }
    uint32_t crc = 0;
    uint64_t folded = 0;
    for (int i = 0; i < ndev; i++) {
        ShardCtx &x = g_shard[i];
        CK(cudaSetDevice(sh[i].device));
        CK(cudaStreamSynchronize(x.copy));
        CK(cudaStreamSynchronize(x.compute));
        stream_len[i] = base[i];
        if (done_len[i]) {
            crc = folded == 0 ? crc_dev[i] : mz_cuda_crc32_combine(crc, crc_dev[i], done_len[i]);
            folded += done_len[i];
        }
    }
    if (crc32) *crc32 = crc;
    cudaSetDevice(prev_dev);
    return MZ_OK;
}

} /* extern "C" */
