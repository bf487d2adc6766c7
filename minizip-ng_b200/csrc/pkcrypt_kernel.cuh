/* pkcrypt_kernel.cuh -- K9: PKWARE traditional encryption (APPNOTE 6.1.5-6.1.6, "ZipCrypto") for a batch of zip entries: what
 * mz_strm_pkcrypt.c:64-102 does per byte with three 32-bit keys,
 *   key stream byte   t = (key2 | 2);  ((t * (t ^ 1)) >> 8) & 0xff          taken BEFORE the plain byte p updates the keys
 *   update_keys(p)    key0 = crc_reg(key0, p)                                 reflected CRC-32 register, no inversions
 *                     key1 = (key1 + (key0 & 0xff)) * 134775813 + 1           mod 2^32
 *                     key2 = crc_reg(key2, key1 >> 24)
 * The keys start from 305419896, 591751049, 878082192 and are first run over the password (the same for every entry, done on
 * the host by the shim).
 *
 * Decryption is serial within an entry: the byte that moves the keys is the OUTPUT. pk_decrypt_kernel is one thread per entry.
 *
 * Encryption is not: the key stream depends on the plaintext only, and each key moves by a map that composes.
 *   key0  is a CRC register fed with the plaintext: linear over GF(2), so over a segment S of the entry
 *         key0_after = key0_before * x^(8|S|) mod P  xor  reg(0, S)                       (crc32_combine's arithmetic)
 *   key1  moves by k -> M k + (M (key0' & 0xff) + 1): affine mod 2^32; a segment's effect is a pair (A, B), k -> A k + B,
 *         and pairs compose. (A, B) only needs key0 at the segment's start.
 *   key2  is a CRC register fed with key1' >> 24: linear again once key1 at the segment's start is known.
 * So an entry is cut into fixed segments (PK_SEG bytes, never crossing entries) and four passes run, one thread per segment,
 * each of the first three followed by an exclusive scan over the segments of each entry (three carries):
 *   pass 1  (reg(0, S), x^(8|S|)) of the plaintext            scan -> key0 at every segment start
 *   pass 2  run key0, build (A, B)                            scan -> key1 at every segment start
 *   pass 3  run key0 and key1, (reg(0, key1>>24 bytes), x^..)  scan -> key2 at every segment start
 *   pass 4  run all three keys and XOR the key stream in place.
 * The per-entry scans are segmented scans over ALL segments of the batch (an entry start resets the carry): within a tile of
 * PK_THREADS segments in the pass kernel itself, across tiles by pk_tile_scan_kernel. The work of a batch therefore does not
 * depend on how it is split into entries: one 256 MiB entry and 4096 entries of 64 KiB are the same segments.
 *
 * The 256-entry CRC table lives in shared memory, replicated once per lane (entry e of lane l at word e * 32 + l, as K1 does):
 * the indices are data-dependent and every lane reads its own bank. */
#ifndef MZ_PKCRYPT_KERNEL_CUH
#define MZ_PKCRYPT_KERNEL_CUH

#include "mzcuda_common.cuh"
#include "crc32_kernel.cuh"

namespace mzc {

constexpr int PK_THREADS = 256;             /* segments per tile = threads per CTA of the pass kernels */
constexpr int PK_TILE_SCAN_THREADS = 1024;
constexpr int PKD_THREADS = 32;             /* decrypt: one warp per CTA, one entry per thread */
constexpr uint32_t PK_SEG = 1024;           /* default segment size (bytes); a power of two, 256 .. 65536 */
constexpr uint32_t PK_MUL = 134775813u;
constexpr uint32_t PK_KEY0 = 305419896u, PK_KEY1 = 591751049u, PK_KEY2 = 878082192u;

/* the three keys after the password (host; the shim runs it once per call) */
inline void pk_host_keys(const char *password, uint32_t k[3]) {
    k[0] = PK_KEY0;
    k[1] = PK_KEY1;
    k[2] = PK_KEY2;
    auto reg = [](uint32_t r, uint32_t b) {
        r ^= b & 0xffu;
        for (int i = 0; i < 8; i++) r = (r >> 1) ^ (CRC_POLY & (0u - (r & 1u)));
        return r;
    };
    for (const unsigned char *p = (const unsigned char *)password; *p; p++) {
        k[0] = reg(k[0], *p);
        k[1] = (k[1] + (k[0] & 0xffu)) * PK_MUL + 1u;
        k[2] = reg(k[2], k[1] >> 24);
    }
}

/* per-lane replicated CRC table, built by the CTA itself: lane l's copy of entry e is word e * 32 + l */
__device__ __forceinline__ void pk_build_table(uint32_t *tab) {
    for (uint32_t i = threadIdx.x; i < 256 * 32; i += blockDim.x) {
        uint32_t r = i >> 5;
        for (int b = 0; b < 8; b++) r = (r >> 1) ^ (CRC_POLY & (0u - (r & 1u)));
        tab[i] = r;
    }
}

struct PkTab {
    const uint32_t *t; /* tab + lane */
    __device__ __forceinline__ uint32_t reg(uint32_t r, uint32_t b) const { return t[((r ^ b) & 0xffu) << 5] ^ (r >> 8); }
};

/* key stream byte of key2 */
__device__ __forceinline__ uint32_t pk_stream(uint32_t k2) {
    const uint32_t t = k2 | 2u;
    return ((t * (t ^ 1u)) >> 8) & 0xffu;
}

/* walk the bytes [p, p + len) in order with 16-byte vector loads (and stores when WRITE) between an unaligned head and tail;
 * f(byte) returns the byte to store */
template <bool WRITE, class F>
__device__ __forceinline__ void pk_walk(uint8_t *p, uint64_t len, F &f) {
    uint64_t head = (16u - ((uintptr_t)p & 15u)) & 15u;
    if (head > len) head = len;
    for (uint64_t i = 0; i < head; i++) {
        const uint32_t o = f((uint32_t)p[i]);
        if (WRITE) p[i] = (uint8_t)o;
    }
    uint4 *q = (uint4 *)(p + head);
    const uint64_t nv = (len - head) >> 4;
    for (uint64_t v = 0; v < nv; v++) {
        uint4 w = q[v];
        uint32_t *ww = &w.x;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t x = ww[j];
            const uint32_t o0 = f(x & 0xffu), o1 = f((x >> 8) & 0xffu), o2 = f((x >> 16) & 0xffu), o3 = f(x >> 24);
            if (WRITE) ww[j] = o0 | (o1 << 8) | (o2 << 16) | (o3 << 24);
        }
        if (WRITE) q[v] = w;
    }
    uint8_t *t = p + head + (nv << 4);
    for (uint64_t i = 0; i < ((len - head) & 15u); i++) {
        const uint32_t o = f((uint32_t)t[i]);
        if (WRITE) t[i] = (uint8_t)o;
    }
}

/* x^(8 n) mod P (reflected; bit 31 = x^0), square and multiply from x^8 */
__device__ __forceinline__ uint32_t pk_xpow8(uint32_t n) {
    uint32_t p = 0x80000000u, b = 0x00800000u;
    for (; n; n >>= 1) {
        if (n & 1u) p = gf2_mulmod(p, b);
        b = gf2_mulmod(b, b);
    }
    return p;
}
/* M^n mod 2^32 */
__device__ __forceinline__ uint32_t pk_mulpow(uint32_t n) {
    uint32_t p = 1u, b = PK_MUL;
    for (; n; n >>= 1) {
        if (n & 1u) p *= b;
        b *= b;
    }
    return p;
}

/* the carries: a segment's map as two words. CRC kind (key0, key2): v.x = reg(0, S), v.y = x^(8|S|); k -> k v.y + v.x.
 * Affine kind (key1): v.x = A, v.y = B; k -> A k + B. combine(a, b) = a first, then b. */
template <int AFFINE>
struct PkOp {
    static __device__ __forceinline__ uint2 identity() { return AFFINE ? make_uint2(1u, 0u) : make_uint2(0u, 0x80000000u); }
    static __device__ __forceinline__ uint2 combine(uint2 a, uint2 b) {
        if (AFFINE) return make_uint2(b.x * a.x, b.x * a.y + b.y);
        return make_uint2(gf2_mulmod(a.x, b.y) ^ b.x, gf2_mulmod(a.y, b.y));
    }
    static __device__ __forceinline__ uint32_t apply(uint2 m, uint32_t k) { return AFFINE ? m.x * k + m.y : gf2_mulmod(k, m.y) ^ m.x; }
};

struct PkParams {
    uint8_t *data;              /* entry e = data[off[e] .. off[e] + len[e]), encrypted in place */
    const uint64_t *off, *len;
    uint32_t n;
    uint32_t seg;               /* segment bytes */
    uint32_t nseg, ntiles;
    uint32_t key0, key1, key2;  /* after the password */
    uint32_t xseg, aseg;        /* x^(8 seg) mod P, M^seg mod 2^32: the maps' multipliers of a full segment */
    const uint64_t *seg_base;   /* n + 1: first segment of entry e (exclusive scan of ceil(len / seg)) */
    uint32_t *seg_count;        /* n */
    uint32_t *seg_entry;        /* nseg */
    uint2 *incl[3];             /* per segment: segmented inclusive scan inside its tile, one per carry */
    uint2 *agg[3];              /* per tile: its inclusive value at the last segment */
    uint32_t *aggf[3];          /* per tile: 1 if an entry starts in it */
    uint2 *pre[3];              /* per tile: the carry from the tiles before it (exclusive) */
    uint32_t *ks0, *ks1;        /* per segment: key0, key1 at its start */
};

__global__ void __launch_bounds__(256) pk_count_kernel(PkParams P) {
    for (uint32_t e = blockIdx.x * blockDim.x + threadIdx.x; e < P.n; e += gridDim.x * blockDim.x)
        P.seg_count[e] = (uint32_t)((P.len[e] + P.seg - 1) / P.seg);
}

/* where segment k lies: its entry, its index inside the entry, its bytes */
struct PkSeg {
    uint32_t e, j;
    uint8_t *p;
    uint32_t len;
};
__device__ __forceinline__ PkSeg pk_seg(const PkParams &P, uint32_t k, uint32_t e) {
    PkSeg s;
    s.e = e;
    s.j = (uint32_t)(k - P.seg_base[e]);
    const uint64_t o = (uint64_t)s.j * P.seg, L = P.len[e];
    s.p = P.data + P.off[e] + o;
    s.len = (uint32_t)(L - o < P.seg ? L - o : P.seg);
    return s;
}

/* segmented inclusive scan of one value per thread over the CTA (Hillis-Steele); thread PK_THREADS - 1 writes the tile's
 * aggregate. Flag = the segment starts its entry. */
template <int AFFINE>
__device__ __forceinline__ void pk_tile_scan(const PkParams &P, int which, uint32_t tile, uint32_t k, uint32_t f, uint2 v, uint2 *s_v, uint32_t *s_f) {
    const uint32_t tid = threadIdx.x;
    s_v[tid] = v;
    s_f[tid] = f;
    __syncthreads();
    for (uint32_t d = 1; d < PK_THREADS; d <<= 1) {
        uint2 nv = v;
        uint32_t nf = f;
        if (tid >= d) {
            const uint2 a = s_v[tid - d];
            const uint32_t af = s_f[tid - d];
            if (!f) nv = PkOp<AFFINE>::combine(a, v);
            nf = f | af;
        }
        __syncthreads();
        v = nv;
        f = nf;
        s_v[tid] = v;
        s_f[tid] = f;
        __syncthreads();
    }
    if (k < P.nseg) P.incl[which][k] = v;
    if (tid == PK_THREADS - 1) {
        P.agg[which][tile] = v;
        P.aggf[which][tile] = f;
    }
}

/* the carry at the start of segment k (exclusive inside its entry) applied to the key's value after the password */
template <int AFFINE>
__device__ __forceinline__ uint32_t pk_start(const PkParams &P, int which, uint32_t k, const PkSeg &s, uint32_t key) {
    if (s.j == 0) return key;
    const uint32_t t = (k - 1) / PK_THREADS;
    uint2 m = P.incl[which][k - 1];
    if (P.seg_base[s.e] < (uint64_t)t * PK_THREADS) m = PkOp<AFFINE>::combine(P.pre[which][t], m); /* the entry began in an earlier tile */
    return PkOp<AFFINE>::apply(m, key);
}

#define PK_TILE_LOOP                                                                 \
    for (uint32_t tile = blockIdx.x; tile < P.ntiles; tile += gridDim.x)

/* pass 1: the plaintext's CRC register per segment; also finds every segment's entry */
__global__ void __launch_bounds__(PK_THREADS) pk_pass1_kernel(PkParams P) {
    __shared__ uint32_t s_tab[256 * 32];
    __shared__ uint2 s_v[PK_THREADS];
    __shared__ uint32_t s_f[PK_THREADS];
    pk_build_table(s_tab);
    __syncthreads();
    const PkTab T{s_tab + lane_id()};
    PK_TILE_LOOP {
        const uint32_t k = tile * PK_THREADS + threadIdx.x;
        uint2 v = PkOp<0>::identity();
        uint32_t f = 1;
        if (k < P.nseg) {
            uint32_t lo = 0, hi = P.n; /* the last entry whose first segment is <= k: seg_base[lo] <= k < seg_base[hi] */
            while (hi - lo > 1) {
                const uint32_t mid = (lo + hi) >> 1;
                if (P.seg_base[mid] <= k) lo = mid;
                else hi = mid;
            }
            P.seg_entry[k] = lo;
            const PkSeg s = pk_seg(P, k, lo);
            uint32_t r = 0;
            auto fn = [&](uint32_t b) { r = T.reg(r, b); return b; };
            pk_walk<false>(s.p, s.len, fn);
            v = make_uint2(r, s.len == P.seg ? P.xseg : pk_xpow8(s.len));
            f = s.j == 0;
        }
        pk_tile_scan<0>(P, 0, tile, k, f, v, s_v, s_f);
    }
}

/* pass 2: key0 at the segment's start; the segment's key1 map (A, B) */
__global__ void __launch_bounds__(PK_THREADS) pk_pass2_kernel(PkParams P) {
    __shared__ uint32_t s_tab[256 * 32];
    __shared__ uint2 s_v[PK_THREADS];
    __shared__ uint32_t s_f[PK_THREADS];
    pk_build_table(s_tab);
    __syncthreads();
    const PkTab T{s_tab + lane_id()};
    PK_TILE_LOOP {
        const uint32_t k = tile * PK_THREADS + threadIdx.x;
        uint2 v = PkOp<1>::identity();
        uint32_t f = 1;
        if (k < P.nseg) {
            const PkSeg s = pk_seg(P, k, P.seg_entry[k]);
            uint32_t k0 = pk_start<0>(P, 0, k, s, P.key0);
            P.ks0[k] = k0;
            uint32_t b1 = 0; /* the map applied to 0 is B */
            auto fn = [&](uint32_t b) {
                k0 = T.reg(k0, b);
                b1 = (b1 + (k0 & 0xffu)) * PK_MUL + 1u;
                return b;
            };
            pk_walk<false>(s.p, s.len, fn);
            v = make_uint2(s.len == P.seg ? P.aseg : pk_mulpow(s.len), b1);
            f = s.j == 0;
        }
        pk_tile_scan<1>(P, 1, tile, k, f, v, s_v, s_f);
    }
}

/* pass 3: key1 at the segment's start; the CRC register of the key1 >> 24 bytes (key2's map) */
__global__ void __launch_bounds__(PK_THREADS) pk_pass3_kernel(PkParams P) {
    __shared__ uint32_t s_tab[256 * 32];
    __shared__ uint2 s_v[PK_THREADS];
    __shared__ uint32_t s_f[PK_THREADS];
    pk_build_table(s_tab);
    __syncthreads();
    const PkTab T{s_tab + lane_id()};
    PK_TILE_LOOP {
        const uint32_t k = tile * PK_THREADS + threadIdx.x;
        uint2 v = PkOp<0>::identity();
        uint32_t f = 1;
        if (k < P.nseg) {
            const PkSeg s = pk_seg(P, k, P.seg_entry[k]);
            uint32_t k0 = P.ks0[k];
            uint32_t k1 = pk_start<1>(P, 1, k, s, P.key1);
            P.ks1[k] = k1;
            uint32_t r = 0;
            auto fn = [&](uint32_t b) {
                k0 = T.reg(k0, b);
                k1 = (k1 + (k0 & 0xffu)) * PK_MUL + 1u;
                r = T.reg(r, k1 >> 24);
                return b;
            };
            pk_walk<false>(s.p, s.len, fn);
            v = make_uint2(r, s.len == P.seg ? P.xseg : pk_xpow8(s.len));
            f = s.j == 0;
        }
        pk_tile_scan<0>(P, 2, tile, k, f, v, s_v, s_f);
    }
}

/* pass 4: all three keys known at the segment's start: encrypt in place */
__global__ void __launch_bounds__(PK_THREADS) pk_pass4_kernel(PkParams P) {
    __shared__ uint32_t s_tab[256 * 32];
    pk_build_table(s_tab);
    __syncthreads();
    const PkTab T{s_tab + lane_id()};
    for (uint32_t k = blockIdx.x * PK_THREADS + threadIdx.x; k < P.nseg; k += gridDim.x * PK_THREADS) {
        const PkSeg s = pk_seg(P, k, P.seg_entry[k]);
        uint32_t k0 = P.ks0[k], k1 = P.ks1[k];
        uint32_t k2 = pk_start<0>(P, 2, k, s, P.key2);
        auto fn = [&](uint32_t b) {
            const uint32_t c = b ^ pk_stream(k2);
            k0 = T.reg(k0, b);
            k1 = (k1 + (k0 & 0xffu)) * PK_MUL + 1u;
            k2 = T.reg(k2, k1 >> 24);
            return c;
        };
        pk_walk<true>(s.p, s.len, fn);
    }
}

/* the carry across tiles: segmented exclusive scan of the tile aggregates, one CTA. Each thread folds a run of tiles, the runs
 * are scanned in shared memory, then each thread walks its run again writing the prefixes. */
template <int AFFINE, int WHICH>
__global__ void __launch_bounds__(PK_TILE_SCAN_THREADS, 1) pk_tile_scan_kernel(PkParams P) {
    __shared__ uint2 s_v[PK_TILE_SCAN_THREADS];
    __shared__ uint32_t s_f[PK_TILE_SCAN_THREADS];
    const uint32_t tid = threadIdx.x;
    const uint32_t per = (P.ntiles + PK_TILE_SCAN_THREADS - 1) / PK_TILE_SCAN_THREADS;
    const uint32_t lo = tid * per;
    const uint2 *agg = P.agg[WHICH];
    const uint32_t *aggf = P.aggf[WHICH];
    uint2 v = PkOp<AFFINE>::identity();
    uint32_t f = 0;
    for (uint32_t i = lo; i < lo + per && i < P.ntiles; i++) {
        v = aggf[i] ? agg[i] : PkOp<AFFINE>::combine(v, agg[i]);
        f |= aggf[i];
    }
    s_v[tid] = v;
    s_f[tid] = f;
    __syncthreads();
    for (uint32_t d = 1; d < PK_TILE_SCAN_THREADS; d <<= 1) {
        uint2 nv = v;
        uint32_t nf = f;
        if (tid >= d) {
            if (!f) nv = PkOp<AFFINE>::combine(s_v[tid - d], v);
            nf = f | s_f[tid - d];
        }
        __syncthreads();
        v = nv;
        f = nf;
        s_v[tid] = v;
        s_f[tid] = f;
        __syncthreads();
    }
    uint2 run = tid ? s_v[tid - 1] : PkOp<AFFINE>::identity(); /* the carry into this thread's run */
    for (uint32_t i = lo; i < lo + per && i < P.ntiles; i++) {
        P.pre[WHICH][i] = run;
        run = aggf[i] ? agg[i] : PkOp<AFFINE>::combine(run, agg[i]);
    }
}

/* ---- decryption: one thread per entry ------------------------------------------------------------------------------------ */
struct PkDecParams {
    uint8_t *data;
    const uint64_t *off, *len;
    uint32_t n;
    uint32_t key0, key1, key2;
};

__global__ void __launch_bounds__(PKD_THREADS) pk_decrypt_kernel(PkDecParams P) {
    __shared__ uint32_t s_tab[256 * 32];
    pk_build_table(s_tab);
    __syncthreads();
    const PkTab T{s_tab + lane_id()};
    for (uint32_t e = blockIdx.x * PKD_THREADS + threadIdx.x; e < P.n; e += gridDim.x * PKD_THREADS) {
        uint32_t k0 = P.key0, k1 = P.key1, k2 = P.key2;
        auto fn = [&](uint32_t c) {
            const uint32_t b = c ^ pk_stream(k2);
            k0 = T.reg(k0, b);
            k1 = (k1 + (k0 & 0xffu)) * PK_MUL + 1u;
            k2 = T.reg(k2, k1 >> 24);
            return b;
        };
        pk_walk<true>(P.data + P.off[e], P.len[e], fn);
    }
}

} // namespace mzc
#endif
