/* mz_zip_cuda.c -- batch zip-entry writer on the reference's raw-entry seam (include/mz_zip_cuda.h).
 *
 * What it replaces, per entry, in the reference: mz_zip_entry_write_open(raw = 0) creating a mz_stream_zlib
 * (mz_zip.c:1771-1773), the caller's write loop feeding it (mz_zip_rw.c:1424-1480), the CRC accumulation
 * (mz_zip.c:2062-2064) and mz_zip_entry_close (mz_zip.c:2116-2160). Here the codec work of MANY entries is one
 * K2+K3 launch + one K1 launch + one K4 launch per round, and the container calls run with raw = 1.
 */
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <sys/random.h>

#include "mz_abi.h"
#include "mz_cuda_batch.h"
#include "mz_zip_cuda.h"

#define ZC_CHUNK 65536u
/* internal flag of the native writer next to MZ_ZIP_CUDA_AES: PKWARE traditional encryption (mz_zip_cuda_write_archive_pkcrypt) */
#define ZA_PKCRYPT 0x100u

/* mz_zip.h:25-51 (mz_zip_file): the raw seam takes this struct by pointer and copies it (mz_zip.c:1939) */
typedef struct zc_file_info_s {
    uint16_t version_madeby;
    uint16_t version_needed;
    uint16_t flag;
    uint16_t compression_method;
    time_t modified_date;
    time_t accessed_date;
    time_t creation_date;
    uint32_t crc;
    int64_t compressed_size;
    int64_t uncompressed_size;
    uint16_t filename_size;
    uint16_t extrafield_size;
    uint16_t comment_size;
    uint32_t disk_number;
    int64_t disk_offset;
    uint16_t internal_fa;
    uint32_t external_fa;
    const char *filename;
    const uint8_t *extrafield;
    const char *comment;
    const char *linkname;
    uint16_t zip64;
    uint16_t aes_version;
    uint8_t aes_strength;
    uint16_t pk_verify;
} zc_file_info;

/* the container stays the reference's: these come from the host program (mz_zip.c:1915, 2056, 2272) */
extern int32_t mz_zip_entry_write_open(void *handle, const void *file_info, int16_t compress_level, uint8_t raw, const char *password)
    __attribute__((weak));
extern int32_t mz_zip_entry_write(void *handle, const void *buf, int32_t len) __attribute__((weak));
extern int32_t mz_zip_entry_close_raw(void *handle, int64_t uncompressed_size, uint32_t crc32) __attribute__((weak));
/* reader side (mz_zip.h:115-172) */
extern int32_t mz_zip_goto_first_entry(void *handle) __attribute__((weak));
extern int32_t mz_zip_goto_next_entry(void *handle) __attribute__((weak));
extern int32_t mz_zip_entry_get_info(void *handle, zc_file_info **file_info) __attribute__((weak));
extern int32_t mz_zip_entry_read_open(void *handle, uint8_t raw, const char *password) __attribute__((weak));
extern int32_t mz_zip_entry_read(void *handle, void *buf, int32_t len) __attribute__((weak));
extern int32_t mz_zip_entry_close(void *handle) __attribute__((weak));

uint32_t mz_zip_cuda_abi_file_info_size(void) {
    return (uint32_t)sizeof(zc_file_info);
}

static double now_ms(void) {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec * 1e3 + (double)ts.tv_nsec * 1e-6;
}

typedef struct zc_bufs_s {
    size_t round_bytes;
    uint32_t max_chunks;
    uint64_t stride;
    uint8_t *h_in, *d_in, *d_slots, *d_out, *h_out;
    uint64_t *h_off, *d_off, *d_joined_off, *h_joined_off;
    uint32_t *h_len, *d_len, *d_out_len, *d_residue, *d_crc, *h_crc;
    uint8_t *h_flags, *d_flags;
    uint64_t *h_eoff, *d_eoff, *h_elen, *d_elen; /* per ENTRY: offset / size of the plain bytes (K7) */
    uint8_t *d_digest, *h_digest;                 /* per entry: 32 bytes */
} zc_bufs;

static void zc_free(zc_bufs *b) {
    mz_cuda_host_free(b->h_in);
    mz_cuda_free(b->d_in);
    mz_cuda_free(b->d_slots);
    mz_cuda_free(b->d_out);
    mz_cuda_host_free(b->h_out);
    mz_cuda_host_free(b->h_off);
    mz_cuda_free(b->d_off);
    mz_cuda_free(b->d_joined_off);
    mz_cuda_host_free(b->h_joined_off);
    mz_cuda_host_free(b->h_len);
    mz_cuda_free(b->d_len);
    mz_cuda_free(b->d_out_len);
    mz_cuda_free(b->d_residue);
    mz_cuda_free(b->d_crc);
    mz_cuda_host_free(b->h_crc);
    mz_cuda_host_free(b->h_flags);
    mz_cuda_free(b->d_flags);
    mz_cuda_host_free(b->h_eoff);
    mz_cuda_free(b->d_eoff);
    mz_cuda_host_free(b->h_elen);
    mz_cuda_free(b->d_elen);
    mz_cuda_free(b->d_digest);
    mz_cuda_host_free(b->h_digest);
    memset(b, 0, sizeof(*b));
}

static int zc_alloc(zc_bufs *b, size_t round_bytes, uint32_t max_chunks, int with_join) {
    memset(b, 0, sizeof(*b));
    b->round_bytes = round_bytes;
    b->max_chunks = max_chunks;
    b->stride = mz_cuda_deflate_slot_bound(ZC_CHUNK);
    const size_t slots = (size_t)max_chunks * b->stride;
    b->h_in = (uint8_t *)mz_cuda_host_alloc(round_bytes + 64);
    b->d_in = (uint8_t *)mz_cuda_malloc(round_bytes + 64);
    b->d_slots = (uint8_t *)mz_cuda_malloc(slots);
    b->d_out = with_join ? (uint8_t *)mz_cuda_malloc(slots) : NULL; /* (the native writer assembles its own region instead) */
    b->h_out = with_join ? (uint8_t *)mz_cuda_host_alloc(slots) : NULL;
    b->h_off = (uint64_t *)mz_cuda_host_alloc((size_t)max_chunks * 8);
    b->d_off = (uint64_t *)mz_cuda_malloc((size_t)max_chunks * 8);
    b->d_joined_off = (uint64_t *)mz_cuda_malloc(((size_t)max_chunks + 1) * 8);
    b->h_joined_off = (uint64_t *)mz_cuda_host_alloc(((size_t)max_chunks + 1) * 8);
    b->h_len = (uint32_t *)mz_cuda_host_alloc((size_t)max_chunks * 4);
    b->d_len = (uint32_t *)mz_cuda_malloc((size_t)max_chunks * 4);
    b->d_out_len = (uint32_t *)mz_cuda_malloc((size_t)max_chunks * 4);
    b->d_residue = (uint32_t *)mz_cuda_malloc((size_t)max_chunks * 4);
    b->d_crc = (uint32_t *)mz_cuda_malloc((size_t)max_chunks * 4);
    b->h_crc = (uint32_t *)mz_cuda_host_alloc((size_t)max_chunks * 4);
    b->h_flags = (uint8_t *)mz_cuda_host_alloc(max_chunks);
    b->d_flags = (uint8_t *)mz_cuda_malloc(max_chunks);
    b->h_eoff = (uint64_t *)mz_cuda_host_alloc((size_t)max_chunks * 8); /* an entry has at least one chunk */
    b->d_eoff = (uint64_t *)mz_cuda_malloc((size_t)max_chunks * 8);
    b->h_elen = (uint64_t *)mz_cuda_host_alloc((size_t)max_chunks * 8);
    b->d_elen = (uint64_t *)mz_cuda_malloc((size_t)max_chunks * 8);
    b->d_digest = (uint8_t *)mz_cuda_malloc((size_t)max_chunks * 32);
    b->h_digest = (uint8_t *)mz_cuda_host_alloc((size_t)max_chunks * 32);
    if (!b->h_in || !b->d_in || !b->d_slots || (with_join && (!b->d_out || !b->h_out)) || !b->h_off || !b->d_off || !b->d_joined_off || !b->h_joined_off ||
        !b->h_len || !b->d_len || !b->d_out_len || !b->d_residue || !b->d_crc || !b->h_crc || !b->h_flags || !b->d_flags || !b->h_eoff ||
        !b->d_eoff || !b->h_elen || !b->d_elen || !b->d_digest || !b->h_digest) {
        zc_free(b);
        return 0;
    }
    return 1;
}

static uint32_t chunks_of(int64_t size) {
    return size <= 0 ? 1u : (uint32_t)(((uint64_t)size + ZC_CHUNK - 1) / ZC_CHUNK);
}

/* one round = consecutive entries that fit the staging buffers; prepared (packed, compressed, downloaded) by a
 * worker thread while the caller's thread hands the previous round to the container */
typedef struct zc_round_s {
    zc_bufs b;
    const mz_cuda_zip_item *items;
    uint32_t count, first, last, nch;
    int16_t level;
    uint32_t flags;
    int32_t device, err;
    double pack_ms, gpu_ms;
} zc_round;

static void *zc_prepare(void *arg) {
    zc_round *r = (zc_round *)arg;
    zc_bufs *b = &r->b;
    int32_t err = mz_cuda_set_device(r->device);
    double t0 = now_ms();
    uint32_t last = r->first, nch = 0;
    size_t pos = 0;
    while (last < r->count) {
        const size_t need = ((size_t)r->items[last].size + 15) & ~(size_t)15;
        const uint32_t c = chunks_of(r->items[last].size);
        if (last > r->first && (pos + need > b->round_bytes || nch + c > b->max_chunks))
            break;
        if (r->items[last].size > 0)
            memcpy(b->h_in + pos, r->items[last].data, (size_t)r->items[last].size);
        b->h_eoff[last - r->first] = pos;
        b->h_elen[last - r->first] = (uint64_t)r->items[last].size;
        int64_t left = r->items[last].size;
        for (uint32_t k = 0; k < c; k++) {
            const uint32_t n = left > (int64_t)ZC_CHUNK ? ZC_CHUNK : (uint32_t)left;
            b->h_off[nch] = pos + (uint64_t)k * ZC_CHUNK;
            b->h_len[nch] = n;
            b->h_flags[nch] = (k + 1 == c ? 1u : 0u) | (k > 0 ? 2u : 0u); /* BFINAL on the entry's last chunk; later chunks of an entry may refer back into the one before (MZ_CUDA_FLAG_DICT) */
            left -= n;
            nch++;
        }
        pos += need;
        last++;
    }
    r->last = last;
    r->nch = nch;
    if (!err) err = mz_cuda_memcpy_h2d(b->d_in, b->h_in, pos + 16, NULL);
    if (!err) err = mz_cuda_memcpy_h2d(b->d_off, b->h_off, (size_t)nch * 8, NULL);
    if (!err) err = mz_cuda_memcpy_h2d(b->d_len, b->h_len, (size_t)nch * 4, NULL);
    if (!err) err = mz_cuda_memcpy_h2d(b->d_flags, b->h_flags, nch, NULL);
    double t1 = now_ms();
    /* device: compress, checksum, join; download */
    if (!err) err = mz_cuda_deflate_chunks(b->d_in, 0, 0, b->d_off, b->d_len, b->d_flags, nch, 0, r->level, b->d_slots, b->stride, b->d_out_len, NULL);
    if (!err) err = mz_cuda_crc32_segments(b->d_in, 0, 0, b->d_off, b->d_len, nch, b->d_residue, b->d_crc, NULL);
    if (!err) err = mz_cuda_concat(b->d_slots, b->stride, b->d_out_len, nch, b->d_joined_off, b->d_out, NULL);
    if (!err && (r->flags & MZ_ZIP_CUDA_HASH_SHA256)) { /* K7: SHA-256 of every entry's plain bytes */
        const uint32_t ne = last - r->first;
        err = mz_cuda_memcpy_h2d(b->d_eoff, b->h_eoff, (size_t)ne * 8, NULL);
        if (!err) err = mz_cuda_memcpy_h2d(b->d_elen, b->h_elen, (size_t)ne * 8, NULL);
        if (!err) err = mz_cuda_sha256_batch(b->d_in, b->d_eoff, b->d_elen, ne, b->d_digest, NULL);
        if (!err) err = mz_cuda_memcpy_d2h(b->h_digest, b->d_digest, (size_t)ne * 32, NULL);
    }
    if (!err) err = mz_cuda_memcpy_d2h(b->h_joined_off, b->d_joined_off, ((size_t)nch + 1) * 8, NULL);
    if (!err) err = mz_cuda_memcpy_d2h(b->h_crc, b->d_crc, (size_t)nch * 4, NULL);
    if (!err) err = mz_cuda_stream_sync(NULL);
    if (!err) err = mz_cuda_memcpy_d2h(b->h_out, b->d_out, (size_t)b->h_joined_off[nch], NULL);
    if (!err) err = mz_cuda_stream_sync(NULL);
    r->pack_ms = t1 - t0;
    r->gpu_ms = now_ms() - t1;
    r->err = err;
    return NULL;
}

int32_t mz_zip_cuda_add_buffers(void *zip_handle, const mz_cuda_zip_item *items, uint32_t count, int16_t level, mz_cuda_zip_stats *stats) {
    return mz_zip_cuda_add_buffers_ex(zip_handle, items, count, level, 0, stats);
}

int32_t mz_zip_cuda_add_buffers_ex(void *zip_handle, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                   mz_cuda_zip_stats *stats) {
    zc_round rd[2];
    int32_t err = MZ_OK;
    mz_cuda_zip_stats st;
    memset(&st, 0, sizeof(st));
    memset(rd, 0, sizeof(rd));
    if (!mz_zip_entry_write_open || !mz_zip_entry_write || !mz_zip_entry_close_raw)
        return MZ_SUPPORT_ERROR; /* no zip container in this process */
    if (!zip_handle || (!items && count))
        return MZ_PARAM_ERROR;
    if (level == MZ_COMPRESS_LEVEL_DEFAULT)
        level = 6;
    if (level < 0 || level > 9)
        return MZ_PARAM_ERROR;
    if (mz_cuda_init() != MZ_OK) {
        fprintf(stderr, "mz_zip_cuda: no usable sm_100 GPU (%s); there is no CPU fallback\n", mz_cuda_last_error());
        return MZ_SUPPORT_ERROR;
    }
    for (uint32_t i = 0; i < count; i++)
        if (!items[i].filename || items[i].size < 0 || (items[i].size > 0 && !items[i].data))
            return MZ_PARAM_ERROR;
    if (count == 0) {
        if (stats)
            *stats = st;
        return MZ_OK;
    }
    size_t round_bytes = 256u << 20;
    {
        const char *v = getenv("MZ_CUDA_ZIP_ROUND_MB");
        if (v && atoll(v) > 0)
            round_bytes = (size_t)atoll(v) << 20;
    }
    /* an entry is never split over rounds: the round must hold the largest one */
    for (uint32_t i = 0; i < count; i++)
        if ((size_t)items[i].size + 16 > round_bytes)
            round_bytes = ((size_t)items[i].size + 16 + 65535) & ~(size_t)65535;
    /* chunks per round: full chunks by size plus one (partial or empty) chunk per entry; size the tables for the
     * densest window of the actual input (entries are packed at 16-byte aligned offsets) */
    uint32_t max_chunks = (uint32_t)(round_bytes / ZC_CHUNK) + 1;
    {
        uint32_t j = 0, ch = 0, best = 0;
        size_t bytes = 0;
        for (uint32_t i = 0; i < count; i++) {
            bytes += ((size_t)items[i].size + 15) & ~(size_t)15;
            ch += chunks_of(items[i].size);
            while (bytes > round_bytes) {
                bytes -= ((size_t)items[j].size + 15) & ~(size_t)15;
                ch -= chunks_of(items[j].size);
                j++;
            }
            if (ch > best)
                best = ch;
        }
        if (best + 1 > max_chunks)
            max_chunks = best + 1;
    }
    const int32_t device = mz_cuda_get_device();
    for (int k = 0; k < 2; k++) {
        if (!zc_alloc(&rd[k].b, round_bytes, max_chunks, 1)) {
            zc_free(&rd[0].b);
            return MZ_MEM_ERROR;
        }
        rd[k].items = items;
        rd[k].count = count;
        rd[k].level = level;
        rd[k].flags = flags;
        rd[k].device = device < 0 ? 0 : device;
    }
    /* round r is prepared by a worker while this thread feeds round r-1 to the container */
    int cur = 0;
    pthread_t th;
    rd[cur].first = 0;
    zc_prepare(&rd[cur]);
    while (err == MZ_OK) {
        zc_round *r = &rd[cur];
        err = r->err;
        if (err)
            break;
        int have_next = r->last < count, started = 0;
        if (have_next) {
            rd[cur ^ 1].first = r->last;
            started = pthread_create(&th, NULL, zc_prepare, &rd[cur ^ 1]) == 0;
            if (!started)
                zc_prepare(&rd[cur ^ 1]);
        }
        /* ---- container: the reference writes headers and copies the finished streams --------------------------- */
        double t2 = now_ms();
        const zc_bufs *b = &r->b;
        uint32_t c0 = 0;
        for (uint32_t i = r->first; i < r->last && err == MZ_OK; i++) {
            const uint32_t c = chunks_of(items[i].size);
            uint32_t crc = b->h_crc[c0];
            for (uint32_t k = 1; k < c; k++)
                crc = mz_cuda_crc32_combine(crc, b->h_crc[c0 + k], b->h_len[c0 + k]);
            if (items[i].size == 0)
                crc = 0;
            const uint8_t *comp = b->h_out + b->h_joined_off[c0];
            const uint64_t csize = b->h_joined_off[c0 + c] - b->h_joined_off[c0];
            zc_file_info fi;
            memset(&fi, 0, sizeof(fi));
            fi.version_madeby = (3u << 8) | 45u; /* MZ_HOST_SYSTEM_UNIX (mz.h:104), zip 4.5 as MZ_VERSION_MADEBY without extra codecs (mz_os.h:27-42) */
            /* MZ_ZIP_FLAG_UTF8 (mz.h:84) | MZ_ZIP_FLAG_DATA_DESCRIPTOR (mz.h:83): like the reference's own compressed
             * entries (mz_zip.c:1992) the sizes follow the data, so close_raw never seeks back to patch the header */
            fi.flag = (1u << 11) | (1u << 3);
            fi.compression_method = 8;           /* MZ_COMPRESS_METHOD_DEFLATE, mz.h:64 */
            fi.modified_date = items[i].modified_date ? (time_t)items[i].modified_date : time(NULL);
            fi.crc = crc;
            fi.compressed_size = (int64_t)csize;
            fi.uncompressed_size = items[i].size;
            fi.external_fa = items[i].external_fa ? items[i].external_fa : (0100644u << 16);
            fi.filename = items[i].filename;
            uint8_t xf[40];
            if (flags & MZ_ZIP_CUDA_HASH_SHA256) {
                /* MZ_ZIP_EXTENSION_HASH (mz.h:93): id, field length 4 + 32, algorithm MZ_HASH_SHA256 (mz.h:131), digest size, digest --
                 * the bytes mz_zip_writer_entry_close assembles (mz_zip_rw.c:1398-1408) */
                static const uint8_t head[8] = {0x51, 0x1a, 36, 0, 23, 0, 32, 0};
                memcpy(xf, head, 8);
                memcpy(xf + 8, b->h_digest + (size_t)(i - r->first) * 32, 32);
                fi.extrafield = xf;
                fi.extrafield_size = 40;
            }
            err = mz_zip_entry_write_open(zip_handle, &fi, level, 1, NULL);
            uint64_t done = 0;
            while (err == MZ_OK && done < csize) {
                const int32_t piece = csize - done > (1u << 30) ? (int32_t)(1u << 30) : (int32_t)(csize - done);
                const int32_t w = mz_zip_entry_write(zip_handle, comp + done, piece);
                if (w != piece)
                    err = w < 0 ? w : MZ_WRITE_ERROR;
                done += (uint64_t)piece;
            }
            if (err == MZ_OK)
                err = mz_zip_entry_close_raw(zip_handle, items[i].size, crc);
            st.bytes_in += (uint64_t)items[i].size;
            st.bytes_out += csize;
            c0 += c;
        }
        st.container_ms += now_ms() - t2;
        st.pack_ms += r->pack_ms;
        st.gpu_ms += r->gpu_ms;
        st.entries += r->last - r->first;
        st.rounds++;
        if (started)
            pthread_join(th, NULL);
        if (!have_next)
            break;
        cur ^= 1;
    }
    zc_free(&rd[0].b);
    zc_free(&rd[1].b);
    if (stats)
        *stats = st;
    return err;
}

/* ---- the native archive writer (mz_zip_cuda_write_archive) ------------------------------------------------------------- */
typedef struct za_meta_s { /* per entry of a round, filled by the worker */
    uint64_t csize, lh_rel; /* compressed bytes; offset of the local header inside the round's region */
    uint32_t crc, lh_size;
} za_meta;

typedef struct za_slot_s {
    zc_bufs b;
    uint32_t *h_out_len;               /* pinned: per chunk */
    uint64_t *h_dst_off, *d_dst_off;   /* per chunk: where its stream goes inside the region */
    uint64_t *h_hdr_off, *d_hdr_off;   /* per entry: where its local header goes */
    uint32_t *h_blob_off, *d_blob_off; /* per entry + 1: header bytes inside the blob */
    uint8_t *h_blob, *d_blob;
    size_t blob_cap;
    uint8_t *d_region, *h_region;
    size_t region_cap;
    za_meta *meta;
    /* the round in flight */
    const mz_cuda_zip_item *items;
    uint32_t first, last, nch;
    uint32_t flags;
    int16_t level;
    int32_t device, err;
    uint64_t region_len;
    double pack_ms, gpu_ms;
    void *stream; /* the slot's own CUDA stream: rounds of different slots (and devices) overlap */
    /* WinZip AES (flag MZ_ZIP_CUDA_AES): per entry a salt, derived keys, where its ciphertext lies in the region, its HMAC */
    const char *password;
    uint32_t strength, pw_len;
    uint8_t *h_salt, *d_salt, *h_keys, *d_keys, *d_pw, *h_mac, *d_mac;
    uint64_t *h_coff, *d_coff, *h_clen, *d_clen;
    /* PKWARE (internal flag ZA_PKCRYPT): the salt, offset and length tables above (10 random header bytes per entry, its
     * encryption header + stream) and K9's workspace */
    uint8_t *d_pkws;
    uint64_t pkws_bytes;
    pthread_t th;
    int running;
    int has_aes; /* the AES buffers exist (pool matching) */
    int has_pk;  /* the PKWARE buffers exist */
} za_slot;

static void put16(uint8_t *p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); }
static void put32(uint8_t *p, uint32_t v) { put16(p, v); put16(p + 2, v >> 16); }
static void put64(uint8_t *p, uint64_t v) { put32(p, (uint32_t)v); put32(p + 4, (uint32_t)(v >> 32)); }

/* mz_zip_time_t_to_dos_date (mz_zip.c): local time, 2-second resolution, years from 1980 */
static uint32_t za_dos_date(int64_t t) {
    static __thread int64_t last_t = -1; /* archives carry few distinct dates: localtime_r once per run of equal ones */
    static __thread uint32_t last_v;
    if (t && t == last_t)
        return last_v;
    time_t tt = (time_t)(t ? t : time(NULL));
    struct tm tmv;
    if (!localtime_r(&tt, &tmv))
        return 0;
    int year = tmv.tm_year >= 1980 ? tmv.tm_year - 1980 : (tmv.tm_year >= 80 ? tmv.tm_year - 80 : 0);
    last_v = ((uint32_t)((tmv.tm_mday) + 32 * (tmv.tm_mon + 1) + 512 * year) << 16) |
             (uint32_t)(tmv.tm_sec / 2 + 32 * tmv.tm_min + 2048 * tmv.tm_hour);
    last_t = t;
    return last_v;
}

static void za_free(za_slot *z) {
    zc_free(&z->b);
    if (z->stream)
        mz_cuda_stream_destroy(z->stream);
    mz_cuda_host_free(z->h_out_len);
    mz_cuda_host_free(z->h_dst_off);
    mz_cuda_free(z->d_dst_off);
    mz_cuda_host_free(z->h_hdr_off);
    mz_cuda_free(z->d_hdr_off);
    mz_cuda_host_free(z->h_blob_off);
    mz_cuda_free(z->d_blob_off);
    mz_cuda_host_free(z->h_blob);
    mz_cuda_free(z->d_blob);
    mz_cuda_free(z->d_region);
    mz_cuda_host_free(z->h_region);
    mz_cuda_host_free(z->h_salt);
    mz_cuda_free(z->d_salt);
    mz_cuda_host_free(z->h_keys);
    mz_cuda_free(z->d_keys);
    mz_cuda_free(z->d_pw);
    mz_cuda_host_free(z->h_mac);
    mz_cuda_free(z->d_mac);
    mz_cuda_host_free(z->h_coff);
    mz_cuda_free(z->d_coff);
    mz_cuda_host_free(z->h_clen);
    mz_cuda_free(z->d_clen);
    mz_cuda_free(z->d_pkws);
    free(z->meta);
    memset(z, 0, sizeof(*z));
}

static int za_alloc(za_slot *z, size_t round_bytes, uint32_t max_chunks, size_t blob_cap, int aes, int pk) {
    memset(z, 0, sizeof(*z));
    z->has_aes = aes;
    z->has_pk = pk;
    if (!zc_alloc(&z->b, round_bytes, max_chunks, 0))
        return 0;
    z->blob_cap = blob_cap;
    z->region_cap = (size_t)max_chunks * z->b.stride + blob_cap + 64;
    z->h_out_len = (uint32_t *)mz_cuda_host_alloc((size_t)max_chunks * 4);
    z->h_dst_off = (uint64_t *)mz_cuda_host_alloc((size_t)max_chunks * 8);
    z->d_dst_off = (uint64_t *)mz_cuda_malloc((size_t)max_chunks * 8);
    z->h_hdr_off = (uint64_t *)mz_cuda_host_alloc((size_t)max_chunks * 8);
    z->d_hdr_off = (uint64_t *)mz_cuda_malloc((size_t)max_chunks * 8);
    z->h_blob_off = (uint32_t *)mz_cuda_host_alloc(((size_t)max_chunks + 1) * 4);
    z->d_blob_off = (uint32_t *)mz_cuda_malloc(((size_t)max_chunks + 1) * 4);
    z->h_blob = (uint8_t *)mz_cuda_host_alloc(blob_cap + 16);
    z->d_blob = (uint8_t *)mz_cuda_malloc(blob_cap + 16);
    z->d_region = (uint8_t *)mz_cuda_malloc(z->region_cap);
    z->h_region = (uint8_t *)mz_cuda_host_alloc(z->region_cap);
    z->meta = (za_meta *)malloc((size_t)max_chunks * sizeof(za_meta));
    z->stream = mz_cuda_stream_create();
    if (aes || pk) {
        z->h_salt = (uint8_t *)mz_cuda_host_alloc((size_t)max_chunks * 16);
        z->h_coff = (uint64_t *)mz_cuda_host_alloc((size_t)max_chunks * 8);
        z->d_coff = (uint64_t *)mz_cuda_malloc((size_t)max_chunks * 8);
        z->h_clen = (uint64_t *)mz_cuda_host_alloc((size_t)max_chunks * 8);
        z->d_clen = (uint64_t *)mz_cuda_malloc((size_t)max_chunks * 8);
        if (!z->h_salt || !z->h_coff || !z->d_coff || !z->h_clen || !z->d_clen) {
            za_free(z);
            return 0;
        }
    }
    if (pk) { /* the encrypted ranges of a round lie inside its region, one per entry (an entry has at least one chunk) */
        z->pkws_bytes = mz_cuda_pkcrypt_workspace_bytes(z->region_cap, max_chunks);
        z->d_pkws = (uint8_t *)mz_cuda_malloc(z->pkws_bytes);
        if (!z->d_pkws) {
            za_free(z);
            return 0;
        }
    }
    if (aes) {
        z->d_salt = (uint8_t *)mz_cuda_malloc((size_t)max_chunks * 16);
        z->h_keys = (uint8_t *)mz_cuda_host_alloc((size_t)max_chunks * MZ_CUDA_WZAES_KEYREC);
        z->d_keys = (uint8_t *)mz_cuda_malloc((size_t)max_chunks * MZ_CUDA_WZAES_KEYREC);
        z->d_pw = (uint8_t *)mz_cuda_malloc(256);
        z->h_mac = (uint8_t *)mz_cuda_host_alloc((size_t)max_chunks * 20);
        z->d_mac = (uint8_t *)mz_cuda_malloc((size_t)max_chunks * 20);
        if (!z->d_salt || !z->h_keys || !z->d_keys || !z->d_pw || !z->h_mac || !z->d_mac) {
            za_free(z);
            return 0;
        }
    }
    if (!z->stream || !z->h_out_len || !z->h_dst_off || !z->d_dst_off || !z->h_hdr_off || !z->d_hdr_off || !z->h_blob_off || !z->d_blob_off || !z->h_blob ||
        !z->d_blob || !z->d_region || !z->h_region || !z->meta) {
        za_free(z);
        return 0;
    }
    return 1;
}

/* Staging pool: a slot is ~130 MiB of page-locked and ~200 MiB of device memory, and making four of them costs more than half a
 * second -- as much as compressing 2 GiB. A process that writes archive after archive keeps up to eight idle slots (per device,
 * matched by capacity); MZ_CUDA_ZIP_POOL=0 turns the pool off, mz_zip_cuda_trim() empties it. */
#define ZA_POOL_MAX 8
static pthread_mutex_t g_za_mu = PTHREAD_MUTEX_INITIALIZER;
static za_slot g_za_pool[ZA_POOL_MAX];
static int g_za_n;

static int za_pool_enabled(void) {
    const char *v = getenv("MZ_CUDA_ZIP_POOL");
    return !(v && v[0] == '0');
}

static int za_acquire(za_slot *z, int32_t dev, size_t round_bytes, uint32_t max_chunks, size_t blob_cap, int aes, int pk) {
    int hit = 0;
    pthread_mutex_lock(&g_za_mu);
    for (int i = 0; i < g_za_n; i++) {
        const za_slot *q = &g_za_pool[i];
        if (q->device == dev && q->b.round_bytes >= round_bytes && q->b.max_chunks >= max_chunks && q->blob_cap >= blob_cap && (q->has_aes || !aes) &&
            (q->has_pk || !pk)) {
            *z = *q;
            g_za_pool[i] = g_za_pool[--g_za_n];
            hit = 1;
            break;
        }
    }
    pthread_mutex_unlock(&g_za_mu);
    if (hit) {
        z->items = NULL;
        z->first = z->last = z->nch = 0;
        z->err = 0;
        z->region_len = 0;
        z->pack_ms = z->gpu_ms = 0;
        z->running = 0;
        z->password = NULL;
        return 1;
    }
    if (!za_alloc(z, round_bytes, max_chunks, blob_cap, aes, pk))
        return 0;
    z->device = dev;
    return 1;
}

static void za_release(za_slot *z) {
    int kept = 0;
    if (z->b.h_in && za_pool_enabled()) {
        pthread_mutex_lock(&g_za_mu);
        if (g_za_n < ZA_POOL_MAX) {
            g_za_pool[g_za_n++] = *z;
            kept = 1;
        }
        pthread_mutex_unlock(&g_za_mu);
    }
    if (kept)
        memset(z, 0, sizeof(*z));
    else
        za_free(z);
}

void mz_zip_cuda_trim(void) {
    const int32_t dev0 = mz_cuda_get_device();
    pthread_mutex_lock(&g_za_mu);
    for (int i = 0; i < g_za_n; i++) {
        mz_cuda_set_device(g_za_pool[i].device);
        za_free(&g_za_pool[i]);
    }
    g_za_n = 0;
    pthread_mutex_unlock(&g_za_mu);
    if (dev0 >= 0)
        mz_cuda_set_device(dev0);
}

/* the hash extra field of an entry (40 bytes) -- the bytes mz_zip_writer_entry_close assembles (mz_zip_rw.c:1398-1408) */
static void za_hash_field(uint8_t *xf, const uint8_t *digest) {
    static const uint8_t head[8] = {0x51, 0x1a, 36, 0, 23, 0, 32, 0};
    memcpy(xf, head, 8);
    memcpy(xf + 8, digest, 32);
}

/* the AES extra field of an entry (11 bytes): id 0x9901, size 7, AE version, vendor "AE", strength, the real method
 * (mz_zip.c:870-885) */
static void za_aes_field(uint8_t *xf, uint32_t strength) {
    const uint8_t f[11] = {0x01, 0x99, 7, 0, 1, 0, 'A', 'E', (uint8_t)strength, 8, 0};
    memcpy(xf, f, 11);
}

/* one round: pack, upload, compress + checksum (+ hash), lay the region out, assemble it on the device, download it */
static void *za_prepare(void *arg) {
    za_slot *z = (za_slot *)arg;
    zc_bufs *b = &z->b;
    int32_t err = mz_cuda_set_device(z->device);
    double t0 = now_ms();
    uint32_t nch = 0;
    size_t pos = 0;
    const uint32_t ne = z->last - z->first;
    for (uint32_t i = z->first; i < z->last; i++) {
        const mz_cuda_zip_item *it = &z->items[i];
        const uint32_t c = chunks_of(it->size);
        if (it->size > 0)
            memcpy(b->h_in + pos, it->data, (size_t)it->size);
        b->h_eoff[i - z->first] = pos;
        b->h_elen[i - z->first] = (uint64_t)it->size;
        int64_t left = it->size;
        for (uint32_t k = 0; k < c; k++) {
            const uint32_t n = left > (int64_t)ZC_CHUNK ? ZC_CHUNK : (uint32_t)left;
            b->h_off[nch] = pos + (uint64_t)k * ZC_CHUNK;
            b->h_len[nch] = n;
            b->h_flags[nch] = (k + 1 == c ? 1u : 0u) | (k > 0 ? 2u : 0u); /* FINAL | DICT, as above */
            left -= n;
            nch++;
        }
        pos += ((size_t)it->size + 15) & ~(size_t)15;
    }
    z->nch = nch;
    if (!err) err = mz_cuda_memcpy_h2d(b->d_in, b->h_in, pos + 16, z->stream);
    if (!err) err = mz_cuda_memcpy_h2d(b->d_off, b->h_off, (size_t)nch * 8, z->stream);
    if (!err) err = mz_cuda_memcpy_h2d(b->d_len, b->h_len, (size_t)nch * 4, z->stream);
    if (!err) err = mz_cuda_memcpy_h2d(b->d_flags, b->h_flags, nch, z->stream);
    double t1 = now_ms();
    const int aes = (z->flags & MZ_ZIP_CUDA_AES) != 0, pk = (z->flags & ZA_PKCRYPT) != 0;
    const uint32_t slen = aes ? 4 * z->strength + 4 : 0; /* MZ_AES_SALT_LENGTH */
    /* bytes between an entry's local header and its stream: AES salt + verifier, or the PKWARE encryption header */
    const uint32_t xenc = aes ? slen + 2 : (pk ? 12u : 0u);
    if (!err && (aes || pk)) { /* fresh random bytes per entry: the AES salt (mz_strm_wzaes.c:85-86), the PKWARE header's first 10 (mz_strm_pkcrypt.c:112-113) */
        size_t got = 0;
        while (got < (size_t)ne * 16) {
            ssize_t k = getrandom(z->h_salt + got, (size_t)ne * 16 - got, 0);
            if (k <= 0) { err = MZ_INTERNAL_ERROR; break; }
            got += (size_t)k;
        }
    }
    if (!err && aes) { /* every entry's keys and password verifier by K8 */
        err = mz_cuda_memcpy_h2d(z->d_salt, z->h_salt, (size_t)ne * 16, z->stream);
        if (!err) err = mz_cuda_memcpy_h2d(z->d_pw, z->password, z->pw_len ? z->pw_len : 1, z->stream);
        if (!err) err = mz_cuda_wzaes_derive(z->d_pw, z->pw_len, z->d_salt, ne, z->strength, z->d_keys, z->stream);
        if (!err) err = mz_cuda_memcpy_d2h(z->h_keys, z->d_keys, (size_t)ne * MZ_CUDA_WZAES_KEYREC, z->stream);
    }
    if (!err) err = mz_cuda_deflate_chunks(b->d_in, 0, 0, b->d_off, b->d_len, b->d_flags, nch, 0, z->level, b->d_slots, b->stride, b->d_out_len, z->stream);
    if (!err) err = mz_cuda_crc32_segments(b->d_in, 0, 0, b->d_off, b->d_len, nch, b->d_residue, b->d_crc, z->stream);
    if (!err && (z->flags & MZ_ZIP_CUDA_HASH_SHA256)) {
        err = mz_cuda_memcpy_h2d(b->d_eoff, b->h_eoff, (size_t)ne * 8, z->stream);
        if (!err) err = mz_cuda_memcpy_h2d(b->d_elen, b->h_elen, (size_t)ne * 8, z->stream);
        if (!err) err = mz_cuda_sha256_batch(b->d_in, b->d_eoff, b->d_elen, ne, b->d_digest, z->stream);
        if (!err) err = mz_cuda_memcpy_d2h(b->h_digest, b->d_digest, (size_t)ne * 32, z->stream);
    }
    if (!err) err = mz_cuda_memcpy_d2h(z->h_out_len, b->d_out_len, (size_t)nch * 4, z->stream);
    if (!err) err = mz_cuda_memcpy_d2h(b->h_crc, b->d_crc, (size_t)nch * 4, z->stream);
    if (!err) err = mz_cuda_stream_sync(z->stream);
    /* host: sizes, CRCs, local headers, the region's layout */
    uint64_t cur = 0, max_clen = 0;
    uint32_t c0 = 0, bo = 0;
    for (uint32_t e = 0; e < ne && !err; e++) {
        const mz_cuda_zip_item *it = &z->items[z->first + e];
        const uint32_t c = chunks_of(it->size);
        uint32_t crc = b->h_crc[c0];
        uint64_t csize = z->h_out_len[c0];
        for (uint32_t k = 1; k < c; k++) {
            crc = mz_cuda_crc32_combine(crc, b->h_crc[c0 + k], b->h_len[c0 + k]);
            csize += z->h_out_len[c0 + k];
        }
        if (it->size == 0)
            crc = 0;
        const size_t nlen = strlen(it->filename);
        const uint32_t xaes = aes ? 11u : 0u;
        const uint32_t xlen = xaes + ((z->flags & MZ_ZIP_CUDA_HASH_SHA256) ? 40u : 0u);
        const uint32_t lh = 30 + (uint32_t)nlen + xlen;
        /* salt | verifier | ciphertext | authentication code, or encryption header | ciphertext */
        const uint64_t stored = csize + (aes ? slen + 2 + 10 : (pk ? 12u : 0u));
        if (bo + lh + xenc > z->blob_cap || stored >= 0xffffffffull) {
            err = MZ_INTERNAL_ERROR;
            break;
        }
        uint8_t *h = z->h_blob + bo;
        put32(h, 0x04034b50u);                       /* MZ_ZIP_MAGIC_LOCALHEADER */
        put16(h + 4, aes ? 51 : 20);                 /* version needed (mz_zip.c:703-725) */
        put16(h + 6, (1u << 11) | (aes || pk ? 1u : 0u)); /* MZ_ZIP_FLAG_UTF8 (| MZ_ZIP_FLAG_ENCRYPTED); no data descriptor: everything is known */
        put16(h + 8, aes ? 99 : 8);                  /* MZ_COMPRESS_METHOD_DEFLATE, or _AES with the real method in the extra field (:728-733) */
        put32(h + 10, za_dos_date(it->modified_date));
        put32(h + 14, crc);                          /* AE-1 (MZ_AES_VERSION 1) keeps the CRC (mz_zip.c:2117-2121) */
        put32(h + 18, (uint32_t)stored);
        put32(h + 22, (uint32_t)it->size);
        put16(h + 26, (uint32_t)nlen);
        put16(h + 28, xlen);
        memcpy(h + 30, it->filename, nlen);
        if (aes)
            za_aes_field(h + 30 + nlen, z->strength);
        if (xlen > xaes)
            za_hash_field(h + 30 + nlen + xaes, b->h_digest + (size_t)e * 32);
        if (aes) { /* salt and password verifier travel with the header blob (mz_strm_wzaes.c:116-125) */
            memcpy(h + lh, z->h_salt + (size_t)e * 16, slen);
            memcpy(h + lh + slen, z->h_keys + (size_t)e * MZ_CUDA_WZAES_KEYREC + 64, 2);
        }
        if (pk) { /* the PKWARE encryption header, still plain: 10 random bytes and the CRC's high bytes -- mz_zip_get_pk_verify for an entry
                   * without a data descriptor (mz_zip.c:192-199); K9 encrypts it with the stream */
            memcpy(h + lh, z->h_salt + (size_t)e * 16, 10);
            h[lh + 10] = (uint8_t)(crc >> 16);
            h[lh + 11] = (uint8_t)(crc >> 24);
            z->h_coff[e] = cur + lh;
            z->h_clen[e] = csize + 12;
        }
        z->h_blob_off[e] = bo;
        z->h_hdr_off[e] = cur;
        z->meta[e].csize = stored;
        z->meta[e].crc = crc;
        z->meta[e].lh_rel = cur;
        z->meta[e].lh_size = lh;
        bo += lh + xenc;
        cur += lh + xenc;
        if (aes) {
            z->h_coff[e] = cur;
            z->h_clen[e] = csize;
            if (csize > max_clen) max_clen = csize;
        }
        for (uint32_t k = 0; k < c; k++) {
            z->h_dst_off[c0 + k] = cur;
            cur += z->h_out_len[c0 + k];
        }
        if (aes)
            cur += 10; /* MZ_AES_AUTHCODE_SIZE */
        c0 += c;
    }
    z->h_blob_off[ne] = bo;
    z->region_len = cur;
    if (!err && cur > z->region_cap)
        err = MZ_INTERNAL_ERROR;
    /* device: streams and headers into place; the finished region comes down in one copy */
    if (!err) err = mz_cuda_memcpy_h2d(z->d_dst_off, z->h_dst_off, (size_t)nch * 8, z->stream);
    if (!err) err = mz_cuda_memcpy_h2d(z->d_hdr_off, z->h_hdr_off, (size_t)ne * 8, z->stream);
    if (!err) err = mz_cuda_memcpy_h2d(z->d_blob_off, z->h_blob_off, ((size_t)ne + 1) * 4, z->stream);
    if (!err) err = mz_cuda_memcpy_h2d(z->d_blob, z->h_blob, (size_t)bo + 16, z->stream);
    if (!err) err = mz_cuda_gather(b->d_slots, b->stride, b->d_out_len, nch, z->d_dst_off, z->d_region, z->stream);
    if (!err) err = mz_cuda_scatter_blobs(z->d_blob, z->d_blob_off, z->d_hdr_off, ne, z->d_region, z->stream);
    if (!err && pk) { /* K9: every entry's encryption header + stream becomes ciphertext in place */
        err = mz_cuda_memcpy_h2d(z->d_coff, z->h_coff, (size_t)ne * 8, z->stream);
        if (!err) err = mz_cuda_memcpy_h2d(z->d_clen, z->h_clen, (size_t)ne * 8, z->stream);
        if (!err) err = mz_cuda_pkcrypt_encrypt(z->d_region, z->d_coff, z->d_clen, ne, z->password, z->d_pkws, z->pkws_bytes, z->stream);
    }
    if (!err && aes) { /* the assembled streams become ciphertext in place; their HMACs follow them down */
        err = mz_cuda_memcpy_h2d(z->d_coff, z->h_coff, (size_t)ne * 8, z->stream);
        if (!err) err = mz_cuda_memcpy_h2d(z->d_clen, z->h_clen, (size_t)ne * 8, z->stream);
        if (!err) err = mz_cuda_wzaes_ctr(z->d_region, z->d_coff, z->d_clen, ne, max_clen, z->d_keys, z->strength, z->stream);
        if (!err) err = mz_cuda_wzaes_hmac(z->d_region, z->d_coff, z->d_clen, ne, z->d_keys, z->strength, z->d_mac, z->stream);
        if (!err) err = mz_cuda_memcpy_d2h(z->h_mac, z->d_mac, (size_t)ne * 20, z->stream);
    }
    if (!err) err = mz_cuda_memcpy_d2h(z->h_region, z->d_region, (size_t)cur, z->stream);
    if (!err) err = mz_cuda_stream_sync(z->stream);
    for (uint32_t e = 0; e < ne && !err && aes; e++) /* authentication code = the first 10 bytes of the HMAC (mz_strm_wzaes.c:243-247) */
        memcpy(z->h_region + z->h_coff[e] + z->h_clen[e], z->h_mac + (size_t)e * 20, 10);
    z->pack_ms = t1 - t0;
    z->gpu_ms = now_ms() - t1;
    z->err = err;
    return NULL;
}

typedef struct za_cd_s {
    uint8_t *p;
    size_t len, cap;
} za_cd;
static uint8_t *za_cd_room(za_cd *cd, size_t n) {
    if (cd->len + n > cd->cap) {
        size_t ncap = cd->cap ? cd->cap * 2 : (1u << 20);
        while (ncap < cd->len + n)
            ncap *= 2;
        uint8_t *q = (uint8_t *)realloc(cd->p, ncap);
        if (!q)
            return NULL;
        cd->p = q;
        cd->cap = ncap;
    }
    uint8_t *r = cd->p + cd->len;
    cd->len += n;
    return r;
}

static int32_t za_write(void *base, const uint8_t *p, uint64_t n) {
    while (n > 0) {
        const int32_t part = n > (1u << 30) ? (int32_t)(1u << 30) : (int32_t)n;
        if (mz_abi_base_write(base, p, part) != part)
            return MZ_WRITE_ERROR;
        p += part;
        n -= (uint64_t)part;
    }
    return MZ_OK;
}

int32_t mz_zip_cuda_write_archive(void *base_stream, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                  mz_cuda_zip_stats *stats) {
    if (flags & MZ_ZIP_CUDA_AES)
        return MZ_PARAM_ERROR; /* needs a password: mz_zip_cuda_write_archive_aes */
    return mz_zip_cuda_write_archive_aes(base_stream, items, count, level, flags, NULL, 0, stats);
}

static int32_t za_write_archive(void *base_stream, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                const char *password, uint8_t aes_strength, mz_cuda_zip_stats *stats);

int32_t mz_zip_cuda_write_archive_aes(void *base_stream, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                      const char *password, uint8_t aes_strength, mz_cuda_zip_stats *stats) {
    return za_write_archive(base_stream, items, count, level, flags & ~ZA_PKCRYPT, password, aes_strength, stats);
}

int32_t mz_zip_cuda_write_archive_pkcrypt(void *base_stream, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                          const char *password, mz_cuda_zip_stats *stats) {
    if ((flags & MZ_ZIP_CUDA_AES) || !password)
        return MZ_PARAM_ERROR;
    return za_write_archive(base_stream, items, count, level, flags | ZA_PKCRYPT, password, 0, stats);
}

static int32_t za_write_archive(void *base_stream, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                const char *password, uint8_t aes_strength, mz_cuda_zip_stats *stats) {
    mz_cuda_zip_stats st;
    int32_t err = MZ_OK;
    memset(&st, 0, sizeof(st));
    if (!base_stream || (!items && count))
        return MZ_PARAM_ERROR;
    if (level == MZ_COMPRESS_LEVEL_DEFAULT)
        level = 6;
    if (level < 0 || level > 9)
        return MZ_PARAM_ERROR;
    const int aes = (flags & MZ_ZIP_CUDA_AES) != 0, pk = (flags & ZA_PKCRYPT) != 0;
    if (aes_strength == 0)
        aes_strength = 3; /* MZ_AES_STRENGTH_256, the reference's default (mz_zip.c:2007-2009) */
    if (aes && (!password || strlen(password) > 128 || aes_strength > 3))
        return MZ_PARAM_ERROR; /* MZ_AES_PW_LENGTH_MAX, mz_strm_wzaes.c:77-79 */
    if (mz_cuda_init() != MZ_OK) {
        fprintf(stderr, "mz_zip_cuda: no usable sm_100 GPU (%s); there is no CPU fallback\n", mz_cuda_last_error());
        return MZ_SUPPORT_ERROR;
    }
    /* 64 MiB rounds, four in preparation: each round's entries are packed into pinned staging by its own worker thread (that copy is
     * the slowest stage of a round), and small rounds keep the page-locked allocations -- and the time to make them -- small */
    size_t round_bytes = 64u << 20;
    {
        const char *v = getenv("MZ_CUDA_ZIP_ROUND_MB");
        if (v && atoll(v) > 0)
            round_bytes = (size_t)atoll(v) << 20;
    }
    size_t max_name = 0;
    for (uint32_t i = 0; i < count; i++) {
        if (!items[i].filename || items[i].size < 0 || (items[i].size > 0 && !items[i].data))
            return MZ_PARAM_ERROR;
        const size_t nl = strlen(items[i].filename);
        if (nl == 0 || nl > 65535)
            return MZ_PARAM_ERROR;
        if (nl > max_name)
            max_name = nl;
        if (items[i].size >= 0xffff0000ll)
            return MZ_SUPPORT_ERROR; /* zip64-sized ENTRIES take the per-entry path (mz_zip_cuda_add_buffers) */
        if ((size_t)items[i].size + 16 > round_bytes)
            round_bytes = ((size_t)items[i].size + 16 + 65535) & ~(size_t)65535;
    }
    /* rounds: consecutive entries that fit the staging buffers; boundaries depend on the sizes alone, so they are fixed up
     * front and several rounds can be prepared at once */
    uint32_t nrounds = 0, rcap = 16;
    uint32_t *rfirst = (uint32_t *)malloc((rcap + 1) * sizeof(uint32_t));
    uint32_t max_chunks = 1, max_entries = 1;
    size_t max_blob = 64;
    if (!rfirst)
        return MZ_MEM_ERROR;
    {
        uint32_t i = 0;
        while (i < count) {
            size_t bytes = 0, blob = 0;
            uint32_t ch = 0, j = i;
            while (j < count) {
                const size_t need = ((size_t)items[j].size + 15) & ~(size_t)15;
                if (j > i && bytes + need > round_bytes)
                    break;
                bytes += need;
                ch += chunks_of(items[j].size);
                blob += 30 + strlen(items[j].filename) + 40 + 11 + 18; /* header, name, hash field, AES field, salt + verifier */
                j++;
            }
            if (nrounds == rcap) {
                rcap *= 2;
                uint32_t *q = (uint32_t *)realloc(rfirst, (rcap + 1) * sizeof(uint32_t));
                if (!q) {
                    free(rfirst);
                    return MZ_MEM_ERROR;
                }
                rfirst = q;
            }
            rfirst[nrounds++] = i;
            if (ch > max_chunks) max_chunks = ch;
            if (j - i > max_entries) max_entries = j - i;
            if (blob > max_blob) max_blob = blob;
            i = j;
        }
        rfirst[nrounds] = count;
    }
    int32_t ndev = 1;
    const int32_t dev0 = mz_cuda_get_device() < 0 ? 0 : mz_cuda_get_device();
    if (flags & MZ_ZIP_CUDA_ALL_DEVICES) {
        ndev = mz_cuda_device_count();
        if (ndev < 1) ndev = 1;
        if (ndev > 8) ndev = 8;
    }
    const double t_setup0 = now_ms();
    const uint32_t want = ndev > 1 ? (uint32_t)ndev * 2 : 4u;
    const uint32_t nslots = want < nrounds ? want : (nrounds ? nrounds : 1);
    za_slot *slots = (za_slot *)calloc(nslots, sizeof(za_slot));
    za_cd cd = {NULL, 0, 0};
    if (!slots) {
        free(rfirst);
        return MZ_MEM_ERROR;
    }
    for (uint32_t k = 0; k < nslots && err == MZ_OK; k++) {
        const int32_t dev = ndev > 1 ? (int32_t)(k % (uint32_t)ndev) : dev0;
        if (mz_cuda_set_device(dev) != MZ_OK || !za_acquire(&slots[k], dev, round_bytes, max_chunks + 1, max_blob, aes, pk)) {
            err = MZ_MEM_ERROR;
            break;
        }
        slots[k].device = dev;
        slots[k].items = items;
        slots[k].level = level;
        slots[k].flags = flags;
        slots[k].password = password;
        slots[k].pw_len = aes ? (uint32_t)strlen(password) : 0;
        slots[k].strength = aes_strength;
    }
    mz_cuda_set_device(dev0);
    uint64_t abs_off = 0;
    uint32_t issued = 0;
    st.setup_ms = now_ms() - t_setup0;
    for (uint32_t r = 0; r < nrounds && err == MZ_OK; r++) {
        /* keep every slot busy: rounds r .. r + nslots - 1 are in preparation */
        while (issued < nrounds && issued < r + nslots) {
            za_slot *z = &slots[issued % nslots];
            z->first = rfirst[issued];
            z->last = rfirst[issued + 1];
            z->running = pthread_create(&z->th, NULL, za_prepare, z) == 0;
            if (!z->running)
                za_prepare(z);
            issued++;
        }
        za_slot *z = &slots[r % nslots];
        if (z->running) {
            pthread_join(z->th, NULL);
            z->running = 0;
        }
        err = z->err;
        if (err)
            break;
        const double t2 = now_ms();
        err = za_write(base_stream, z->h_region, z->region_len);
        /* central directory records of the round (mz_zip.c:594-919 with local = 0) */
        for (uint32_t e = 0; e < z->last - z->first && err == MZ_OK; e++) {
            const mz_cuda_zip_item *it = &items[z->first + e];
            const za_meta *m = &z->meta[e];
            const uint64_t lh_off = abs_off + m->lh_rel;
            const int z64 = lh_off >= 0xffffffffull;
            const size_t nlen = strlen(it->filename);
            const uint32_t xhash = (flags & MZ_ZIP_CUDA_HASH_SHA256) ? 40u : 0u;
            const uint32_t xlen = (z64 ? 4u + 24u : 0u) + (aes ? 11u : 0u) + xhash;
            uint8_t *h = za_cd_room(&cd, 46 + nlen + xlen);
            if (!h) {
                err = MZ_MEM_ERROR;
                break;
            }
            put32(h, 0x02014b50u);                   /* MZ_ZIP_MAGIC_CENTRALHEADER */
            put16(h + 4, (3u << 8) | 45u);           /* made by: MZ_HOST_SYSTEM_UNIX, 4.5 */
            put16(h + 6, aes ? 51 : (z64 ? 45 : 20));
            put16(h + 8, (1u << 11) | (aes || pk ? 1u : 0u));
            put16(h + 10, aes ? 99 : 8);
            put32(h + 12, za_dos_date(it->modified_date));
            put32(h + 16, m->crc);
            put32(h + 20, z64 ? 0xffffffffu : (uint32_t)m->csize); /* with a zip64 field both sizes move into it (mz_zip.c:519-548) */
            put32(h + 24, z64 ? 0xffffffffu : (uint32_t)it->size);
            put16(h + 28, (uint32_t)nlen);
            put16(h + 30, xlen);
            put16(h + 32, 0);                        /* comment */
            put16(h + 34, 0);                        /* disk number start */
            put16(h + 36, 0);                        /* internal attributes */
            put32(h + 38, it->external_fa ? it->external_fa : (0100644u << 16));
            put32(h + 42, z64 ? 0xffffffffu : (uint32_t)lh_off);
            memcpy(h + 46, it->filename, nlen);
            uint8_t *x = h + 46 + nlen;
            if (z64) {                               /* MZ_ZIP_EXTENSION_ZIP64: uncompressed, compressed, header offset */
                put16(x, 0x0001);
                put16(x + 2, 24);
                put64(x + 4, (uint64_t)it->size);
                put64(x + 12, m->csize);
                put64(x + 20, lh_off);
                x += 28;
            }
            if (aes) {
                za_aes_field(x, aes_strength);
                x += 11;
            }
            if (xhash)
                za_hash_field(x, z->b.h_digest + (size_t)e * 32);
            st.bytes_in += (uint64_t)it->size;
            st.bytes_out += m->csize;
        }
        abs_off += z->region_len;
        st.container_ms += now_ms() - t2;
        st.pack_ms += z->pack_ms;
        st.gpu_ms += z->gpu_ms;
        st.entries += z->last - z->first;
        st.rounds++;
    }
    for (uint32_t k = 0; k < nslots; k++)
        if (slots[k].running) {
            pthread_join(slots[k].th, NULL);
            slots[k].running = 0;
        }
    /* central directory + end records (mz_zip.c:1102-1234) */
    if (err == MZ_OK) {
        const uint64_t cd_off = abs_off, cd_size = cd.len;
        uint8_t tail[56 + 20 + 22];
        size_t tl = 0;
        err = za_write(base_stream, cd.p, cd.len);
        if (cd_off >= 0xffffffffull || count >= 0xffffu) {
            uint8_t *q = tail;
            put32(q, 0x06064b50u);                   /* MZ_ZIP_MAGIC_ENDHEADER64 */
            put64(q + 4, 44);
            put16(q + 12, (3u << 8) | 45u);
            put16(q + 14, 45);
            put32(q + 16, 0);
            put32(q + 20, 0);
            put64(q + 24, count);
            put64(q + 32, count);
            put64(q + 40, cd_size);
            put64(q + 48, cd_off);
            q += 56;
            put32(q, 0x07064b50u);                   /* MZ_ZIP_MAGIC_ENDLOCHEADER64 */
            put32(q + 4, 0);
            put64(q + 8, cd_off + cd_size);
            put32(q + 16, 1);
            tl = 76;
        }
        uint8_t *q = tail + tl;
        put32(q, 0x06054b50u);                       /* MZ_ZIP_MAGIC_ENDHEADER */
        put16(q + 4, 0);
        put16(q + 6, 0);
        put16(q + 8, count >= 0xffffu ? 0xffffu : count);
        put16(q + 10, count >= 0xffffu ? 0xffffu : count);
        put32(q + 12, (uint32_t)cd_size);
        put32(q + 16, cd_off >= 0xffffffffull ? 0xffffffffu : (uint32_t)cd_off);
        put16(q + 20, 0);
        tl += 22;
        if (err == MZ_OK)
            err = za_write(base_stream, tail, tl);
    }
    const double t_setup1 = now_ms();
    for (uint32_t k = 0; k < nslots; k++) {
        mz_cuda_set_device(slots[k].device);
        za_release(&slots[k]);
    }
    mz_cuda_set_device(dev0);
    st.setup_ms += now_ms() - t_setup1;
    free(slots);
    free(cd.p);
    free(rfirst);
    if (stats)
        *stats = st;
    return err;
}

/* ---- batch extraction ------------------------------------------------------------------------------------------ */
typedef struct zx_entry_s {
    uint64_t coff, csize, ooff, usize; /* offsets inside the round's compressed / plain buffers */
    uint32_t crc, name_off;
    uint16_t method;
    uint8_t has_sha;
    uint8_t aes;     /* 0, or the WinZip AES strength 1..3: the stored bytes are salt | verifier | ciphertext | authentication code */
    uint8_t pk;      /* PKWARE traditional encryption: the stored bytes are the 12-byte encryption header | ciphertext */
    uint16_t pk_verify, version_needed;
    uint8_t sha[32]; /* expected SHA-256 from the MZ_ZIP_EXTENSION_HASH extra field */
} zx_entry;

typedef struct zx_bufs_s {
    size_t comp_cap, out_cap;
    uint32_t max_entries;
    uint8_t *h_comp, *d_comp, *d_out, *h_out;
    mz_cuda_inflate_job *h_job, *d_job;
    mz_cuda_inflate_state *h_state, *d_state;
    uint64_t *h_off, *d_off;
    uint32_t *h_len, *d_len, *d_residue, *d_crc, *h_crc;
    uint64_t *h_len64, *d_len64;
    uint8_t *d_digest, *h_digest;
    /* WinZip AES entries of the round, grouped by strength (K8) */
    uint8_t *h_salt, *d_salt, *h_keys, *d_keys, *d_pw, *h_mac, *d_mac;
    uint64_t *h_coff, *d_coff, *h_clen, *d_clen;
    uint32_t *aes_idx;
    zx_entry *ent;
    char *names;
    size_t names_cap;
} zx_bufs;

static void zx_free(zx_bufs *b) {
    mz_cuda_host_free(b->h_comp);
    mz_cuda_free(b->d_comp);
    mz_cuda_free(b->d_out);
    mz_cuda_host_free(b->h_out);
    mz_cuda_host_free(b->h_job);
    mz_cuda_free(b->d_job);
    mz_cuda_host_free(b->h_state);
    mz_cuda_free(b->d_state);
    mz_cuda_host_free(b->h_off);
    mz_cuda_free(b->d_off);
    mz_cuda_host_free(b->h_len);
    mz_cuda_free(b->d_len);
    mz_cuda_free(b->d_residue);
    mz_cuda_free(b->d_crc);
    mz_cuda_host_free(b->h_crc);
    mz_cuda_host_free(b->h_len64);
    mz_cuda_free(b->d_len64);
    mz_cuda_free(b->d_digest);
    mz_cuda_host_free(b->h_digest);
    mz_cuda_host_free(b->h_salt);
    mz_cuda_free(b->d_salt);
    mz_cuda_host_free(b->h_keys);
    mz_cuda_free(b->d_keys);
    mz_cuda_free(b->d_pw);
    mz_cuda_host_free(b->h_mac);
    mz_cuda_free(b->d_mac);
    mz_cuda_host_free(b->h_coff);
    mz_cuda_free(b->d_coff);
    mz_cuda_host_free(b->h_clen);
    mz_cuda_free(b->d_clen);
    free(b->aes_idx);
    free(b->ent);
    free(b->names);
    memset(b, 0, sizeof(*b));
}

/* the K8 tables, made when the first encrypted entry turns up */
static int zx_alloc_aes(zx_bufs *b) {
    const size_t n = b->max_entries;
    if (b->aes_idx)
        return 1;
    b->h_salt = (uint8_t *)mz_cuda_host_alloc(n * 16);
    b->d_salt = (uint8_t *)mz_cuda_malloc(n * 16);
    b->h_keys = (uint8_t *)mz_cuda_host_alloc(n * MZ_CUDA_WZAES_KEYREC);
    b->d_keys = (uint8_t *)mz_cuda_malloc(n * MZ_CUDA_WZAES_KEYREC);
    b->d_pw = (uint8_t *)mz_cuda_malloc(256);
    b->h_mac = (uint8_t *)mz_cuda_host_alloc(n * 20);
    b->d_mac = (uint8_t *)mz_cuda_malloc(n * 20);
    b->h_coff = (uint64_t *)mz_cuda_host_alloc(n * 8);
    b->d_coff = (uint64_t *)mz_cuda_malloc(n * 8);
    b->h_clen = (uint64_t *)mz_cuda_host_alloc(n * 8);
    b->d_clen = (uint64_t *)mz_cuda_malloc(n * 8);
    b->aes_idx = (uint32_t *)malloc(n * 4);
    return b->h_salt && b->d_salt && b->h_keys && b->d_keys && b->d_pw && b->h_mac && b->d_mac && b->h_coff && b->d_coff && b->h_clen && b->d_clen &&
           b->aes_idx;
}

static int zx_alloc(zx_bufs *b, size_t comp_cap, size_t out_cap, uint32_t max_entries) {
    memset(b, 0, sizeof(*b));
    b->comp_cap = comp_cap;
    b->out_cap = out_cap;
    b->max_entries = max_entries;
    b->names_cap = (size_t)max_entries * 64;
    b->h_comp = (uint8_t *)mz_cuda_host_alloc(comp_cap + 64);
    b->d_comp = (uint8_t *)mz_cuda_malloc(comp_cap + 64);
    b->d_out = (uint8_t *)mz_cuda_malloc(out_cap + 512);
    b->h_out = (uint8_t *)mz_cuda_host_alloc(out_cap + 512);
    b->h_job = (mz_cuda_inflate_job *)mz_cuda_host_alloc((size_t)max_entries * sizeof(mz_cuda_inflate_job));
    b->d_job = (mz_cuda_inflate_job *)mz_cuda_malloc((size_t)max_entries * sizeof(mz_cuda_inflate_job));
    b->h_state = (mz_cuda_inflate_state *)mz_cuda_host_alloc((size_t)max_entries * sizeof(mz_cuda_inflate_state));
    b->d_state = (mz_cuda_inflate_state *)mz_cuda_malloc((size_t)max_entries * sizeof(mz_cuda_inflate_state));
    b->h_off = (uint64_t *)mz_cuda_host_alloc((size_t)max_entries * 8);
    b->d_off = (uint64_t *)mz_cuda_malloc((size_t)max_entries * 8);
    b->h_len = (uint32_t *)mz_cuda_host_alloc((size_t)max_entries * 4);
    b->d_len = (uint32_t *)mz_cuda_malloc((size_t)max_entries * 4);
    b->d_residue = (uint32_t *)mz_cuda_malloc((size_t)max_entries * 4);
    b->d_crc = (uint32_t *)mz_cuda_malloc((size_t)max_entries * 4);
    b->h_crc = (uint32_t *)mz_cuda_host_alloc((size_t)max_entries * 4);
    b->h_len64 = (uint64_t *)mz_cuda_host_alloc((size_t)max_entries * 8);
    b->d_len64 = (uint64_t *)mz_cuda_malloc((size_t)max_entries * 8);
    b->d_digest = (uint8_t *)mz_cuda_malloc((size_t)max_entries * 32);
    b->h_digest = (uint8_t *)mz_cuda_host_alloc((size_t)max_entries * 32);
    b->ent = (zx_entry *)malloc((size_t)max_entries * sizeof(zx_entry));
    b->names = (char *)malloc(b->names_cap);
    if (!b->h_comp || !b->d_comp || !b->d_out || !b->h_out || !b->h_job || !b->d_job || !b->h_state || !b->d_state || !b->h_off || !b->d_off ||
        !b->h_len || !b->d_len || !b->d_residue || !b->d_crc || !b->h_crc || !b->h_len64 || !b->d_len64 || !b->d_digest || !b->h_digest ||
        !b->ent || !b->names) {
        zx_free(b);
        return 0;
    }
    return 1;
}

/* PKWARE key schedule on the host, for the 12 header bytes of each entry (APPNOTE 6.1.5-6.1.6, mz_strm_pkcrypt.c:64-102) */
static uint32_t zx_pk_reg(uint32_t r, uint32_t b) {
    r ^= b & 0xffu;
    for (int i = 0; i < 8; i++)
        r = (r >> 1) ^ (0xedb88320u & (0u - (r & 1u)));
    return r;
}
static uint32_t zx_pk_decode(uint32_t k[3], uint32_t c) {
    const uint32_t t = k[2] | 2u, p = (c ^ ((t * (t ^ 1u)) >> 8)) & 0xffu;
    k[0] = zx_pk_reg(k[0], p);
    k[1] = (k[1] + (k[0] & 0xffu)) * 134775813u + 1u;
    k[2] = zx_pk_reg(k[2], k[1] >> 24);
    return p;
}

/* decode + checksum + deliver the entries collected in b->ent[0..n) */
static int32_t zx_flush(zx_bufs *b, uint32_t n, size_t comp_used, size_t out_used, const char *password, mz_cuda_zip_entry_cb cb, void *userdata,
                        mz_cuda_zip_stats *st) {
    int32_t err = MZ_OK;
    uint32_t njobs = 0;
    double t0 = now_ms();
    if (n == 0)
        return MZ_OK;
    err = mz_cuda_memcpy_h2d(b->d_comp, b->h_comp, comp_used + 32, NULL);
    /* PKWARE entries (mz_strm_pkcrypt.c): every encryption header of the round is checked before anything is launched -- its
     * decrypted last byte against the verifier, and the byte before it too for version_needed < 2 (:154-161) -- so a wrong password
     * fails with MZ_PASSWORD_ERROR, not a decode error (except with probability 256^-n). Then K9 decrypts header + stream in place. */
    uint32_t m = 0;
    for (uint32_t i = 0; i < n && !err; i++) {
        zx_entry *e = &b->ent[i];
        if (!e->pk)
            continue;
        uint32_t k[3] = {305419896u, 591751049u, 878082192u}, hdr[12];
        for (const unsigned char *q = (const unsigned char *)password; *q; q++) {
            k[0] = zx_pk_reg(k[0], *q);
            k[1] = (k[1] + (k[0] & 0xffu)) * 134775813u + 1u;
            k[2] = zx_pk_reg(k[2], k[1] >> 24);
        }
        for (int j = 0; j < 12; j++)
            hdr[j] = zx_pk_decode(k, b->h_comp[e->coff + j]);
        if (hdr[11] != (e->pk_verify & 0xffu) || (e->version_needed < 2 && hdr[10] != (uint32_t)(e->pk_verify >> 8)))
            err = MZ_PASSWORD_ERROR;
        b->h_coff[m] = e->coff;
        b->h_clen[m++] = e->csize;
    }
    if (!err && m) {
        err = mz_cuda_memcpy_h2d(b->d_coff, b->h_coff, (size_t)m * 8, NULL);
        if (!err) err = mz_cuda_memcpy_h2d(b->d_clen, b->h_clen, (size_t)m * 8, NULL);
        if (!err) err = mz_cuda_pkcrypt_decrypt(b->d_comp, b->d_coff, b->d_clen, m, password, NULL);
        if (!err) err = mz_cuda_stream_sync(NULL); /* (the tables are reused below) */
        for (uint32_t i = 0; i < n; i++)
            if (b->ent[i].pk) { /* from here on the entry is its compressed stream */
                b->ent[i].coff += 12;
                b->ent[i].csize -= 12;
            }
    }
    /* WinZip AES entries first (mz_strm_wzaes.c): keys from password + salt, verifier, HMAC of the ciphertext against the stored
     * authentication code, then the ciphertext becomes the compressed stream in place. One pass per strength present. */
    for (uint32_t strength = 1; strength <= 3 && !err; strength++) {
        const uint32_t slen = 4 * strength + 4;
        uint32_t m = 0;
        uint64_t max_clen = 0;
        for (uint32_t i = 0; i < n; i++) {
            zx_entry *e = &b->ent[i];
            if (e->aes != strength)
                continue;
            memcpy(b->h_salt + (size_t)m * 16, b->h_comp + e->coff, slen);
            b->h_coff[m] = e->coff + slen + 2;
            b->h_clen[m] = e->csize - slen - 12;
            if (b->h_clen[m] > max_clen) max_clen = b->h_clen[m];
            b->aes_idx[m++] = i;
        }
        if (m == 0)
            continue;
        const size_t pwl = strlen(password);
        err = mz_cuda_memcpy_h2d(b->d_salt, b->h_salt, (size_t)m * 16, NULL);
        if (!err) err = mz_cuda_memcpy_h2d(b->d_pw, password, pwl ? pwl : 1, NULL);
        if (!err) err = mz_cuda_wzaes_derive(b->d_pw, (uint32_t)pwl, b->d_salt, m, strength, b->d_keys, NULL);
        if (!err) err = mz_cuda_memcpy_d2h(b->h_keys, b->d_keys, (size_t)m * MZ_CUDA_WZAES_KEYREC, NULL);
        if (!err) err = mz_cuda_memcpy_h2d(b->d_coff, b->h_coff, (size_t)m * 8, NULL);
        if (!err) err = mz_cuda_memcpy_h2d(b->d_clen, b->h_clen, (size_t)m * 8, NULL);
        if (!err) err = mz_cuda_wzaes_hmac(b->d_comp, b->d_coff, b->d_clen, m, b->d_keys, strength, b->d_mac, NULL);
        if (!err) err = mz_cuda_memcpy_d2h(b->h_mac, b->d_mac, (size_t)m * 20, NULL);
        if (!err) err = mz_cuda_wzaes_ctr(b->d_comp, b->d_coff, b->d_clen, m, max_clen, b->d_keys, strength, NULL);
        if (!err) err = mz_cuda_stream_sync(NULL);
        for (uint32_t k = 0; k < m && !err; k++) {
            zx_entry *e = &b->ent[b->aes_idx[k]];
            if (memcmp(b->h_keys + (size_t)k * MZ_CUDA_WZAES_KEYREC + 64, b->h_comp + e->coff + slen, 2) != 0)
                err = MZ_PASSWORD_ERROR; /* mz_strm_wzaes.c:133-134 */
            else if (memcmp(b->h_mac + (size_t)k * 20, b->h_comp + b->h_coff[k] + b->h_clen[k], 10) != 0)
                err = MZ_CRC_ERROR;      /* :252-254 */
            e->coff = b->h_coff[k];      /* from here on the entry is its compressed stream */
            e->csize = b->h_clen[k];
        }
    }
    if (err)
        return err;
    memset(b->h_state, 0, (size_t)n * sizeof(mz_cuda_inflate_state));
    for (uint32_t i = 0; i < n; i++) {
        const zx_entry *e = &b->ent[i];
        b->h_off[i] = e->ooff;
        b->h_len[i] = (uint32_t)e->usize;
        if (e->method == 8) {
            mz_cuda_inflate_job *j = &b->h_job[njobs];
            j->d_in = b->d_comp + e->coff;
            j->in_base = 0;
            j->in_avail = e->csize;
            j->d_out = b->d_out + e->ooff;
            j->out_base = 0;
            j->out_cap = e->usize;
            j->in_final = 1;
            j->flags = 0;
            njobs++;
        }
    }
    /* stored entries: their bytes are the plain bytes */
    for (uint32_t i = 0; i < n && !err; i++)
        if (b->ent[i].method == 0 && b->ent[i].usize)
            err = mz_cuda_memcpy_d2d(b->d_out + b->ent[i].ooff, b->d_comp + b->ent[i].coff, (size_t)b->ent[i].usize, NULL);
    if (!err && njobs) {
        err = mz_cuda_memcpy_h2d(b->d_job, b->h_job, (size_t)njobs * sizeof(mz_cuda_inflate_job), NULL);
        if (!err) err = mz_cuda_memcpy_h2d(b->d_state, b->h_state, (size_t)njobs * sizeof(mz_cuda_inflate_state), NULL);
        if (!err) err = mz_cuda_inflate_streams(b->d_job, b->d_state, njobs, NULL);
        if (!err) err = mz_cuda_memcpy_d2h(b->h_state, b->d_state, (size_t)njobs * sizeof(mz_cuda_inflate_state), NULL);
    }
    if (!err) err = mz_cuda_memcpy_h2d(b->d_off, b->h_off, (size_t)n * 8, NULL);
    if (!err) err = mz_cuda_memcpy_h2d(b->d_len, b->h_len, (size_t)n * 4, NULL);
    if (!err) err = mz_cuda_crc32_segments(b->d_out, 0, 0, b->d_off, b->d_len, n, b->d_residue, b->d_crc, NULL);
    if (!err) err = mz_cuda_memcpy_d2h(b->h_crc, b->d_crc, (size_t)n * 4, NULL);
    int any_sha = 0;
    for (uint32_t i = 0; i < n; i++) {
        any_sha |= b->ent[i].has_sha;
        b->h_len64[i] = b->ent[i].usize;
    }
    if (!err && any_sha) { /* K7 over the round's plain bytes */
        err = mz_cuda_memcpy_h2d(b->d_len64, b->h_len64, (size_t)n * 8, NULL);
        if (!err) err = mz_cuda_sha256_batch(b->d_out, b->d_off, b->d_len64, n, b->d_digest, NULL);
        if (!err) err = mz_cuda_memcpy_d2h(b->h_digest, b->d_digest, (size_t)n * 32, NULL);
    }
    if (!err) err = mz_cuda_memcpy_d2h(b->h_out, b->d_out, out_used, NULL);
    if (!err) err = mz_cuda_stream_sync(NULL);
    double t1 = now_ms();
    if (err)
        return err;
    uint32_t jk = 0;
    for (uint32_t i = 0; i < n; i++) {
        const zx_entry *e = &b->ent[i];
        if (e->method == 8) {
            const mz_cuda_inflate_state *s = &b->h_state[jk++];
            /* the stream must end, produce exactly the recorded size and use exactly the recorded bytes (mz_zip.c:2116-2128 checks
             * the same three things through total_in / total_out / crc) */
            if (s->status != 1 || s->out_pos != e->usize || ((s->in_bitpos + 7) >> 3) != e->csize)
                return s->status < 0 ? s->status : MZ_DATA_ERROR;
        }
        const uint32_t crc = e->usize ? b->h_crc[i] : 0u;
        if (crc != e->crc)
            return MZ_CRC_ERROR;
        if (e->has_sha && memcmp(b->h_digest + (size_t)i * 32, e->sha, 32) != 0)
            return MZ_CRC_ERROR; /* mz_zip_reader_entry_close: hash mismatch -> MZ_CRC_ERROR (mz_zip_rw.c:444-447) */
    }
    double t2 = now_ms();
    for (uint32_t i = 0; i < n; i++) {
        const zx_entry *e = &b->ent[i];
        if (cb) {
            err = cb(userdata, b->names + e->name_off, b->h_out + e->ooff, (int64_t)e->usize, e->crc);
            if (err)
                return err;
        }
        st->bytes_in += e->csize;
        st->bytes_out += e->usize;
    }
    st->gpu_ms += t1 - t0;
    st->container_ms += now_ms() - t2;
    st->entries += n;
    st->rounds++;
    return MZ_OK;
}

int32_t mz_zip_cuda_extract_all(void *zip_handle, mz_cuda_zip_entry_cb cb, void *userdata, mz_cuda_zip_stats *stats) {
    return mz_zip_cuda_extract_all_aes(zip_handle, NULL, cb, userdata, stats);
}

static int32_t zx_extract(void *zip_handle, const char *password, int allow_pk, mz_cuda_zip_entry_cb cb, void *userdata, mz_cuda_zip_stats *stats);

int32_t mz_zip_cuda_extract_all_aes(void *zip_handle, const char *password, mz_cuda_zip_entry_cb cb, void *userdata, mz_cuda_zip_stats *stats) {
    return zx_extract(zip_handle, password, 0, cb, userdata, stats);
}

int32_t mz_zip_cuda_extract_all_encrypted(void *zip_handle, const char *password, mz_cuda_zip_entry_cb cb, void *userdata, mz_cuda_zip_stats *stats) {
    return zx_extract(zip_handle, password, 1, cb, userdata, stats);
}

/* the entry walk of both: allow_pk = 0 keeps mz_zip_cuda_extract_all_aes's contract (PKWARE entries: MZ_SUPPORT_ERROR) */
static int32_t zx_extract(void *zip_handle, const char *password, int allow_pk, mz_cuda_zip_entry_cb cb, void *userdata, mz_cuda_zip_stats *stats) {
    zx_bufs b;
    mz_cuda_zip_stats st;
    int32_t err;
    memset(&st, 0, sizeof(st));
    if (!mz_zip_goto_first_entry || !mz_zip_goto_next_entry || !mz_zip_entry_get_info || !mz_zip_entry_read_open || !mz_zip_entry_read ||
        !mz_zip_entry_close)
        return MZ_SUPPORT_ERROR; /* no zip container in this process */
    if (!zip_handle)
        return MZ_PARAM_ERROR;
    if (mz_cuda_init() != MZ_OK) {
        fprintf(stderr, "mz_zip_cuda: no usable sm_100 GPU (%s); there is no CPU fallback\n", mz_cuda_last_error());
        return MZ_SUPPORT_ERROR;
    }
    size_t comp_cap = 128u << 20, out_cap = 512u << 20;
    {
        const char *v = getenv("MZ_CUDA_ZIP_ROUND_MB");
        if (v && atoll(v) > 0) {
            comp_cap = (size_t)atoll(v) << 20;
            out_cap = comp_cap * 4;
        }
    }
    const uint32_t max_entries = 65536;
    if (!zx_alloc(&b, comp_cap, out_cap, max_entries))
        return MZ_MEM_ERROR;
    uint32_t n = 0;
    size_t comp_used = 0, out_used = 0, names_used = 0;
    err = mz_zip_goto_first_entry(zip_handle);
    while (err == MZ_OK) {
        zc_file_info *fi = NULL;
        double t0 = now_ms();
        err = mz_zip_entry_get_info(zip_handle, &fi);
        if (err != MZ_OK)
            break;
        const int enc = (fi->flag & 1u) != 0;
        const int pk = enc && !fi->aes_version && allow_pk; /* PKWARE traditional encryption */
        /* salt + verifier + authentication code, or the PKWARE encryption header */
        const uint32_t aes_over = pk ? 12u : (enc ? 4u * fi->aes_strength + 4u + 12u : 0u);
        if (enc && (fi->aes_version || pk) && !password) {
            err = MZ_PASSWORD_ERROR; /* encrypted and no password given */
            break;
        }
        if (pk && fi->compressed_size < 12) {
            err = MZ_FORMAT_ERROR; /* shorter than its own encryption header */
            break;
        }
        if ((enc && !pk && (!fi->aes_version || fi->aes_strength < 1 || fi->aes_strength > 3 || strlen(password) > 128 ||
                            fi->compressed_size < (int64_t)aes_over)) ||
            (fi->compression_method != 0 && fi->compression_method != 8) || fi->compressed_size < 0 ||
            fi->uncompressed_size < 0 || fi->uncompressed_size > (1ll << 30) || fi->compressed_size > (1ll << 30)) {
            err = MZ_SUPPORT_ERROR; /* PKWARE-encrypted, another codec, or too large for the batch path */
            break;
        }
        if (enc && !zx_alloc_aes(&b)) {
            err = MZ_MEM_ERROR;
            break;
        }
        if (fi->compression_method == 0 && fi->compressed_size - (int64_t)aes_over != fi->uncompressed_size) {
            err = MZ_FORMAT_ERROR;
            break;
        }
        const size_t csz = (size_t)fi->compressed_size, usz = (size_t)fi->uncompressed_size;
        const size_t cneed = (csz + 32 + 15) & ~(size_t)15, oneed = (usz + 15) & ~(size_t)15; /* K5 reads up to 16 bytes past a stream */
        const size_t nlen = strlen(fi->filename) + 1;
        if (cneed > b.comp_cap || oneed > b.out_cap) { /* one entry larger than a round: not batched */
            err = MZ_SUPPORT_ERROR;
            break;
        }
        if (n == b.max_entries || comp_used + cneed > b.comp_cap || out_used + oneed > b.out_cap || names_used + nlen > b.names_cap) {
            err = zx_flush(&b, n, comp_used, out_used, password, cb, userdata, &st);
            if (err)
                break;
            n = 0;
            comp_used = out_used = names_used = 0;
        }
        zx_entry *e = &b.ent[n];
        e->coff = comp_used;
        e->csize = csz;
        e->ooff = out_used;
        e->usize = usz;
        e->crc = fi->crc;
        e->method = fi->compression_method;
        e->name_off = (uint32_t)names_used;
        e->has_sha = 0;
        e->aes = enc && !pk ? fi->aes_strength : 0;
        e->pk = (uint8_t)pk;
        e->pk_verify = fi->pk_verify;
        e->version_needed = fi->version_needed;
        /* extra fields are {id u16, size u16, data}; find MZ_ZIP_EXTENSION_HASH with algorithm SHA-256 (mz_zip_rw.c:478-510) */
        for (uint32_t xo = 0; fi->extrafield && xo + 4 <= fi->extrafield_size;) {
            const uint8_t *x = fi->extrafield + xo;
            const uint32_t id = x[0] | (x[1] << 8), xs = x[2] | (x[3] << 8);
            if (xo + 4 + xs > fi->extrafield_size)
                break;
            if (id == 0x1a51 && xs >= 4 + 32 && (x[4] | (x[5] << 8)) == 23 && (x[6] | (x[7] << 8)) == 32) {
                memcpy(e->sha, x + 8, 32);
                e->has_sha = 1;
                break;
            }
            xo += 4 + xs;
        }
        memcpy(b.names + names_used, fi->filename, nlen);
        /* the compressed bytes, untouched, through the raw seam */
        if (csz) {
            err = mz_zip_entry_read_open(zip_handle, 1, NULL);
            size_t got = 0;
            while (err == MZ_OK && got < csz) {
                const int32_t want = csz - got > (1u << 30) ? (int32_t)(1u << 30) : (int32_t)(csz - got);
                const int32_t r = mz_zip_entry_read(zip_handle, b.h_comp + comp_used + got, want);
                if (r <= 0) {
                    err = r < 0 ? r : MZ_READ_ERROR;
                    break;
                }
                got += (size_t)r;
            }
            const int32_t cerr = mz_zip_entry_close(zip_handle);
            if (err == MZ_OK && cerr != MZ_OK)
                err = cerr;
            if (err != MZ_OK)
                break;
        }
        memset(b.h_comp + comp_used + csz, 0, cneed - csz);
        comp_used += cneed;
        out_used += oneed;
        names_used += nlen;
        n++;
        st.pack_ms += now_ms() - t0;
        err = mz_zip_goto_next_entry(zip_handle);
    }
    if (err == MZ_END_OF_LIST)
        err = zx_flush(&b, n, comp_used, out_used, password, cb, userdata, &st);
    zx_free(&b);
    if (stats)
        *stats = st;
    return err;
}
