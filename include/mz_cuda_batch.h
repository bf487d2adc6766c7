/* mz_cuda_batch.h -- device-pointer batch API of the B200 DEFLATE + CRC-32 backend (C ABI).
 *
 * ADDITIVE to the reference: minizip-ng has no batch interface (SURVEY.md section 8b "Beyond the vtbl").
 * It exists so that (a) the vtbl stream (mz_strm_cuda.h) has something to drive, (b) kernels can be
 * measured on device-resident buffers against the HBM roofline, (c) chunks / zip entries can be sharded
 * over GPUs. Plain pointers and sizes only; `stream` is a cudaStream_t passed as void* (NULL = default).
 * All functions return MZ_OK (0) or a negative MZ_* code (mz.h:21-47); MZ_CUDA_ERROR details are
 * available from mz_cuda_last_error().  Device pointers must belong to the CURRENT CUDA device.
 */
#ifndef MZ_CUDA_BATCH_H
#define MZ_CUDA_BATCH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MZ_CUDA_CHUNK_MAX    65536u /* largest independent DEFLATE chunk */
#define MZ_CUDA_FLAG_FINAL   1u     /* chunk ends its stream (BFINAL, no sync marker) */
#define MZ_CUDA_FLAG_DICT    2u     /* the 32 KiB in front of the chunk (same buffer) are earlier bytes of the SAME stream: at levels 6-9 the
                                    * chunk may refer back into them (zlib's sliding window across our chunk boundaries). In `last_flags` of a
                                    * uniform partition it applies to every chunk: the buffer is one stream. */

/* ---- runtime ---------------------------------------------------------------------------------- */
int32_t mz_cuda_init(void);                 /* idempotent, thread-safe; MZ_SUPPORT_ERROR without a usable GPU */
int32_t mz_cuda_device_count(void);
int32_t mz_cuda_set_device(int32_t ordinal);
int32_t mz_cuda_get_device(void);           /* the calling thread's current device, -1 on failure */
const char *mz_cuda_last_error(void);
int32_t mz_cuda_sm_count(void);

void *mz_cuda_malloc(size_t bytes);         /* device memory; NULL on failure */
void mz_cuda_free(void *dptr);
void *mz_cuda_host_alloc(size_t bytes);     /* pinned host memory */
void mz_cuda_host_free(void *hptr);
int32_t mz_cuda_memcpy_h2d(void *dptr, const void *hptr, size_t bytes, void *stream);  /* async on stream */
int32_t mz_cuda_memcpy_d2h(void *hptr, const void *dptr, size_t bytes, void *stream);  /* async on stream */
int32_t mz_cuda_memcpy_d2d(void *dst, const void *src, size_t bytes, void *stream);
int32_t mz_cuda_memset(void *dptr, int value, size_t bytes, void *stream);
int32_t mz_cuda_host_is_pinned(const void *hptr);           /* 1 if page-locked and usable for async copies */
int32_t mz_cuda_stream_sync(void *stream);
void *mz_cuda_stream_create(void);
void mz_cuda_stream_destroy(void *stream);
void *mz_cuda_event_create(void);
void mz_cuda_event_destroy(void *event);
int32_t mz_cuda_event_record(void *event, void *stream);
int32_t mz_cuda_event_sync(void *event);
int32_t mz_cuda_event_query(void *event); /* 1 = complete, 0 = not yet, < 0 = MZ_* error */
float mz_cuda_event_elapsed_ms(void *start, void *stop); /* syncs on stop */

/* ---- K1: CRC-32 ---------------------------------------------------------------------------------
 * Segments: either a uniform partition (d_off = d_len = NULL: segment i = bytes [i*seg_size, ...) of
 * total_len) or explicit per-segment offsets/lengths (device arrays). d_residue[i] = pure residue
 * R(segment) (init 0, no final xor) -- the linear quantity that folds; d_crc[i] (optional) = the value
 * mz_crypt_crc32_update(0, segment, len) returns (mz_crypt.c:35). */
int32_t mz_cuda_crc32_segments(const void *d_in, uint64_t total_len, uint64_t seg_size, const uint64_t *d_off,
                               const uint32_t *d_len, uint32_t nseg, uint32_t *d_residue, uint32_t *d_crc, void *stream);
/* fold the residues of a UNIFORM partition: d_out2[0] = residue of the whole buffer, d_out2[1] = crc32(0, buffer) */
int32_t mz_cuda_crc32_fold(const uint32_t *d_residue, uint32_t nseg, uint64_t seg_size, uint64_t total_len, uint32_t *d_out2,
                           void *stream);
/* whole device buffer, synchronous: *crc = mz_crypt_crc32_update(value, buffer, len) */
int32_t mz_cuda_crc32_device(const void *d_in, uint64_t len, uint32_t value, uint32_t *crc);
/* same, enqueued on `stream` and synchronised on it only (the scratch buffer is shared: one caller per device at a time) */
int32_t mz_cuda_crc32_device_stream(const void *d_in, uint64_t len, uint32_t value, uint32_t *crc, void *stream);
/* host arithmetic: crc(A||B) from crc(A), crc(B), |B|  (the "polynomial combine" of the north star) */
uint32_t mz_cuda_crc32_combine(uint32_t crc_a, uint32_t crc_b, uint64_t len_b);

/* ---- K2+K3: DEFLATE encode of independent chunks --------------------------------------------------
 * Chunk i (<= MZ_CUDA_CHUNK_MAX bytes) is compressed into slot i = d_slots + i*slot_stride
 * (slot_stride >= mz_cuda_deflate_slot_bound(chunk size), multiple of 16; d_slots 16-byte aligned);
 * d_out_len[i] = bytes written. Every slot is a byte-aligned piece of raw RFC1951 data: non-final
 * chunks end with a sync-flush marker, chunks flagged FINAL end with BFINAL. Uniform partition when
 * d_off == NULL (then only the last chunk gets the FINAL bit of `last_flags`). level 0 = stored, 1 = candidates at every second
 * position, 2-3 = every position, 4-5 = + one-step lazy evaluation, 6-9 = + the previous 32 KiB as history (inside a chunk: its
 * first half for its second; with MZ_CUDA_FLAG_DICT also the bytes in front of the chunk). */
uint64_t mz_cuda_deflate_slot_bound(uint32_t chunk_size);
int32_t mz_cuda_deflate_chunks(const void *d_in, uint64_t total_len, uint32_t chunk_size, const uint64_t *d_off,
                               const uint32_t *d_len, const uint8_t *d_flags, uint32_t nchunks, uint32_t last_flags,
                               int32_t level, void *d_slots, uint64_t slot_stride, uint32_t *d_out_len, void *stream);
/* ---- K4: join slots into one contiguous stream ------------------------------------------------------
 * d_offsets: nchunks+1 uint64 (scratch/out): d_offsets[i] = position of chunk i in d_dst, [nchunks] = total. */
int32_t mz_cuda_concat(const void *d_slots, uint64_t slot_stride, const uint32_t *d_out_len, uint32_t nchunks,
                       uint64_t *d_offsets, void *d_dst, void *stream);

/* ---- multi-GPU: chunk-sharded DEFLATE, all-gather on the copy engines ---------------------------------------------------
 * Chunks are independent, so device r of N owns a contiguous chunk range; the only exchange is the all-gather of the joined
 * bitstreams and of the per-chunk {crc32, in_len, out_len} rows. It is done with peer-to-peer copies (cudaMemcpyPeerAsync /
 * IPC-mapped destinations): the copy engines move the bytes over NVLink while every SM keeps compressing -- an SM-based
 * collective cannot co-reside with the 2 x 111 KB deflate CTAs and serialises with them.
 *
 * (a) one process, N devices (a C host):  mz_cuda_deflate_sharded()
 * (b) one process per device (torchrun):  export / open IPC handles of the gathered buffers once, then mz_cuda_memcpy_peer(). */
typedef struct mz_cuda_shard {
    int32_t device;          /* CUDA ordinal */
    const void *d_in;        /* this device's shard of the input (on `device`), 16-byte aligned */
    uint64_t len;            /* bytes; every shard but the last must be a multiple of 64 KiB */
    void *d_gathered;        /* on `device`: receives EVERY device's joined stream; device r's stream starts at region_off[r] */
    uint64_t gathered_cap;
    uint32_t *d_rows;        /* on `device`: receives every device's rows {crc32, in_len, out_len} (3 x uint32 per chunk), in
                                global chunk order (device r's rows start at chunk index = sum of earlier devices' chunks) */
} mz_cuda_shard;
/* Compress + CRC + join every shard on its device (level 0..9, BFINAL on the globally last chunk) and all-gather: after the
 * call every device holds all streams and all rows. region_off[r], stream_len[r] (arrays of ndev, host) describe where device
 * r's stream lies in every gathered buffer: region_off[r] = sum over earlier devices of mz_cuda_gather_region_bound(len);
 * the rank-ordered concatenation of the N streams is ONE valid raw DEFLATE stream. *crc32 = CRC-32 of the whole input
 * (host fold of the per-device CRCs). `pieces` >= 1: each shard is compressed in that many pieces and a finished piece
 * travels while the next one is being compressed. Synchronous. */
uint64_t mz_cuda_gather_region_bound(uint64_t shard_len);
int32_t mz_cuda_deflate_sharded(const mz_cuda_shard *shards, int32_t ndev, int32_t level, int32_t pieces, uint64_t *region_off,
                                uint64_t *stream_len, uint32_t *crc32);
/* IPC: handle64 = 64 opaque bytes to hand to the other processes; open() maps a peer's allocation into this process (peer
 * access is enabled lazily); memcpy_peer() = cudaMemcpyAsync between any two device pointers of this process's address space
 * (own or IPC-mapped), executed by a copy engine. The exported pointer must come from mz_cuda_malloc(). */
int32_t mz_cuda_ipc_export(const void *dptr, void *handle64);
int32_t mz_cuda_ipc_open(const void *handle64, void **dptr);
int32_t mz_cuda_ipc_close(void *dptr);
int32_t mz_cuda_memcpy_peer(void *dst, const void *src, size_t bytes, void *stream);
int32_t mz_cuda_stream_wait_event(void *stream, void *event);

/* ---- K7: SHA-256 of independent buffers ----------------------------------------------------------------------
 * Message i = d_in[d_off[i] .. d_off[i] + d_len[i]); d_digest receives n x 32 bytes (the digest as the standard prints it).
 * This is the per-entry hash of the reference's zip writer / reader (MZ_ZIP_EXTENSION_HASH, mz_zip_rw.c:1339-1420, :410-450),
 * batched like the per-entry CRC. */
int32_t mz_cuda_sha256_batch(const void *d_in, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, void *d_digest, void *stream);

/* K8: the arithmetic of WinZip AES entries (mz_strm_wzaes.c) for a batch of zip entries, every entry with its own salt.
 * strength = MZ_AES_STRENGTH_128 / _192 / _256 (1 / 2 / 3, mz.h:117-119): key 16 / 24 / 32 bytes, salt 8 / 12 / 16 bytes.
 *   derive: PBKDF2-HMAC-SHA1, 1000 iterations (mz_strm_wzaes.c:95-97) of the password with salt e (d_salts + 16 e) into the key
 *           record d_keys + MZ_CUDA_WZAES_KEYREC * e: encryption key at +0, authentication key at +32, 2-byte verifier at +64.
 *   ctr:    XOR entry e's bytes d_data[d_off[e] .. + d_len[e]) in place with the AES-CTR key stream of its encryption key
 *           (counter little-endian, first block 1, mz_strm_wzaes.c:147-171) -- encrypts and decrypts. max_len >= every d_len[e].
 *   hmac:   HMAC-SHA1 (authentication key) of entry e's bytes -> d_mac + 20 e; the entry stores the first 10 (:236-256). */
#define MZ_CUDA_WZAES_KEYREC 80
int32_t mz_cuda_wzaes_derive(const void *d_password, uint32_t pw_len, const void *d_salts, uint32_t n, uint32_t strength, void *d_keys, void *stream);
int32_t mz_cuda_wzaes_ctr(void *d_data, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, uint64_t max_len, const void *d_keys, uint32_t strength,
                          void *stream);
int32_t mz_cuda_wzaes_hmac(const void *d_data, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, const void *d_keys, uint32_t strength, void *d_mac,
                           void *stream);

/* K9: PKWARE traditional encryption (APPNOTE 6.1, "ZipCrypto"; mz_strm_pkcrypt.c) of a batch of zip entries, in place: entry e is
 * d_data[d_off[e] .. + d_len[e]), i.e. its 12-byte encryption header followed by its (compressed) bytes. `password` is a host C
 * string (NULL: MZ_PARAM_ERROR); every entry starts from the same keys after the password, as the reference's do.
 *   encrypt: segmented (the key stream depends on the plaintext only): every entry is cut into fixed segments and four passes
 *            with three carry scans run over all segments of the batch, so the time follows the total bytes, not the largest
 *            entry. Needs a device workspace of mz_cuda_pkcrypt_workspace_bytes(sum of d_len, n) bytes; the call synchronises
 *            `stream` once, to learn the segment count (MZ_PARAM_ERROR if the workspace is too small for it).
 *   decrypt: one thread per entry (the byte that moves the keys is the output); no workspace. The caller checks the verifier
 *            byte(s) at the end of each decrypted header. */
uint64_t mz_cuda_pkcrypt_workspace_bytes(uint64_t total_len, uint32_t n);
int32_t mz_cuda_pkcrypt_encrypt(void *d_data, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, const char *password, void *d_workspace,
                                uint64_t workspace_bytes, void *stream);
int32_t mz_cuda_pkcrypt_decrypt(void *d_data, const uint64_t *d_off, const uint64_t *d_len, uint32_t n, const char *password, void *stream);

/* K4 with caller-given destinations: slot i goes to d_dst + d_offsets[i] (no scan) -- the zip archive writer interleaves the
 * entries' streams with their local headers; and n small blobs (blob i = d_blob[d_blob_off[i] .. d_blob_off[i+1])) scattered to
 * d_dst + d_dst_off[i] (the headers themselves). */
int32_t mz_cuda_gather(const void *d_slots, uint64_t slot_stride, const uint32_t *d_out_len, uint32_t nchunks, const uint64_t *d_offsets,
                       void *d_dst, void *stream);
int32_t mz_cuda_scatter_blobs(const void *d_blob, const uint32_t *d_blob_off, const uint64_t *d_dst_off, uint32_t n, void *d_dst, void *stream);

/* ---- K5: DEFLATE decode of independent raw streams (resumable) ---------------------------------------- */
typedef struct mz_cuda_inflate_job {
    const void *d_in;    /* d_in[0] = stream byte `in_base`; readable (zero padded) 16 bytes past in_avail */
    uint64_t in_base;
    uint64_t in_avail;
    void *d_out;         /* d_out[0] = output byte `out_base`; keeps >= 32 KiB of history once out_pos > 0 */
    uint64_t out_base;
    uint64_t out_cap;
    uint32_t in_final;   /* no more input will follow */
    uint32_t flags;      /* MZ_CUDA_INFLATE_STOP_AT_BLOCK: return (why = 3) after the next completed block */
} mz_cuda_inflate_job;
#define MZ_CUDA_INFLATE_STOP_AT_BLOCK 1u

typedef struct mz_cuda_inflate_state {
    uint64_t in_bitpos;  /* consumed bits of the raw stream (TOTAL_IN = ceil(in_bitpos / 8) at END) */
    uint64_t out_pos;    /* produced bytes (TOTAL_OUT) */
    int32_t status;      /* 0 running, 1 end of stream, MZ_DATA_ERROR (-3), MZ_BUF_ERROR (-5) */
    int32_t why;         /* when running: 1 needs input, 2 needs output space, 3 stopped at a block boundary */
    uint32_t phase, last_block, stored_remaining, nlit, ndist, blocks;
    uint8_t lens[320];
} mz_cuda_inflate_state;

int32_t mz_cuda_inflate_streams(const mz_cuda_inflate_job *d_jobs, mz_cuda_inflate_state *d_states, uint32_t nstreams,
                                void *stream);

/* ---- K6: one long foreign stream, segment-speculative (csrc/inflate_spec_kernel.cuh) ------------------------
 * One ROUND decodes as much of the compressed window d_in[0..in_avail) as can be proven, starting at the block
 * boundary `start_bit` (absolute bit; the serial decoder's state must be at a block header), into
 * d_out[out_pos - out_base ...) up to absolute position out_end. 32 KiB of history before out_pos must be present
 * in d_out (as for K5). The summary says how far the round got; the caller continues from there with another
 * round or with mz_cuda_inflate_streams (which also owns every error / end-of-input decision: a round that
 * meets anything unusual just stops early). d_in must be 4-byte aligned with 16 readable bytes past in_avail. */
typedef struct mz_cuda_spec_summary {
    uint64_t end_bit;    /* absolute bit position reached (a block boundary, or the end of the stream) */
    uint64_t total_out;  /* bytes written from out_pos on */
    uint32_t nchain;     /* segments proven and emitted; 0 = no progress, use the serial decoder */
    int32_t status;      /* 0 running, 1 end of stream */
    uint32_t blocks;
    uint32_t flags;      /* != 0: internal cross-check failed, the round's output must be discarded */
    uint32_t candidates;
    uint32_t pad;
} mz_cuda_spec_summary;
uint64_t mz_cuda_inflate_spec_workspace_bytes(uint32_t max_segments);
int32_t mz_cuda_inflate_spec_round(const void *d_in, uint64_t in_base, uint64_t in_avail, uint32_t in_final, uint64_t start_bit,
                                   uint64_t seg_bytes, uint32_t nseg, void *d_out, uint64_t out_base, uint64_t out_pos,
                                   uint64_t out_end, void *d_workspace, uint32_t max_segments, mz_cuda_spec_summary *d_summary,
                                   void *stream);

#ifdef __cplusplus
}
#endif
#endif
