/* mz_zip_cuda.h -- batch zip-entry writer on the reference's RAW-entry seam (SURVEY.md 8f.1, config C4).
 *
 * The reference compresses a zip entry by pushing its bytes through mz_stream_zlib, one entry at a time
 * (mz_zip_entry_write_open -> mz_zip_entry_write -> mz_zip_entry_close, mz_zip.c:1915,2056,2269). This routine keeps
 * the container code exactly where it is and only moves the codec work: all entries of a batch are DEFLATE-compressed
 * and CRC'd on the GPU in ONE launch each (every entry its own raw stream: 64 KiB chunks joined by sync markers,
 * BFINAL on the entry's last chunk), then handed to the reference through its raw seam
 *     mz_zip_entry_write_open(handle, &file_info, level, raw = 1, NULL)     mz_zip.c:1915
 *     mz_zip_entry_write(handle, compressed, size)                          mz_zip.c:2056
 *     mz_zip_entry_close_raw(handle, uncompressed_size, crc32)              mz_zip.c:2272
 * so local headers, zip64 decisions and the central directory stay the reference's own code.
 *
 * Linking: the three functions above (plus nothing else) are taken from the HOST program, which links the
 * reference's mz_zip.c. They are declared weak here, so libmz_strm_cuda.so still loads in a process that has no
 * zip container (the call then returns MZ_SUPPORT_ERROR).
 */
#ifndef MZ_ZIP_CUDA_H
#define MZ_ZIP_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mz_cuda_zip_item {
    const char *filename;    /* utf-8, null terminated (stored with MZ_ZIP_FLAG_UTF8) */
    const void *data;        /* host memory, `size` bytes (may be NULL when size == 0) */
    int64_t size;
    int64_t modified_date;   /* unix time; 0 = now */
    uint32_t external_fa;    /* 0 = regular file 0644 */
    uint32_t reserved;
} mz_cuda_zip_item;

typedef struct mz_cuda_zip_stats {
    uint64_t bytes_in, bytes_out;
    uint32_t entries, rounds;
    double pack_ms, gpu_ms, container_ms; /* host packing + upload, device work + download, reference container calls */
    double setup_ms;                      /* native writer: creating and releasing the page-locked / device staging of the call */
} mz_cuda_zip_stats;

/* Append `count` entries to the zip that `zip_handle` (an open mz_zip writer, mz_zip.c:1237 mz_zip_open) is writing.
 * level: 0..9 or -1 (= 6), as mz_zip_entry_write_open takes it. Returns MZ_OK or the first error (MZ_* codes).
 * stats may be NULL. */
int32_t mz_zip_cuda_add_buffers(void *zip_handle, const mz_cuda_zip_item *items, uint32_t count, int16_t level,
                                mz_cuda_zip_stats *stats);

/* Same, with options. MZ_ZIP_CUDA_HASH_SHA256: every entry also gets the SHA-256 of its plain bytes, computed on the GPU in
 * the same round (K7) and stored in the MZ_ZIP_EXTENSION_HASH extra field (id 0x1a51: algorithm 23, digest size 32, digest)
 * exactly as the reference's zip writer stores it when built with a crypto provider (mz_zip_rw.c:1339-1420); the reference's
 * reader then verifies it on extraction (mz_zip_rw.c:410-450), and so does mz_zip_cuda_extract_all. */
#define MZ_ZIP_CUDA_HASH_SHA256 1u
int32_t mz_zip_cuda_add_buffers_ex(void *zip_handle, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                   mz_cuda_zip_stats *stats);

/* ---- a whole archive, natively (scope row f1, "if the container is the limit") ------------------------------------------
 * With 100 000 small entries the reference's per-entry container calls (mz_zip_entry_write_open / _write / _close_raw: three
 * calls and ~28 us per entry) cost ten times the GPU work. This call writes the COMPLETE archive itself to `base_stream` (any
 * mz_stream object: file, buffered, memory): local headers (mz_zip.c:594-919 layout: no data descriptor -- sizes and CRC are
 * known before a byte is written --, UTF-8 flag, version 20, or 45 with a zip64 extra field), the entries' DEFLATE streams,
 * the central directory and the end records incl. the zip64 end record + locator when there are >= 65535 entries or the
 * directory starts beyond 4 GiB (mz_zip.c:1102-1234, zip64 rules :551-592). A round's region [header | stream | header | ...]
 * is assembled ON THE DEVICE (K4 gather with explicit destinations + a header scatter) and goes to base in one write.
 * MZ_ZIP_CUDA_ALL_DEVICES: rounds are prepared round-robin on every visible GPU (entries shard across the GPUs; the archive
 * itself is one serial byte stream written in order). Entries must be smaller than 4 GiB - 64 KiB. */
#define MZ_ZIP_CUDA_ALL_DEVICES 2u
int32_t mz_zip_cuda_write_archive(void *base_stream, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                  mz_cuda_zip_stats *stats);
/* The native writer keeps the staging of finished calls (page-locked + device buffers, up to eight round slots per process) for
 * the next call; this frees them. MZ_CUDA_ZIP_POOL=0 in the environment turns the pool off. */
void mz_zip_cuda_trim(void);

/* The same archive with every entry WinZip-AES encrypted after compression (scope row f4, the part that follows the codec): what
 * the reference does per entry by stacking mz_stream_wzaes under the codec (mz_zip.c:1734-1741, mz_strm_wzaes.c) -- a random salt,
 * PBKDF2-HMAC-SHA1 (1000 iterations) of the password, AES in counter mode over the compressed stream, HMAC-SHA1 of the ciphertext
 * -- done for all entries of a round by three kernels (K8, include/mz_cuda_batch.h). Entry layout and headers as the reference
 * writes them: method 99 + the 0x9901 extra field (AE-1, strength, real method 8), flag bit 0, version needed 51, stored size =
 * salt + 2-byte verifier + ciphertext + 10-byte authentication code, CRC kept (mz_zip.c:703-733, :870-885).
 * flags must contain MZ_ZIP_CUDA_AES; aes_strength = 1 / 2 / 3 (AES-128 / 192 / 256; 0 = 3, the reference's default);
 * password up to 128 bytes. */
#define MZ_ZIP_CUDA_AES 4u
int32_t mz_zip_cuda_write_archive_aes(void *base_stream, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                      const char *password, uint8_t aes_strength, mz_cuda_zip_stats *stats);

/* The same archive with every entry encrypted by PKWARE traditional encryption (APPNOTE 6.1, "ZipCrypto"; scope row f4): what the
 * reference does per entry by stacking mz_stream_pkcrypt under the codec (mz_zip.c:1733-1755, mz_strm_pkcrypt.c), and what
 * `minizip -p` without -s, Info-ZIP `zip -e` and the Windows shell write. Each entry's stored bytes are the 12-byte encryption
 * header (10 random bytes, then the CRC's bytes 2 and 3: the verifier of an entry without a data descriptor, mz_zip.c:192-199)
 * followed by the DEFLATE stream, both encrypted with the keys of the password by K9 (include/mz_cuda_batch.h) on the device.
 * Headers: flag bit 0, method 8, version needed 20 (45 with zip64), CRC kept, compressed size = stream + 12.
 * flags may contain MZ_ZIP_CUDA_HASH_SHA256 and MZ_ZIP_CUDA_ALL_DEVICES; MZ_ZIP_CUDA_AES or a NULL password: MZ_PARAM_ERROR.
 * PKWARE encryption is weak by today's standards (known-plaintext attacks); it is offered because it is what most readers
 * expect. */
int32_t mz_zip_cuda_write_archive_pkcrypt(void *base_stream, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                          const char *password, mz_cuda_zip_stats *stats);

/* ---- batch extraction (scope row f2): the reverse direction ---------------------------------------------------
 * The reference extracts entry by entry: mz_zip_entry_read_open(raw=0) creates a mz_stream_zlib, the caller's loop
 * reads through it, mz_zip_entry_close compares the CRC (mz_zip_rw.c:818-909, mz_zip.c:2116-2128). Here the central
 * directory is still walked by the reference's own reader (mz_zip_goto_first_entry / _next_entry /
 * mz_zip_entry_get_info, mz_zip.c:2320-2400) and the compressed bytes are fetched through the raw seam
 * (mz_zip_entry_read_open(raw=1) / mz_zip_entry_read, mz_zip.c:1874,2031), but all entries of a round are inflated by
 * ONE K5 launch and checksummed by ONE K1 launch; the CRCs are compared with the headers on the host (MZ_CRC_ERROR on
 * the first mismatch, MZ_DATA_ERROR if a stream does not decode to exactly its recorded size). An entry that carries a
 * SHA-256 in a MZ_ZIP_EXTENSION_HASH extra field has that verified too (K7 over the round's plain bytes; MZ_CRC_ERROR on a
 * mismatch, as mz_zip_reader_entry_close reports it, mz_zip_rw.c:430-450).
 * `cb` is called once per entry in archive order with the plain bytes (valid during the call only); a non-zero return
 * stops the extraction and is returned. Entries that are encrypted, use another method than STORE/DEFLATE, or exceed
 * 1 GiB are not batched: the call returns MZ_SUPPORT_ERROR (use the per-entry stream path for such archives). */
typedef int32_t (*mz_cuda_zip_entry_cb)(void *userdata, const char *filename, const void *data, int64_t size, uint32_t crc32);
int32_t mz_zip_cuda_extract_all(void *zip_handle, mz_cuda_zip_entry_cb cb, void *userdata, mz_cuda_zip_stats *stats);

/* The same for archives whose entries are WinZip-AES encrypted (any strength; written by this library, by the reference or by
 * WinZip): the stored bytes still come through the raw seam (mz_zip_entry_read_open(raw = 1, password = NULL) hands out the
 * encrypted bytes, mz_zip.c:1727-1731), K8 derives every entry's keys from password + salt, the 2-byte verifier is compared
 * (MZ_PASSWORD_ERROR, mz_strm_wzaes.c:133-134), the HMAC-SHA1 of the ciphertext is compared with the stored authentication code
 * (MZ_CRC_ERROR, :252-254), the ciphertext is decrypted in place and decoded like any other entry. The HOST program's container
 * must be built with HAVE_WZAES (otherwise its reader refuses such entries before this code sees them). PKWARE-encrypted entries
 * return MZ_SUPPORT_ERROR here (mz_zip_cuda_extract_all_encrypted reads them); encrypted entries without a password
 * MZ_PASSWORD_ERROR. */
int32_t mz_zip_cuda_extract_all_aes(void *zip_handle, const char *password, mz_cuda_zip_entry_cb cb, void *userdata, mz_cuda_zip_stats *stats);

/* The same for archives with plain, WinZip-AES and PKWARE-encrypted entries in any mix. A PKWARE entry (flag bit 0, no AES extra
 * field) needs a password (MZ_PASSWORD_ERROR without one) and at least its 12-byte header (MZ_FORMAT_ERROR; for STORE the stored
 * size must be the plain size + 12). Per round every PKWARE header is decrypted and its verifier checked before any decoding --
 * the last header byte against the entry's pk_verify, and the byte before it too when version_needed < 2, the reference's rules
 * (mz_strm_pkcrypt.c:154-161; the reader takes pk_verify from the CRC, or from the DOS time with a data descriptor) -- a mismatch
 * is MZ_PASSWORD_ERROR. Then K9 decrypts the stored bytes in place, one thread per entry, and the entry is decoded and checked like
 * any other. PKWARE has no MAC: damaged ciphertext shows as MZ_DATA_ERROR or MZ_CRC_ERROR. The HOST program's container must be
 * built with HAVE_PKCRYPT (it fills pk_verify) and, for AES entries, HAVE_WZAES. */
int32_t mz_zip_cuda_extract_all_encrypted(void *zip_handle, const char *password, mz_cuda_zip_entry_cb cb, void *userdata, mz_cuda_zip_stats *stats);

/* sizeof the mz_zip_file mirror this library was built with: the host asserts it equals sizeof(mz_zip_file) */
uint32_t mz_zip_cuda_abi_file_info_size(void);

#ifdef __cplusplus
}
#endif
#endif
