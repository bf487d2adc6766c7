/* zipbatch_pkshim.c -- TEST / BENCH INFRASTRUCTURE: puts the PKWARE entry points behind the C4 driver's WinZip AES modes.
 *
 * Preloaded (LD_PRELOAD) into oracle/_ref/zipbatch_cudae or zipbatch_emue, this library takes the place of the two AES entry points
 * the driver calls with a password:
 *   native_aes[_sha]   mz_zip_cuda_write_archive_aes  -> mz_zip_cuda_write_archive_pkcrypt (the AES flag dropped, SHA-256 kept)
 *   extract_aes        mz_zip_cuda_extract_all_aes    -> mz_zip_cuda_extract_all_encrypted
 * so the same driver, data generator and JSON lines serve the PKWARE tests. extract_ref_aes needs no shim: the reference's own loop
 * with the password reads PKWARE entries too (the driver's container is built with HAVE_PKCRYPT). Calls without a password go to
 * the library's own functions (the plain writer and extractor reach these names internally). Built by the tests with only the
 * project's headers: gcc -shared -fPIC zipbatch_pkshim.c -I include -ldl. */
#define _GNU_SOURCE
#include <dlfcn.h>
#include <stddef.h>
#include <stdint.h>

#include "mz_zip_cuda.h"

typedef int32_t (*write_aes_fn)(void *, const mz_cuda_zip_item *, uint32_t, int16_t, uint32_t, const char *, uint8_t, mz_cuda_zip_stats *);
typedef int32_t (*extract_aes_fn)(void *, const char *, mz_cuda_zip_entry_cb, void *, mz_cuda_zip_stats *);

int32_t mz_zip_cuda_write_archive_aes(void *base_stream, const mz_cuda_zip_item *items, uint32_t count, int16_t level, uint32_t flags,
                                      const char *password, uint8_t aes_strength, mz_cuda_zip_stats *stats) {
    if (!password) {
        write_aes_fn real = (write_aes_fn)dlsym(RTLD_NEXT, "mz_zip_cuda_write_archive_aes");
        return real ? real(base_stream, items, count, level, flags, password, aes_strength, stats) : -109;
    }
    return mz_zip_cuda_write_archive_pkcrypt(base_stream, items, count, level, flags & ~MZ_ZIP_CUDA_AES, password, stats);
}

int32_t mz_zip_cuda_extract_all_aes(void *zip_handle, const char *password, mz_cuda_zip_entry_cb cb, void *userdata, mz_cuda_zip_stats *stats) {
    if (!password) {
        extract_aes_fn real = (extract_aes_fn)dlsym(RTLD_NEXT, "mz_zip_cuda_extract_all_aes");
        return real ? real(zip_handle, password, cb, userdata, stats) : -109;
    }
    return mz_zip_cuda_extract_all_encrypted(zip_handle, password, cb, userdata, stats);
}
