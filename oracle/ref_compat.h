/*
 * oracle/ref_compat.h -- TEST INFRASTRUCTURE ONLY (never linked into the product).
 *
 * Force-included (-include) when the *unmodified* reference sources under
 * /root/reference/Gemini/src are compiled into oracle/_ref/.  It contains no
 * reference code; it only restores the toolchain assumptions the reference was
 * written against (CUDA <= 11.4 headers, glibc < 2.34):
 *
 *  - CUDA 12 maps `cuGetProcAddress` to the 5-argument `cuGetProcAddress_v2`
 *    (cuda.h:156).  The reference declares and defines the legacy 4-argument
 *    entry point (reference hook.cpp:79, 875-980), so the macro is removed and
 *    the legacy prototype is given C linkage here, exactly as the old cuda.h did.
 *  - comm.cpp:130 uses `errno` without including <cerrno>.
 *  - The hook reads its pod manager's address from the absolute path
 *    /kubeshare/library/schedulerIP.txt (hook.cpp:162, 233-237), which only root can
 *    create outside a KubeShare pod.  The Makefile routes that one path through
 *    ref_compat_path(): with REF_KUBESHARE_ROOT set, /kubeshare/... is looked up
 *    under that directory instead.
 *
 * The missing glibc-private symbols (__libc_dlsym, __libc_dlopen_mode), the
 * missing non-debug hDEBUG overload and the cuGetProcAddress_v2 export live in
 * oracle/ref_compat.cpp.
 */
#ifndef GEMHOOK_ORACLE_REF_COMPAT_H
#define GEMHOOK_ORACLE_REF_COMPAT_H

#include <cerrno>

extern "C" const char *ref_compat_path(const char *path);

#ifdef REF_COMPAT_WITH_CUDA
#include <cuda.h>
#undef cuGetProcAddress
extern "C" CUresult CUDAAPI cuGetProcAddress(const char *symbol, void **pfn, int cudaVersion,
                                             cuuint64_t flags);
#endif

#endif
