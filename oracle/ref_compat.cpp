/*
 * oracle/ref_compat.cpp -- TEST INFRASTRUCTURE ONLY (never linked into the product).
 *
 * Link-time shims that let the unmodified reference hook (reference hook.cpp,
 * predictor.cpp, comm.cpp, debug.cpp) exist on this image (glibc 2.39, CUDA 12.9).
 * Nothing here changes the reference's algorithm; each shim only supplies a symbol
 * the reference expects from an older platform:
 *
 *  1. __libc_dlsym / __libc_dlopen_mode (reference hook.cpp:66-84) were removed
 *     in glibc 2.34.  They are re-provided on top of dlvsym/dlopen.
 *  2. In a non-_DEBUG build debug.cpp:66 defines hDEBUG with a 3-argument prefix
 *     while debug.h:33 declares (and every caller uses) the 4-argument one, so an
 *     -O2 build has an undefined symbol.  An empty 4-argument hDEBUG is provided
 *     (same behaviour as the intended empty stub).
 *  3. CUDA >= 12 runtimes resolve driver entry points through
 *     cuGetProcAddress_v2 (5 args).  The reference only exports the 4-argument
 *     legacy symbol (hook.cpp:875), so a CUDA-12 cudart would bypass every hook
 *     and the "reference overhead" would be a meaningless 0 %.  The _v2 export
 *     below delegates to the reference's own cuGetProcAddress, which performs the
 *     pointer swap (hook.cpp:885-970).  Driver-API clients (our storm app) do not
 *     need it: they bind the interposed symbols directly.
 *  4. ref_compat_path (ref_compat.h): /kubeshare/<rest> -> $REF_KUBESHARE_ROOT/<rest>
 *     when that variable is set, so the hook runs without root.
 */
#include <cuda.h>
#include <dlfcn.h>
#include <stdlib.h>
#include <string.h>

#include <string>

#undef cuGetProcAddress
extern "C" CUresult CUDAAPI cuGetProcAddress(const char *symbol, void **pfn, int cudaVersion,
                                             cuuint64_t flags);

typedef void *(*dlsym_fn)(void *, const char *);

static dlsym_fn true_dlsym() {
  static dlsym_fn fn = nullptr;
  if (!fn) {
    fn = (dlsym_fn)dlvsym(RTLD_NEXT, "dlsym", "GLIBC_2.2.5");
    if (!fn) fn = (dlsym_fn)dlvsym(RTLD_NEXT, "dlsym", "GLIBC_2.34");
  }
  return fn;
}

extern "C" CUresult CUDAAPI cuGetProcAddress_v2(const char *symbol, void **pfn, int cudaVersion,
                                                cuuint64_t flags,
                                                CUdriverProcAddressQueryResult *symbolStatus) {
  if (symbol && pfn && strcmp(symbol, "cuGetProcAddress") == 0) {
    // A CUDA-12 runtime asks the resolver for the resolver itself.  The reference would store what the driver answers
    // -- the 5-argument cuGetProcAddress_v2 -- and later call it through its 4-argument type (hook.cpp:879-885): the
    // fifth argument (where the driver WRITES the query result) is then whatever the register happens to hold.  The -O2
    // build survived that by luck, the DEBUG=1 (-O0) build crashed inside libcuda on the GPU box.  Answering here keeps
    // the reference on its own first branch (the legacy 4-argument entry point from dlsym) for every later lookup.
    *pfn = (void *)&cuGetProcAddress_v2;
    if (symbolStatus) *symbolStatus = CU_GET_PROC_ADDRESS_SUCCESS;
    return CUDA_SUCCESS;
  }
  CUresult r = cuGetProcAddress(symbol, pfn, cudaVersion, flags);
  if (symbolStatus)
    *symbolStatus = (r == CUDA_SUCCESS && pfn && *pfn) ? CU_GET_PROC_ADDRESS_SUCCESS
                                                       : CU_GET_PROC_ADDRESS_SYMBOL_NOT_FOUND;
  return r;
}

// dlsym as seen by the reference's real_dlsym(): identical to the libc one except that a
// lookup of "cuGetProcAddress_v2" lands on the export above (see 3.).
static void *compat_dlsym(void *handle, const char *symbol) {
  if (symbol && strcmp(symbol, "cuGetProcAddress_v2") == 0) return (void *)&cuGetProcAddress_v2;
  return true_dlsym()(handle, symbol);
}

extern "C" void *__libc_dlsym(void *map, const char *name) {
  (void)map;
  if (name && strcmp(name, "dlsym") == 0) return (void *)&compat_dlsym;
  return true_dlsym()(RTLD_NEXT, name);
}

extern "C" void *__libc_dlopen_mode(const char *name, int mode) {
  // the reference asks for unversioned dev names (hook.cpp:75-77); fall back to the sonames
  void *h = dlopen(name, mode);
  if (!h && name && strcmp(name, "libcuda.so") == 0) h = dlopen("libcuda.so.1", mode);
  if (!h && name && strcmp(name, "libdl.so") == 0) h = dlopen("libdl.so.2", mode);
  return h;
}

#ifndef _DEBUG
void hDEBUG(const char *, const char *, long, const char *, ...) {}
#endif

extern "C" const char *ref_compat_path(const char *path) {
  const char *root = getenv("REF_KUBESHARE_ROOT");
  if (!root || strncmp(path, "/kubeshare/", 11) != 0) return path;
  return (new std::string(std::string(root) + (path + 10)))->c_str();  // called once, at static initialisation
}
