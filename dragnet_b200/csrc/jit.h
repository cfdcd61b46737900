/*
 * jit.h: run-time compilation of a scan's record templates (tmpl.h / fast.h)
 * into the matcher of scan_kernel_j -- the F kernel with its interpreted trie
 * walk replaced by straight-line code with the literals as immediates.
 *
 * What is generated at run time is ONLY the matcher, dng_jmatch(): a few
 * hundred lines from the trie blob plus the wildcard scanners of fscan.cuh
 * (embedded as text).  NVRTC turns it into LTO-IR and nvJitLink optimises it
 * together with the LTO-IR build of the kernel that ships inside the library
 * (fast_jit.cu): the matcher is inlined into the record loop and registers are
 * allocated across it.  Everything else -- chunk pipeline, newline index,
 * stages, tally, miss handling -- is the code of scan_kernel_f; its rare paths
 * (fast_jit_cold.cu) are compiled ahead of time and only linked.  Results cannot depend on this choice: the generated
 * matcher accepts exactly what fmatch() accepts (same trie, same scanners) and
 * everything it rejects is parsed by the general code.
 *
 * Kernels are cached per process by a hash of the generated source.  Both
 * libraries are dlopen()ed; without them (or with DNG_JIT=0) scans use the
 * interpreted matcher.
 */
#ifndef DNG_JIT_H
#define DNG_JIT_H

#include <cuda_runtime.h>

#include <atomic>
#include <memory>
#include <string>

#include "fast.h"

namespace dng {

struct JitKernels {
	cudaLibrary_t lib = nullptr;
	cudaKernel_t kern = nullptr;	/* dng_scan_kernel_j for one slice size */
	std::atomic<int> state{0};	/* 0 being built, 1 ready, 2 failed */
	bool ok = false;
	std::string err;
	double compile_ms = 0, link_ms = 0;
};

/* the CUDA source of dng_jmatch() for an F trie blob (tmpl_build, compact)
 * and of the plan constant the kernel is specialised to (null: left out);
 * `prelude` replaces the device definitions the generated code builds on
 * (tests/hostcheck compiles the same code for the host with its own).  With a
 * value dictionary (dict->ncols != 0) and jit_dense() on, dng_jcode() looks the
 * record's key up in it (the kernel's dense counters). */
std::string jit_source(const u8 *blob, size_t bytes, const FPlan *plan,
    const char *prelude = nullptr, const FDict *dict = nullptr);

/*
 * Dense keys (fast.h FDict) in the run-time linked kernel: DNG_DENSE, default
 * 1; 0 turns them off (the hashed tally for every key).  Bits of a value other
 * than 0 and 1 pick variants: 2 keeps the hashed path for keys outside the
 * dictionary inline instead of calling it, 4 adds the lanes of a warp that
 * share a counter together before the shared-memory add.
 */
unsigned jit_dense();

/*
 * The kernels for this source on device `dev`, from the cache or built now:
 * on the caller's thread if `wait` (then state is 1 or 2 on return), else on a
 * worker thread (state 0 until it is done: the caller keeps using the
 * interpreted matcher meanwhile).  smem_max = dynamic shared memory the
 * kernels may be launched with.
 */
std::shared_ptr<JitKernels> jit_request(const std::string &source, int nsl,
    int dev, int smem_max, bool wait);

/* load the two compiler libraries now, on this thread (they are dlopen()ed
 * once per process); false if they are not there */
bool jit_prepare();

/* only compile + link, to `cubin` (no device needed: tests); nsl = 16-byte
 * units per lane slice: 7, 9, 11 or 13 */
bool jit_build(const std::string &source, int nsl, std::string &cubin,
    std::string &err, double *compile_ms, double *link_ms);

} /* namespace dng */

#endif
