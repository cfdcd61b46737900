/*
 * fast_jit_cold.cu: the rare paths of the run-time linked F kernel
 * (fast_jit.cu), compiled ahead of time as relocatable SASS: a key the inline
 * tally tier has no room for, a record the miss list has no room for (the
 * general parser, from HBM), the end-of-launch flush of the tally cache; with
 * dense keys, the key of a record outside the dictionary and the flush of the
 * dense counters.
 */
#define DNG_NO_GENERAL_KERNELS
#include "fast_kernel.cuh"

using namespace dng;

extern "C" __device__ void dng_cold_slow_add(FSmem m, const FPlan *F,
    u32 defmask, u32 klen, STab stab, const GTable *gt)
{
	fslow_add(m, F, defmask, klen, stab, gt);
}

extern "C" __device__ void dng_cold_miss(const u8 *data,
    unsigned long long start, unsigned long long beg, unsigned long long end,
    const DevPlan *plan, STab stab, const GTable *gt,
    unsigned long long *counters)
{
	fmiss_inline(data, start, beg, end, plan, stab, gt, counters);
}

extern "C" __device__ void dng_cold_flush(STab stab, u32 s1slots, u32 sslots,
    const GTable *tab)
{
	flush_tally(stab, s1slots, sslots, *tab);
}

/* hash + tally of a record's key (false: too long for the F path, a miss) */
extern "C" __device__ u32 dng_cold_key(FSmem m, const FPlan *F, u32 defmask,
    STab stab, const GTable *gt, u32 over_sa)
{
	u32 h, klen;
	if (!fkey_hash(m, *F, defmask, h, klen))
		return 0;
	ftally(m, *F, F, defmask, h, klen, stab, *gt, over_sa);
	return 1;
}

/*
 * The dense counters of the CTA -> the global table, keyed by the bytes
 * fkey_write() gives the same values: a key counted densely here and hashed
 * in another CTA (or launch) is one entry.  Counters at zero add nothing.
 */
extern "C" __device__ void dng_cold_dense_flush(u32 dense_sa, const FDict *D,
    const GTable *gt)
{
	const u32 total = D->total;
	for (u32 i = threadIdx.x; i < total; i += blockDim.x) {
		const u32 c = lds32(dense_sa + 4 * i);
		if (!c)
			continue;
		__align__(8) u8 kbuf[F_MAXKEY + 16];
		const u32 klen = fdense_key(*D, i, kbuf);
		const unsigned long long *kw = (const unsigned long long *)kbuf;
		global_add(*gt, key_hash_words(kw, klen), kbuf, klen,
		    (unsigned long long)c);
	}
}
