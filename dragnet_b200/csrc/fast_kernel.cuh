/*
 * fast_kernel.cuh: scan_kernel_f, the F path's kernel (fast.h), and
 * scan_miss_kernel, which hands the records it did not take to the general
 * per-record code.
 *
 * Geometry: one persistent 896-thread CTA per SM; every WARP is its own
 * pipeline, as in scan_kernel_w, over SEGMENTS of consecutive chunks:
 *
 *   - a chunk is 32 lane slices of NSL x 16 bytes (the host picks NSL so that
 *     a chunk holds just under 32 average records), staged by one TMA bulk
 *     copy into the warp's private buffer behind a 512-byte pre-lap;
 *   - the record that straddles two chunks of a segment never goes back to
 *     HBM: before the next chunk is staged, the warp copies the last 512 bytes
 *     of its buffer into the pre-lap (shared -> shared) and carries the start
 *     of the open record over.  Only a segment's first chunk stages its
 *     pre-lap from HBM;
 *   - newline index: every lane tests its slice 16 bytes at a time with one
 *     "any byte == '\n'" SWAR test per word (exact analysis only where it
 *     fires), a shuffle scan orders the hits, lanes write their (<= 4)
 *     positions; record r of the chunk goes to lane r;
 *   - fmatch() -> fstage() -> fkey_hash() / tally (fast.cuh): captures are one
 *     word per path in shared memory ([path][thread]: conflict free), the key
 *     is hashed and compared in place against the CTA's tally cache;
 *   - a record the F path does not decide is appended to the miss list
 *     (absolute offsets) and parsed by scan_miss_kernel right after this
 *     kernel; if the list is full it is parsed here, out of line, from HBM.
 *
 * Bound: HBM read of the input, once (+ 512 bytes per segment).
 */
#ifndef DNG_FAST_KERNEL_CUH
#define DNG_FAST_KERNEL_CUH

#include <stddef.h>

#include "scan_kernel.cuh"
#include "fast.cuh"

namespace dng {

#define DNG_F_NT F_NT			/* threads per CTA */
#define DNG_F_NW (DNG_F_NT / 32)
#define DNG_F_PRE 512			/* pre-lap bytes = longest straddling head */
#define DNG_F_SLACK 64
#define DNG_F_NLCAP 128			/* newline positions per chunk */
#define DNG_F_MAXLINE DNG_F_PRE		/* host: sampled lines must be shorter */
#define DNG_F_SEG 16			/* chunks per segment (at most) */

struct MissEnt {
	unsigned long long beg;		/* ~0: unknown, before `end` */
	unsigned long long end;		/* the record's newline (or end of input) */
};

struct FScanArgs {
	const u8 *data;			/* 16-byte aligned */
	unsigned long long start;	/* first valid byte (< 16) */
	unsigned long long nbytes;	/* end of valid bytes */
	const FPlan *fplan;
	const DevPlan *plan;		/* the full plan (global): overflow path */
	const u8 *tmpl;			/* F trie blob or null */
	u32 tmpl_bytes;
	u32 leaf_off, pool_off;		/* its THdr's, for the kernel's convenience */
	unsigned long long *counters;
	GTable tab;
	u32 nchunks, seg;		/* chunks, chunks per segment */
	u32 final;
	u32 s1slots, sslots;
	u32 ndense;			/* dense counters (FDict::total; 0: none),
					 * rounded up to a multiple of 4 */
	const FDict *dict;
	u32 nrows;			/* capture rows (FPlan::nrows) */
	MissEnt *miss;
	u32 miss_cap;
	u32 *miss_n;
	u32 *seg_next;			/* segment queue: zero at launch */
};

/* per-warp shared memory: buffer, newline positions, mbarrier */
template <int NSL>
struct FWarpSmem {
	static constexpr u32 CHUNK = 32 * 16 * NSL;
	static constexpr u32 BUF = DNG_F_PRE + CHUNK + DNG_F_SLACK;
	static constexpr u32 BYTES = (BUF + 2 * DNG_F_NLCAP + 16 + 127) & ~127u;
};

static constexpr u32 FPLAN_SMEM = (sizeof (FPlan) + 127) & ~127u;

/* (nw = warps of the launch: DNG_F_NW, or fewer -- the capture rows keep
 * their stride -- when the tally cache needs the room) */
template <int NSL>
static inline size_t fkernel_smem(u32 tmpl_bytes, u32 s1slots, u32 sslots,
    u32 nrows, u32 nw = DNG_F_NW, u32 ndense = 0)
{
	return FPLAN_SMEM + tmpl_bytes + (size_t)s1slots * sizeof (SSlot1) +
	    (size_t)sslots * sizeof (SSlot) + (size_t)ndense * 4 +
	    (size_t)nrows * DNG_F_NT * 4 + (size_t)nw * FWarpSmem<NSL>::BYTES;
}

/* mbarrier / TMA helpers on 32-bit shared addresses (no generic pointers to
 * keep alive across the record loop) */
__device__ __forceinline__ void mbar_init_sa(u32 bar, u32 count)
{
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;"
	    :: "r"(bar), "r"(count) : "memory");
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_expect_tx_sa(u32 bar, u32 bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
	    :: "r"(bar), "r"(bytes) : "memory");
}

__device__ __forceinline__ void tma_load_1d_sa(u32 dst, const void *src,
    u32 bytes, u32 bar)
{
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::"
	    "complete_tx::bytes [%0], [%1], %2, [%3];"
	    :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

__device__ __forceinline__ void mbar_wait_sa(u32 bar, u32 parity)
{
	asm volatile(
	    "{\n"
	    ".reg .pred p;\n"
	    "WAIT_%=:\n"
	    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
	    "@p bra DONE_%=;\n"
	    "bra WAIT_%=;\n"
	    "DONE_%=:\n"
	    "}\n"
	    :: "r"(bar), "r"(parity) : "memory");
}

__device__ __forceinline__ void sts8(u32 addr, u32 v)
{
	asm volatile("st.shared.u8 [%0], %1;" :: "r"(addr), "r"(v) : "memory");
}

__device__ __forceinline__ void sts16(u32 addr, u32 v)
{
	asm volatile("st.shared.u16 [%0], %1;" :: "r"(addr), "r"(v) : "memory");
}

__device__ __forceinline__ void sts128(u32 addr, uint4 v)
{
	asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};"
	    :: "r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ void sts32(u32 addr, u32 v)
{
	asm volatile("st.shared.u32 [%0], %1;" :: "r"(addr), "r"(v) : "memory");
}

/* shared-memory access for fmatch()/fstage()/fkey_*() */
struct FSmem {
	u32 ra;			/* record start (shared address) */
	u32 nodes, leaves, pool;
	u32 caps;		/* this thread's capture column */

	typedef TmplSmem::Cur Cur;
	__device__ __forceinline__ Cur cursor(u32 off) const
	{
		Cur c;
		const u32 a = ra + off;
		c.sh = (a & 3) * 8;
		c.wa = (a & ~3u) + 4;
		c.w0 = lds32(c.wa - 4);
		c.w1 = lds32(c.wa);
		return c;
	}
	/* aligned words (fscan.cuh) */
	struct ACur {
		u32 wa, k;
		__device__ __forceinline__ u32 next()
		{
			const u32 v = lds32(wa);
			wa += 4;
			return v;
		}
	};
	__device__ __forceinline__ ACur acursor(u32 off) const
	{
		ACur c;
		const u32 a = ra + off;
		c.k = a & 3;
		c.wa = a & ~3u;
		return c;
	}
	__device__ __forceinline__ u32 apos(const ACur &c) const
	{
		return c.wa - 4 - ra;
	}
	__device__ __forceinline__ u32 byte(u32 off) const { return lds8(ra + off); }
	__device__ __forceinline__ u32 word(u32 off) const
	{
		Cur c = cursor(off);
		return c.next();
	}
	__device__ __forceinline__ const u8 *ptr(u32 off) const
	{
		return (const u8 *)__cvta_shared_to_generic(ra + off);
	}
	__device__ __forceinline__ TQuad node(u32 i) const
	{
		const uint4 v = lds128(nodes + i * 16);
		TQuad q;
		q.x = v.x; q.y = v.y; q.z = v.z; q.w = v.w;
		return q;
	}
	__device__ __forceinline__ u32 litw(u32 off) const { return lds32(pool + off); }
	__device__ __forceinline__ u32 leaf(u32 i) const { return lds32(leaves + 4 * i); }
	__device__ __forceinline__ u32 pool32(u32 off) const { return lds32(pool + off); }
	__device__ __forceinline__ void setcap(u32 p, u32 v) const
	{
		sts32(caps + p * (DNG_F_NT * 4), v);
	}
	__device__ __forceinline__ u32 getcap(u32 p) const
	{
		return lds32(caps + p * (DNG_F_NT * 4));
	}
};

/* a tally slot's inline key, any alignment */
struct FKeySmem {
	u32 ka;
	typedef TmplSmem::Cur Cur;
	__device__ __forceinline__ Cur cursor(u32 off) const
	{
		Cur c;
		const u32 a = ka + off;
		c.sh = (a & 3) * 8;
		c.wa = (a & ~3u) + 4;
		c.w0 = lds32(c.wa - 4);
		c.w1 = lds32(c.wa);
		return c;
	}
};

#ifdef DNG_JIT_HOT
/*
 * The link-time-optimised build of the kernel (fast_jit.cu) keeps its rare,
 * large paths out of the optimiser's way: they are compiled ahead of time
 * (fast_jit_cold.cu) and only linked in.
 */
extern "C" __device__ void dng_cold_slow_add(FSmem m, const FPlan *F,
    u32 defmask, u32 klen, STab stab, const GTable *gt);
extern "C" __device__ void dng_cold_miss(const u8 *data,
    unsigned long long start, unsigned long long beg, unsigned long long end,
    const DevPlan *plan, STab stab, const GTable *gt,
    unsigned long long *counters);
extern "C" __device__ void dng_cold_flush(STab stab, u32 s1slots, u32 sslots,
    const GTable *tab);
extern "C" __device__ u32 dng_cold_key(FSmem m, const FPlan *F, u32 defmask,
    STab stab, const GTable *gt, u32 over_sa);
extern "C" __device__ void dng_cold_dense_flush(u32 dense_sa, const FDict *D,
    const GTable *gt);
/*
 * The scan's plan as a CONSTANT of the generated code (jit.cpp writes it out
 * with its initialiser): after link-time optimisation the stage and key code
 * below is specialised to it -- column loops unrolled, kinds and entry points
 * folded, absent filters gone.  (The copy in shared memory is still what the
 * rare paths are handed.)
 */
extern "C" __constant__ const FPlan dng_jplan;
/*
 * Dense keys (fast.h FDict), generated with the matcher when the scan learned
 * a value dictionary: dng_jcode() = the record's dense counter, or ~0u.
 * dng_jdense (jit.h jit_dense()): 0 no dictionary; bit 0 dense counters, bit 1
 * keys outside the dictionary hashed inline rather than by a call to
 * dng_cold_key(), bit 2 lanes with the same counter added up first.
 */
extern "C" __constant__ const unsigned dng_jdense;
extern "C" __device__ unsigned dng_jcode(unsigned ra, unsigned dm,
    unsigned caps);
#define fslow_add dng_cold_slow_add
#define fmiss_inline dng_cold_miss
#else
/* first sighting of a key in this CTA, or a key the inline tier has no room
 * for: materialise it and take the general tally path */
__device__ __noinline__ void fslow_add(FSmem m, const FPlan *F, u32 defmask,
    u32 klen, STab stab, const GTable *gt)
{
	__align__(8) u8 kbuf[F_MAXKEY + 16];
	fkey_write(m, *F, defmask, kbuf);
	const unsigned long long *kw = (const unsigned long long *)kbuf;
	shared_add(stab, *gt, key_hash_words(kw, klen), kw, klen, 1);
}

#endif /* DNG_JIT_HOT */

__device__ __forceinline__ unsigned long long lds64_acquire(u32 addr)
{
	unsigned long long v;
	asm volatile("ld.acquire.cta.shared.u64 %0, [%1];" : "=l"(v) : "r"(addr)
	    : "memory");
	return v;
}

__device__ __forceinline__ void sts64_release(u32 addr, unsigned long long v)
{
	asm volatile("st.release.cta.shared.u64 [%0], %1;" :: "r"(addr), "l"(v)
	    : "memory");
}

/*
 * Count the record's key: the CTA's inline tier, probed with the F hash.  A
 * slot's tag is published with release semantics once its key is written and
 * read with acquire semantics (plain shared loads and stores in SASS: no
 * fence on the path every record takes).
 */
__device__ __forceinline__ void ftally(FSmem &m, const FPlan &F,
    const FPlan *Fcold, u32 defmask, u32 h, u32 klen, const STab &stab,
    const GTable &gt, u32 over_sa)
{
	if (klen <= DNG_SKEY) {
		const unsigned long long claim = (unsigned long long)(h | 1u);
		u32 idx = (h >> 7) & stab.mask1;
		for (u32 probe = 0; probe < 8; probe++) {
			SSlot1 *s = &stab.s1[idx];
			const u32 sa = smem_u32(s);
			unsigned long long tag = lds64_acquire(sa);
			if (tag == 0) {
				const unsigned long long old =
				    atomicCAS(&s->tag, 0ull, claim);
				if (old == 0) {
					s->klen = klen;
					fkey_write(m, F, defmask, (u8 *)s->key);
					atomicAdd(&s->count, 1u);
					sts64_release(sa, claim | DNG_READY);
					return;
				}
				tag = old;
			}
			if ((tag & ~DNG_READY) == claim) {
				while (!(tag & DNG_READY))
					tag = lds64_acquire(sa);
				if (lds32(sa + (u32)offsetof(SSlot1, klen)) == klen) {
					FKeySmem k;
					k.ka = sa + (u32)offsetof(SSlot1, key);
					if (fkey_equal(m, F, defmask, k)) {
						atomicAdd(&s->count, 1u);
						return;
					}
				}
			}
			idx = (idx + 1) & stab.mask1;
		}
	}
	/* (counted: the host gives the cache more room if this is common) */
	asm volatile("red.shared.add.u32 [%0], 1;" :: "r"(over_sa) : "memory");
	fslow_add(m, Fcold, defmask, klen, stab, &gt);
}

#ifndef DNG_JIT_HOT
/*
 * A record the miss list had no room for: the general parser, from HBM, right
 * here.  Entirely out of line, with its own counters (added to the global
 * ones directly), so that the kernel's per-thread state stays in registers.
 */
__device__ __noinline__ void fmiss_inline(const u8 *data,
    unsigned long long start, unsigned long long beg, unsigned long long end,
    const DevPlan *plan, STab stab, const GTable *gt,
    unsigned long long *counters)
{
	u32 mctr[(MAX_METRICS - 1) * MCTR_PER];
	for (int k = 0; k < (MAX_METRICS - 1) * MCTR_PER; k++)
		mctr[k] = 0;
	LocalCounters C;
	C.lines = C.invalid_json = C.invalid_point = 0;
	C.ds_filtered = C.ds_failedeval = C.user_filtered = 0;
	C.user_failedeval = C.synth_undef = C.synth_baddate = 0;
	C.time_filtered = C.time_failedeval = C.aggr = C.slow = 0;
	C.unsupported = 0;
	unsigned long long q = beg;
	u32 nlong = 0;
	if (q == ~0ull) {
		q = end;
		while (q > start && data[q - 1] != '\n')
			q--;
		nlong = 1;
	}
	scan_one_global(data + q, (u32)min((unsigned long long)DNG_MAXREC,
	    end - q), *plan, stab, *gt, C, mctr);
	const u32 vals[CTR_TMPL] = { C.lines, C.invalid_json, C.invalid_point,
	    C.ds_filtered, C.ds_failedeval, C.user_filtered, C.user_failedeval,
	    C.synth_undef, C.synth_baddate, C.time_filtered, C.time_failedeval,
	    C.aggr, C.slow, C.unsupported, nlong };
	for (int k = 0; k < CTR_TMPL; k++)
		if (vals[k])
			atomicAdd(&counters[k], (unsigned long long)vals[k]);
}

#endif /* DNG_JIT_HOT */

/* append to the miss list, or parse here when it is full */
__device__ __forceinline__ void fmiss_put(const FScanArgs &a, const STab &stab,
    u32 at, unsigned long long beg, unsigned long long end)
{
	if (at < a.miss_cap) {
		MissEnt e;
		e.beg = beg;
		e.end = end;
		a.miss[at] = e;
	} else {
		fmiss_inline(a.data, a.start, beg, end, a.plan, stab, &a.tab,
		    a.counters);
	}
}

/*
 * The matcher the run-time compiler generates for one scan's templates
 * (jit.cpp): fmatch() with the trie turned into straight-line code, literals as
 * immediates.  Returns 0, or 1 | defmask << 1.  Only the relocatable build of
 * this file (fast_jit.cu) calls it; it is resolved when that build is linked
 * with the generated code.
 */
extern "C" __device__ unsigned dng_jmatch(unsigned ra, unsigned len,
    unsigned active, unsigned caps);

template <int NSL, bool JIT>
__device__ __forceinline__ void fscan_body(const FScanArgs &a)
{
	typedef FWarpSmem<NSL> WS;
	constexpr u32 CHUNK = WS::CHUNK, SLICE = 16 * NSL, D0 = DNG_F_PRE;
	extern __shared__ __align__(128) u8 smem[];
#ifdef DNG_JIT_HOT
	const FPlan &F = dng_jplan;
#else
	const FPlan &F = *(const FPlan *)smem;
#endif
	u8 *sp = smem + FPLAN_SMEM;
	const u32 tmpl_sa = smem_u32(sp);
	sp += a.tmpl_bytes;
	STab stab;
	stab.s1 = (SSlot1 *)sp;
	sp += a.s1slots * sizeof (SSlot1);
	stab.s = (SSlot *)sp;
	sp += a.sslots * sizeof (SSlot);
	const u32 dense_sa = smem_u32(sp);
	sp += a.ndense * 4;
	stab.mask1 = a.s1slots - 1;
	stab.mask = a.sslots - 1;
	const u32 caps_sa = smem_u32(sp);
	sp += a.nrows * DNG_F_NT * 4;

	const u32 tid = threadIdx.x;
	const u32 lane = tid & 31, wid = tid >> 5;
	/* this warp's buffer, newline positions (u16) and mbarrier: shared
	 * addresses */
	const u32 sb = smem_u32(sp) + wid * WS::BYTES;
	const u32 nlpos = sb + WS::BUF;
	const u32 mbar = sb + WS::BUF + 2 * DNG_F_NLCAP;

	{	/* plan, templates -> shared; clear the tally cache */
		const uint4 *src = (const uint4 *)a.fplan;
		uint4 *dst = (uint4 *)smem;
		for (u32 i = tid; i < FPLAN_SMEM / 16; i += blockDim.x)
			dst[i] = src[i];
		const uint4 *tsrc = (const uint4 *)a.tmpl;
		uint4 *tdst = (uint4 *)(smem + FPLAN_SMEM);
		for (u32 i = tid; i < a.tmpl_bytes / 16; i += blockDim.x)
			tdst[i] = tsrc[i];
		const uint4 z = make_uint4(0, 0, 0, 0);
		uint4 *tz = (uint4 *)stab.s1;
		/* (and the dense counters behind it) */
		const u32 tab_bytes = a.s1slots * (u32)sizeof (SSlot1) +
		    a.sslots * (u32)sizeof (SSlot) + a.ndense * 4;
		for (u32 i = tid; i < tab_bytes / 16; i += blockDim.x)
			tz[i] = z;
		if (lane == 0)
			mbar_init_sa(mbar, 1);
		/* the quotes after the buffer that end a runaway string scan
		 * (fscan.cuh) */
		if (lane < DNG_F_SLACK / 4)
			sts32(sb + D0 + CHUNK + 4 * lane, 0x22222222u);
	}
	__syncthreads();

	const bool use_tmpl = a.tmpl_bytes != 0;
	FSmem m;
	m.ra = 0;
	m.nodes = tmpl_sa + (u32)sizeof (THdr);
	m.leaves = tmpl_sa + a.leaf_off;
	m.pool = tmpl_sa + a.pool_off;
	m.caps = caps_sa + tid * 4;

	/* counters: records taken and aggregated per warp (the same value in
	 * every lane); the drop counters and `slow` in shared memory */
	__shared__ u32 s_drop[16];
	if (tid < 16)
		s_drop[tid] = 0;
	u32 ntmpl = 0, naggr = 0, parity = 0;
	const u32 ltmask = (1u << lane) - 1;

	/*
	 * Segments are handed out through a counter: a warp that finishes
	 * early takes the next one, so that the launch ends within a segment's
	 * time of its last warp (static shares left 13% of the warp time parked
	 * at the final barrier).  The first round is implicit -- warp gw takes
	 * segment gw, spread over the SMs -- the counter hands out the rest.
	 */
	const u32 nwarps = gridDim.x * (blockDim.x >> 5);
	const u32 gw = wid * gridDim.x + blockIdx.x;
	const u32 nseg = (a.nchunks + a.seg - 1) / a.seg;

	for (u32 seg = gw; seg < nseg; ) {
		const u32 ch0 = seg * a.seg;
		const u32 ch1 = min(ch0 + a.seg, a.nchunks);
		/* the open record: where it starts in the buffer (may be
		 * negative: before it), and in the input if that is known */
		int beg0 = 0;
		unsigned long long open_abs = ~0ull;
		for (u32 ch = ch0; ch < ch1; ch++) {
			const unsigned long long g0 = (unsigned long long)ch * CHUNK;
			const u32 dlen = (u32)min((unsigned long long)CHUNK,
			    a.nbytes - g0);
			const u32 bulk = dlen & ~15u;
			const bool first = ch == ch0;

			__syncwarp();
			if (!first) {
				/* the tail of the previous chunk becomes the
				 * pre-lap of this one */
				const uint4 v = lds128(sb + D0 + CHUNK - DNG_F_PRE +
				    16 * lane);
				__syncwarp();
				sts128(sb + 16 * lane, v);
				__syncwarp();
			}
			if (lane == 0) {
				const u32 pre = (first && g0) ? DNG_F_PRE : 0;
				asm volatile("fence.proxy.async.shared::cta;"
				    ::: "memory");
				if (bulk + pre) {
					mbar_expect_tx_sa(mbar, bulk + pre);
					if (bulk)
						tma_load_1d_sa(sb + D0, a.data + g0,
						    bulk, mbar);
					if (pre)
						tma_load_1d_sa(sb, a.data + g0 -
						    DNG_F_PRE, DNG_F_PRE, mbar);
				}
				/* start pulling this warp's next chunk into L2 */
				const unsigned long long nx = g0 + CHUNK;
				if (ch + 1 < ch1 && nx + CHUNK <= a.nbytes)
					asm volatile("cp.async.bulk.prefetch.L2."
					    "global [%0], %1;" :: "l"(a.data + nx),
					    "r"(CHUNK) : "memory");
			}
			for (u32 i = bulk + lane; i < dlen; i += 32)
				sts8(sb + D0 + i, a.data[g0 + i]);
			/* (a short last chunk: the sentinel right behind it) */
			if (dlen < CHUNK && lane < 16)
				sts8(sb + D0 + dlen + lane, '"');
			if (bulk || (first && g0)) {
				mbar_wait_sa(mbar, parity);
				parity ^= 1;
			}
			__syncwarp();

			/* valid bytes of the buffer: [lo, hi) */
			const u32 lo = g0 ? 0 : D0 + (u32)a.start;
			const u32 hi = D0 + dlen;
			if (first) {
				/* where the open record starts: after the last
				 * newline of the pre-lap, which the lanes search
				 * together (16 bytes each) */
				beg0 = (int)lo;
				open_abs = a.start;
				if (g0) {
					const uint4 v = lds128(sb + D0 - 16 * (lane + 1));
					const u32 wd[4] = { v.x, v.y, v.z, v.w };
					u32 mine = 0;
#pragma unroll
					for (int j = 3; j >= 0; j--) {
						const u32 mk = nl_mask(wd[j]);
						if (mk && !mine)
							mine = D0 - 16 * (lane + 1) +
							    4 * j + ((31 - __clz(mk)) >> 3) + 1;
					}
					const u32 best = __reduce_max_sync(0xffffffffu,
					    mine);
					beg0 = best ? (int)best : -1;
					open_abs = best ? g0 - D0 + best : ~0ull;
				}
			}

			/* ---- newline index ---- */
			/*
			 * Bit j of hot: 16-byte unit j of the lane's slice holds a
			 * newline (a SWAR test with no false negatives); the units
			 * it flags are then looked at exactly, twice: to count, and
			 * -- once a shuffle scan has ordered the lanes -- to write
			 * the positions.
			 */
			const u32 c0 = D0 + lane * SLICE;
			u32 hot = 0, cnt = 0, one = 0;
#pragma unroll
			for (u32 j = 0; j < (u32)NSL; j++) {
				/* any byte <= '\n' in these 16?  (b - 0x0b borrows
				 * exactly for those; a borrow into the next byte can
				 * only add a flag) */
				const uint4 v = lds128(sb + c0 + 16 * j);
				u32 t = (v.x - 0x0b0b0b0bu) & ~v.x;
				t |= (v.y - 0x0b0b0b0bu) & ~v.y;
				t |= (v.z - 0x0b0b0b0bu) & ~v.z;
				t |= (v.w - 0x0b0b0b0bu) & ~v.w;
				if (t & 0x80808080u)
					hot |= 1u << j;
			}
#pragma unroll 1
			for (u32 hm = hot; hm; hm &= hm - 1) {
				const u32 p = c0 + 16 * (__ffs(hm) - 1);
				const uint4 v = lds128(sb + p);
				if (p >= lo && p + 16 <= hi) {
					const u32 m0 = nl_mask(v.x), m1 = nl_mask(v.y);
					const u32 m2 = nl_mask(v.z), m3 = nl_mask(v.w);
					const u32 k = __popc(m0) + __popc(m1) +
					    __popc(m2) + __popc(m3);
					/* (the usual case, one newline per lane: its
					 * position right away) */
					if (k == 1)
						one = p + (m0 ? 0 : m1 ? 4 : m2 ? 8 : 12) +
						    ((__ffs(m0 | m1 | m2 | m3) - 1) >> 3);
					cnt += k;
				} else {
					/* the ends of the input: byte by byte */
					for (u32 x = 0; x < 16; x++)
						cnt += p + x >= lo && p + x < hi &&
						    lds8(sb + p + x) == '\n';
				}
			}
			/* an unterminated final line ends at a virtual newline:
			 * it is never templated (nothing terminates its scans) */
			const bool lastch = ch + 1 == a.nchunks;
			bool vnl = false;
			if (lastch && a.final && hi > lo)
				vnl = lds8(sb + hi - 1) != '\n';

			u32 incl = cnt;
#pragma unroll
			for (int d = 1; d < 32; d <<= 1) {
				const u32 y = __shfl_up_sync(0xffffffffu, incl, d);
				if (lane >= (u32)d)
					incl += y;
			}
			const u32 mybase = incl - cnt;
			const u32 total = __shfl_sync(0xffffffffu, incl, 31);
			const bool dense = total > DNG_F_NLCAP;
			if (dense) {
				/*
				 * Degenerate input (lines of a few bytes): one lane
				 * walks the chunk and hands every record to the
				 * general parser.
				 */
				if (lane == 0) {
					unsigned long long b = open_abs;
					for (u32 p = max(lo, D0); p < hi; p++) {
						if (lds8(sb + p) != '\n')
							continue;
						const unsigned long long e = g0 - D0 + p;
						fmiss_put(a, stab, atomicAdd(a.miss_n, 1u),
						    b, e);
						b = e + 1;
					}
					open_abs = b;
				}
				open_abs = __shfl_sync(0xffffffffu, open_abs, 0);
				/* (beg0 of the next chunk is recomputed below) */
				int last = -1;
				for (int p = (int)hi - 1; p >= (int)max(lo, D0); p--)
					if (lds8(sb + p) == '\n') {
						last = p;
						break;
					}
				if (last >= 0)
					beg0 = last + 1;
			} else if (total) {
				if (cnt == 1 && one) {
					sts16(nlpos + 2 * mybase, one);
				} else if (cnt) {
					u32 idx = mybase;
#pragma unroll 1
					for (u32 hm = hot; hm; hm &= hm - 1) {
						const u32 p = c0 + 16 * (__ffs(hm) - 1);
#pragma unroll 1
						for (u32 q = 0; q < 4; q++) {
							u32 mk = nl_mask(lds32(sb + p + 4 * q));
#pragma unroll 1
							for (; mk; mk &= mk - 1) {
								const u32 pos = p + 4 * q +
								    ((__ffs(mk) - 1) >> 3);
								if (pos >= lo && pos < hi)
									sts16(nlpos + 2 * idx++,
									    pos);
							}
						}
					}
				}
				__syncwarp();

				for (u32 rb = 0; rb < total; rb += 32) {
					const u32 r = rb + lane;
					const bool have = r < total;
					int beg = 0;
					u32 end = 0;
					if (have) {
						end = lds16(nlpos + 2 * r);
						beg = r ? (int)lds16(nlpos + 2 * r - 2) + 1 :
						    beg0;
					}
					/* (captures carry 12-bit offsets and lengths) */
					const bool inbuf = have && beg >= 0 &&
					    end - (u32)beg <= F_MAXLINE;
					const u32 len = inbuf ? end - (u32)beg : 0;
					m.ra = sb + (inbuf ? (u32)beg : 0);
					u32 defmask = 0;
					u32 fo = FO_MISS;
					bool matched;
					if (JIT) {
						const u32 r_ = dng_jmatch(m.ra, len, inbuf,
						    m.caps);
						matched = r_ & 1;
						defmask = r_ >> 1;
					} else {
						matched = use_tmpl &&
						    fmatch(m, len, inbuf, defmask);
					}
					u32 dc = ~0u;	/* dense counter */
					if (matched) {
						double s0, s1;
						fo = fstage(m, F, defmask, s0, s1);
						u32 h = 0, klen = 0, slow = 0;
						if (fo == FO_AGGR && !fprep(m, F, defmask,
						    s0, s1, slow))
							fo = FO_MISS;
#ifdef DNG_JIT_HOT
						if (fo == FO_AGGR && (dng_jdense & 1))
							dc = dng_jcode(m.ra, defmask, m.caps);
						if (dc != ~0u) {
							/* (counted below) */
						} else if (fo == FO_AGGR &&
						    (dng_jdense & 3) == 1) {
							/* a key outside the dictionary:
							 * out of line, so that the loop
							 * is the dense path's size */
							if (!dng_cold_key(m, (const FPlan *)smem,
							    defmask, stab, &a.tab,
							    smem_u32(&s_drop[15])))
								fo = FO_MISS;
						} else
#endif
						if (fo == FO_AGGR) {
							if (!fkey_hash(m, F, defmask, h, klen))
								fo = FO_MISS;
							else
								ftally(m, F, (const FPlan *)smem,
								    defmask, h, klen, stab, a.tab,
								    smem_u32(&s_drop[15]));
						}
						if (fo == FO_AGGR && slow)
							atomicAdd(&s_drop[1], 1u);
					}
#ifdef DNG_JIT_HOT
					/* dense counters (u32, per launch: like the
					 * inline tally tier's) */
					if (dng_jdense & 4) {
						const u32 peers = __match_any_sync(
						    0xffffffffu, dc);
						if (dc != ~0u && !(peers & ltmask))
							asm volatile("red.shared.add.u32 "
							    "[%0], %1;" :: "r"(dense_sa +
							    4 * dc), "r"(__popc(peers))
							    : "memory");
					} else if (dc != ~0u) {
						asm volatile("red.shared.add.u32 [%0], 1;"
						    :: "r"(dense_sa + 4 * dc) : "memory");
					}
#endif
					const bool done = fo != FO_MISS;
					ntmpl += __popc(__ballot_sync(0xffffffffu, done));
					naggr += __popc(__ballot_sync(0xffffffffu,
					    fo == FO_AGGR));
					{
						/* dropped records: one shared atomic per
						 * outcome present in the warp */
						u32 dm = __ballot_sync(0xffffffffu,
						    fo >= FO_DS_FILTERED);
						while (dm) {
							const u32 f0 = __shfl_sync(0xffffffffu,
							    fo, __ffs(dm) - 1);
							const u32 same = __ballot_sync(
							    0xffffffffu, fo == f0);
							if (lane == 0)
								atomicAdd(&s_drop[f0],
								    (u32)__popc(same));
							dm &= ~same;
						}
					}
					/* what the F path did not take */
					const bool miss = have && !done;
					const u32 mm = __ballot_sync(0xffffffffu, miss);
					if (mm) {
						u32 base = 0;
						if (lane == 0)
							base = atomicAdd(a.miss_n,
							    (u32)__popc(mm));
						base = __shfl_sync(0xffffffffu, base, 0);
						if (miss)
							fmiss_put(a, stab, base +
							    __popc(mm & ltmask), r ? g0 - D0 +
							    (u32)beg : open_abs, g0 - D0 + end);
					}
				}
				__syncwarp();
				const u32 lastnl = lds16(nlpos + 2 * (total - 1));
				beg0 = (int)lastnl + 1;
				open_abs = g0 - D0 + lastnl + 1;
				__syncwarp();
			}
			if (vnl && lane == 0) {
				/* the unterminated tail [open, end of input) */
				fmiss_put(a, stab, atomicAdd(a.miss_n, 1u), open_abs,
				    a.nbytes);
			}
			/* the open record, seen from the next chunk's buffer */
			beg0 -= (int)CHUNK;
			if (beg0 < 0)
				beg0 = -1;
		}
		/* the next segment nobody has taken yet */
		if (lane == 0)
			seg = nwarps + atomicAdd(a.seg_next, 1u);
		seg = __shfl_sync(0xffffffffu, seg, 0);
	}

#ifdef DNG_JIT_HOT
	__syncthreads();
	if (a.ndense)
		dng_cold_dense_flush(dense_sa, a.dict, &a.tab);
	dng_cold_flush(stab, a.s1slots, a.sslots, &a.tab);
#else
	flush_tally(stab, a.s1slots, a.sslots, a.tab);
#endif
	if (lane == 0) {
		if (ntmpl) {
			atomicAdd(&a.counters[CTR_LINES], (unsigned long long)ntmpl);
			atomicAdd(&a.counters[CTR_TMPL], (unsigned long long)ntmpl);
		}
		if (naggr)
			atomicAdd(&a.counters[CTR_AGGR], (unsigned long long)naggr);
	}
	if (tid == 15 && s_drop[15])
		atomicAdd(&a.counters[CTR_OVER], (unsigned long long)s_drop[15]);
	if (tid < 15 && s_drop[tid]) {
		/* FO_* -> CTR_*; s_drop[1] = records that took a slow conversion */
		const int ctr = tid == 1 ? (int)CTR_SLOW :
		    tid == FO_DS_FILTERED ? (int)CTR_DS_FILTERED :
		    tid == FO_DS_FAILED ? (int)CTR_DS_FAILED :
		    tid == FO_USER_FILTERED ? (int)CTR_USER_FILTERED :
		    tid == FO_USER_FAILED ? (int)CTR_USER_FAILED :
		    tid == FO_SYNTH_UNDEF ? (int)CTR_SYNTH_UNDEF :
		    tid == FO_SYNTH_BADDATE ? (int)CTR_SYNTH_BADDATE :
		    tid == FO_TIME_FILTERED ? (int)CTR_TIME_FILTERED :
		    tid == FO_TIME_FAILED ? (int)CTR_TIME_FAILED : -1;
		if (ctr >= 0)
			atomicAdd(&a.counters[ctr], (unsigned long long)s_drop[tid]);
	}
}

#ifndef DNG_JIT_HOT
template <int NSL>
__global__ void __launch_bounds__(DNG_F_NT, 1)
scan_kernel_f(const FScanArgs a)
{
	fscan_body<NSL, false>(a);
}
#endif

#ifndef DNG_JIT_HOT
/* ---- the records the F path did not take ------------------------------------ */

struct FMissArgs {
	const u8 *data;
	unsigned long long start;
	const DevPlan *plan;
	u32 plan_bytes;
	unsigned long long *counters;
	GTable tab;
	u32 s1slots, sslots;
	const MissEnt *miss;
	const u32 *miss_n;
	u32 miss_cap;
};

#define DNG_MISS_NT 256

__global__ void __launch_bounds__(DNG_MISS_NT)
scan_miss_kernel(const FMissArgs a)
{
	const u32 n = min(*a.miss_n, a.miss_cap);
	if (blockIdx.x * DNG_MISS_NT >= n)
		return;
	extern __shared__ __align__(128) u8 smem[];
	DevPlan *sp = (DevPlan *)smem;
	STab stab;
	stab.s1 = (SSlot1 *)(smem + a.plan_bytes);
	stab.s = (SSlot *)(smem + a.plan_bytes + a.s1slots * sizeof (SSlot1));
	stab.mask1 = a.s1slots - 1;
	stab.mask = a.sslots - 1;
	const u32 tid = threadIdx.x;
	{
		const uint4 *src = (const uint4 *)a.plan;
		uint4 *dst = (uint4 *)sp;
		for (u32 i = tid; i < a.plan_bytes / 16; i += DNG_MISS_NT)
			dst[i] = src[i];
		const uint4 z = make_uint4(0, 0, 0, 0);
		uint4 *tz = (uint4 *)stab.s1;
		const u32 tab_bytes = a.s1slots * (u32)sizeof (SSlot1) +
		    a.sslots * (u32)sizeof (SSlot);
		for (u32 i = tid; i < tab_bytes / 16; i += DNG_MISS_NT)
			tz[i] = z;
	}
	__syncthreads();
	const DevPlan &P = *sp;
	LocalCounters C;
	C.lines = C.invalid_json = C.invalid_point = 0;
	C.ds_filtered = C.ds_failedeval = C.user_filtered = 0;
	C.user_failedeval = C.synth_undef = C.synth_baddate = 0;
	C.time_filtered = C.time_failedeval = C.aggr = C.slow = 0;
	C.unsupported = 0;
	u32 nlong = 0;
	u32 mctr[(MAX_METRICS - 1) * MCTR_PER];
	for (int k = 0; k < (MAX_METRICS - 1) * MCTR_PER; k++)
		mctr[k] = 0;
	for (u32 i = blockIdx.x * DNG_MISS_NT + tid; i < n;
	    i += gridDim.x * DNG_MISS_NT) {
		const MissEnt e = a.miss[i];
		unsigned long long q = e.beg;
		if (q == ~0ull) {
			q = e.end;
			while (q > a.start && a.data[q - 1] != '\n')
				q--;
			nlong++;
		}
		scan_one_global(a.data + q, (u32)min((unsigned long long)
		    DNG_MAXREC, e.end - q), P, stab, a.tab, C, mctr);
	}
	flush_tally(stab, a.s1slots, a.sslots, a.tab);
	flush_counters(a.counters, C, nlong, 0);
}

#endif /* DNG_JIT_HOT */

} /* namespace dng */
#endif
