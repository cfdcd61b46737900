/*
 * api.cu: the C ABI of libdragnet_gpu.so (include/dragnet_gpu.h).
 *
 * Host-side plumbing only: device buffers, the H2D ring that keeps PCIe busy
 * while the previous chunk is being scanned, line carry between chunks
 * (lstream semantics, lib/format-json.js:32-33), kernel launches, result
 * download.  There is deliberately no host execution path for records: if no
 * CUDA device is usable, dng_scan_open() fails.
 */
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <map>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/dragnet_gpu.h"
#include "plan.h"
#include "result.h"
#include "scan_kernel.cuh"
#include "fast_kernel.cuh"
#include "jit.h"
#include "gen.cuh"

using namespace dng;

namespace {

const size_t RING_SLOTS = 3;
const size_t CARRY_ROOM = (size_t)DNG_MAXREC + 4096;	/* room before a chunk */

size_t env_size(const char *name, size_t dflt)
{
	const char *v = getenv(name);
	if (!v || !*v)
		return dflt;
	return (size_t)strtoull(v, nullptr, 0);
}

/*
 * Scan buffers (table, key arena, carry, H2D ring, pinned staging) have the
 * same few sizes for every scan, and cudaMalloc / cudaMallocHost / cudaFree
 * cost milliseconds each: destroyed scans park their buffers here and the
 * next scan on that device takes them back.  Bounded (DNG_CACHE_BYTES, default
 * 2 GiB per kind); dng_release_cached() empties it.
 */
struct BufCache {
	std::mutex mu;
	std::multimap<std::pair<int, size_t>, void *> idle;	/* (device|-1 host, bytes) */
	std::map<void *, std::pair<int, size_t>> live;
	size_t idle_dev = 0, idle_host = 0;
};

BufCache &buf_cache()
{
	static BufCache *c = new BufCache();	/* outlives static destructors */
	return *c;
}

cudaError_t cached_alloc(int device, void **p, size_t n)
{
	BufCache &c = buf_cache();
	{
		std::lock_guard<std::mutex> g(c.mu);
		auto it = c.idle.find(std::make_pair(device, n));
		if (it != c.idle.end()) {
			*p = it->second;
			c.idle.erase(it);
			(device < 0 ? c.idle_host : c.idle_dev) -= n;
			c.live[*p] = std::make_pair(device, n);
			return cudaSuccess;
		}
	}
	cudaError_t e = device < 0 ? cudaMallocHost(p, n) : cudaMalloc(p, n);
	if (e == cudaSuccess) {
		std::lock_guard<std::mutex> g(c.mu);
		c.live[*p] = std::make_pair(device, n);
	}
	return e;
}

void cached_free(void *p)
{
	if (!p)
		return;
	static const size_t limit = env_size("DNG_CACHE_BYTES", (size_t)2 << 30);
	BufCache &c = buf_cache();
	int device = 0;
	{
		std::lock_guard<std::mutex> g(c.mu);
		auto it = c.live.find(p);
		if (it == c.live.end())
			return;
		device = it->second.first;
		size_t n = it->second.second;
		c.live.erase(it);
		size_t &idle = device < 0 ? c.idle_host : c.idle_dev;
		if (idle + n <= limit) {
			idle += n;
			c.idle.insert(std::make_pair(std::make_pair(device, n), p));
			return;
		}
	}
	if (device < 0)
		cudaFreeHost(p);
	else
		cudaFree(p);
}

#define DEV_ALLOC(s, p, n) cached_alloc((s)->device, (void **)(p), (n))
#define HOST_ALLOC(p, n) cached_alloc(-1, (void **)(p), (n))

void set_err(char *err, size_t errlen, const char *fmt, const char *a = "")
{
	if (err && errlen)
		snprintf(err, errlen, fmt, a);
}

} /* namespace */

/* the same buffer cache for the library's other translation units (merge.cu) */
cudaError_t dng_cached_alloc(int device, void **p, size_t n)
{
	return cached_alloc(device, p, n);
}

void dng_cached_free(void *p)
{
	cached_free(p);
}


struct dng_scan {
	dng_plan plan;
	int device = 0;
	int sm_count = 0;
	u32 plan_bytes = 0, sslots = 0, s1slots = 0;
	cudaStream_t stream = nullptr, copy_stream = nullptr;
	cudaStream_t own_stream = nullptr;
	DevPlan *d_plan = nullptr;
	GTable tab{};
	unsigned long long *d_counters = nullptr;
	unsigned long long *d_nl = nullptr;	/* find_nl scratch (2) */
	size_t table_cap = 0;
	/* H2D ring */
	size_t ring_cap = 0;
	u8 *d_ring[RING_SLOTS] = {};
	u8 *h_stage[RING_SLOTS] = {};
	cudaEvent_t ev_ready[RING_SLOTS] = {}, ev_free[RING_SLOTS] = {};
	bool slot_used[RING_SLOTS] = {};
	size_t next_slot = 0;
	/* carry: the unterminated tail of everything fed so far */
	u8 *d_carry = nullptr;
	size_t carry_len = 0;
	u8 *d_side = nullptr;		/* carry + head of a device chunk */
	/* pinned block ring of dng_scan_feed_file's reader threads */
	u8 *file_buf = nullptr;
	cudaEvent_t file_done[32] = {};
	/* stats */
	std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pairs;
	std::vector<cudaEvent_t> ev_pool;
	double kernel_ms = 0;
	uint64_t launches = 0, kernel_bytes = 0, bytes_fed = 0;
	uint64_t aux_launches = 0;	/* resolve / find_nl / compact kernels */
	cudaEvent_t ev_init = nullptr;	/* setup enqueued by dng_scan_open */
	bool finished = false;
	/* record templates (tmpl.h), learned from the head of the input */
	bool tmpl_enabled = true, tmpl_tried = false;
	/* kernel geometry: per-warp chunks for short lines, CTA tiles otherwise */
	bool warp_kernel = false;
	u32 wslice = DNG_W_SLICE_MAX;	/* bytes per lane of a warp's chunk */
	int kernel_pref = 0;		/* DNG_KERNEL: 0 auto, 1 tile, 2 warp, 3 fast */
	u32 w_sslots = 0, w_s1slots = 0;
	/* counters of finished launches, copied to pinned memory after every
	 * launch: lets the host notice that the input changed character */
	unsigned long long *h_live = nullptr;
	unsigned long long learn_lines = 0, learn_tmpl = 0;
	unsigned long long seen_lines = 0, seen_long = 0;
	int relearns = 0;
	u8 *d_tmpl = nullptr;
	u32 tmpl_bytes = 0, ntemplates = 0;
	/* the F path (fast.h): its plan, its templates, its miss list */
	FPlan fplan;
	FPlan *d_fplan = nullptr;
	u8 *d_ftmpl = nullptr;
	u32 ftmpl_bytes = 0, nftemplates = 0, ftmpl_leaf_off = 0, ftmpl_pool_off = 0;
	/* dense keys: the value dictionary the compiled matcher was generated
	 * with (ncols = 0: none), on the device for the end-of-launch flush */
	FDict fdict{};
	FDict *d_fdict = nullptr;
	bool f_kernel = false;
	u32 f_nt = DNG_F_NT;		/* threads of its CTA: DNG_F_NT, or 768 when
					 * the tally cache needs the shared memory */
	unsigned long long seen_over = 0, seen_aggr = 0;
	bool f_probed = false;
	u32 f_nsl = 13;			/* 16-byte units per lane slice */
	double mean_line = 224;		/* of the sample the templates came from */
	u32 f_smem_max = 0;		/* dynamic shared memory a CTA may ask for */
	/* run-time compiled matcher (jit.h): 0 off, 1 in the background, 2 wait */
	int jit_mode = 1;
	std::shared_ptr<JitKernels> jit;
	uint64_t jit_launches = 0;
	MissEnt *d_miss = nullptr;
	u32 *d_miss_n = nullptr;
	u32 miss_cap = 0;
	unsigned long long seen_tmpl = 0;
	std::string err;
	int err_code = 0;

	int fail(int code, const std::string &m) {
		if (!err_code) {
			err_code = code;
			err = m;
		}
		return code;
	}
	int cuda(cudaError_t e, const char *what) {
		if (e == cudaSuccess)
			return 0;
		return fail(DNG_ECUDA, std::string(what) + ": " +
		    cudaGetErrorString(e));
	}
};

#define CK(s, call) do { if ((s)->cuda((call), #call)) return (s)->err_code; } while (0)

namespace {

cudaEvent_t get_event(dng_scan *s)
{
	if (!s->ev_pool.empty()) {
		cudaEvent_t e = s->ev_pool.back();
		s->ev_pool.pop_back();
		return e;
	}
	cudaEvent_t e;
	cudaEventCreate(&e);
	return e;
}

/* shared memory set aside for the template trie when sizing the tally cache */
static constexpr size_t TMPL_RESERVE = 4096;

/* the record parser's view of one sample line per template candidate */
__global__ void resolve_pairs_kernel(const DevPlan *plan, const u8 *lines,
    const u32 *se, u32 n, TResolved *out)
{
	u32 i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n)
		return;
	RecState R;
	parse_record(lines + se[2 * i], se[2 * i + 1] - se[2 * i], *plan, R);
	out[i].flags = R.flags;
	out[i].set_mask = R.set_mask;
	for (int k = 0; k < MAX_SLOTS; k++)
		out[i].slots[k] = ((R.set_mask >> k) & 1) ? R.slots[k] : 0;
}

/*
 * The F path's templates (fast.h): the same candidates, their captures indexed
 * by path, compact literals.  The F kernel is chosen when they cover the
 * sample (results never depend on that choice, only the speed does).
 */
/*
 * What a scan of this plan found out about its tally cache (f_nt), kept for
 * the scans of the same plan that follow in this process: they start with it
 * and need no probe launch.
 */
static std::mutex g_fnt_mu;
static std::map<unsigned long long, u32> g_fnt_memo;

static unsigned long long fplan_hash(const FPlan &F)
{
	unsigned long long h = 1469598103934665603ull;
	const u8 *p = (const u8 *)&F;
	for (size_t i = 0; i < sizeof (F); i++)
		h = (h ^ p[i]) * 1099511628211ull;
	return h;
}

static void fnt_remember(const dng_scan *s)
{
	std::lock_guard<std::mutex> g(g_fnt_mu);
	g_fnt_memo[fplan_hash(s->fplan)] = s->f_nt;
}

int learn_ftemplates(dng_scan *s, const std::vector<TCandidate> &cands,
    const std::vector<TResolved> &res, size_t sampled_lines, const u8 *head,
    size_t nhead)
{
	std::vector<TResolved> fres(res.size());
	for (size_t i = 0; i < res.size(); i++)
		fplan_resolve(s->plan.dev, res[i], fres[i]);
	std::vector<u8> blob, accepted;
	u32 nt = 0;
	tmpl_build(cands, fres, TMPL_RESERVE, blob, &nt, true, &accepted);
	cached_free(s->d_ftmpl);
	s->d_ftmpl = nullptr;
	s->ftmpl_bytes = 0;
	s->nftemplates = 0;
	if (!blob.empty()) {
		const THdr *th = (const THdr *)blob.data();
		s->ftmpl_leaf_off = th->leaf_off;
		s->ftmpl_pool_off = th->pool_off;
	}
	size_t covered = 0;
	for (size_t i = 0; i < cands.size(); i++)
		if (accepted[i])
			covered += cands[i].count;
	/* the breakdown's values, for the compiled matcher's dense keys */
	memset(&s->fdict, 0, sizeof (s->fdict));
	if (s->jit_mode && !blob.empty() && jit_dense())
		fdict_learn(s->fplan, blob.data(), head, nhead, s->fdict);
	if (!blob.empty()) {
		size_t padded = (blob.size() + 127) & ~(size_t)127;
		blob.resize(padded, 0);
		CK(s, DEV_ALLOC(s, &s->d_ftmpl, padded));
		CK(s, cudaMemcpyAsync(s->d_ftmpl, blob.data(), padded,
		    cudaMemcpyHostToDevice, s->stream));
		if (s->fdict.ncols) {
			if (!s->d_fdict)
				CK(s, DEV_ALLOC(s, &s->d_fdict, sizeof (FDict)));
			CK(s, cudaMemcpyAsync(s->d_fdict, &s->fdict,
			    sizeof (FDict), cudaMemcpyHostToDevice, s->stream));
		}
		CK(s, cudaStreamSynchronize(s->stream));
		s->ftmpl_bytes = (u32)padded;
		s->nftemplates = nt;
	}
	s->jit.reset();
	if (s->jit_mode && !blob.empty())
		s->jit = jit_request(jit_source(blob.data(), blob.size(), &s->fplan,
		    nullptr, &s->fdict), (int)s->f_nsl, s->device,
		    (int)s->f_smem_max, s->jit_mode == 2);
	if (s->kernel_pref == 0)
		s->f_kernel = s->warp_kernel && !blob.empty() &&
		    covered * 10 >= sampled_lines * 9 &&
		    s->mean_line * DNG_F_NLCAP >= 32.0 * 16 * s->f_nsl * 1.5;
	return 0;
}

/*
 * Learn record templates from the head of the first data this scan sees
 * (device memory): skeletons on the host (lexical only), what their
 * wildcards mean to the plan from the device's own parser.  Failure to learn
 * anything is not an error: the kernel then parses every record itself.
 */
int learn_templates(dng_scan *s, const u8 *data, unsigned long long start,
    unsigned long long nbytes)
{
	s->tmpl_tried = true;
	if (!s->tmpl_enabled && s->kernel_pref != 0)
		return 0;
	size_t n = (size_t)std::min<unsigned long long>(nbytes - start,
	    TMPL_SAMPLE_BYTES);
	/* pinned (and cached) so that the copy is a plain DMA */
	u8 *hbuf = nullptr;
	CK(s, HOST_ALLOC(&hbuf, TMPL_SAMPLE_BYTES));
	struct Release {
		u8 *p;
		~Release() { cached_free(p); }
	} release{hbuf};
	CK(s, cudaMemcpyAsync(hbuf, data + start, n, cudaMemcpyDeviceToHost,
	    s->stream));
	CK(s, cudaStreamSynchronize(s->stream));
	struct { u8 *p; u8 *data() const { return p; }
	    u8 operator[](size_t i) const { return p[i]; } } head{hbuf};
	if (s->kernel_pref == 0) {
		/* short lines: every warp stages its own chunk (scan_kernel_w);
		 * otherwise CTA-wide tiles, whose window holds long lines */
		size_t longest = 0, run = 0;
		for (size_t i = 0; i < n; i++) {
			if (head[i] == '\n') {
				longest = std::max(longest, run);
				run = 0;
			} else {
				run++;
			}
		}
		longest = std::max(longest, run);
		s->warp_kernel = longest <= DNG_W_MAXLINE;
	}
	{
		/* chunk size: the lane slice (16 x odd bytes) whose chunk holds
		 * the most records per 32-lane pass, given the mean line */
		size_t nl = 0;
		for (size_t i = 0; i < n; i++)
			nl += head[i] == '\n';
		double mean = nl ? (double)n / (double)nl : 224.0;
		s->mean_line = mean;
		double best = -1;
		for (u32 sl = 112; sl <= DNG_W_SLICE_MAX; sl += 32) {
			double recs = 32.0 * sl / mean;
			double passes = ceil((recs + 1.5) / 32.0);
			double util = recs / (32.0 * passes);
			if (util >= best) {
				best = util;
				s->wslice = sl;
			}
		}
		/* the F kernel indexes at most DNG_F_NLCAP lines per chunk:
		 * the largest such slice with the best lane use */
		best = -1;
		s->f_nsl = 7;
		for (u32 sl = 112; sl <= DNG_W_SLICE_MAX; sl += 32) {
			double recs = 32.0 * sl / mean;
			double passes = ceil((recs + 1.5) / 32.0);
			double util = recs / (32.0 * passes);
			if (recs * 1.25 <= DNG_F_NLCAP && util >= best) {
				best = util;
				s->f_nsl = sl / 16;
			}
		}
	}
	if (!s->tmpl_enabled)
		return 0;
	std::vector<TCandidate> cands;
	size_t sampled_lines = 0;
	tmpl_candidates(head.data(), n, TMPL_MAX_LEAVES, cands, &sampled_lines);
	if (cands.empty())
		return 0;
	std::vector<u8> lines;
	std::vector<u32> offs(1, 0);
	for (const TCandidate &c : cands) {
		lines.insert(lines.end(), c.sample.begin(), c.sample.end());
		lines.push_back('\n');
		offs.push_back((u32)lines.size());
	}
	u8 *d_lines = nullptr;
	u32 *d_offs = nullptr;
	TResolved *d_res = nullptr;
	std::vector<TResolved> res(cands.size());
	/* constant sizes, so that the buffer cache can hand them back */
	cudaError_t e = DEV_ALLOC(s, &d_lines,
	    (size_t)TMPL_MAX_LEAVES * (TMPL_MAX_LINE + 1) + 16);
	if (e == cudaSuccess)
		e = DEV_ALLOC(s, &d_offs, 2 * (TMPL_MAX_LEAVES + 1) * sizeof (u32));
	if (e == cudaSuccess)
		e = DEV_ALLOC(s, &d_res, TMPL_MAX_LEAVES * sizeof (TResolved));
	if (e == cudaSuccess)
		e = cudaMemcpyAsync(d_lines, lines.data(), lines.size(),
		    cudaMemcpyHostToDevice, s->stream);
	/* line i = [offs[i], offs[i + 1] - 1): keep starts and ends apart */
	std::vector<u32> se;
	for (size_t i = 0; i < cands.size(); i++) {
		se.push_back(offs[i]);
		se.push_back(offs[i + 1] - 1);
	}
	if (e == cudaSuccess)
		e = cudaMemcpyAsync(d_offs, se.data(), se.size() * sizeof (u32),
		    cudaMemcpyHostToDevice, s->stream);
	if (e == cudaSuccess) {
		s->aux_launches++;
		resolve_pairs_kernel<<<1, 32, 0, s->stream>>>(s->d_plan, d_lines,
		    d_offs, (u32)cands.size(), d_res);
		e = cudaGetLastError();
	}
	if (e == cudaSuccess)
		e = cudaMemcpyAsync(res.data(), d_res,
		    res.size() * sizeof (TResolved), cudaMemcpyDeviceToHost,
		    s->stream);
	if (e == cudaSuccess)
		e = cudaStreamSynchronize(s->stream);
	cached_free(d_lines);
	cached_free(d_offs);
	cached_free(d_res);
	if (e != cudaSuccess)
		return s->cuda(e, "template resolve");
	if (s->fplan.ok && learn_ftemplates(s, cands, res, sampled_lines,
	    head.data(), n))
		return s->err_code;
	std::vector<u8> blob;
	u32 nt = 0;
	tmpl_build(cands, res, TMPL_RESERVE, blob, &nt);
	if (blob.empty())
		return 0;
	size_t padded = (blob.size() + 127) & ~(size_t)127;
	blob.resize(padded, 0);
	/* (the stream is idle here: a blob being replaced is not in use) */
	cached_free(s->d_tmpl);
	s->d_tmpl = nullptr;
	s->tmpl_bytes = 0;
	CK(s, DEV_ALLOC(s, &s->d_tmpl, padded));
	CK(s, cudaMemcpyAsync(s->d_tmpl, blob.data(), padded,
	    cudaMemcpyHostToDevice, s->stream));
	CK(s, cudaStreamSynchronize(s->stream));
	s->tmpl_bytes = (u32)padded;
	s->ntemplates = nt;
	return 0;
}

template <int NSL>
void launch_fkernel(dng_scan *s, const FScanArgs &a, u32 grid)
{
	scan_kernel_f<NSL><<<grid, s->f_nt, fkernel_smem<NSL>(a.tmpl_bytes,
	    a.s1slots, a.sslots, a.nrows, s->f_nt / 32, a.ndense),
	    s->stream>>>(a);
}

/* tally-cache sizes of the F kernel: what its buffers (and dense counters)
 * leave */
template <int NSL>
void fkernel_slots(const dng_scan *s, u32 nrows, u32 tmpl_room, u32 ndense,
    u32 *s1, u32 *s2)
{
	const size_t fixed = fkernel_smem<NSL>(tmpl_room, 0, 0, nrows,
	    s->f_nt / 32, ndense);
	const size_t room = s->f_smem_max > fixed ? s->f_smem_max - fixed : 0;
	u32 n1 = 32;
	while (n1 < 1024 && (size_t)n1 * 2 * sizeof (SSlot1) +
	    DNG_SSLOTS_MIN * sizeof (SSlot) <= room * 3 / 4)
		n1 *= 2;
	const size_t left = room - std::min(room, (size_t)n1 * sizeof (SSlot1));
	u32 n2 = DNG_SSLOTS_MIN;
	while (n2 * 2 <= DNG_SSLOTS_MAX && (size_t)n2 * 2 * sizeof (SSlot) <= left)
		n2 *= 2;
	*s1 = n1;
	*s2 = n2;
}

/*
 * The F path over data[start, nbytes): scan_kernel_f, then scan_miss_kernel
 * for what it did not take (it exits at once when the list is empty).
 */
int launch_fscan(dng_scan *s, const u8 *data, unsigned long long start,
    unsigned long long nbytes, bool final)
{
	if (!s->d_miss) {
		s->miss_cap = (u32)env_size("DNG_MISS_CAP", (size_t)4 << 20);
		CK(s, DEV_ALLOC(s, &s->d_miss, (size_t)s->miss_cap *
		    sizeof (MissEnt)));
		CK(s, DEV_ALLOC(s, &s->d_miss_n, 64));
		CK(s, cudaMemsetAsync(s->d_miss_n, 0, 64, s->stream));
	}
	/* the kernel wants the first valid byte inside the first 16 */
	const unsigned long long skip = start & ~15ull;
	data += skip;
	start -= skip;
	nbytes -= skip;
	FScanArgs a;
	a.data = data;
	a.start = start;
	a.nbytes = nbytes;
	a.fplan = s->d_fplan;
	a.plan = s->d_plan;
	a.tmpl = s->d_ftmpl;
	a.tmpl_bytes = s->ftmpl_bytes;
	a.leaf_off = s->ftmpl_leaf_off;
	a.pool_off = s->ftmpl_pool_off;
	a.counters = s->d_counters;
	a.tab = s->tab;
	a.final = final ? 1 : 0;
	a.nrows = s->fplan.nrows;
	a.miss = s->d_miss;
	a.miss_cap = s->miss_cap;
	a.miss_n = s->d_miss_n;
	const u32 nsl = s->f_nsl;
	const unsigned long long chunk = 32ull * 16 * nsl;
	a.nchunks = (u32)((nbytes + chunk - 1) / chunk);
	const u32 nw = s->f_nt / 32;
	const u32 grid = std::min<u32>((a.nchunks + nw - 1) / nw,
	    (u32)s->sm_count);
	/* segments: long enough to amortise the pre-lap, short enough to keep
	 * every warp of the grid busy */
	const u32 nwarps = grid * nw;
	a.seg = std::max<u32>(1, std::min<u32>(DNG_F_SEG,
	    a.nchunks / (nwarps * 8)));
	/* the segment queue: [1] of the miss counter's allocation */
	a.seg_next = s->d_miss_n + 1;
	cudaMemsetAsync(s->d_miss_n, 0, 2 * sizeof (u32), s->stream);
	cudaEvent_t e0 = get_event(s), e1 = get_event(s);
	cudaEventRecord(e0, s->stream);
	/* the matcher compiled for these templates, once it is there */
	const bool jit = s->jit && s->jit->state.load() == 1 && s->ftmpl_bytes;
	/* (the compiled matcher has the templates in its code: no trie in shared
	 * memory, more of it for the tally cache) */
	const u32 tmpl_room = jit ? 0 : (u32)TMPL_RESERVE;
	if (jit)
		a.tmpl_bytes = 0;
	/* (dense counters: only the compiled matcher has the dictionary) */
	a.ndense = jit && s->fdict.ncols ? (s->fdict.total + 3) & ~3u : 0;
	a.dict = a.ndense ? s->d_fdict : nullptr;
	size_t smem = 0;
	switch (nsl) {
	case 7:
		fkernel_slots<7>(s, a.nrows, tmpl_room, a.ndense, &a.s1slots,
		    &a.sslots);
		smem = fkernel_smem<7>(a.tmpl_bytes, a.s1slots, a.sslots, a.nrows,
		    s->f_nt / 32, a.ndense);
		if (!jit)
			launch_fkernel<7>(s, a, grid);
		break;
	case 9:
		fkernel_slots<9>(s, a.nrows, tmpl_room, a.ndense, &a.s1slots,
		    &a.sslots);
		smem = fkernel_smem<9>(a.tmpl_bytes, a.s1slots, a.sslots, a.nrows,
		    s->f_nt / 32, a.ndense);
		if (!jit)
			launch_fkernel<9>(s, a, grid);
		break;
	case 11:
		fkernel_slots<11>(s, a.nrows, tmpl_room, a.ndense, &a.s1slots,
		    &a.sslots);
		smem = fkernel_smem<11>(a.tmpl_bytes, a.s1slots, a.sslots, a.nrows,
		    s->f_nt / 32, a.ndense);
		if (!jit)
			launch_fkernel<11>(s, a, grid);
		break;
	default:
		fkernel_slots<13>(s, a.nrows, tmpl_room, a.ndense, &a.s1slots,
		    &a.sslots);
		smem = fkernel_smem<13>(a.tmpl_bytes, a.s1slots, a.sslots, a.nrows,
		    s->f_nt / 32, a.ndense);
		if (!jit)
			launch_fkernel<13>(s, a, grid);
		break;
	}
	cudaError_t le = cudaSuccess;
	if (jit) {
		void *args[] = { &a };
		le = cudaLaunchKernel((const void *)s->jit->kern, dim3(grid),
		    dim3(s->f_nt), args, smem, s->stream);
		s->jit_launches++;
	}
	if (le == cudaSuccess)
		le = cudaGetLastError();
	FMissArgs ma;
	ma.data = data;
	ma.start = start;
	ma.plan = s->d_plan;
	ma.plan_bytes = s->plan_bytes;
	ma.counters = s->d_counters;
	ma.tab = s->tab;
	ma.s1slots = 64;
	ma.sslots = 1024;
	ma.miss = s->d_miss;
	ma.miss_n = s->d_miss_n;
	ma.miss_cap = s->miss_cap;
	if (le == cudaSuccess) {
		scan_miss_kernel<<<s->sm_count * 2, DNG_MISS_NT, s->plan_bytes +
		    ma.s1slots * sizeof (SSlot1) + ma.sslots * sizeof (SSlot),
		    s->stream>>>(ma);
		le = cudaGetLastError();
	}
	cudaEventRecord(e1, s->stream);
	if (!s->h_live && HOST_ALLOC(&s->h_live, NCTR * sizeof (unsigned long long))
	    == cudaSuccess)
		memset(s->h_live, 0, NCTR * sizeof (unsigned long long));
	if (s->h_live)
		cudaMemcpyAsync(s->h_live, s->d_counters,
		    NCTR * sizeof (unsigned long long), cudaMemcpyDeviceToHost,
		    s->stream);
	s->ev_pairs.emplace_back(e0, e1);
	s->launches++;
	s->aux_launches++;
	s->kernel_bytes += nbytes - start;
	return s->cuda(le, "scan_kernel_f launch");
}

/* launch the scan kernel over data[start, nbytes) */
int launch_scan(dng_scan *s, const u8 *data, unsigned long long start,
    unsigned long long nbytes, bool final)
{
	if (nbytes <= start)
		return 0;
	if (!s->tmpl_tried) {
		if (learn_templates(s, data, start, nbytes))
			return s->err_code;
	} else if (s->h_live) {
		/*
		 * Input that changes character mid-stream (another file,
		 * another producer): many lines longer than a warp's pre-lap
		 * -> the tile kernel from here on; most records missing the
		 * templates -> learn again from this data (a few times at most;
		 * each costs a stream synchronisation).
		 */
		const volatile unsigned long long *lv = s->h_live;
		const unsigned long long lines = lv[CTR_LINES];
		const unsigned long long nlong = lv[CTR_LONG];
		if (lines - s->seen_lines >= 64) {
			/* over the launches that finished since the last look */
			if (s->warp_kernel && s->kernel_pref == 0 &&
			    (nlong - s->seen_long) * 16 > lines - s->seen_lines)
				s->warp_kernel = false;
			s->seen_lines = lines;
			s->seen_long = nlong;
		}
		/* keys the F kernel's inline tally tier had no room for: with 28
		 * warps it is small; 24 leave it 30 KB more */
		if (s->f_nt > 768 && lv[CTR_AGGR] - s->seen_aggr >= 4096) {
			if ((lv[CTR_OVER] - s->seen_over) * 64 >
			    lv[CTR_AGGR] - s->seen_aggr)
				s->f_nt = 768;
			s->seen_over = lv[CTR_OVER];
			s->seen_aggr = lv[CTR_AGGR];
			fnt_remember(s);
		}
		const unsigned long long dl = lines - s->learn_lines;
		/* the F path only pays while it takes nearly every record: with
		 * more than a few percent going through the miss list, learn
		 * again; if that was already done, leave it to the general
		 * kernels (whose second tier runs from shared memory) */
		if (s->f_kernel && s->kernel_pref == 0 && dl > 200000 &&
		    (dl - (lv[CTR_TMPL] - s->learn_tmpl)) * 16 > dl &&
		    s->relearns >= 1)
			s->f_kernel = false;
		const bool fweak = s->f_kernel && s->kernel_pref == 0 &&
		    (dl - (lv[CTR_TMPL] - s->learn_tmpl)) * 16 > dl;
		if (s->tmpl_enabled && s->relearns < 3 && dl > 200000 &&
		    ((lv[CTR_TMPL] - s->learn_tmpl) * 2 < dl || fweak)) {
			s->relearns++;
			const bool wk = s->warp_kernel;
			if (learn_templates(s, data, start, nbytes))
				return s->err_code;
			if (!wk && s->kernel_pref == 0)
				s->warp_kernel = false;	/* long lines were seen */
			/* the stream is idle: the counters below are current */
			s->learn_lines = lv[CTR_LINES];
			s->learn_tmpl = lv[CTR_TMPL];
		}
	}
	/* (a plan with many capture rows leaves the F kernel's buffers no room) */
	if (s->f_kernel && s->fplan.ok &&
	    fkernel_smem<13>(TMPL_RESERVE, 32, DNG_SSLOTS_MIN, s->fplan.nrows) >
	    s->f_smem_max)
		s->f_kernel = false;
	if (s->f_kernel && s->fplan.ok)
		return launch_fscan(s, data, start, nbytes, final);
	ScanArgs a;
	a.data = data;
	a.start = start;
	a.nbytes = nbytes;
	a.plan = s->d_plan;
	a.counters = s->d_counters;
	a.tab = s->tab;
	a.final = final ? 1 : 0;
	a.plan_bytes = s->plan_bytes;
	a.tmpl = s->d_tmpl;
	a.tmpl_bytes = s->tmpl_bytes;
	a.wslice = DNG_W_SLICE_MAX;
	cudaEvent_t e0 = get_event(s), e1 = get_event(s);
	if (s->warp_kernel) {
		const unsigned long long chunk = 32ull * s->wslice;
		a.wslice = s->wslice;
		a.ntiles = (u32)((nbytes + chunk - 1) / chunk);
		a.sslots = s->w_sslots;
		a.s1slots = s->w_s1slots;
		u32 grid = std::min<u32>((a.ntiles + DNG_NW - 1) / DNG_NW,
		    (u32)s->sm_count);
		cudaEventRecord(e0, s->stream);
		scan_kernel_w<<<grid, DNG_NT, SMEM_W_FIXED + s->plan_bytes +
		    s->tmpl_bytes + a.sslots * sizeof (SSlot) +
		    a.s1slots * sizeof (SSlot1), s->stream>>>(a);
	} else {
		a.ntiles = (u32)((nbytes + DNG_TILE - 1) / DNG_TILE);
		a.sslots = s->sslots;
		a.s1slots = s->s1slots;
		u32 grid = std::min<u32>(a.ntiles,
		    (u32)s->sm_count * DNG_CTAS_PER_SM);
		cudaEventRecord(e0, s->stream);
		scan_kernel<<<grid, DNG_NT, SMEM_FIXED + s->plan_bytes +
		    s->tmpl_bytes + a.sslots * sizeof (SSlot) +
		    a.s1slots * sizeof (SSlot1), s->stream>>>(a);
	}
	cudaEventRecord(e1, s->stream);
	if (!s->h_live && HOST_ALLOC(&s->h_live, NCTR * sizeof (unsigned long long))
	    == cudaSuccess)
		memset(s->h_live, 0, NCTR * sizeof (unsigned long long));
	if (s->h_live)
		cudaMemcpyAsync(s->h_live, s->d_counters,
		    NCTR * sizeof (unsigned long long), cudaMemcpyDeviceToHost,
		    s->stream);
	s->ev_pairs.emplace_back(e0, e1);
	s->launches++;
	s->kernel_bytes += nbytes - start;
	return s->cuda(cudaGetLastError(), "scan_kernel launch");
}

void drain_events(dng_scan *s)
{
	for (auto &p : s->ev_pairs) {
		float ms = 0;
		if (cudaEventElapsedTime(&ms, p.first, p.second) == cudaSuccess)
			s->kernel_ms += ms;
		s->ev_pool.push_back(p.first);
		s->ev_pool.push_back(p.second);
	}
	s->ev_pairs.clear();
}

/*
 * One piece of host input (<= ring_cap bytes) whose bytes up to `upto`
 * (exclusive; ends just after a newline) are complete lines.  The previous
 * carry is prepended on the device; bytes [upto, len) become the new carry.
 */
int feed_piece(dng_scan *s, const u8 *buf, size_t len, size_t upto, bool pinned)
{
	size_t slot = s->next_slot;
	s->next_slot = (slot + 1) % RING_SLOTS;
	if (s->slot_used[slot])
		CK(s, cudaEventSynchronize(s->ev_free[slot]));
	const u8 *src = buf;
	if (!pinned) {
		memcpy(s->h_stage[slot], buf, len);
		src = s->h_stage[slot];
	}
	u8 *dst = s->d_ring[slot] + CARRY_ROOM;
	CK(s, cudaMemcpyAsync(dst, src, len, cudaMemcpyHostToDevice,
	    s->copy_stream));
	CK(s, cudaEventRecord(s->ev_ready[slot], s->copy_stream));
	CK(s, cudaStreamWaitEvent(s->stream, s->ev_ready[slot], 0));
	if (upto > 0) {
		u8 *begin = dst - s->carry_len;
		if (s->carry_len)
			CK(s, cudaMemcpyAsync(begin, s->d_carry, s->carry_len,
			    cudaMemcpyDeviceToDevice, s->stream));
		u8 *base = (u8 *)((uintptr_t)begin & ~(uintptr_t)15);
		if (launch_scan(s, base, (unsigned long long)(begin - base),
		    (unsigned long long)(dst + upto - base), false))
			return s->err_code;
		s->carry_len = 0;
	}
	if (len > upto) {
		size_t tail = len - upto;
		if (s->carry_len + tail > DNG_MAXREC)
			return s->fail(DNG_ELIMIT, "input line longer than 16 MiB");
		CK(s, cudaMemcpyAsync(s->d_carry + s->carry_len, dst + upto, tail,
		    cudaMemcpyDeviceToDevice, s->stream));
		s->carry_len += tail;
	}
	CK(s, cudaEventRecord(s->ev_free[slot], s->stream));
	s->slot_used[slot] = true;
	return 0;
}

int feed_host(dng_scan *s, const void *vbuf, size_t len, bool pinned)
{
	if (s->err_code)
		return s->err_code;
	if (s->finished)
		return s->fail(DNG_EINVAL, "scan already finished");
	const u8 *buf = (const u8 *)vbuf;
	s->bytes_fed += len;
	while (len > 0) {
		size_t n = std::min(len, s->ring_cap);
		/* complete lines end at the last '\n' of the piece */
		const void *nl = memrchr(buf, '\n', n);
		size_t upto = nl ? (size_t)((const u8 *)nl - buf) + 1 : 0;
		int rc = feed_piece(s, buf, n, upto, pinned);
		if (rc)
			return rc;
		buf += n;
		len -= n;
	}
	return 0;
}

} /* namespace */

extern "C" {

const char *dng_version(void)
{
	return "dragnet-b200 0.1 (sm_100a)";
}

int dng_plan_create(const char *plan_json, dng_plan **out, char *err,
    size_t errlen)
{
	if (!plan_json || !out) {
		set_err(err, errlen, "null argument");
		return DNG_EINVAL;
	}
	dng_plan *p = new dng_plan();
	int rc = dng_plan_compile(plan_json, p, err, errlen);
	if (rc) {
		delete p;
		return rc;
	}
	*out = p;
	return DNG_OK;
}

void dng_plan_destroy(dng_plan *plan)
{
	delete plan;
}

int dng_device_count(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess)
		return 0;
	return n;
}

int dng_scan_open(const dng_plan *plan, int device, dng_scan **out, char *err,
    size_t errlen)
{
	if (!plan || !out) {
		set_err(err, errlen, "null argument");
		return DNG_EINVAL;
	}
	int ndev = 0;
	cudaError_t e = cudaGetDeviceCount(&ndev);
	if (e != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
		set_err(err, errlen, "no usable CUDA device (%s); "
		    "libdragnet_gpu has no CPU fallback", e != cudaSuccess ?
		    cudaGetErrorString(e) : "device index out of range");
		return DNG_ENODEV;
	}
	dng_scan *s = new dng_scan();
	s->plan = *plan;
	s->device = device;
	int rc = 0;
	do {
		if ((rc = s->cuda(cudaSetDevice(device), "cudaSetDevice")))
			break;
		/* cudaGetDeviceProperties costs about a millisecond: once
		 * per device */
		static std::mutex prop_mu;
		static std::map<int, cudaDeviceProp> props;
		cudaDeviceProp prop;
		{
			std::lock_guard<std::mutex> g(prop_mu);
			auto it = props.find(device);
			if (it == props.end()) {
				if ((rc = s->cuda(cudaGetDeviceProperties(&prop,
				    device), "cudaGetDeviceProperties")))
					break;
				props[device] = prop;
			} else {
				prop = it->second;
			}
		}
		s->sm_count = prop.multiProcessorCount;
		if (const char *ev = getenv("DNG_TEMPLATES"))
			s->tmpl_enabled = atoi(ev) != 0;
		s->plan_bytes = devplan_smem_bytes(plan->dev);
		{
			/* the tally cache takes whatever shared memory is left
			 * when two CTAs share an SM (1 KB is reserved per CTA) */
			size_t per_cta = prop.sharedMemPerMultiprocessor /
			    DNG_CTAS_PER_SM - 1024 - 256;
			/* a single block may not exceed the opt-in limit, which
			 * also covers the kernel's static shared variables */
			per_cta = std::min(per_cta,
			    (size_t)prop.sharedMemPerBlockOptin - 1024 - 512);
			size_t used = SMEM_FIXED + s->plan_bytes + TMPL_RESERVE;
			size_t room = per_cta > used ? per_cta - used : 0;
			/* tier 1: 128 inline-key slots (64 when tight); tier 2:
			 * as many compact slots as still fit (power of two) */
			s->s1slots = room >= 24576 ? 256 : room >= 12288 ? 128 : 64;
			size_t t1 = (size_t)s->s1slots * sizeof (SSlot1);
			size_t left = room > t1 ? room - t1 : 0;
			u32 n = DNG_SSLOTS_MIN;
			while (n * 2 <= DNG_SSLOTS_MAX &&
			    (size_t)n * 2 * sizeof (SSlot) <= left)
				n *= 2;
			s->sslots = n;
			/* the per-warp kernel's fixed part differs: size its
			 * tally cache separately */
			size_t usedw = SMEM_W_FIXED + s->plan_bytes + TMPL_RESERVE;
			size_t roomw = per_cta > usedw ? per_cta - usedw : 0;
			s->w_s1slots = roomw >= 24576 ? 256 : roomw >= 12288 ? 128 : 64;
			size_t t1w = (size_t)s->w_s1slots * sizeof (SSlot1);
			size_t leftw = roomw > t1w ? roomw - t1w : 0;
			u32 nw = DNG_SSLOTS_MIN;
			while (nw * 2 <= DNG_SSLOTS_MAX &&
			    (size_t)nw * 2 * sizeof (SSlot) <= leftw)
				nw *= 2;
			s->w_sslots = nw;
		}
		/* a fan-out plan runs a long stage list per record and tallies
		 * many tuples: measured 1.2-2x faster on CTA tiles (whose
		 * warps move through the stages together and whose tally cache
		 * is larger) than on per-warp chunks */
		if (plan->dev.nmetrics > 1)
			s->kernel_pref = 1;
		if (const char *ev = getenv("DNG_KERNEL")) {
			/* tuning/testing: force one kernel geometry */
			s->kernel_pref = !strcmp(ev, "tile") ? 1 :
			    !strcmp(ev, "warp") ? 2 : !strcmp(ev, "fast") ? 3 : 0;
			s->warp_kernel = s->kernel_pref == 2;
		}
		/* the F path (fast.h), for the plans it models */
		fplan_build(plan->dev, s->fplan);
		/* three columns and more: keys are many more often than not,
		 * start with the larger tally cache (f_nt) */
		if (s->fplan.ncols >= 3)
			s->f_nt = 768;
		{
			std::lock_guard<std::mutex> g(g_fnt_mu);
			auto it = g_fnt_memo.find(fplan_hash(s->fplan));
			if (it != g_fnt_memo.end()) {
				s->f_nt = it->second;
				s->f_probed = true;
			}
		}
		if (const char *ev = getenv("DNG_F_WARPS")) {
			s->f_nt = atoi(ev) >= 28 ? DNG_F_NT : 768;
			s->f_probed = true;
		}
		if (getenv("DNG_FAST") && atoi(getenv("DNG_FAST")) == 0)
			s->fplan.ok = 0;
		if (const char *ev = getenv("DNG_JIT"))
			s->jit_mode = !strcmp(ev, "sync") || !strcmp(ev, "wait") ? 2 :
			    (!strcmp(ev, "0") || !strcmp(ev, "off")) ? 0 : 1;
		if (s->kernel_pref == 3) {
			/* forced: every eligible plan takes it, whatever the
			 * templates cover; others choose as usual */
			s->f_kernel = s->fplan.ok != 0;
			if (!s->f_kernel)
				s->kernel_pref = plan->dev.nmetrics > 1 ? 1 : 0;
		}
		s->f_smem_max = (u32)prop.sharedMemPerBlockOptin - 1024;
		{
			cudaError_t fe = cudaFuncSetAttribute(scan_kernel_f<7>,
			    cudaFuncAttributeMaxDynamicSharedMemorySize,
			    (int)s->f_smem_max);
			if (fe == cudaSuccess)
				fe = cudaFuncSetAttribute(scan_kernel_f<9>,
				    cudaFuncAttributeMaxDynamicSharedMemorySize,
				    (int)s->f_smem_max);
			if (fe == cudaSuccess)
				fe = cudaFuncSetAttribute(scan_kernel_f<11>,
				    cudaFuncAttributeMaxDynamicSharedMemorySize,
				    (int)s->f_smem_max);
			if (fe == cudaSuccess)
				fe = cudaFuncSetAttribute(scan_kernel_f<13>,
				    cudaFuncAttributeMaxDynamicSharedMemorySize,
				    (int)s->f_smem_max);
			if (fe == cudaSuccess)
				fe = cudaFuncSetAttribute(scan_miss_kernel,
				    cudaFuncAttributeMaxDynamicSharedMemorySize,
				    (int)s->f_smem_max);
			if ((rc = s->cuda(fe, "cudaFuncSetAttribute")))
				break;
		}
		if ((rc = s->cuda(cudaFuncSetAttribute(scan_kernel,
		    cudaFuncAttributeMaxDynamicSharedMemorySize,
		    (int)prop.sharedMemPerBlockOptin - 1024),
		    "cudaFuncSetAttribute")))
			break;
		if ((rc = s->cuda(cudaFuncSetAttribute(scan_kernel_w,
		    cudaFuncAttributeMaxDynamicSharedMemorySize,
		    (int)prop.sharedMemPerBlockOptin - 1024),
		    "cudaFuncSetAttribute")))
			break;
		if (SMEM_FIXED + s->plan_bytes + TMPL_RESERVE +
		    s->sslots * sizeof (SSlot) + s->s1slots * sizeof (SSlot1) >
		    prop.sharedMemPerBlockOptin - 1024) {
			rc = s->fail(DNG_ELIMIT, "plan does not fit in shared "
			    "memory (fixed " + std::to_string(SMEM_FIXED) +
			    " + plan " + std::to_string(s->plan_bytes) +
			    " + tier2 " + std::to_string(s->sslots) + " + tier1 " +
			    std::to_string(s->s1slots) + " slots > " +
			    std::to_string(prop.sharedMemPerBlockOptin) + ")");
			break;
		}
		if (SMEM_W_FIXED + s->plan_bytes + TMPL_RESERVE +
		    s->w_sslots * sizeof (SSlot) +
		    s->w_s1slots * sizeof (SSlot1) >
		    prop.sharedMemPerBlockOptin - 1024) {
			/* no room for the per-warp geometry with this plan */
			s->kernel_pref = 1;
			s->warp_kernel = false;
		}
		if ((rc = s->cuda(cudaStreamCreateWithFlags(&s->stream,
		    cudaStreamNonBlocking), "cudaStreamCreate")))
			break;
		s->own_stream = s->stream;
		if ((rc = s->cuda(cudaStreamCreateWithFlags(&s->copy_stream,
		    cudaStreamNonBlocking), "cudaStreamCreate")))
			break;
		if ((rc = s->cuda(DEV_ALLOC(s, &s->d_plan, sizeof (DevPlan) + 256),
		    "cudaMalloc plan")))
			break;
		if (s->fplan.ok) {
			if ((rc = s->cuda(DEV_ALLOC(s, &s->d_fplan, FPLAN_SMEM),
			    "cudaMalloc fplan")))
				break;
			if ((rc = s->cuda(cudaMemcpyAsync(s->d_fplan, &s->fplan,
			    sizeof (FPlan), cudaMemcpyHostToDevice, s->stream),
			    "fplan upload")))
				break;
		}
		/* s->plan is this scan's own copy: safe to upload from */
		if ((rc = s->cuda(cudaMemcpyAsync(s->d_plan, &s->plan.dev,
		    sizeof (DevPlan), cudaMemcpyHostToDevice, s->stream),
		    "plan upload")))
			break;
		size_t cap = env_size("DNG_TABLE_CAP", (size_t)1 << 20);
		size_t c2 = 1024;
		while (c2 < cap)
			c2 <<= 1;
		s->table_cap = c2;
		size_t arena = env_size("DNG_ARENA_BYTES", (size_t)64 << 20);
		if ((rc = s->cuda(DEV_ALLOC(s, &s->tab.entries,
		    c2 * sizeof (GEntry)), "cudaMalloc table")))
			break;
		if ((rc = s->cuda(DEV_ALLOC(s, &s->tab.arena, arena),
		    "cudaMalloc arena")))
			break;
		if ((rc = s->cuda(DEV_ALLOC(s, &s->tab.misc, 16 * sizeof (u32)),
		    "cudaMalloc misc")))
			break;
		s->tab.mask = (u32)(c2 - 1);
		s->tab.arena_cap = (u32)arena;
		cudaMemsetAsync(s->tab.entries, 0, c2 * sizeof (GEntry), s->stream);
		cudaMemsetAsync(s->tab.misc, 0, 16 * sizeof (u32), s->stream);
		const size_t nctr = NCTR + (MAX_METRICS - 1) * MCTR_PER;
		if ((rc = s->cuda(DEV_ALLOC(s, &s->d_counters,
		    nctr * sizeof (unsigned long long)), "cudaMalloc counters")))
			break;
		cudaMemsetAsync(s->d_counters, 0,
		    nctr * sizeof (unsigned long long), s->stream);
		if ((rc = s->cuda(DEV_ALLOC(s, &s->d_nl,
		    2 * sizeof (unsigned long long)), "cudaMalloc nl")))
			break;
		if ((rc = s->cuda(DEV_ALLOC(s, &s->d_carry, CARRY_ROOM + 64),
		    "cudaMalloc carry")))
			break;
		s->ring_cap = env_size("DNG_RING_BYTES", (size_t)64 << 20);
		/* whichever stream the scan ends up on waits for this setup */
		if ((rc = s->cuda(cudaEventCreateWithFlags(&s->ev_init,
		    cudaEventDisableTiming), "cudaEventCreate")))
			break;
		rc = s->cuda(cudaEventRecord(s->ev_init, s->stream), "init");
	} while (0);
	if (rc) {
		set_err(err, errlen, "%s", s->err.c_str());
		dng_scan_destroy(s);
		return rc;
	}
	*out = s;
	set_err(err, errlen, "");
	return DNG_OK;
}

int dng_scan_set_stream(dng_scan *s, void *cuda_stream)
{
	if (!s)
		return DNG_EINVAL;
	if (s->launches || s->bytes_fed)
		return s->fail(DNG_EINVAL, "dng_scan_set_stream after a feed");
	s->stream = (cudaStream_t)cuda_stream;
	CK(s, cudaStreamWaitEvent(s->stream, s->ev_init, 0));
	return DNG_OK;
}

static int ensure_ring(dng_scan *s, bool need_stage)
{
	for (size_t i = 0; i < RING_SLOTS; i++) {
		if (!s->d_ring[i]) {
			CK(s, DEV_ALLOC(s, &s->d_ring[i], CARRY_ROOM +
			    s->ring_cap + 64));
			CK(s, cudaEventCreateWithFlags(&s->ev_ready[i],
			    cudaEventDisableTiming));
			CK(s, cudaEventCreateWithFlags(&s->ev_free[i],
			    cudaEventDisableTiming));
		}
		if (need_stage && !s->h_stage[i])
			CK(s, HOST_ALLOC(&s->h_stage[i], s->ring_cap));
	}
	return 0;
}

int dng_scan_feed(dng_scan *s, const void *buf, size_t len)
{
	if (!s || (!buf && len))
		return DNG_EINVAL;
	cudaSetDevice(s->device);
	if (ensure_ring(s, true))
		return s->err_code;
	return feed_host(s, buf, len, false);
}

int dng_scan_feed_pinned(dng_scan *s, const void *buf, size_t len)
{
	if (!s || (!buf && len))
		return DNG_EINVAL;
	cudaSetDevice(s->device);
	if (ensure_ring(s, false))
		return s->err_code;
	return feed_host(s, buf, len, true);
}

/*
 * Sequential fallback for inputs that cannot be pread (pipes, /dev/stdin):
 * read(2) into two pinned buffers, DMA from one while filling the other.
 */
static int feed_fd_sequential(dng_scan *s, int fd, const char *path)
{
	size_t cap = std::min(s->ring_cap, (size_t)16 << 20);
	u8 *bufs[2] = { nullptr, nullptr };
	cudaEvent_t done[2] = { nullptr, nullptr };
	bool inflight[2] = { false, false };
	int rc = 0;
	for (int i = 0; i < 2 && !rc; i++) {
		rc = s->cuda(cudaMallocHost(&bufs[i], cap), "cudaMallocHost");
		if (!rc)
			rc = s->cuda(cudaEventCreateWithFlags(&done[i],
			    cudaEventDisableTiming), "cudaEventCreate");
	}
	int which = 0;
	while (!rc) {
		if (inflight[which]) {
			rc = s->cuda(cudaEventSynchronize(done[which]),
			    "copy sync");
			if (rc)
				break;
		}
		ssize_t n = read(fd, bufs[which], cap);
		if (n < 0) {
			rc = s->fail(DNG_EIO, std::string("read ") + path + ": " +
			    strerror(errno));
			break;
		}
		if (n == 0)
			break;
		rc = feed_host(s, bufs[which], (size_t)n, true);
		if (!rc)
			rc = s->cuda(cudaEventRecord(done[which], s->copy_stream),
			    "cudaEventRecord");
		inflight[which] = true;
		which ^= 1;
	}
	cudaStreamSynchronize(s->copy_stream);
	for (int i = 0; i < 2; i++) {
		if (bufs[i])
			cudaFreeHost(bufs[i]);
		if (done[i])
			cudaEventDestroy(done[i]);
	}
	return rc;
}

/*
 * Regular files: a few reader threads pread() fixed-size blocks into a ring of
 * pinned buffers (the page cache memcpy is the slow part of reading, so it is
 * spread over cores) while this thread feeds completed blocks, in order, to
 * the H2D ring.  The reference reads with 2 concurrent 16 KB-request streams
 * (lib/datasource-file.js:262-266).
 */
static int feed_file_parallel(dng_scan *s, int fd, size_t size, const char *path)
{
	const size_t BLK = (size_t)4 << 20;
	const size_t NSLOT = 32;	/* 128 MiB of pinned ring */
	const size_t LAG = 6;		/* blocks kept back for in-flight DMA */
	const size_t GROUP = 4;		/* ready neighbours fed as one chunk */
	if (!s->file_buf) {
		CK(s, HOST_ALLOC(&s->file_buf, NSLOT * BLK));
		for (size_t i = 0; i < NSLOT; i++)
			CK(s, cudaEventCreateWithFlags(&s->file_done[i],
			    cudaEventDisableTiming));
	}
	const size_t nblocks = (size + BLK - 1) / BLK;
	/* 16 readers measured best on the 128-core B200 host (21 GB/s from
	 * tmpfs); more threads contend in the page cache */
	size_t nthreads = env_size("DNG_READ_THREADS", 16);
	nthreads = std::max<size_t>(1, std::min(nthreads, std::min(nblocks,
	    NSLOT - LAG)));
	std::mutex mu;
	std::condition_variable cv;
	size_t next_block = 0;		/* next block a reader takes */
	size_t released = NSLOT;	/* blocks < released may be (re)filled */
	std::vector<ssize_t> got(nblocks, -2);	/* -2 pending, -1 error */
	int read_errno = 0;
	bool abort_all = false;
	auto reader = [&]() {
		for (;;) {
			size_t b;
			{
				std::unique_lock<std::mutex> lk(mu);
				b = next_block++;
				if (b >= nblocks)
					return;
				cv.wait(lk, [&] { return b < released ||
				    abort_all; });
				if (abort_all)
					return;
			}
			size_t want = std::min(BLK, size - b * BLK), have = 0;
			u8 *dst = s->file_buf + (b % NSLOT) * BLK;
			int err = 0;
			while (have < want) {
				ssize_t n = pread(fd, dst + have, want - have,
				    (off_t)(b * BLK + have));
				if (n < 0) {
					if (errno == EINTR)
						continue;
					err = errno;
					break;
				}
				if (n == 0)
					break;	/* file shrank */
				have += (size_t)n;
			}
			std::lock_guard<std::mutex> lk(mu);
			if (err) {
				read_errno = err;
				got[b] = -1;
			} else {
				got[b] = (ssize_t)have;
			}
			cv.notify_all();
		}
	};
	std::vector<std::thread> pool;
	for (size_t i = 0; i < nthreads; i++)
		pool.emplace_back(reader);
	int rc = 0;
	size_t b = 0;
	while (b < nblocks && !rc) {
		/* block b, plus ready full neighbours that are contiguous in
		 * the ring, go down as one chunk */
		size_t k = 0, bytes = 0;
		{
			std::unique_lock<std::mutex> lk(mu);
			cv.wait(lk, [&] { return got[b] != -2; });
			while (k < GROUP && b + k < nblocks &&
			    got[b + k] != -2 && (b + k) % NSLOT >= b % NSLOT) {
				if (got[b + k] < 0) {
					if (k == 0)
						rc = s->fail(DNG_EIO,
						    std::string("read ") + path +
						    ": " + strerror(read_errno));
					break;
				}
				bytes += (size_t)got[b + k];
				k++;
				if ((size_t)got[b + k - 1] != BLK)
					break;	/* short block: last one */
			}
		}
		if (rc)
			break;
		if (bytes)
			rc = feed_host(s, s->file_buf + (b % NSLOT) * BLK, bytes,
			    true);
		for (size_t j = 0; j < k && !rc; j++)
			rc = s->cuda(cudaEventRecord(
			    s->file_done[(b + j) % NSLOT], s->copy_stream),
			    "cudaEventRecord");
		b += k;
		/* slots LAG blocks behind have certainly been DMA'd: hand them
		 * back to the readers */
		if (!rc && b > LAG) {
			size_t old = b - LAG - 1;
			rc = s->cuda(cudaEventSynchronize(
			    s->file_done[old % NSLOT]), "copy sync");
			std::lock_guard<std::mutex> lk(mu);
			released = old + NSLOT + 1;
			cv.notify_all();
		}
	}
	{
		std::lock_guard<std::mutex> lk(mu);
		abort_all = true;
		cv.notify_all();
	}
	for (auto &t : pool)
		t.join();
	/* the pinned ring is reused by the next file: drain its copies */
	cudaStreamSynchronize(s->copy_stream);
	return rc;
}

int dng_scan_feed_file(dng_scan *s, const char *path)
{
	if (!s || !path)
		return DNG_EINVAL;
	cudaSetDevice(s->device);
	if (ensure_ring(s, false))
		return s->err_code;
	int fd = open(path, O_RDONLY);
	if (fd < 0)
		return s->fail(DNG_EIO, std::string("open ") + path + ": " +
		    strerror(errno));
	struct stat st;
	int rc;
	if (fstat(fd, &st) == 0 && S_ISREG(st.st_mode) && st.st_size > 0)
		rc = feed_file_parallel(s, fd, (size_t)st.st_size, path);
	else
		rc = feed_fd_sequential(s, fd, path);
	close(fd);
	return rc;
}

int dng_scan_feed_device(dng_scan *s, const void *devbuf, size_t len)
{
	if (!s || (!devbuf && len))
		return DNG_EINVAL;
	if (s->err_code)
		return s->err_code;
	if (s->finished)
		return s->fail(DNG_EINVAL, "scan already finished");
	if ((uintptr_t)devbuf & 15)
		return s->fail(DNG_EINVAL, "device buffer must be 16-byte "
		    "aligned");
	if (len == 0)
		return 0;
	/*
	 * A CTA's tally cache counts in 32 bits and is flushed once per launch.
	 * With weight-1 records that cannot wrap within a launch over any buffer
	 * HBM holds; with json-skinner weights (up to 255 take the cache) a
	 * launch is kept to 4 GiB: 29 MB per CTA, under 2^32 / 255 records of
	 * even the shortest point line.
	 */
	const size_t LAUNCH_MAX = (size_t)4 << 30;
	if (s->plan.dev.format == FMT_SKINNER && len > LAUNCH_MAX) {
		for (size_t off = 0; off < len; off += LAUNCH_MAX) {
			int rc = dng_scan_feed_device(s, (const u8 *)devbuf + off,
			    std::min(LAUNCH_MAX, len - off));
			if (rc)
				return rc;
		}
		return 0;
	}
	cudaSetDevice(s->device);
	/*
	 * A large buffer would be ONE launch: nothing learnt from it could
	 * help it.  Its head goes first, as a launch of its own, and what that
	 * one counted (keys that overflowed the F kernel's tally cache: f_nt)
	 * is looked at before the rest is launched.
	 */
	const size_t PROBE = (size_t)64 << 20;
	if (!s->f_probed && s->fplan.ok && s->f_nt > 768 && len > 4 * PROBE) {
		s->f_probed = true;
		int rc = dng_scan_feed_device(s, devbuf, PROBE);
		if (rc)
			return rc;
		CK(s, cudaStreamSynchronize(s->stream));
		return dng_scan_feed_device(s, (const u8 *)devbuf + PROBE,
		    len - PROBE);
	}
	const u8 *d = (const u8 *)devbuf;
	s->bytes_fed += len;
	/* locate the first and last newline (windows first, then all) */
	unsigned long long init[2] = { ~0ull, 0 }, got[2];
	const unsigned long long W = 1 << 20;
	for (int attempt = 0; attempt < 2; attempt++) {
		CK(s, cudaMemcpyAsync(s->d_nl, init, sizeof (init),
		    cudaMemcpyHostToDevice, s->stream));
		if (attempt == 0) {
			s->aux_launches++;
			find_nl_kernel<<<64, 256, 0, s->stream>>>(d, 0,
			    std::min<unsigned long long>(len, W), s->d_nl,
			    s->d_nl + 1);
			if (len > W) {
				s->aux_launches++;
				find_nl_kernel<<<64, 256, 0, s->stream>>>(d,
				    len - W, len, s->d_nl, s->d_nl + 1);
			}
		} else {
			s->aux_launches++;
			find_nl_kernel<<<1024, 256, 0, s->stream>>>(d, 0, len,
			    s->d_nl, s->d_nl + 1);
		}
		CK(s, cudaMemcpyAsync(got, s->d_nl, sizeof (got),
		    cudaMemcpyDeviceToHost, s->stream));
		CK(s, cudaStreamSynchronize(s->stream));
		/* with windows: `first` is only trustworthy if it fell in the
		 * head window, `last` if it fell in the tail window */
		bool first_ok = got[0] != ~0ull && (len <= W || got[0] < W);
		bool last_ok = got[1] != 0 && (len <= W || got[1] > len - W);
		if ((first_ok && last_ok) || attempt == 1 || len <= W)
			break;
	}
	if (got[0] == ~0ull) {
		/* no newline at all: the whole chunk extends the carry */
		if (s->carry_len + len > DNG_MAXREC)
			return s->fail(DNG_ELIMIT, "input line longer than 16 MiB");
		CK(s, cudaMemcpyAsync(s->d_carry + s->carry_len, d, len,
		    cudaMemcpyDeviceToDevice, s->stream));
		s->carry_len += len;
		return 0;
	}
	unsigned long long first = got[0], last = got[1];
	unsigned long long start = 0;
	if (s->carry_len) {
		/* finish the carried line in a side buffer */
		size_t head = (size_t)first + 1;
		if (s->carry_len + head > DNG_MAXREC)
			return s->fail(DNG_ELIMIT, "input line longer than 16 MiB");
		if (!s->d_side)
			CK(s, DEV_ALLOC(s, &s->d_side, CARRY_ROOM + 64));
		CK(s, cudaMemcpyAsync(s->d_side, s->d_carry, s->carry_len,
		    cudaMemcpyDeviceToDevice, s->stream));
		CK(s, cudaMemcpyAsync(s->d_side + s->carry_len, d, head,
		    cudaMemcpyDeviceToDevice, s->stream));
		if (launch_scan(s, s->d_side, 0, s->carry_len + head, false))
			return s->err_code;
		s->carry_len = 0;
		start = head;
	}
	if (launch_scan(s, d, start, last, false))
		return s->err_code;
	if (last < len) {
		size_t tail = len - (size_t)last;
		if (tail > DNG_MAXREC)
			return s->fail(DNG_ELIMIT, "input line longer than 16 MiB");
		CK(s, cudaMemcpyAsync(s->d_carry, d + last, tail,
		    cudaMemcpyDeviceToDevice, s->stream));
		s->carry_len = tail;
	}
	return 0;
}

int dng_scan_sync(dng_scan *s)
{
	if (!s)
		return DNG_EINVAL;
	cudaSetDevice(s->device);
	CK(s, cudaStreamSynchronize(s->copy_stream));
	CK(s, cudaStreamSynchronize(s->stream));
	drain_events(s);
	return s->err_code;
}

static int flush_tail(dng_scan *s)
{
	if (s->finished)
		return 0;
	s->finished = true;
	if (s->carry_len) {
		/* lstream emits the final unterminated line */
		if (launch_scan(s, s->d_carry, 0, s->carry_len, true))
			return s->err_code;
		s->carry_len = 0;
	}
	return 0;
}

int dng_scan_counters(dng_scan *s, dng_counters *out)
{
	if (!s || !out)
		return DNG_EINVAL;
	cudaSetDevice(s->device);
	if (dng_scan_sync(s))
		return s->err_code;
	unsigned long long c[NCTR];
	CK(s, cudaMemcpy(c, s->d_counters, sizeof (c), cudaMemcpyDeviceToHost));
	memset(out, 0, sizeof (*out));
	out->lines = c[CTR_LINES];
	out->invalid_json = c[CTR_INVALID_JSON];
	out->invalid_point = c[CTR_INVALID_POINT];
	out->ds_filtered = c[CTR_DS_FILTERED];
	out->ds_failedeval = c[CTR_DS_FAILED];
	out->user_filtered = c[CTR_USER_FILTERED];
	out->user_failedeval = c[CTR_USER_FAILED];
	out->synth_undef = c[CTR_SYNTH_UNDEF];
	out->synth_baddate = c[CTR_SYNTH_BADDATE];
	out->time_filtered = c[CTR_TIME_FILTERED];
	out->time_failedeval = c[CTR_TIME_FAILED];
	out->aggr_ninputs = c[CTR_AGGR];
	out->slowpath_records = c[CTR_SLOW];
	out->unsupported = c[CTR_UNSUPPORTED];
	out->long_records = c[CTR_LONG];
	out->bytes = s->bytes_fed;
	uint64_t n = out->lines - out->invalid_json - out->invalid_point;
	const DevPlan &P = s->plan.dev;
	if (P.ds_entry >= 0) {
		out->ds_ninputs = n;
		n -= out->ds_filtered + out->ds_failedeval;
	}
	if (P.metric[0].user_entry >= 0) {
		out->user_ninputs = n;
		n -= out->user_filtered + out->user_failedeval;
	}
	if (P.metric[0].nsyn) {
		out->synth_ninputs = n;
		n -= out->synth_undef + out->synth_baddate;
	}
	if (P.metric[0].time_entry >= 0)
		out->time_ninputs = n;
	return DNG_OK;
}

int dng_scan_counters_metric(dng_scan *s, int m, dng_counters *out)
{
	if (!s || !out || m < 0 || m >= s->plan.dev.nmetrics)
		return DNG_EINVAL;
	int rc = dng_scan_counters(s, out);
	if (rc || m == 0)
		return rc;
	unsigned long long c[MCTR_PER];
	CK(s, cudaMemcpy(c, s->d_counters + NCTR + (m - 1) * MCTR_PER,
	    sizeof (c), cudaMemcpyDeviceToHost));
	const Metric &M = s->plan.dev.metric[m];
	uint64_t n = out->lines - out->invalid_json - out->invalid_point -
	    out->ds_filtered - out->ds_failedeval;
	out->user_ninputs = out->synth_ninputs = out->time_ninputs = 0;
	out->user_filtered = c[0];
	out->user_failedeval = c[1];
	out->synth_undef = c[2];
	out->synth_baddate = c[3];
	out->time_filtered = c[4];
	out->time_failedeval = c[5];
	out->aggr_ninputs = c[6];
	if (M.user_entry >= 0) {
		out->user_ninputs = n;
		n -= c[0] + c[1];
	}
	if (M.nsyn) {
		out->synth_ninputs = n;
		n -= c[2] + c[3];
	}
	if (M.time_entry >= 0)
		out->time_ninputs = n;
	return DNG_OK;
}

int dng_scan_finish(dng_scan *s, dng_result **out)
{
	if (!s || !out)
		return DNG_EINVAL;
	if (s->err_code)
		return s->err_code;
	cudaSetDevice(s->device);
	if (flush_tail(s))
		return s->err_code;
	if (dng_scan_sync(s))
		return s->err_code;
	u32 misc[4];
	CK(s, cudaMemcpy(misc, s->tab.misc, sizeof (misc),
	    cudaMemcpyDeviceToHost));
	if (misc[2] & ST_TABLE_FULL)
		return s->fail(DNG_ELIMIT, "too many distinct tuples for the "
		    "device table (raise DNG_TABLE_CAP)");
	if (misc[2] & ST_ARENA_FULL)
		return s->fail(DNG_ELIMIT, "group-key arena exhausted (raise "
		    "DNG_ARENA_BYTES)");
#ifdef DNG_PROFILE_PHASES
	{	/* tuning builds only: where a tile's cycles go (see scan_kernel) */
		unsigned long long pc[NCTR];
		CK(s, cudaMemcpy(pc, s->d_counters, sizeof (pc),
		    cudaMemcpyDeviceToHost));
		double nw = (double)pc[18] ? (double)pc[18] : 1;
		fprintf(stderr, "phases: per warp-tile cycles: load-wait %.0f "
		    "index %.0f records-busy %.0f records-phase %.0f total %.0f "
		    "(%llu warp-tiles)\n", pc[19] / nw, pc[20] / nw, pc[16] / nw,
		    pc[17] / nw, pc[21] / nw, pc[18]);
	}
#endif
	dng_counters c;
	if (dng_scan_counters(s, &c))
		return s->err_code;
	if (c.unsupported)
		return s->fail(DNG_EUNSUPPORTED, "input contains records the "
		    "device path cannot decide yet (" +
		    std::to_string(c.unsupported) + "): nesting deeper than 64, "
		    "a group key longer than 512 bytes, a line >= 16 MiB, an "
		    "array where an index/length lookup is needed, or a date "
		    "string outside the ISO format (V8's legacy Date.parse "
		    "forms are not restated)");
	u32 n = misc[1];
	dng_result *r = new dng_result();
	r->init_from_plan(&s->plan);
	if (n) {
		OutEntry *d_out = nullptr;
		u32 *d_n = nullptr;
		size_t cap_out = 4096;		/* few sizes: cache-friendly */
		while (cap_out < n)
			cap_out <<= 1;
		CK(s, DEV_ALLOC(s, &d_out, cap_out * sizeof (OutEntry)));
		CK(s, DEV_ALLOC(s, &d_n, 16));
		CK(s, cudaMemsetAsync(d_n, 0, sizeof (u32), s->stream));
		s->aux_launches++;
		compact_kernel<<<256, 256, 0, s->stream>>>(s->tab.entries,
		    s->tab.mask + 1, d_out, d_n);
		std::vector<OutEntry> ents(n);
		std::vector<u8> arena(misc[0]);
		CK(s, cudaMemcpyAsync(ents.data(), d_out,
		    (size_t)n * sizeof (OutEntry), cudaMemcpyDeviceToHost,
		    s->stream));
		if (misc[0])
			CK(s, cudaMemcpyAsync(arena.data(), s->tab.arena, misc[0],
			    cudaMemcpyDeviceToHost, s->stream));
		CK(s, cudaStreamSynchronize(s->stream));
		cached_free(d_out);
		cached_free(d_n);
		r->keys.reserve(n);
		r->values.reserve(n);
		for (u32 i = 0; i < n; i++) {
			r->keys.emplace_back((const char *)arena.data() +
			    ents[i].koff, ents[i].klen);
			r->values.push_back(ents[i].count);
		}
	}
	r->finalize();
	*out = r;
	return DNG_OK;
}

const char *dng_scan_error(const dng_scan *s)
{
	return s ? s->err.c_str() : "null scan";
}

int dng_scan_set_templates(dng_scan *s, int enable)
{
	if (!s)
		return DNG_EINVAL;
	if (s->tmpl_tried)
		return s->fail(DNG_EINVAL, "templates are fixed once data has "
		    "been fed");
	s->tmpl_enabled = enable != 0;
	return DNG_OK;
}

int dng_scan_template_stats(dng_scan *s, uint64_t *templates,
    uint64_t *templated_records)
{
	if (!s)
		return DNG_EINVAL;
	cudaSetDevice(s->device);
	if (dng_scan_sync(s))
		return s->err_code;
	unsigned long long c = 0;
	CK(s, cudaMemcpy(&c, s->d_counters + CTR_TMPL, sizeof (c),
	    cudaMemcpyDeviceToHost));
	if (templates)
		*templates = s->ntemplates;
	if (templated_records)
		*templated_records = c;
	return DNG_OK;
}

uint64_t dng_scan_launch_count(const dng_scan *s)
{
	return s ? s->launches + s->aux_launches : 0;
}

int dng_scan_kernel_kind(const dng_scan *s)
{
	if (!s)
		return DNG_EINVAL;
	return s->f_kernel && s->fplan.ok ? 2 : s->warp_kernel ? 1 : 0;
}

int dng_scan_jit_stats(dng_scan *s, int *state, uint64_t *launches,
    double *compile_ms, double *link_ms, char *err, size_t errlen)
{
	if (!s)
		return DNG_EINVAL;
	const int st = s->jit ? s->jit->state.load() : 0;
	if (state)
		*state = st;
	if (launches)
		*launches = s->jit_launches;
	if (compile_ms)
		*compile_ms = st ? s->jit->compile_ms : 0;
	if (link_ms)
		*link_ms = st ? s->jit->link_ms : 0;
	set_err(err, errlen, "%s", st == 2 ? s->jit->err.c_str() : "");
	return DNG_OK;
}

int dng_scan_kernel_stats(dng_scan *s, double *kernel_ms, uint64_t *launches,
    uint64_t *kernel_bytes)
{
	if (!s)
		return DNG_EINVAL;
	cudaSetDevice(s->device);
	if (dng_scan_sync(s))
		return s->err_code;
	if (kernel_ms)
		*kernel_ms = s->kernel_ms;
	if (launches)
		*launches = s->launches;
	if (kernel_bytes)
		*kernel_bytes = s->kernel_bytes;
	return DNG_OK;
}

void dng_release_cached(void)
{
	BufCache &c = buf_cache();
	std::multimap<std::pair<int, size_t>, void *> idle;
	{
		std::lock_guard<std::mutex> g(c.mu);
		idle.swap(c.idle);
		c.idle_dev = c.idle_host = 0;
	}
	for (auto &kv : idle) {
		if (kv.first.first < 0) {
			cudaFreeHost(kv.second);
		} else {
			cudaSetDevice(kv.first.first);
			cudaFree(kv.second);
		}
	}
}

void dng_scan_destroy(dng_scan *s)
{
	if (!s)
		return;
	cudaSetDevice(s->device);
	if (s->stream)
		cudaStreamSynchronize(s->stream);
	if (s->own_stream && s->own_stream != s->stream)
		cudaStreamSynchronize(s->own_stream);
	if (s->copy_stream)
		cudaStreamSynchronize(s->copy_stream);
	drain_events(s);
	if (s->ev_init)
		cudaEventDestroy(s->ev_init);
	for (auto e : s->ev_pool)
		cudaEventDestroy(e);
	for (size_t i = 0; i < RING_SLOTS; i++) {
		if (s->d_ring[i]) {
			cached_free(s->d_ring[i]);
			cudaEventDestroy(s->ev_ready[i]);
			cudaEventDestroy(s->ev_free[i]);
		}
		if (s->h_stage[i])
			cached_free(s->h_stage[i]);
	}
	if (s->file_buf) {
		cached_free(s->file_buf);
		for (int i = 0; i < 32; i++)
			cudaEventDestroy(s->file_done[i]);
	}
	cached_free(s->h_live);
	cached_free(s->d_plan);
	cached_free(s->d_tmpl);
	cached_free(s->d_fplan);
	cached_free(s->d_ftmpl);
	cached_free(s->d_fdict);
	cached_free(s->d_miss);
	cached_free(s->d_miss_n);
	cached_free(s->tab.entries);
	cached_free(s->tab.arena);
	cached_free(s->tab.misc);
	cached_free(s->d_counters);
	cached_free(s->d_nl);
	cached_free(s->d_carry);
	cached_free(s->d_side);
	if (s->own_stream)
		cudaStreamDestroy(s->own_stream);
	if (s->copy_stream)
		cudaStreamDestroy(s->copy_stream);
	delete s;
}

void *dng_pinned_alloc(size_t len)
{
	void *p = nullptr;
	if (cudaMallocHost(&p, len) != cudaSuccess)
		return nullptr;
	return p;
}

void dng_pinned_free(void *p)
{
	if (p)
		cudaFreeHost(p);
}

/* ---- results ------------------------------------------------------------ */

size_t dng_result_count(const dng_result *r)
{
	return r ? r->keys.size() : 0;
}

size_t dng_result_ncols(const dng_result *r)
{
	size_t n = 0;
	for (int m = 0; r && m < r->nmetrics; m++)
		n = std::max(n, (size_t)r->ncols[m]);
	return n;		/* widest metric; == ncols for a plain scan */
}

size_t dng_result_nmetrics(const dng_result *r)
{
	return r ? (size_t)r->nmetrics : 0;
}

size_t dng_result_ncols_metric(const dng_result *r, int m)
{
	return r && m >= 0 && m < r->nmetrics ? (size_t)r->ncols[m] : 0;
}

int dng_result_metric(const dng_result *r, size_t i)
{
	return r && i < r->metric.size() ? r->metric[i] : -1;
}

int dng_result_get(const dng_result *r, size_t i, const char **strs,
    size_t *strlens, uint8_t *is_number, double *numvals, uint64_t *value)
{
	if (!r || i >= r->keys.size())
		return DNG_EINVAL;
	for (int j = 0; j < r->ncols[r->metric[i]]; j++) {
		const dng_result::Cell &c = r->cells[r->cell0[i] + j];
		if (is_number)
			is_number[j] = c.is_number;
		if (numvals)
			numvals[j] = c.num;
		if (strs)
			strs[j] = c.is_number ? nullptr :
			    r->keys[i].data() + c.off;
		if (strlens)
			strlens[j] = c.is_number ? 0 : c.len;
	}
	if (value)
		*value = r->values[i];
	return DNG_OK;
}

void dng_result_destroy(dng_result *r)
{
	delete r;
}

/* ---- synthetic input ------------------------------------------------------ */

void dng_gen_defaults(dng_gen_params *p)
{
	p->seed = 0xD5A60000ull;
	p->total_records = 1000;
	p->time_min_ms = 1401570000000ll;	/* 2014-05-31T21:00:00Z */
	p->time_max_ms = 1401580799000ll;	/* 2014-05-31T23:59:59Z */
	p->string_latency = 0;
}

int dng_gen_host(const dng_gen_params *p, uint64_t first, uint64_t count,
    void *buf, size_t cap, size_t *len)
{
	if (!p || !buf || !len)
		return DNG_EINVAL;
	char *o = (char *)buf;
	size_t n = 0;
	char tmp[GEN_MAXREC];
	for (uint64_t j = first; j < first + count; j++) {
		int k = gen_record(*p, j, tmp);
		if (n + (size_t)k > cap)
			return DNG_ELIMIT;
		memcpy(o + n, tmp, (size_t)k);
		n += (size_t)k;
	}
	*len = n;
	return DNG_OK;
}

} /* extern "C" */

namespace {

__global__ void gen_len_kernel(dng_gen_params p, uint64_t first, uint64_t count,
    unsigned long long *block_sums, u32 *lens)
{
	__shared__ u32 red[256 / 32];
	uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	char tmp[GEN_MAXREC];
	u32 k = 0;
	if (j < count) {
		k = (u32)gen_record(p, first + j, tmp);
		lens[j] = k;
	}
	u32 v = k;
	for (int d = 16; d > 0; d >>= 1)
		v += __shfl_xor_sync(0xffffffffu, v, d);
	if ((threadIdx.x & 31) == 0)
		red[threadIdx.x >> 5] = v;
	__syncthreads();
	if (threadIdx.x == 0) {
		u32 t = 0;
		for (int i = 0; i < 256 / 32; i++)
			t += red[i];
		block_sums[blockIdx.x] = t;
	}
}

__global__ void gen_write_kernel(dng_gen_params p, uint64_t first,
    uint64_t count, const unsigned long long *block_offs, const u32 *lens,
    char *out)
{
	__shared__ u32 soff[256];
	uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
	u32 k = j < count ? lens[j] : 0;
	soff[threadIdx.x] = k;
	__syncthreads();
	/* exclusive scan within the block (serial by thread 0: 256 adds) */
	if (threadIdx.x == 0) {
		u32 acc = 0;
		for (int i = 0; i < 256; i++) {
			u32 t = soff[i];
			soff[i] = acc;
			acc += t;
		}
	}
	__syncthreads();
	if (j < count) {
		char tmp[GEN_MAXREC];
		int n = gen_record(p, first + j, tmp);
		char *dst = out + block_offs[blockIdx.x] + soff[threadIdx.x];
		for (int i = 0; i < n; i++)
			dst[i] = tmp[i];
	}
}

} /* namespace */

extern "C" int dng_gen_device(const dng_gen_params *p, int device,
    uint64_t first, uint64_t count, void *devbuf, size_t cap, size_t *len)
{
	if (!p || !devbuf || !len)
		return DNG_EINVAL;
	if (cudaSetDevice(device) != cudaSuccess)
		return DNG_ENODEV;
	if (count == 0) {
		*len = 0;
		return DNG_OK;
	}
	u32 nblocks = (u32)((count + 255) / 256);
	unsigned long long *d_sums = nullptr;
	u32 *d_lens = nullptr;
	int rc = DNG_OK;
	if (cudaMalloc(&d_sums, (size_t)nblocks * 8) != cudaSuccess ||
	    cudaMalloc(&d_lens, (size_t)count * 4) != cudaSuccess) {
		cudaFree(d_sums);
		cudaFree(d_lens);
		return DNG_ENOMEM;
	}
	gen_len_kernel<<<nblocks, 256>>>(*p, first, count, d_sums, d_lens);
	std::vector<unsigned long long> sums(nblocks);
	if (cudaMemcpy(sums.data(), d_sums, (size_t)nblocks * 8,
	    cudaMemcpyDeviceToHost) != cudaSuccess)
		rc = DNG_ECUDA;
	unsigned long long acc = 0;
	for (u32 i = 0; i < nblocks; i++) {
		unsigned long long t = sums[i];
		sums[i] = acc;
		acc += t;
	}
	if (!rc && acc > cap)
		rc = DNG_ELIMIT;
	if (!rc) {
		cudaMemcpy(d_sums, sums.data(), (size_t)nblocks * 8,
		    cudaMemcpyHostToDevice);
		gen_write_kernel<<<nblocks, 256>>>(*p, first, count, d_sums,
		    d_lens, (char *)devbuf);
		if (cudaDeviceSynchronize() != cudaSuccess)
			rc = DNG_ECUDA;
		*len = (size_t)acc;
	}
	cudaFree(d_sums);
	cudaFree(d_lens);
	return rc;
}
