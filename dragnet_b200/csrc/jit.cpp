/*
 * jit.cpp: see jit.h.  Host code only: source generation from a trie blob,
 * NVRTC + nvJitLink through dlopen, the per-process kernel cache.
 */
#include <dlfcn.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <chrono>
#include <functional>
#include <map>
#include <mutex>
#include <set>
#include <vector>

#include "jit.h"
#include "fast.h"
#include "tmpl.h"

/* jit_blob.S: the LTO-IR builds of the kernel (fast_jit.cu), its rare paths as
 * SASS (fast_jit_cold.cu) and fscan.cuh as text */
#define BLOB(n) extern "C" const unsigned char n[]; \
	extern "C" const unsigned char n##_end[];
BLOB(dng_jit_hot7) BLOB(dng_jit_hot9) BLOB(dng_jit_hot11) BLOB(dng_jit_hot13)
BLOB(dng_jit_cold)
#undef BLOB
extern "C" const char dng_fscan_src[];
extern "C" const char dng_fscan_src_end[];

namespace dng {

namespace {

/* what fscan.cuh expects from its includer, for NVRTC (no headers at all) */
const char *PRELUDE =
"typedef unsigned char u8;\n"
"typedef unsigned int u32;\n"
"typedef unsigned long long u64;\n"
"#define DNG_HD __device__ __forceinline__\n"
"#ifdef DNG_JIT_SHARED_SCAN\n"
"#define DNG_FSCAN_FN __device__ __noinline__\n"
"#endif\n"

"enum { T_UNDEF = 0, T_NULL = 1, T_FALSE = 2, T_TRUE = 3, T_NUM = 4, T_STR = 5 };\n"
"#define DNG_FCAP(type, off, len, flag) \\\n"
"	((u32)(off) | ((u32)(len) << 12) | ((u32)(type) << 24) | ((u32)(flag) << 27))\n"
"DNG_HD bool is_hex(u32 c)\n"
"{\n"
"	return (c >= '0' && c <= '9') || ((c | 0x20) >= 'a' && (c | 0x20) <= 'f');\n"
"}\n"
"DNG_HD u32 tm_isdigit(u32 c) { return c - '0' <= 9u; }\n"
"DNG_HD u32 nondigit_mask(u32 w)\n"
"{\n"
"	const u32 x = w ^ 0x30303030u;\n"
"	return (((x & 0x7f7f7f7fu) + 0x76767676u) | x) & 0x80808080u;\n"
"}\n"
"DNG_HD u32 low_flag_byte(u32 m) { return (__ffs(m) - 8) >> 3; }\n"
"DNG_HD u32 jlds32(u32 a)\n"
"{\n"
"	u32 v;\n"
"	asm volatile(\"ld.shared.u32 %0, [%1];\" : \"=r\"(v) : \"r\"(a));\n"
"	return v;\n"
"}\n"
"DNG_HD u32 jlds8(u32 a)\n"
"{\n"
"	u32 v;\n"
"	asm volatile(\"ld.shared.u8 %0, [%1];\" : \"=r\"(v) : \"r\"(a));\n"
"	return v;\n"
"}\n"
"DNG_HD void jsts32(u32 a, u32 v)\n"
"{\n"
"	asm volatile(\"st.shared.u32 [%0], %1;\" :: \"r\"(a), \"r\"(v) : \"memory\");\n"
"}\n"
"/* the record in shared memory (fast_kernel.cuh FSmem) */\n"
"struct JMem {\n"
"	u32 ra;\n"
"	struct Cur {\n"
"		u32 wa, w0, w1, sh;\n"
"		DNG_HD u32 next()\n"
"		{\n"
"			const u32 d = __funnelshift_r(w0, w1, sh);\n"
"			w0 = w1;\n"
"			wa += 4;\n"
"			w1 = jlds32(wa);\n"
"			return d;\n"
"		}\n"
"	};\n"
"	DNG_HD Cur cursor(u32 off) const\n"
"	{\n"
"		Cur c;\n"
"		const u32 a = ra + off;\n"
"		c.sh = (a & 3) * 8;\n"
"		c.wa = (a & ~3u) + 4;\n"
"		c.w0 = jlds32(c.wa - 4);\n"
"		c.w1 = jlds32(c.wa);\n"
"		return c;\n"
"	}\n"
"	struct ACur {\n"
"		u32 wa, k;\n"
"		DNG_HD u32 next() { const u32 v = jlds32(wa); wa += 4; return v; }\n"
"	};\n"
"	DNG_HD ACur acursor(u32 off) const\n"
"	{\n"
"		ACur c;\n"
"		const u32 a = ra + off;\n"
"		c.k = a & 3;\n"
"		c.wa = a & ~3u;\n"
"		return c;\n"
"	}\n"
"	DNG_HD u32 apos(const ACur &c) const { return c.wa - 4 - ra; }\n"
"	DNG_HD u32 byte(u32 off) const { return jlds8(ra + off); }\n"
"	DNG_HD u32 word(u32 off) const { Cur c = cursor(off); return c.next(); }\n"
"};\n";

void appendf(std::string &s, const char *fmt, ...)
    __attribute__((format(printf, 2, 3)));

void appendf(std::string &s, const char *fmt, ...)
{
	char buf[512];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(buf, sizeof (buf), fmt, ap);
	va_end(ap);
	s += buf;
}

} /* namespace */

/*
 * The generated matcher is fmatch() (fast.cuh) with the trie unrolled into a
 * state machine in topological order: one block per node,
 *
 *     if (st == i) { literal at p against immediates; wildcard scan;
 *                    capture; st = successor | dispatched child | DONE
 *                    -- or, on a mismatch, st = alt sibling | FAIL }
 *
 * emitted in node order, which is breadth first: every edge (successor,
 * dispatched child, `alt` sibling) leads to a higher index, so ONE pass over
 * the blocks carries every lane along its own path, and the lanes of a warp
 * meet again in front of every block (a __syncwarp(): the function is called
 * by all 32 lanes, with `active` clear for those without a record).
 *
 * A string wildcard takes its closing quote with it (the literals that follow
 * one lose their first byte), so that what follows `"caller":"x"` and
 * `"caller":null` is the same text; a block whose only way on is a block
 * nothing else leads to continues with that block's body (no meeting needed
 * where nobody can join); literals short enough for the slack behind the
 * buffer are compared without asking whether the record is that long (its
 * '\n' differs from every literal byte).
 *
 * Equivalent subtrees are emitted once: records that differ in an optional
 * field take different blocks for it and the same blocks again for what
 * follows, with the whole warp.  To make the tails of such templates
 * identical the paths a template defines are accumulated along the way (a bit
 * per capturing node) instead of being a constant of the leaf; this is checked
 * here against the leaf masks and falls back to them if it ever differs.
 */
namespace {

struct JN {
	std::string lit;
	u32 kind, cap;
	bool leaf;
	u32 leaf_mask;
	int next, alt;			/* node indexes, -1 none */
	u32 dk;				/* dispatch byte offset */
	std::vector<std::pair<u32, int>> disp;	/* byte -> child */
	bool has_disp;
};

/* the children a record can move to from n (after n matched) */
void successors(const JN &n, std::vector<int> &out)
{
	out.clear();
	if (n.leaf)
		return;
	if (n.has_disp) {
		for (auto &d : n.disp)
			out.push_back(d.second);
	} else {
		out.push_back(n.next);
	}
}

} /* namespace */

/*
 * The plan, written out as the constant the LTO build of the kernel refers to
 * (fast_kernel.cuh dng_jplan): the same bytes as the FPlan the scan uploads,
 * field by field, under struct declarations that are checked against the
 * library's by size.
 */
static void plan_source(const FPlan &F, std::string &s)
{
	s += "struct Src { u8 kind; u8 idx; };\n"
	    "/* (binary64 fields as their bit patterns: NaN and infinity have no\n"
	    " * literal; same layout as the double the kernel reads) */\n"
	    "struct Leaf { u64 cnum; unsigned short coff, clen; short jt, jf; "
	    "u8 op; u8 cstr; Src src; u32 pad; };\n"
	    "struct Col { u64 step; Src src; u8 kind; u8 pad[5]; };\n"
	    "struct alignas(16) FPlan { Leaf code[16]; Col col[6]; "
	    "u8 syn_path[2]; short ds_entry, user_entry, time_entry; "
	    "u8 nsyn, ncols, npaths, ok; u8 ord_row[6]; u8 nrows, ncode; u8 pad[4]; "
	    "char pool[512]; };\n";
	appendf(s, "static_assert(sizeof (Leaf) == %zu && sizeof (Col) == %zu && "
	    "sizeof (FPlan) == %zu, \"plan layout\");\n", sizeof (Leaf),
	    sizeof (Col), sizeof (FPlan));
	static_assert(F_MAXCODE == 16 && F_MAXCOLS == 6 && F_MAXSYN == 2 &&
	    F_POOL == 512, "plan_source() spells these out");
	s += "extern \"C\" __constant__ const FPlan dng_jplan = {\n	{\n";
	for (int i = 0; i < F_MAXCODE; i++) {
		const Leaf &l = F.code[i];
		u64 cb;
		memcpy(&cb, &l.cnum, 8);
		appendf(s, "		{ 0x%016llxull, %u, %u, %d, %d, %u, %u, { %u, %u }, 0 },\n",
		    (unsigned long long)cb, (unsigned)l.coff, (unsigned)l.clen, (int)l.jt,
		    (int)l.jf, (unsigned)l.op, (unsigned)l.cstr,
		    (unsigned)l.src.kind, (unsigned)l.src.idx);
	}
	s += "	},\n	{\n";
	for (int i = 0; i < F_MAXCOLS; i++) {
		const Col &c = F.col[i];
		u64 sb;
		memcpy(&sb, &c.step, 8);
		appendf(s, "		{ 0x%016llxull, { %u, %u }, %u, { 0, 0, 0, 0, 0 } },\n",
		    (unsigned long long)sb, (unsigned)c.src.kind, (unsigned)c.src.idx,
		    (unsigned)c.kind);
	}
	appendf(s, "	},\n	{ %u, %u }, %d, %d, %d, %u, %u, %u, %u,\n",
	    (unsigned)F.syn_path[0], (unsigned)F.syn_path[1], (int)F.ds_entry,
	    (int)F.user_entry, (int)F.time_entry, (unsigned)F.nsyn,
	    (unsigned)F.ncols, (unsigned)F.npaths, (unsigned)F.ok);
	appendf(s, "	{ %u, %u, %u, %u, %u, %u }, %u, %u, { 0, 0, 0, 0 },\n	{ ",
	    (unsigned)F.ord_row[0], (unsigned)F.ord_row[1],
	    (unsigned)F.ord_row[2], (unsigned)F.ord_row[3],
	    (unsigned)F.ord_row[4], (unsigned)F.ord_row[5], (unsigned)F.nrows,
	    (unsigned)F.ncode);
	for (int i = 0; i < F_POOL; i++)
		appendf(s, "%d,%s", (int)(signed char)F.pool[i],
		    i % 32 == 31 ? "\n	  " : "");
	s += " }\n};\n";
}

unsigned jit_dense()
{
	const char *v = getenv("DNG_DENSE");
	return v ? (unsigned)atoi(v) : 1u;
}

/*
 * dng_jcode(): the record's dense counter (fast.h FDict), or ~0u when a piece of
 * its key is not in the dictionary.  The same pieces as fpiece() (fast.cuh):
 * the record's bytes for a string or a plain integer -- by length, then word by
 * word against immediates -- and the constant a null / boolean / missing value
 * stands for.  fprep() has already turned away every other form.
 */
static void dense_source(const FDict &D, std::string &s)
{
	s += "extern \"C\" __device__ unsigned dng_jcode(unsigned ra, unsigned dm, "
	    "unsigned caps)\n{\n	JMem m;\n	m.ra = ra;\n	u32 idx = 0;\n";
	for (u32 j = 0; j < D.ncols; j++) {
		const u32 p = D.path[j];
		appendf(s, "	{	/* column %u: path %u, %u values */\n", j, p,
		    D.n[j]);
		appendf(s, "	const u32 cw = (dm >> %uu) & 1u ? jlds32(caps + %uu) "
		    ": 0u;\n", p, p * (u32)F_NT * 4u);
		s += "	const u32 t = (cw >> 24) & 7u, n = (cw >> 12) & 0xfffu;\n"
		    "	u32 c = 0xffffffffu;\n"
		    "	if (t == T_STR || t == T_NUM) {\n"
		    "		JMem::Cur k = m.cursor(cw & 0xfffu);\n"
		    "		switch (n) {\n";
		std::map<u32, std::vector<u32>> bylen;
		for (u32 c = 0; c < D.n[j]; c++)
			bylen[D.len[j][c]].push_back(c);
		for (auto &bl : bylen) {
			const u32 L = bl.first, nw = (L + 3) / 4;
			appendf(s, "		case %u: {\n", L);
			for (u32 w = 0; w < nw; w++) {
				if (w + 1 == nw && (L & 3))
					appendf(s, "			const u32 w%u = k.next() & "
					    "0x%08xu;\n", w, (1u << (8 * (L & 3))) - 1);
				else
					appendf(s, "			const u32 w%u = k.next();\n",
					    w);
			}
			bool first = true;
			for (u32 c : bl.second) {
				s += first ? "			if (" : "			else if (";
				first = false;
				if (nw == 0)
					s += "true";
				for (u32 w = 0; w < nw; w++) {
					u32 lit = 0;
					for (u32 x = 0; x < 4 && 4 * w + x < L; x++)
						lit |= (u32)D.val[j][c][4 * w + x] <<
						    (8 * x);
					appendf(s, "%sw%u == 0x%08xu", w ? " && " : "",
					    w, lit);
				}
				appendf(s, ")\n				c = %uu;\n",
				    c * D.stride[j]);
			}
			s += "			break;\n		}\n";
		}
		s += "		}\n	}\n";
		/* the constants of fpiece() */
		static const struct { u32 t; const char *v; } K[] = {
			{ T_UNDEF, "undefined" }, { T_NULL, "null" },
			{ T_TRUE, "true" }, { T_FALSE, "false" } };
		for (auto &kc : K)
			for (u32 c = 0; c < D.n[j]; c++)
				if (D.len[j][c] == strlen(kc.v) &&
				    !memcmp(D.val[j][c], kc.v, D.len[j][c]))
					appendf(s, "	if (t == %uu)\n		c = %uu;\n",
					    kc.t, c * D.stride[j]);
		s += "	if (c == 0xffffffffu)\n		return c;\n	idx += c;\n	}\n";
	}
	s += "	return idx;\n}\n";
}

std::string jit_source(const u8 *blob, size_t bytes, const FPlan *plan,
    const char *prelude, const FDict *dict)
{
	std::string s;
	s += "/* generated by libdragnet_gpu (jit.cpp) */\n";
	/*
	 * One copy of each scanner, called, instead of one inlined into every
	 * block?  Measured on B200 (100 M rows): with one or two columns the
	 * kernel's loop is 37 KB of code against 32 KB of instruction cache and
	 * the calls cost more than the misses they save (configs[2]: -7 %);
	 * with three columns the unrolled key code makes it 40 KB, the hit rate
	 * falls from 84 % to 62 %, the L1.5's fetch rate becomes the bound and
	 * the shared copies win (configs[4]: +13 %).  (Sharing the number
	 * scanner alone: -2 % and -4 % on configs[2] and [1].)
	 * DNG_JIT_SHARED=0|1 forces.
	 */
	bool shared = plan && plan->ncols >= 3;
	if (const char *sh = getenv("DNG_JIT_SHARED"))
		shared = atoi(sh) == 1;
	if (!prelude && shared)
		s += "#define DNG_JIT_SHARED_SCAN\n";
	s += prelude ? prelude : PRELUDE;
	if (plan)
		plan_source(*plan, s);
	s.append(dng_fscan_src, (size_t)(dng_fscan_src_end - dng_fscan_src));
	/*
	 * Dense keys: the kernel refers to both symbols, so the device build
	 * always has them -- without a dictionary dng_jdense = 0 and the lookup
	 * is dead code.  The dictionary is part of the text, hence of the
	 * kernel cache's key.
	 */
	const unsigned mode = jit_dense();
	const bool dense = dict && dict->ncols && mode;
	if (plan)
		appendf(s, "\nextern \"C\" __constant__ const unsigned dng_jdense = "
		    "%uu;\n", dense ? mode | 1u : 0u);
	if (dense)
		dense_source(*dict, s);
	else if (plan)
		s += "extern \"C\" __device__ unsigned dng_jcode(unsigned, unsigned, "
		    "unsigned)\n{\n	return 0xffffffffu;\n}\n";
	s += "\nextern \"C\" __device__ unsigned dng_jmatch(unsigned ra, "
	    "unsigned len, unsigned active, unsigned caps)\n{\n"
	    "	JMem m;\n	m.ra = ra;\n"
	    "	u32 p = 0, q = 0, val = 0, dm = 0, res = 0;\n";
	if (bytes < sizeof (THdr)) {
		s += "	return 0;\n}\n";
		return s;
	}
	THdr h;
	memcpy(&h, blob, sizeof (h));
	const TNode *tn = (const TNode *)(blob + sizeof (THdr));
	const u8 *pool = blob + h.pool_off;
	auto pool32 = [&](u32 off) {
		u32 v;
		memcpy(&v, pool + off, 4);
		return v;
	};
	const u32 N = h.nnodes;
	std::vector<JN> nd(N);
	bool str_takes_quote = false;
	for (u32 i = 0; i < N; i++) {
		const TNode &t = tn[i];
		JN &n = nd[i];
		n.lit.assign((const char *)pool + t.lit, t.len);
		n.kind = t.kind;
		n.cap = t.cap;
		n.leaf = (t.next & TN_LEAF) != 0;
		n.leaf_mask = 0;
		if (n.leaf)
			memcpy(&n.leaf_mask, blob + h.leaf_off +
			    4 * (t.next & 0x7fff), 4);
		n.next = n.leaf ? -1 : (int)t.next;
		n.alt = t.alt == TN_NOALT ? -1 : (int)t.alt;
		n.has_disp = !n.leaf && t.disp != TN_NODISP;
		n.dk = 0;
		if (n.has_disp) {
			const u32 head = pool32(4u * t.disp);
			n.dk = head & 0xffff;
			/* (a byte listed twice: the later entry wins, as in
			 * tmpl_dispatch) */
			std::map<u32, int> ent;
			for (u32 x = 0; x < (head >> 16); x++) {
				const u32 e = pool32(4u * t.disp + 4 + 4 * x);
				ent[e & 0xff] = (int)(e >> 16);
			}
			for (auto &kv : ent)
				n.disp.push_back(kv);
		}
	}
	/* a string takes its closing quote with it */
	{
		std::vector<int> succ;
		bool okq = true;
		std::vector<char> strip(N, 0);
		for (u32 i = 0; i < N && okq; i++) {
			if (nd[i].kind != TK_STR)
				continue;
			if (nd[i].leaf) {	/* (cannot be: a string ends in '"') */
				okq = false;
				break;
			}
			successors(nd[i], succ);
			for (int c0 : succ)
				for (int c = c0; c >= 0; c = nd[c].alt) {
					if (nd[c].lit.empty() || nd[c].lit[0] != '"')
						okq = false;
					strip[c] = 1;
				}
			if (nd[i].has_disp && nd[i].dk == 0)
				okq = false;
		}
		for (u32 i = 0; i < N && okq; i++) {
			if (strip[i])
				nd[i].lit.erase(0, 1);
			if (nd[i].kind == TK_STR && nd[i].has_disp)
				nd[i].dk--;
		}
		str_takes_quote = okq;
	}
	/* do the captures along every way to a leaf add up to its mask? */
	bool accumulate = true;
	{
		std::vector<std::pair<int, u32>> stack;
		std::vector<int> succ;
		stack.push_back(std::make_pair(0, 0u));
		size_t steps = 0;
		while (!stack.empty() && accumulate && steps++ < 100000) {
			const int i = stack.back().first;
			u32 acc = stack.back().second;
			stack.pop_back();
			const JN &n = nd[i];
			if (n.alt >= 0)
				stack.push_back(std::make_pair(n.alt, acc));
			if (n.cap)
				acc |= 1u << (n.cap - 1);
			if (n.leaf) {
				if (acc != n.leaf_mask)
					accumulate = false;
				continue;
			}
			successors(n, succ);
			for (int c : succ)
				stack.push_back(std::make_pair(c, acc));
		}
		if (steps >= 100000)
			accumulate = false;
	}
	/* equivalence classes of subtrees, highest index = representative */
	std::vector<int> canon(N);
	{
		std::map<std::string, int> seen;
		std::vector<std::string> sig(N);
		for (int i = (int)N - 1; i >= 0; i--) {
			const JN &n = nd[i];
			std::string g;
			char buf[64];
			snprintf(buf, sizeof (buf), "%zu:", n.lit.size());
			g += buf;
			g += n.lit;
			snprintf(buf, sizeof (buf), "|k%u|c%u|", n.kind, n.cap);
			g += buf;
			if (n.leaf) {
				snprintf(buf, sizeof (buf), "L%x", accumulate ? 0u :
				    n.leaf_mask);
				g += buf;
			} else if (n.has_disp) {
				snprintf(buf, sizeof (buf), "D%u", n.dk);
				g += buf;
				for (auto &d : n.disp) {
					snprintf(buf, sizeof (buf), ",%u>%d", d.first,
					    canon[d.second]);
					g += buf;
				}
			} else {
				snprintf(buf, sizeof (buf), "N%d", canon[n.next]);
				g += buf;
			}
			snprintf(buf, sizeof (buf), "|a%d", n.alt < 0 ? -1 :
			    canon[n.alt]);
			g += buf;
			auto it = seen.find(g);
			if (it == seen.end()) {
				seen[g] = i;
				canon[i] = i;
			} else {
				canon[i] = it->second;
			}
		}
	}
	/* the blocks some record can reach */
	std::vector<char> live(N, 0);
	{
		std::vector<int> stack(1, canon[0]), succ;
		while (!stack.empty()) {
			const int i = stack.back();
			stack.pop_back();
			if (live[i])
				continue;
			live[i] = 1;
			if (nd[i].alt >= 0)
				stack.push_back(canon[nd[i].alt]);
			successors(nd[i], succ);
			for (int c : succ)
				stack.push_back(canon[c]);
		}
	}
	const u32 FAIL = 0xffffu, DONE = 0xfffeu;
	/* who leads to whom (over the blocks that are emitted) */
	std::vector<u32> indeg(N, 0);
	std::vector<char> alt_target(N, 0);
	{
		std::vector<int> succ;
		for (u32 i = 0; i < N; i++) {
			if (!live[i])
				continue;
			if (nd[i].alt >= 0) {
				indeg[canon[nd[i].alt]]++;
				alt_target[canon[nd[i].alt]] = 1;
			}
			successors(nd[i], succ);
			for (int c : succ)
				indeg[canon[c]]++;
		}
		indeg[canon[0]]++;
	}
	/* may block v's body follow its only predecessor's in place? */
	auto inlinable = [&](int v) {
		return indeg[v] == 1 && !alt_target[v] && nd[v].alt < 0;
	};
	std::vector<char> emitted(N, 0);
	/* the body of node i (inside a do { } while (0) that a mismatch breaks
	 * out of), then what follows it */
	std::function<void(u32, bool)> body = [&](u32 i, bool head) {
		const JN &n = nd[i];
		const u32 L = (u32)n.lit.size();
		emitted[i] = 1;
		appendf(s, "			/* node %u */\n", i);
		if (L) {
			/* (longer than the slack behind the buffer: ask) */
			if (L > 48)
				appendf(s, "			if (p + %uu > len)\n"
				    "				break;\n", L);
			s += "			{\n			const u32 a_ = ra + p, sh = (a_ & 3) * 8, "
			    "wa = a_ & ~3u;\n			u32 w0 = jlds32(wa), w1, "
			    "diff;\n";
			const u32 nw = (L + 3) / 4;
			for (u32 k = 0; k < nw; k++) {
				/* registers alternate so that no moves are needed */
				const char *lo = (k & 1) ? "w1" : "w0";
				const char *hi = (k & 1) ? "w0" : "w1";
				u32 lit = 0;
				for (u32 x = 0; x < 4 && 4 * k + x < L; x++)
					lit |= (u32)(u8)n.lit[4 * k + x] << (8 * x);
				appendf(s, "			%s = jlds32(wa + %uu);\n", hi,
				    4 * k + 4);
				s += k == 0 ? "			diff = " : "			diff |= ";
				if (k == nw - 1 && (L & 3))
					appendf(s, "(__funnelshift_r(%s, %s, sh) ^ "
					    "0x%08xu) & 0x%08xu;\n", lo, hi, lit,
					    (1u << (8 * (L & 3))) - 1);
				else
					appendf(s, "__funnelshift_r(%s, %s, sh) ^ "
					    "0x%08xu;\n", lo, hi, lit);
			}
			s += "			if (diff)\n				break;\n			}\n";
			appendf(s, "			q = p + %uu;\n", L);
		} else {
			s += "			q = p;\n";
		}
		if (n.kind == TK_STR) {
			s += "			if (!fscan_str(m, q, val))\n"
			    "				break;\n";
			if (str_takes_quote)
				s += "			q++;\n";
		} else if (n.kind == TK_BARE) {
			s += "			if (!fscan_bare(m, q, val))\n"
			    "				break;\n";
		}
		if (n.cap) {
			appendf(s, "			jsts32(caps + %uu, val);\n",
			    (u32)(n.cap - 1) * (u32)F_NT * 4u);
			if (accumulate)
				appendf(s, "			dm |= 0x%xu;\n",
				    1u << (n.cap - 1));
		}
		s += "			p = q;\n";
		if (n.leaf) {
			appendf(s, "			st = %uu;\n", DONE);
			if (accumulate)
				s += "			if (p == len)\n"
				    "				res = 1u | (dm << 1);\n";
			else
				appendf(s, "			if (p == len)\n"
				    "				res = 0x%xu;\n",
				    1u | (n.leaf_mask << 1));
		} else if (n.has_disp) {
			appendf(s, "			st = %uu;\n", FAIL);
			if (n.dk > 48)
				appendf(s, "			if (p + %uu >= len)\n"
				    "				break;\n", n.dk);
			appendf(s, "			const u32 db%u = m.byte(p + %uu);\n",
			    i, n.dk);
			for (auto &d : n.disp)
				appendf(s, "			if (db%u == %uu)\n"
				    "				st = %uu;\n", i, d.first,
				    (u32)canon[d.second]);
		} else {
			const int nx = canon[n.next];
			if (inlinable(nx) && !emitted[nx]) {
				/* (a later mismatch fails the record, whatever
				 * sibling this block had) */
				if (head && n.alt >= 0)
					appendf(s, "			st = %uu;\n", FAIL);
				body((u32)nx, false);
			} else {
				appendf(s, "			st = %uu;\n", (u32)nx);
			}
		}
	};
	appendf(s, "	u32 st = active ? %uu : %uu;\n", (u32)canon[0], FAIL);
	for (u32 i = 0; i < N; i++) {
		if (!live[i] || emitted[i])
			continue;
		const JN &n = nd[i];
		const u32 onfail = n.alt < 0 ? FAIL : (u32)canon[n.alt];
		/* every lane of the warp is here (jump threading would
		 * otherwise keep apart the lanes that arrive from different
		 * blocks, all the way to the end) */
		s += "	__syncwarp();\n";
		appendf(s, "	if (st == %uu) {\n		st = %uu;\n", i, onfail);
		/* the body runs inside do { } while (0): a mismatch breaks out
		 * with st = the alt sibling / FAIL */
		s += "		do {\n";
		body(i, true);
		s += "		} while (0);\n	}\n";
	}
	s += "	return res;\n}\n";
	return s;
}

namespace {

typedef struct _nvrtcProgram *nvrtcProgram;
typedef struct nvJitLink *nvJitLinkHandle;

struct Libs {
	void *rtc = nullptr, *jl = nullptr;
	int (*CreateProgram)(nvrtcProgram *, const char *, const char *, int,
	    const char *const *, const char *const *) = nullptr;
	int (*CompileProgram)(nvrtcProgram, int, const char *const *) = nullptr;
	int (*GetLTOIRSize)(nvrtcProgram, size_t *) = nullptr;
	int (*GetLTOIR)(nvrtcProgram, char *) = nullptr;
	int (*GetProgramLogSize)(nvrtcProgram, size_t *) = nullptr;
	int (*GetProgramLog)(nvrtcProgram, char *) = nullptr;
	int (*DestroyProgram)(nvrtcProgram *) = nullptr;
	int (*LCreate)(nvJitLinkHandle *, uint32_t, const char **) = nullptr;
	int (*LAddData)(nvJitLinkHandle, int, const void *, size_t,
	    const char *) = nullptr;
	int (*LComplete)(nvJitLinkHandle) = nullptr;
	int (*LCubinSize)(nvJitLinkHandle, size_t *) = nullptr;
	int (*LCubin)(nvJitLinkHandle, void *) = nullptr;
	int (*LErrSize)(nvJitLinkHandle, size_t *) = nullptr;
	int (*LErr)(nvJitLinkHandle, char *) = nullptr;
	int (*LDestroy)(nvJitLinkHandle *) = nullptr;
	std::string err;
	bool ok = false;
};

void *open_lib(const char *soname)
{
	/* the toolkit this library was built with first (a process may have an
	 * older copy loaded under the same soname), then the loader's choice */
	std::vector<std::string> dirs;
	if (const char *h = getenv("CUDA_HOME"))
		dirs.push_back(std::string(h) + "/lib64/");
	dirs.push_back("/usr/local/cuda/lib64/");
	dirs.push_back("");
	for (const std::string &d : dirs) {
		void *p = dlopen((d + soname).c_str(), RTLD_NOW | RTLD_LOCAL);
		if (p)
			return p;
	}
	return nullptr;
}

/* nvJitLink's entry points are versioned: __nvJitLinkCreate_12_N */
void *jl_sym(void *lib, const char *name)
{
	for (int v = 0; v <= 12; v++) {
		char buf[96];
		snprintf(buf, sizeof (buf), "__%s_12_%d", name, v);
		if (void *p = dlsym(lib, buf))
			return p;
	}
	return dlsym(lib, name);
}

Libs &libs()
{
	static Libs L;
	static std::once_flag once;
	std::call_once(once, [] {
		L.rtc = open_lib("libnvrtc.so.12");
		L.jl = open_lib("libnvJitLink.so.12");
		if (!L.rtc || !L.jl) {
			L.err = std::string("cannot load ") +
			    (!L.rtc ? "libnvrtc.so.12" : "libnvJitLink.so.12");
			return;
		}
#define RTC(field, name) \
	*(void **)&L.field = dlsym(L.rtc, name); \
	if (!L.field) { L.err = "missing " name; return; }
		RTC(CreateProgram, "nvrtcCreateProgram")
		RTC(CompileProgram, "nvrtcCompileProgram")
		RTC(GetLTOIRSize, "nvrtcGetLTOIRSize")
		RTC(GetLTOIR, "nvrtcGetLTOIR")
		RTC(GetProgramLogSize, "nvrtcGetProgramLogSize")
		RTC(GetProgramLog, "nvrtcGetProgramLog")
		RTC(DestroyProgram, "nvrtcDestroyProgram")
#undef RTC
#define JL(field, name) \
	*(void **)&L.field = jl_sym(L.jl, name); \
	if (!L.field) { L.err = "missing " name; return; }
		JL(LCreate, "nvJitLinkCreate")
		JL(LAddData, "nvJitLinkAddData")
		JL(LComplete, "nvJitLinkComplete")
		JL(LCubinSize, "nvJitLinkGetLinkedCubinSize")
		JL(LCubin, "nvJitLinkGetLinkedCubin")
		JL(LErrSize, "nvJitLinkGetErrorLogSize")
		JL(LErr, "nvJitLinkGetErrorLog")
		JL(LDestroy, "nvJitLinkDestroy")
#undef JL
		L.ok = true;
	});
	return L;
}

double now_ms()
{
	return std::chrono::duration<double, std::milli>(
	    std::chrono::steady_clock::now().time_since_epoch()).count();
}

} /* namespace */

bool jit_prepare()
{
	return libs().ok;
}

bool jit_build(const std::string &source, int nsl, std::string &cubin,
    std::string &err, double *compile_ms, double *link_ms)
{
	Libs &L = libs();
	if (!L.ok) {
		err = L.err;
		return false;
	}
	const unsigned char *hot, *hot_end;
	switch (nsl) {
	case 7: hot = dng_jit_hot7; hot_end = dng_jit_hot7_end; break;
	case 9: hot = dng_jit_hot9; hot_end = dng_jit_hot9_end; break;
	case 11: hot = dng_jit_hot11; hot_end = dng_jit_hot11_end; break;
	case 13: hot = dng_jit_hot13; hot_end = dng_jit_hot13_end; break;
	default:
		err = "no kernel for this slice size";
		return false;
	}
	/* one build at a time: two links running side by side (scans started in
	 * quick succession, each with its compiler thread) have crashed inside
	 * libnvJitLink */
	static std::mutex build_mu;
	std::lock_guard<std::mutex> build_lock(build_mu);
	const double t0 = now_ms();
	nvrtcProgram prog = nullptr;
	if (L.CreateProgram(&prog, source.c_str(), "dng_jmatch.cu", 0, nullptr,
	    nullptr) != 0) {
		err = "nvrtcCreateProgram failed";
		return false;
	}
	/* LTO-IR, within the register budget of the kernel it becomes part of
	 * (__launch_bounds__(F_NT = 896, 1): 72 registers) */
	const char *opts[] = { "-arch=sm_100a", "-rdc=true", "-dlto",
	    "-maxrregcount=72", "-std=c++17", "-lineinfo" };
	const int rc = L.CompileProgram(prog, 6, opts);
	if (rc != 0) {
		size_t n = 0;
		L.GetProgramLogSize(prog, &n);
		std::string log(n, '\0');
		if (n)
			L.GetProgramLog(prog, &log[0]);
		err = "nvrtcCompileProgram: " + log;
		L.DestroyProgram(&prog);
		return false;
	}
	size_t n = 0;
	L.GetLTOIRSize(prog, &n);
	std::string ir(n, '\0');
	L.GetLTOIR(prog, &ir[0]);
	L.DestroyProgram(&prog);
	const double t1 = now_ms();
	if (compile_ms)
		*compile_ms = t1 - t0;

	nvJitLinkHandle h = nullptr;
	const char *lopts[] = { "-arch=sm_100a", "-lto", "-maxrregcount=72",
	    "-lineinfo" };
	if (L.LCreate(&h, 4, lopts) != 0) {
		err = "nvJitLinkCreate failed";
		return false;
	}
	const int IN_CUBIN = 1, IN_LTOIR = 3, IN_FATBIN = 4;
	int lrc = L.LAddData(h, IN_FATBIN, hot, (size_t)(hot_end - hot),
	    "fast_jit");
	if (lrc == 0)
		lrc = L.LAddData(h, IN_LTOIR, ir.data(), ir.size(), "dng_jmatch");
	if (lrc == 0)
		lrc = L.LAddData(h, IN_CUBIN, dng_jit_cold,
		    (size_t)(dng_jit_cold_end - dng_jit_cold), "fast_jit_cold");
	if (lrc == 0)
		lrc = L.LComplete(h);
	if (lrc != 0) {
		size_t en = 0;
		L.LErrSize(h, &en);
		std::string log(en, '\0');
		if (en)
			L.LErr(h, &log[0]);
		err = "nvJitLink: " + log;
		L.LDestroy(&h);
		return false;
	}
	size_t cn = 0;
	L.LCubinSize(h, &cn);
	cubin.assign(cn, '\0');
	L.LCubin(h, &cubin[0]);
	L.LDestroy(&h);
	if (link_ms)
		*link_ms = now_ms() - t1;
	return true;
}

} /* namespace dng */
