/*
 * fast.cuh: the per-record code of the F path (fast.h): fmatch() walks the F
 * template trie for one record and stores the plan's paths as captures;
 * fstage() runs the reference's stages on them (lib/stream-scan.js:56-86:
 * datasource filter, user filter, lib/stream-synthetic.js:37-85 dates, time
 * bounds); fkey_*() hash / compare / write the record's group key
 * (lib/dragnet-impl.js:48-51, lib/dragnet.js:52-71 bucketizers) piece by piece
 * without materialising it.
 *
 * Everything here only has to be right when it says yes: whatever it cannot
 * decide exactly is reported as a miss and redone by record.cuh, whose
 * semantics (and key encoding) these functions reproduce for the value forms
 * they accept.  Host + device like record.cuh, so tests/hostcheck can run the
 * same logic against the oracle without a GPU.
 *
 * M supplies memory: the record (a '\n' follows its last byte), the trie blob,
 * the record's captures.
 */
#ifndef DNG_FAST_CUH
#define DNG_FAST_CUH

#include "fast.h"
#include "tmpl.cuh"

/*
 * Loops over the plan (its three filters, its synthetic fields, its columns):
 * rolled up in the ahead-of-time build, where the plan is data and unrolling
 * only multiplies the interpretive code; fully unrolled in the link-time
 * optimised build (fast_jit.cu), where the plan is a constant and every
 * iteration folds to the few instructions its column or filter needs.
 */
#ifdef DNG_JIT_HOT
#define DNG_PLAN_LOOP _Pragma("unroll")
#else
#define DNG_PLAN_LOOP _Pragma("unroll 1")
#endif

namespace dng {

#include "fscan.cuh"		/* (includes nothing: lives in this namespace) */

DNG_HD u32 fcap_off(u32 c) { return c & 0xfff; }
DNG_HD u32 fcap_len(u32 c) { return (c >> 12) & 0xfff; }
DNG_HD u32 fcap_type(u32 c) { return (c >> 24) & 7; }
DNG_HD u32 fcap_flag(u32 c) { return c >> 27; }

/*
 * Match one record against the F trie.  Same trie format and the same walk as
 * tmpl_match() (tmpl.cuh) with two differences: literals are plain words
 * (tmpl_build's compact pool: no per-word masks, only the last word of a
 * literal is masked), and a node's `cap` is 1 + the PATH its wildcard
 * supplies.  On success *defmask = the paths this template defines.
 * Every lane of the warp must call this (active = false without a record).
 */
template <class M>
DNG_HD bool fmatch(M &m, u32 len, bool active, u32 &defmask)
{
	u32 p = 0;
	bool matched = false;
	TQuad nd = m.node(0);
	while (DNG_WARP_ANY(active)) {
		if (active) {
			/* the likely successor is fetched while this node is matched */
			const u32 succ = nd.y & 0xffff;
			const TQuad nx = m.node(succ & TN_LEAF ? 0 : succ);
			const u32 lit = nd.x & 0xffff, L = nd.x >> 16;
			bool ok = p + L <= len;
			if (ok && L) {
				typename M::Cur c = m.cursor(p);
				u32 diff = 0;
				const u32 nfull = L >> 2;
				/* (short, warp-uniform trip counts: rolled up, the
				 * loop is a dozen instructions instead of pages of
				 * unrolled stages to branch through) */
#pragma unroll 1
				for (u32 k = 0; k < nfull; k++)
					diff |= c.next() ^ m.litw(lit + 4 * k);
				if (L & 3)
					diff |= (c.next() ^ m.litw(lit + 4 * nfull)) &
					    ((1u << (8 * (L & 3))) - 1);
				ok = diff == 0;
			}
			u32 q = p + L;
			u32 val = 0;
			const u32 kind = nd.z & 0xff;
			if (ok && kind == TK_STR)
				ok = fscan_str(m, q, val);
			else if (ok && kind == TK_BARE)
				ok = fscan_bare(m, q, val);
			if (!ok) {
				const u32 alt = nd.y >> 16;
				active = alt != TN_NOALT;
				nd = m.node(active ? alt : 0);
			} else {
				const u32 cap = (nd.z >> 8) & 0xff;
				if (cap)
					m.setcap(cap - 1, val);
				p = q;
				const u32 disp = nd.w >> 16;
				if (succ & TN_LEAF) {
					active = false;
					if (p == len) {
						defmask = m.leaf(succ & 0x7fff);
						matched = true;
					}
				} else if (disp != TN_NODISP) {
					const u32 ch = tmpl_dispatch(m, disp, p, len);
					active = ch != TN_NOALT;
					nd = m.node(active ? ch : 0);
				} else {
					nd = nx;
				}
			}
		}
	}
	return matched;
}

/* [-]digits (a "simple integer" capture: at most 15 of them) as a double */
template <class M>
DNG_HD double fsimple_int(M &m, u32 off, u32 n)
{
	const u32 neg = m.byte(off) == '-';
	u32 i = neg, hi = 0, lo = 0;
	/* the first nine digits and the rest, 32 bits each: every product and
	 * sum below is an integer < 2^53, exact in binary64 */
	const u32 split = n - i > 9 ? i + 9 : n;
#pragma unroll 1
	for (; i < split; i++)
		hi = hi * 10 + (m.byte(off + i) - '0');
	double d = (double)hi;
#pragma unroll 1
	for (; i < n; i++) {
		lo = lo * 10 + (m.byte(off + i) - '0');
		d *= 10.0;
	}
	d += (double)lo;
	return neg ? -d : d;
}

/* ToNumber of a capture (not an escaped string / container) */
template <class M>
DNG_HD double fnumber(M &m, u32 cw)
{
	const u32 t = fcap_type(cw), off = fcap_off(cw), n = fcap_len(cw);
	switch (t) {
	case T_TRUE:
		return 1.0;
	case T_NUM:
		if (fcap_flag(cw))
			return fsimple_int(m, off, n);
		return dng_parse_decimal(m.ptr(off), (int)n);
	case T_STR:
		return dng_string_to_number(m.ptr(off), (int)n);
	default:
		return 0.0;		/* null, false */
	}
}

/* record bytes [off, off + n) == pool bytes at coff (4-byte aligned, zero
 * padded)? */
template <class M>
DNG_HD bool fbytes_equal(M &m, u32 off, const char *cst, u32 n)
{
	typename M::Cur c = m.cursor(off);
	const u32 *cw = (const u32 *)cst;
	u32 diff = 0;
	const u32 nfull = n >> 2;
	for (u32 k = 0; k < nfull; k++)
		diff |= c.next() ^ cw[k];
	if (n & 3)
		diff |= (c.next() ^ cw[nfull]) & ((1u << (8 * (n & 3))) - 1);
	return diff == 0;
}

/* one krill leaf (record.cuh eval_leaf): 1 true, 0 false, -1 evaluation
 * failed; miss is set when the value's form is not the F path's to decide */
template <class M>
DNG_HD int feval_leaf(M &m, const FPlan &F, const Leaf &lf, u32 defmask,
    double s0, double s1, bool &miss)
{
	if (lf.op == OP_TRUE)
		return 1;
	u32 cw = 0, t;
	double x = 0;
	bool havenum = false;
	if (lf.src.kind == SRC_SYNTH) {
		t = T_NUM;
		x = lf.src.idx ? s1 : s0;
		havenum = true;
	} else if (lf.src.kind == SRC_PATH && ((defmask >> lf.src.idx) & 1)) {
		cw = m.getcap(lf.src.idx);
		t = fcap_type(cw);
	} else {
		return -1;
	}
	const u32 off = fcap_off(cw), n = fcap_len(cw);
	const bool str = t == T_STR;
	if ((str && fcap_flag(cw)) || t == T_OBJ || t == T_ARR) {
		miss = true;
		return 0;
	}
	const char *cst = F.pool + lf.coff;
	if (lf.op == OP_EQ || lf.op == OP_NE) {
		int eq;
		if (t == T_NULL) {
			eq = 0;
		} else if (str && lf.cstr) {
			eq = n == lf.clen && fbytes_equal(m, off, cst, n);
		} else {
			if (!havenum)
				x = fnumber(m, cw);
			eq = x == lf.cnum;
		}
		return lf.op == OP_EQ ? eq : !eq;
	}
	if (str && lf.cstr) {
		const int c = utf16_cmp(m.ptr(off), n, (const u8 *)cst, lf.clen);
		switch (lf.op) {
		case OP_LT: return c < 0;
		case OP_LE: return c <= 0;
		case OP_GT: return c > 0;
		default: return c >= 0;
		}
	}
	if (!havenum)
		x = fnumber(m, cw);
	const double y = lf.cnum;
	switch (lf.op) {
	case OP_LT: return x < y;
	case OP_LE: return x <= y;
	case OP_GT: return x > y;
	default: return x >= y;
	}
}

/* a filter program (record.cuh eval_program): 1 pass, 0 filtered out, -1
 * failed */
template <class M>
DNG_HD int feval(M &m, const FPlan &F, int entry, u32 defmask, double s0,
    double s1, bool &miss)
{
	int pc = entry;
#ifdef DNG_JIT_HOT
	/* the plan is a constant here: one block per leaf, in order (jumps
	 * only go forward), each folded down to its own comparison */
#pragma unroll
	for (int i = 0; i < F_MAXCODE; i++) {
		if (i >= (int)F.ncode || pc != i)
			continue;
		const Leaf &lf = F.code[i];
		const int r = feval_leaf(m, F, lf, defmask, s0, s1, miss);
		if (miss)
			return 0;
		if (r < 0)
			return -1;
		pc = r ? lf.jt : lf.jf;
	}
#else
	while (pc >= 0) {
		const Leaf &lf = F.code[pc];
		const int r = feval_leaf(m, F, lf, defmask, s0, s1, miss);
		if (miss)
			return 0;
		if (r < 0)
			return -1;
		pc = r ? lf.jt : lf.jf;
	}
#endif
	return pc == -1;
}

/*
 * "YYYY-MM-DDTHH:MM:SS.mmmZ" (what machine-written logs carry) without the
 * general parser; anything else goes through dng_date_parse().
 */
template <class M>
DNG_HD bool fdate(M &m, u32 off, u32 n, int64_t *ms)
{
	if (n == 24) {
		typename M::Cur c = m.cursor(off);
		const u32 w0 = c.next(), w1 = c.next(), w2 = c.next();
		const u32 w3 = c.next(), w4 = c.next(), w5 = c.next();
		/* digits where digits belong, punctuation in between */
		const u32 nd = nondigit_mask(w0) |
		    nondigit_mask((w1 & 0x00ffff00u) | 0x30000030u) |
		    nondigit_mask((w2 & 0xff00ffffu) | 0x00300000u) |
		    nondigit_mask((w3 & 0xffff00ffu) | 0x00003000u) |
		    nondigit_mask((w4 & 0x00ffff00u) | 0x30000030u) |
		    nondigit_mask((w5 & 0x00ffffffu) | 0x30000000u);
		const bool punct = (w1 & 0xff0000ffu) == 0x2d00002du &&	/* - - */
		    (w2 & 0x00ff0000u) == 0x00540000u &&		/* T */
		    (w3 & 0x0000ff00u) == 0x00003a00u &&		/* : */
		    (w4 & 0xff0000ffu) == 0x2e00003au &&		/* : . */
		    (w5 >> 24) == 'Z';
		if (!nd && punct) {
#define DNG_D(w, k) ((int)(((w) >> (8 * (k))) & 0xf))
			const int y = DNG_D(w0, 0) * 1000 + DNG_D(w0, 1) * 100 +
			    DNG_D(w0, 2) * 10 + DNG_D(w0, 3);
			const int mo = DNG_D(w1, 1) * 10 + DNG_D(w1, 2);
			const int dd = DNG_D(w2, 0) * 10 + DNG_D(w2, 1);
			const int hh = DNG_D(w2, 3) * 10 + DNG_D(w3, 0);
			const int mi = DNG_D(w3, 2) * 10 + DNG_D(w3, 3);
			const int ss = DNG_D(w4, 1) * 10 + DNG_D(w4, 2);
			const int msec = DNG_D(w5, 0) * 100 + DNG_D(w5, 1) * 10 +
			    DNG_D(w5, 2);
#undef DNG_D
			if (mo >= 1 && mo <= 12 && dd >= 1 && dd <= 31 &&
			    hh <= 23 && mi <= 59 && ss <= 59) {
				*ms = (int64_t)days_from_civil(y, mo, dd) *
				    86400000ll + (int64_t)(((hh * 60 + mi) * 60 +
				    ss) * 1000 + msec);
				return true;
			}
		}
	}
	return dng_date_parse(m.ptr(off), (int)n, ms);
}

/*
 * The stages in front of the aggregator for a matched record.  Returns the
 * record's fate (FO_*); FO_AGGR means its group key is to be counted.  s0/s1
 * receive the synthetic fields.  Nothing is counted here: the caller bumps
 * the counter the outcome names, so a miss leaves no trace.
 */
template <class M>
DNG_HD u32 fstage(M &m, const FPlan &F, u32 defmask, double &s0, double &s1)
{
	bool miss = false;
	s0 = s1 = 0;
	/* datasource filter, user filter, [dates,] time filter: one copy of
	 * the evaluator for the three */
DNG_PLAN_LOOP
	for (u32 k = 0; k < 3; k++) {
		if (k == 2 && F.nsyn) {
			/* lib/stream-synthetic.js:37-85: only the first error
			 * of a record is counted, but every field is looked at */
			u32 err = 0;
DNG_PLAN_LOOP
			for (u32 j = 0; j < F.nsyn; j++) {
				const u32 pi = F.syn_path[j];
				double v = 0;
				u32 e = 0;
				if (pi == 0xff || !((defmask >> pi) & 1)) {
					e = FO_SYNTH_UNDEF;
				} else {
					const u32 cw = m.getcap(pi);
					const u32 t = fcap_type(cw);
					if (t == T_NUM) {
						v = fnumber(m, cw);
					} else if (t == T_STR) {
						if (fcap_flag(cw))
							return FO_MISS;
						int64_t ms = 0;
						if (fdate(m, fcap_off(cw), fcap_len(cw),
						    &ms))
							v = floor((double)ms / 1000.0);
						else if (dng_date_maybe_legacy(m.ptr(
						    fcap_off(cw)), (int)fcap_len(cw)))
							return FO_MISS;	/* (jsdate.cuh) */
						else
							e = FO_SYNTH_BADDATE;
					} else if (t == T_OBJ || t == T_ARR) {
						return FO_MISS;
					} else {
						e = FO_SYNTH_BADDATE;
					}
				}
				if (e && !err)
					err = e;
				if (j == 0)
					s0 = v;
				else
					s1 = v;
			}
			if (err)
				return err;
		}
		const int entry = k == 0 ? F.ds_entry : k == 1 ? F.user_entry :
		    F.time_entry;
		if (entry < 0)
			continue;
		const int r = feval(m, F, entry, defmask, s0, s1, miss);
		if (miss)
			return FO_MISS;
		if (r <= 0) {
			const u32 base = k == 0 ? FO_DS_FILTERED : k == 1 ?
			    FO_USER_FILTERED : FO_TIME_FILTERED;
			return base + (r < 0);
		}
	}
	return FO_AGGR;
}

/*
 * The group key (record.cuh process_metric's encoding), column by column:
 * discrete = u16 length + the bytes of String(value), taken from the record
 * or from the plan's constants; bucketized = 0xFFFF + the ordinal's binary64.
 *
 * fprep() looks at every column once: false = the F path does not build this
 * key (miss).  Ordinals are computed here and parked in two capture rows of
 * their own (FPlan::ord_row), so that hashing, comparing and writing the key
 * are cheap, cannot fail and agree with each other.
 */
template <class M>
DNG_HD bool fprep(M &m, const FPlan &F, u32 defmask, double s0, double s1,
    u32 &slow)
{
DNG_PLAN_LOOP
	for (u32 j = 0; j < F.ncols; j++) {
		const Col &col = F.col[j];
		u32 cw = DNG_FCAP(T_UNDEF, 0, 0, 0);
		const bool synth = col.src.kind == SRC_SYNTH;
		if (col.src.kind == SRC_PATH && ((defmask >> col.src.idx) & 1))
			cw = m.getcap(col.src.idx);
		const u32 t = fcap_type(cw);
		if (t == T_OBJ || t == T_ARR || (t == T_STR && fcap_flag(cw)))
			return false;
		if (col.kind == COL_DISCRETE) {
			/* Number::toString of anything but a plain integer, and
			 * of a date: the general path */
			if (synth || (t == T_NUM && !fcap_flag(cw)))
				return false;
			continue;
		}
		double x;
		if (synth) {
			x = col.src.idx ? s1 : s0;
		} else if (t == T_UNDEF) {
			x = dng_nan();
		} else {
			if (t == T_STR)
				slow = 1;	/* (as value_to_number counts it) */
			x = fnumber(m, cw);
		}
		const double ord = col.kind == COL_P2 ? p2_ordinal(x) :
		    linear_ordinal(x, col.step);
		const u64 b = ord != ord ? 0x7ff8000000000000ull :
		    double_to_bits(ord);
		m.setcap(F.ord_row[j], (u32)b);
		m.setcap(F.ord_row[j] + 1u, (u32)(b >> 32));
	}
	return true;
}

struct FPiece {
	u32 kind;		/* 0 record bytes, 1 pool constant, 2 ordinal */
	u32 off, n;		/* kind 0/1 */
	u32 lo, hi;		/* kind 2 */
};

/* column j's piece of the key, after fprep() said yes */
template <class M>
DNG_HD void fpiece(M &m, const FPlan &F, u32 j, u32 defmask, FPiece &pc)
{
	const Col &col = F.col[j];
	pc.lo = pc.hi = pc.off = pc.n = 0;
	if (col.kind != COL_DISCRETE) {
		pc.kind = 2;
		pc.lo = m.getcap(F.ord_row[j]);
		pc.hi = m.getcap(F.ord_row[j] + 1u);
		return;
	}
	u32 cw = DNG_FCAP(T_UNDEF, 0, 0, 0);
	if (col.src.kind == SRC_PATH && ((defmask >> col.src.idx) & 1))
		cw = m.getcap(col.src.idx);
	const u32 t = fcap_type(cw);
	if (t == T_STR || t == T_NUM) {
		pc.kind = 0;
		pc.off = fcap_off(cw);
		pc.n = fcap_len(cw);
		return;
	}
	pc.kind = 1;
	pc.off = t == T_UNDEF ? FC_UNDEFINED : t == T_NULL ? FC_NULL :
	    t == T_TRUE ? FC_TRUE : FC_FALSE;
	pc.n = t == T_UNDEF ? 9 : t == T_FALSE ? 5 : 4;
}

DNG_HD u32 fmix(u32 h, u32 w)
{
	h = (h ^ w) * 0x9E3779B1u;
	return h ^ (h >> 15);
}

/* a piece's bytes as words from its start (the last one zero padded): the
 * record through a cursor, constants straight from the 4-byte aligned pool */
template <class M>
struct FWords {
	typename M::Cur c;
	const u32 *cw;
	u32 left;
	bool rec;
	DNG_HD FWords(M &m, const FPlan &F, const FPiece &pc, u32 skip)
	{
		rec = pc.kind == 0;
		left = pc.n - skip;
		cw = (const u32 *)(F.pool + pc.off);
		c = m.cursor(rec ? pc.off + skip : 0);
	}
	/* (constants are only ever read from their start: skip = 0) */
	DNG_HD u32 next()
	{
		u32 w = rec ? c.next() : *cw++;
		if (left < 4)
			w &= (1u << (8 * left)) - 1;
		left -= left < 4 ? left : 4;
		return w;
	}
};

/*
 * Hash and length of the record's group key (false: longer than the F path
 * carries).  The hash is a function of the key's content only (lengths,
 * bytes, ordinals), so equal keys hash alike whatever record they come from.
 */
template <class M>
DNG_HD bool fkey_hash(M &m, const FPlan &F, u32 defmask, u32 &hash, u32 &klen)
{
	u32 h = 0x2545F491u, kl = 0;
DNG_PLAN_LOOP
	for (u32 j = 0; j < F.ncols; j++) {
		FPiece pc;
		fpiece(m, F, j, defmask, pc);
		if (pc.kind == 2) {
			h = fmix(fmix(fmix(h, 0xffff0000u), pc.lo), pc.hi);
			kl += 10;
			continue;
		}
		h = fmix(h, pc.n);
		FWords<M> ws(m, F, pc, 0);
#pragma unroll 1
		for (u32 k = 0; k < pc.n; k += 4)
			h = fmix(h, ws.next());
		kl += 2 + pc.n;
	}
	h ^= h >> 16;
	h *= 0x85ebca6bu;
	h ^= h >> 13;
	hash = h;
	klen = kl;
	return kl <= F_MAXKEY;
}

/* byte i of a discrete piece */
template <class M>
DNG_HD u32 fpiece_byte(M &m, const FPlan &F, const FPiece &pc, u32 i)
{
	return pc.kind == 0 ? m.byte(pc.off + i) : (u32)(u8)F.pool[pc.off + i];
}

/*
 * Is the stored key K (its bytes through K.cursor(offset).next(), any
 * alignment) this record's key?  The caller has compared the lengths.
 */
template <class M, class K>
DNG_HD bool fkey_equal(M &m, const FPlan &F, u32 defmask, K &k)
{
	u32 o = 0, diff = 0;
DNG_PLAN_LOOP
	for (u32 j = 0; j < F.ncols; j++) {
		FPiece pc;
		fpiece(m, F, j, defmask, pc);
		typename K::Cur kc = k.cursor(o);
		if (pc.kind == 2) {
			const u32 a = kc.next(), b = kc.next(), c = kc.next();
			diff |= (a ^ (0xffffu | (pc.lo << 16))) |
			    (b ^ ((pc.lo >> 16) | (pc.hi << 16))) |
			    ((c ^ (pc.hi >> 16)) & 0xffffu);
			o += 10;
			continue;
		}
		/* u16 length, then the bytes: the first word holds two of them */
		const u32 n = pc.n;
		u32 first = n;
		if (n > 0)
			first |= fpiece_byte(m, F, pc, 0) << 16;
		if (n > 1)
			first |= fpiece_byte(m, F, pc, 1) << 24;
		const u32 fm = n >= 2 ? ~0u : n == 1 ? 0x00ffffffu : 0x0000ffffu;
		diff |= (kc.next() ^ first) & fm;
		if (n > 2) {
			if (pc.kind == 0) {
				FWords<M> ws(m, F, pc, 2);
				const u32 r = n - 2;
#pragma unroll 1
				for (u32 i = 0; i < r; i += 4) {
					const u32 mk = i + 4 <= r ? ~0u :
					    (1u << (8 * (r & 3))) - 1;
					diff |= (kc.next() ^ ws.next()) & mk;
				}
			} else {
				/* constants ("undefined", "false", ...) */
				const u32 r = n - 2;
#pragma unroll 1
				for (u32 i = 0; i < r; i += 4) {
					u32 w = 0;
					for (u32 x = 0; x < 4 && i + x < r; x++)
						w |= fpiece_byte(m, F, pc, 2 + i + x)
						    << (8 * x);
					const u32 mk = i + 4 <= r ? ~0u :
					    (1u << (8 * (r & 3))) - 1;
					diff |= (kc.next() ^ w) & mk;
				}
			}
		}
		o += 2 + n;
	}
	return diff == 0;
}

/* a discrete piece of the key at out + o: u16 length, then byte(k), k < n;
 * returns the offset after it */
template <class B>
DNG_HD u32 fkey_put(u8 *out, u32 o, u32 n, const B &byte)
{
	out[o] = (u8)n;
	out[o + 1] = (u8)(n >> 8);
#pragma unroll 1
	for (u32 k = 0; k < n; k++)
		out[o + 2 + k] = (u8)byte(k);
	return o + 2 + n;
}

/* zero padding to a multiple of 8 */
DNG_HD void fkey_pad(u8 *out, u32 o)
{
	while (o & 7)
		out[o++] = 0;
}

template <class M>
struct FPieceBytes {
	M *m;
	const FPlan *F;
	const FPiece *pc;
	DNG_HD u32 operator()(u32 k) const { return fpiece_byte(*m, *F, *pc, k); }
};

/* the key's bytes (record.cuh process_metric's encoding), zero padded to a
 * multiple of 8; out has room for F_MAXKEY + 8 */
template <class M>
DNG_HD void fkey_write(M &m, const FPlan &F, u32 defmask, u8 *out)
{
	u32 o = 0;
DNG_PLAN_LOOP
	for (u32 j = 0; j < F.ncols; j++) {
		FPiece pc;
		fpiece(m, F, j, defmask, pc);
		if (pc.kind == 2) {
			out[o] = 0xff;
			out[o + 1] = 0xff;
			for (u32 k = 0; k < 4; k++) {
				out[o + 2 + k] = (u8)(pc.lo >> (8 * k));
				out[o + 6 + k] = (u8)(pc.hi >> (8 * k));
			}
			o += 10;
			continue;
		}
		FPieceBytes<M> b;
		b.m = &m;
		b.F = &F;
		b.pc = &pc;
		o = fkey_put(out, o, pc.n, b);
	}
	fkey_pad(out, o);
}

struct FDictBytes {
	const u8 *v;
	DNG_HD u32 operator()(u32 k) const { return v[k]; }
};

/* the key of dense counter `idx` (FDict) as fkey_write() writes it: the
 * dictionary values of its codes; returns the key's length */
DNG_HD u32 fdense_key(const FDict &D, u32 idx, u8 *out)
{
	u32 o = 0;
	for (u32 j = 0; j < D.ncols; j++) {
		const u32 c = idx / D.stride[j] % D.n[j];
		FDictBytes b;
		b.v = D.val[j][c];
		o = fkey_put(out, o, D.len[j][c], b);
	}
	fkey_pad(out, o);
	return o;
}

#ifndef __CUDACC__
/* host access (tests/hostcheck only) */
struct FastHostMem : TmplHostMem {
	u32 caps[F_MAXROWS];
	const u8 *ptr(u32 off) const { return rec + off; }
	u32 litw(u32 off) const { return pool32(off); }
	void setcap(u32 p, u32 v) { caps[p] = v; }
	u32 getcap(u32 p) const { return caps[p]; }
};
struct FastHostKey {
	const u8 *key;
	u32 len;
	struct Cur {
		const FastHostKey *k;
		u32 off;
		u32 next() {
			u32 w = 0;
			for (u32 x = 0; x < 4; x++)
				if (off + x < k->len)
					w |= (u32)k->key[off + x] << (8 * x);
			off += 4;
			return w;
		}
	};
	Cur cursor(u32 off) const { Cur c; c.k = this; c.off = off; return c; }
};
#endif

} /* namespace dng */
#endif
