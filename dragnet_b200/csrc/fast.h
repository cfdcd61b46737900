/*
 * fast.h: the F path -- the lean first tier of the scan for templated input.
 *
 * The general kernels (scan_kernel.cuh) carry every record through a RecState
 * (32 slots + synthetic doubles, in local memory), a byte-wise key buffer and
 * the full stage code.  Almost every record of a machine-written log needs
 * none of that: it matches one of a few templates (tmpl.h), the values the
 * plan wants are plain strings or short integers, and its group key is one of
 * a handful already in the CTA's tally cache.  The F path is what is left when
 * everything else is taken out:
 *
 *   - a template trie whose captures are indexed by the plan's PATHS, not its
 *     slots: which slot supplies a dotted path (jsprim.pluck's whole-key-first
 *     precedence, lib/stream-synthetic.js:47) is a property of the template,
 *     so it is resolved when the template is built and a record only ever
 *     stores the winning value (one 32-bit word per path, in shared memory);
 *   - the stages (lib/stream-scan.js:56-86: datasource filter, user filter,
 *     synthetic dates, time bounds, group key) evaluated straight from those
 *     captures, the key hashed and compared piece by piece in place -- it is
 *     only materialised the first time a CTA sees it.
 *
 * A record the F path cannot decide EXACTLY (no template, an escaped string
 * or a container where a value is needed, a key too long ...) is a "miss":
 * it leaves no trace in the F path and is parsed by the general code
 * (parse_record and the stages of record.cuh) from the miss list, so results
 * never depend on which tier a record took.  Plans the F path does not model
 * (several metrics, json-skinner input, discrete date columns ...) are not
 * eligible and keep using the general kernels.
 */
#ifndef DNG_FAST_H
#define DNG_FAST_H

#include "plan.h"
#include "tmpl.h"

namespace dng {

enum : int {
	F_MAXPATHS = 8, F_MAXCODE = 16, F_MAXCOLS = 6, F_MAXSYN = 2,
	F_POOL = 512, F_MAXKEY = 256,
	F_MAXLINE = 4095,		/* longest line the F path matches */
	F_MAXROWS = F_MAXPATHS + 2 * F_MAXCOLS,	/* capture rows: paths, ordinals */
	F_NT = 896			/* threads of the F kernels' CTA: 28 warps,
					 * 72 registers a thread (measured against 24
					 * warps of 80: +5 % records/s) */
};

/* offsets of the constant strings every FPlan pool starts with */
enum : u16 { FC_UNDEFINED = 0, FC_NULL = 12, FC_TRUE = 16, FC_FALSE = 20,
	FC_END = 28 };

/*
 * The part of a DevPlan the F path evaluates, with sources given as PATH
 * indexes (captures) or synthetic indexes.  Same Leaf / Col layout as plan.h;
 * constants re-based into the small pool.
 */
struct alignas(16) FPlan {
	Leaf code[F_MAXCODE];
	Col col[F_MAXCOLS];
	u8 syn_path[F_MAXSYN];		/* path supplying synthetic j, 0xff = none */
	int16_t ds_entry, user_entry, time_entry;
	u8 nsyn, ncols, npaths, ok;
	u8 ord_row[F_MAXCOLS];		/* bucketized column j parks its ordinal in
					 * capture rows ord_row[j], + 1 */
	u8 nrows;			/* capture rows in all */
	u8 ncode;			/* leaves in code[]; jumps only go forward */
	u8 pad[4];
	char pool[F_POOL];
};

/*
 * Dense keys: the values the breakdown columns take in the head of the input,
 * learned per column (fdict_learn).  A record whose pieces are all in it is
 * counted at index sum_j code_j * stride[j] of a per-CTA array of u32 counters
 * instead of being hashed and probed; val[j][c] holds the bytes fkey_write()
 * would write for code c (String(value), or "null" ...), sorted by bytes.
 */
/* (24 bytes: the operation names of a web service's log, "deletepublicstorage"
 * ..., are longer than 16) */
enum : int { F_DICT_VALS = 15, F_DICT_BYTES = 24, F_DENSE_MAX = 1024 };

struct alignas(16) FDict {
	u32 ncols;			/* 0: no dictionary */
	u32 total;			/* counters: the product of n[] */
	u32 n[F_MAXCOLS];		/* values of column j */
	u32 stride[F_MAXCOLS];
	u8 path[F_MAXCOLS];		/* column j's path (capture row) */
	u8 len[F_MAXCOLS][F_DICT_VALS];
	u8 val[F_MAXCOLS][F_DICT_VALS][F_DICT_BYTES];
};

/*
 * A capture: what the matcher stores for a path of the record at hand.
 * off(12) | len(12) << 12 | type(3) << 24 | flag << 27; off is relative to the
 * record.  flag = VF_ESCAPED for strings, "simple integer" for numbers.
 */
#define DNG_FCAP(type, off, len, flag) \
	((u32)(off) | ((u32)(len) << 12) | ((u32)(type) << 24) | ((u32)(flag) << 27))

/* outcome of the stages for one record */
enum : u32 {
	FO_AGGR = 0, FO_MISS, FO_DS_FILTERED, FO_DS_FAILED, FO_USER_FILTERED,
	FO_USER_FAILED, FO_SYNTH_UNDEF, FO_SYNTH_BADDATE, FO_TIME_FILTERED,
	FO_TIME_FAILED
};

} /* namespace dng */

#include <vector>

namespace dng {

/* the F plan of a compiled plan; ok = 0 when the plan is not eligible */
void fplan_build(const DevPlan &P, FPlan &F);

/*
 * The parser's captures of a template's sample line (slot indexed) as the F
 * path wants them: path indexed, winners only.  False if the template cannot
 * be an F template (a needed path resolves to a container).
 */
bool fplan_resolve(const DevPlan &P, const TResolved &in, TResolved &out);

/*
 * The value dictionary of an F plan whose columns are all discrete with a path
 * source, from the lines of head[0, n) that the F trie `blob` (tmpl_build,
 * compact) takes to the aggregator (fdict.cpp).  False, and D.ncols = 0, unless
 * every column has at most F_DICT_VALS values of at most F_DICT_BYTES bytes
 * covering 99 % of those records, in at most F_DENSE_MAX counters.
 */
bool fdict_learn(const FPlan &F, const u8 *blob, const u8 *head, size_t n,
    FDict &D);

} /* namespace dng */

#endif
