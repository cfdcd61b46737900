/*
 * fdict.cpp: the value dictionary of the dense keys (fast.h FDict), learned on
 * the host by the host instantiation of the F path's own per-record code
 * (fast.cuh: fmatch, fstage, fprep, fpiece), so that a value is what the
 * kernel would put into the key, byte for byte.
 */
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "fast.cuh"

namespace dng {

namespace {

/* the lines of the head looked at: enough for a breakdown's few values (~70
 * records of the benchmark's shape see all of C5's 10 x 4 x 5), few enough to
 * keep learning cheap next to the rest of a scan's set-up -- it runs once per
 * scan, and 64 KB added 0.11 ms to every scan of the benchmark on B200's host */
constexpr size_t DICT_SAMPLE_BYTES = 16 * 1024;

} /* namespace */

bool fdict_learn(const FPlan &F, const u8 *blob, const u8 *head, size_t n,
    FDict &D)
{
	memset(&D, 0, sizeof (D));
	if (!F.ok || F.ncols == 0 || !blob)
		return false;
	for (u32 j = 0; j < F.ncols; j++)
		if (F.col[j].kind != COL_DISCRETE || F.col[j].src.kind != SRC_PATH)
			return false;
	n = std::min(n, DICT_SAMPLE_BYTES);
	const u32 nc = F.ncols;
	/* per column: value -> records; per record: its values */
	std::vector<std::map<std::string, u32>> freq(nc);
	std::vector<std::string> recs;		/* nc values per record */
	size_t nrec = 0;
	size_t pos = 0;
	while (pos < n) {
		const u8 *nl = (const u8 *)memchr(head + pos, '\n', n - pos);
		if (!nl)
			break;
		const size_t end = (size_t)(nl - head);
		const u32 len = (u32)(end - pos);
		const u8 *rec = head + pos;
		pos = end + 1;
		if (len > F_MAXLINE)
			continue;
		FastHostMem fm;
		fm.rec = rec;
		fm.len = len;
		fm.blob = blob;
		u32 defmask = 0, slow = 0;
		double s0 = 0, s1 = 0;
		if (!fmatch(fm, len, true, defmask) ||
		    fstage(fm, F, defmask, s0, s1) != FO_AGGR ||
		    !fprep(fm, F, defmask, s0, s1, slow))
			continue;
		nrec++;
		for (u32 j = 0; j < nc; j++) {
			FPiece pc;
			fpiece(fm, F, j, defmask, pc);
			const char *b = pc.kind == 0 ? (const char *)rec + pc.off :
			    F.pool + pc.off;
			std::string v(b, pc.n);
			freq[j][v]++;
			recs.push_back(v);
		}
	}
	if (nrec == 0)
		return false;
	/* per column the most frequent values that fit, then sorted by bytes:
	 * the codes depend on the head alone */
	std::vector<std::vector<std::string>> vals(nc);
	u32 total = 1;
	for (u32 j = 0; j < nc; j++) {
		std::vector<std::pair<u32, std::string>> byf;
		for (auto &kv : freq[j])
			if (kv.first.size() <= (size_t)F_DICT_BYTES)
				byf.push_back(std::make_pair(kv.second, kv.first));
		std::sort(byf.begin(), byf.end(), [](const std::pair<u32,
		    std::string> &a, const std::pair<u32, std::string> &b) {
			return a.first != b.first ? a.first > b.first :
			    a.second < b.second;
		});
		if (byf.size() > (size_t)F_DICT_VALS)
			byf.resize(F_DICT_VALS);
		for (auto &p : byf)
			vals[j].push_back(p.second);
		std::sort(vals[j].begin(), vals[j].end());
		if (vals[j].empty())
			return false;
		total *= (u32)vals[j].size();
		if (total > (u32)F_DENSE_MAX)
			return false;
	}
	size_t covered = 0;
	for (size_t r = 0; r < nrec; r++) {
		bool in = true;
		for (u32 j = 0; j < nc && in; j++)
			in = std::binary_search(vals[j].begin(), vals[j].end(),
			    recs[r * nc + j]);
		covered += in;
	}
	if (covered * 100 < nrec * 99)
		return false;
	D.ncols = nc;
	D.total = total;
	u32 stride = 1;
	for (int j = (int)nc - 1; j >= 0; j--) {
		D.n[j] = (u32)vals[j].size();
		D.stride[j] = stride;
		D.path[j] = F.col[j].src.idx;
		stride *= D.n[j];
		for (u32 c = 0; c < D.n[j]; c++) {
			D.len[j][c] = (u8)vals[j][c].size();
			memcpy(D.val[j][c], vals[j][c].data(), vals[j][c].size());
		}
	}
	return true;
}

} /* namespace dng */
