/*
 * densecheck: TEST-ONLY host check of the dense keys (fast.h FDict) without a
 * GPU.  Not part of libdragnet_gpu.so.
 *
 *   densecheck PLAN.json LEARN_FILE DATA_FILE [device]
 *
 * Learns the F templates of DATA_FILE's head and the value dictionary of
 * LEARN_FILE's head (fdict_learn), generates dng_jmatch() and dng_jcode() with
 * that dictionary (jit.cpp), compiles them for the host and, for every record
 * of DATA_FILE the F path counts, checks
 *   - dng_jcode() against the dictionary looked up from fpiece()'s bytes;
 *   - the key fdense_key() rebuilds for that counter against fkey_write().
 * With `device`, the same source must also build and link for sm_100a
 * (DNG_DENSECHECK_DUMP=PREFIX writes PREFIX.cu and PREFIX.cubin).
 * Prints one JSON line: records counted, dense hits, dictionary size.
 */
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include <dlfcn.h>
#include <unistd.h>

#include "../../dragnet_b200/csrc/record.cuh"
#include "../../dragnet_b200/csrc/tmpl.cuh"
#include "../../dragnet_b200/csrc/fast.cuh"
#include "../../dragnet_b200/csrc/jit.h"
#include "../../include/dragnet_gpu.h"

using namespace dng;

/* the generated code's device accessors on a byte array (as in hostcheck) */
static const char *HOST_PRELUDE =
"#include <stdint.h>\n#include <string.h>\n"
"typedef uint8_t u8; typedef uint32_t u32; typedef uint64_t u64;\n"
"#define DNG_HD static inline\n#define __device__\n#define __syncwarp()\n"
"enum { T_UNDEF = 0, T_NULL = 1, T_FALSE = 2, T_TRUE = 3, T_NUM = 4, T_STR = 5 };\n"
"#define DNG_FCAP(type, off, len, flag) \\\n"
"	((u32)(off) | ((u32)(len) << 12) | ((u32)(type) << 24) | ((u32)(flag) << 27))\n"
"DNG_HD bool is_hex(u32 c) { return (c >= '0' && c <= '9') || ((c | 0x20) >= 'a' && (c | 0x20) <= 'f'); }\n"
"DNG_HD u32 tm_isdigit(u32 c) { return c - '0' <= 9u; }\n"
"DNG_HD u32 nondigit_mask(u32 w) { const u32 x = w ^ 0x30303030u; return (((x & 0x7f7f7f7fu) + 0x76767676u) | x) & 0x80808080u; }\n"
"DNG_HD u32 low_flag_byte(u32 m) { u32 k = 0; while (!((m >> (8 * k + 7)) & 1)) k++; return k; }\n"
"extern \"C\" unsigned char *dng_jit_host_mem;\nunsigned char *dng_jit_host_mem;\n"
"DNG_HD u32 jlds32(u32 a) { u32 v; memcpy(&v, dng_jit_host_mem + a, 4); return v; }\n"
"DNG_HD u32 jlds8(u32 a) { return dng_jit_host_mem[a]; }\n"
"DNG_HD void jsts32(u32 a, u32 v) { memcpy(dng_jit_host_mem + a, &v, 4); }\n"
"DNG_HD u32 __funnelshift_r(u32 lo, u32 hi, u32 sh) { return sh ? (lo >> sh) | (hi << (32 - sh)) : lo; }\n"
"struct JMem {\n	u32 ra;\n	struct Cur { u32 wa, w0, w1, sh;\n"
"		u32 next() { const u32 d = __funnelshift_r(w0, w1, sh); w0 = w1; wa += 4; w1 = jlds32(wa); return d; } };\n"
"	Cur cursor(u32 off) const { Cur c; const u32 a = ra + off; c.sh = (a & 3) * 8; c.wa = (a & ~3u) + 4;\n"
"		c.w0 = jlds32(c.wa - 4); c.w1 = jlds32(c.wa); return c; }\n"
"	struct ACur { u32 wa, k; u32 next() { const u32 v = jlds32(wa); wa += 4; return v; } };\n"
"	ACur acursor(u32 off) const { ACur c; const u32 a = ra + off; c.k = a & 3; c.wa = a & ~3u; return c; }\n"
"	u32 apos(const ACur &c) const { return c.wa - 4 - ra; }\n"
"	u32 byte(u32 off) const { return jlds8(ra + off); }\n"
"	u32 word(u32 off) const { Cur c = cursor(off); return c.next(); }\n};\n";

typedef unsigned (*jmatch_fn)(unsigned, unsigned, unsigned, unsigned);
typedef unsigned (*jcode_fn)(unsigned, unsigned, unsigned);

static std::string slurp(const char *path)
{
	std::ifstream f(path, std::ios::binary);
	std::stringstream ss;
	ss << f.rdbuf();
	return ss.str();
}

/* the F trie of a head, as api.cu learns it (the parser on the host) */
static std::vector<u8> ftemplates(const dng_plan &plan, const std::string &d)
{
	std::vector<TCandidate> cands;
	tmpl_candidates((const u8 *)d.data(), std::min<size_t>(d.size(),
	    TMPL_SAMPLE_BYTES), TMPL_MAX_LEAVES, cands);
	std::vector<TResolved> res(cands.size());
	for (size_t i = 0; i < cands.size(); i++) {
		static RecState R;
		TResolved r0;
		parse_record((const u8 *)cands[i].sample.data(),
		    (u32)cands[i].sample.size(), plan.dev, R);
		r0.flags = R.flags;
		r0.set_mask = R.set_mask;
		memcpy(r0.slots, R.slots, sizeof (R.slots));
		fplan_resolve(plan.dev, r0, res[i]);
	}
	std::vector<u8> blob;
	tmpl_build(cands, res, 60000, blob, nullptr, true);
	return blob;
}

int main(int argc, char **argv)
{
	if (argc < 4) {
		fprintf(stderr, "usage: densecheck PLAN.json LEARN DATA [device]\n");
		return 2;
	}
	static dng_plan plan;
	char err[256];
	if (dng_plan_compile(slurp(argv[1]).c_str(), &plan, err, sizeof (err))) {
		fprintf(stderr, "plan: %s\n", err);
		return 1;
	}
	static FPlan FP;
	fplan_build(plan.dev, FP);
	const std::string learn = slurp(argv[2]), data = slurp(argv[3]);
	const std::vector<u8> lblob = ftemplates(plan, learn);
	const std::vector<u8> fblob = ftemplates(plan, data);
	static FDict D;
	if (!FP.ok || lblob.empty() || fblob.empty() ||
	    !fdict_learn(FP, lblob.data(), (const u8 *)learn.data(),
	    std::min<size_t>(learn.size(), TMPL_SAMPLE_BYTES), D)) {
		printf("{\"dict\":0}\n");
		return 0;
	}
	if (argc > 4) {
		std::string cubin, e;
		double cms = 0, lms = 0;
		const std::string dev = jit_source(fblob.data(), fblob.size(), &FP,
		    nullptr, &D);
		if (dev.find("dng_jdense = 0u") != std::string::npos) {
			fprintf(stderr, "device source without dense keys\n");
			return 3;
		}
		if (!jit_build(dev, 13, cubin, e, &cms, &lms)) {
			fprintf(stderr, "jit_build: %s\n", e.c_str());
			return 4;
		}
		fprintf(stderr, "jit: nvrtc %.0f ms, link %.0f ms, cubin %zu bytes\n",
		    cms, lms, cubin.size());
		/* DNG_DENSECHECK_DUMP=PREFIX: the source and the linked kernel */
		if (const char *dump = getenv("DNG_DENSECHECK_DUMP")) {
			FILE *d1 = fopen((std::string(dump) + ".cu").c_str(), "w");
			FILE *d2 = fopen((std::string(dump) + ".cubin").c_str(), "w");
			if (d1 && d2) {
				fwrite(dev.data(), 1, dev.size(), d1);
				fwrite(cubin.data(), 1, cubin.size(), d2);
			}
			if (d1)
				fclose(d1);
			if (d2)
				fclose(d2);
		}
	}
	const std::string host = jit_source(fblob.data(), fblob.size(), nullptr,
	    HOST_PRELUDE, &D);
	char dir[] = "/tmp/dng_dense_XXXXXX";
	if (!mkdtemp(dir))
		return 4;
	const std::string src = std::string(dir) + "/jc.cpp";
	const std::string so = std::string(dir) + "/jc.so";
	FILE *f = fopen(src.c_str(), "w");
	fwrite(host.data(), 1, host.size(), f);
	fclose(f);
	const std::string cmd = "g++ -std=c++17 -O1 -w -shared -fPIC -o " + so +
	    " " + src;
	if (system(cmd.c_str()) != 0) {
		fprintf(stderr, "host build of the generated code failed\n");
		return 4;
	}
	void *h = dlopen(so.c_str(), RTLD_NOW);
	unlink(src.c_str());
	unlink(so.c_str());
	rmdir(dir);
	if (!h)
		return 4;
	unsigned char **jmem = (unsigned char **)dlsym(h, "dng_jit_host_mem");
	jmatch_fn jm = (jmatch_fn)dlsym(h, "dng_jmatch");
	jcode_fn jc = (jcode_fn)dlsym(h, "dng_jcode");
	if (!jmem || !jm || !jc)
		return 4;
	static unsigned char jbuf[65536];
	*jmem = jbuf;

	unsigned long nrec = 0, ndense = 0;
	size_t pos = 0;
	while (pos < data.size()) {
		const size_t nl = data.find('\n', pos);
		if (nl == std::string::npos)
			break;
		const u32 len = (u32)(nl - pos);
		const u8 *rec = (const u8 *)data.data() + pos;
		pos = nl + 1;
		if (len > 4095)
			continue;
		/* the record at an odd address, '\n' and the sentinel quotes
		 * after it, captures in rows of F_NT */
		const u32 ra = 1027, caps = 32768;
		memcpy(jbuf + ra, rec, len);
		jbuf[ra + len] = '\n';
		memset(jbuf + ra + len + 1, '"', 64);
		const unsigned r = jm(ra, len, 1, caps);
		if (!(r & 1))
			continue;
		FastHostMem fm;
		fm.rec = rec;
		fm.len = len;
		fm.blob = fblob.data();
		const u32 defmask = r >> 1;
		for (u32 k = 0; k < F_MAXPATHS; k++)
			memcpy(&fm.caps[k], jbuf + caps + k * F_NT * 4, 4);
		double s0 = 0, s1 = 0;
		u32 slow = 0, hh = 0, klen = 0;
		if (fstage(fm, FP, defmask, s0, s1) != FO_AGGR ||
		    !fprep(fm, FP, defmask, s0, s1, slow) ||
		    !fkey_hash(fm, FP, defmask, hh, klen))
			continue;
		nrec++;
		/* the counter by the book: every piece in the dictionary */
		u32 want = 0;
		for (u32 j = 0; j < D.ncols && want != ~0u; j++) {
			FPiece pc;
			fpiece(fm, FP, j, defmask, pc);
			const char *b = pc.kind == 0 ? (const char *)rec + pc.off :
			    FP.pool + pc.off;
			u32 c = 0;
			while (c < D.n[j] && !(D.len[j][c] == pc.n &&
			    !memcmp(D.val[j][c], b, pc.n)))
				c++;
			want = c < D.n[j] ? want + c * D.stride[j] : ~0u;
		}
		const u32 got = jc(ra, defmask, caps);
		if (got != want) {
			fprintf(stderr, "dng_jcode: %u, expected %u: %.*s\n", got,
			    want, (int)len, rec);
			return 3;
		}
		if (got == ~0u)
			continue;
		ndense++;
		u8 k1[F_MAXKEY + 16], k2[F_MAXKEY + 16];
		memset(k1, 0xee, sizeof (k1));
		memset(k2, 0xee, sizeof (k2));
		fkey_write(fm, FP, defmask, k1);
		const u32 dl = fdense_key(D, got, k2);
		if (dl != klen || memcmp(k1, k2, (klen + 7) & ~7u)) {
			fprintf(stderr, "fdense_key differs from fkey_write: %.*s\n",
			    (int)len, rec);
			return 3;
		}
	}
	printf("{\"dict\":%u,\"records\":%lu,\"dense\":%lu}\n", D.total, nrec,
	    ndense);
	return 0;
}
