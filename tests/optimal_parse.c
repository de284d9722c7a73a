/*
 * TEST INFRASTRUCTURE ONLY - the CPU parse that pins mg_anneal_optimal_init (tests/test_optimal_parse.py compiles it
 * into a temporary directory and loads it with ctypes; the product never links it).
 *
 * It is built from the oracle port's own pricing: the whole port is included, so Index, Model, bit_price,
 * length_price, tree_price, next_ctx and code_packet are the ones the port's cost uses, and this file only adds the
 * semantics of include/megalania_cuda.h mg_anneal_optimal_init with one region, written sequentially.  The device
 * parse must equal it packet for packet.
 */
#include "../oracle/mg_oracle.c"

/* The shortest-path parse with one region (lc = 0): blocks of 4096 bytes priced with the model at the block's
 * start, cheapest path per block, exact model through it.  max_occ 0 = 64. */
void cpu_optimal_slab(const uint8_t* data, size_t n, uint32_t max_occ, MgoPacket* slab);
/* Its match list of position pos: up to cap (len, distance - 1) pairs into out[2 * i], rising in both; returns the
 * count. */
size_t cpu_match_list(const uint8_t* data, size_t n, size_t pos, uint32_t max_occ, uint32_t* out, size_t cap);

/* ---- shortest-path parse (mg_anneal_optimal_init) ---------------------------------------- */
#define OPT_BLOCK 4096 /* nodes per block: csrc/mg_kernels.cuh OPT_BLOCK */
#define OPT_LIST 32    /* match-list entries per position: csrc/mg_kernels.cuh OPT_LIST */
#define OPT_INF 0xffffffffu

typedef struct {
	uint32_t len, dist; /* dist = distance - 1 */
} OptEntry;

/* The match list of pos: the nearest max_occ earlier occurrences of its bigram, nearest first; an entry is kept only
 * when it is longer than every earlier one, and the walk stops at an entry of min(273, n - pos) bytes or at cap. */
static size_t opt_match_list(const Index* ix, size_t pos, uint32_t max_occ, OptEntry* out, size_t cap)
{
	const uint8_t* data = ix->data;
	size_t n = ix->n;
	if (pos == 0 || pos + 1 >= n) return 0;
	if (max_occ == 0) max_occ = 64;
	unsigned key = (unsigned)data[pos] << 8 | data[pos + 1];
	uint32_t first = ix->start[key], lo = first, hi = ix->start[key + 1];
	while (lo < hi) { /* the first occurrence at or after pos */
		uint32_t mid = lo + (hi - lo) / 2;
		if (ix->occ[mid] < pos) lo = mid + 1;
		else hi = mid;
	}
	size_t limit = n - pos < 273 ? n - pos : 273, count = 0, best = 0;
	for (uint32_t i = lo, visited = 0; i > first && visited < max_occ; visited++) {
		size_t o = ix->occ[--i];
		size_t len = 2;
		while (len < limit && data[pos + len] == data[o + len]) len++;
		if (len <= best) continue;
		if (count == cap) break;
		out[count].len = (uint32_t)len;
		out[count].dist = (uint32_t)(pos - o - 1);
		count++;
		best = len;
		if (len >= limit) break;
	}
	return count;
}

size_t cpu_match_list(const uint8_t* data, size_t n, size_t pos, uint32_t max_occ, uint32_t* out, size_t cap)
{
	Index ix;
	index_build(&ix, data, n);
	OptEntry* e = malloc(sizeof(OptEntry) * (cap ? cap : 1));
	size_t count = opt_match_list(&ix, pos, max_occ, e, cap);
	for (size_t i = 0; i < count; i++) {
		out[2 * i] = e[i].len;
		out[2 * i + 1] = e[i].dist;
	}
	free(e);
	index_free(&ix);
	return count;
}

typedef struct {
	uint32_t cost;
	MgoPacket pk; /* the packet that reached the node */
	uint8_t ctx;
	uint32_t rep[4];
} OptNode;

/* price of a literal at pos under the block-start probabilities of m, with the node's state and rep0 */
static uint32_t opt_literal_price(const Model* m, const uint32_t* litp, unsigned ctx, size_t pos, uint32_t rep0)
{
	uint32_t c = bit_price(m, S_ISMATCH + (ctx << 4), 0);
	unsigned byte = m->data[pos];
	if (ctx < 7) return c + litp[byte];
	unsigned mbyte = m->data[pos - rep0 - 1];
	int matched = 1;
	unsigned node = 1;
	for (int i = 7; i >= 0; i--) {
		unsigned bit = (byte >> i) & 1;
		unsigned slot = node;
		if (matched) {
			unsigned mbit = (mbyte >> i) & 1;
			slot += (1 + mbit) << 8;
			matched = (mbit == bit);
		}
		c += bit_price(m, S_LIT + slot, bit);
		node = (node << 1) | bit;
	}
	return c;
}

static void opt_relax(OptNode* nodes, size_t t, uint32_t cost, const OptNode* from, MgoPacket pk)
{
	OptNode* v = &nodes[t];
	if (cost >= v->cost) return;
	v->cost = cost;
	v->pk = pk;
	v->ctx = (uint8_t)next_ctx(from->ctx, pk.type);
	memcpy(v->rep, from->rep, sizeof(v->rep));
	if (pk.type == T_MATCH) {
		v->rep[3] = v->rep[2];
		v->rep[2] = v->rep[1];
		v->rep[1] = v->rep[0];
		v->rep[0] = pk.dist;
	} else if (pk.type == T_LONG_REP) {
		uint32_t d = v->rep[pk.dist];
		for (unsigned i = pk.dist; i > 0; i--) v->rep[i] = v->rep[i - 1];
		v->rep[0] = d;
	}
}

void cpu_optimal_slab(const uint8_t* data, size_t n, uint32_t max_occ, MgoPacket* slab)
{
	Index ix;
	index_build(&ix, data, n);
	Model m;
	Sink s;
	model_init(&m, data, n);
	sink_init(&s, SINK_COST);
	for (size_t i = 0; i < n; i++) slab[i] = mk(T_LITERAL, 0, 1);
	OptNode* nodes = malloc(sizeof(OptNode) * (OPT_BLOCK + 1));
	OptEntry list[OPT_LIST];
	uint32_t lenp[274], replenp[274], slotp[4][64], alignp[16], litp[256];
	while (m.pos < n) {
		const size_t p = m.pos, B = n - p < OPT_BLOCK ? n - p : OPT_BLOCK;
		/* static price tables from the model at the block's start */
		for (unsigned l = 2; l <= 273; l++) {
			lenp[l] = length_price(&m, S_LEN, l);
			replenp[l] = length_price(&m, S_REPLEN, l);
		}
		for (unsigned c = 0; c < 4; c++)
			for (unsigned ps = 0; ps < 64; ps++) slotp[c][ps] = tree_price(&m, S_POSSLOT + c * 64, 6, ps);
		for (unsigned a = 0; a < 16; a++) alignp[a] = tree_rev_price(&m, S_ALIGN, 4, a);
		for (unsigned b = 0; b < 256; b++) litp[b] = tree_price(&m, S_LIT, 8, b);
		nodes[0].cost = 0;
		nodes[0].ctx = m.ctx;
		memcpy(nodes[0].rep, m.rep, sizeof(m.rep));
		for (size_t j = 1; j <= B; j++) nodes[j].cost = OPT_INF;
		for (size_t j = 0; j < B; j++) {
			const OptNode* u = &nodes[j];
			const size_t i = p + j;
			const unsigned ctx = u->ctx;
			const uint32_t c0 = u->cost;
			opt_relax(nodes, j + 1, c0 + opt_literal_price(&m, litp, ctx, i, u->rep[0]), u, mk(T_LITERAL, 0, 1));
			const uint32_t is_rep = bit_price(&m, S_ISMATCH + (ctx << 4), 1) + bit_price(&m, S_ISREP + ctx, 1);
			if (i >= (size_t)u->rep[0] + 1 && data[i] == data[i - u->rep[0] - 1])
				opt_relax(nodes, j + 1,
				          c0 + is_rep + bit_price(&m, S_ISREPG0 + ctx, 0) + bit_price(&m, S_ISREP0LONG + (ctx << 4), 0), u,
				          mk(T_SHORT_REP, 0, 1));
			const size_t maxl = B - j < 273 ? B - j : 273;
			size_t rl[4];
			uint32_t rep_head[4];
			for (unsigned r = 0; r < 4; r++) {
				rl[r] = 0;
				if (i >= (size_t)u->rep[r] + 1)
					while (rl[r] < maxl && data[i + rl[r]] == data[i + rl[r] - u->rep[r] - 1]) rl[r]++;
				if (r == 0) {
					rep_head[r] = is_rep + bit_price(&m, S_ISREPG0 + ctx, 0) + bit_price(&m, S_ISREP0LONG + (ctx << 4), 1);
				} else {
					rep_head[r] = is_rep + bit_price(&m, S_ISREPG0 + ctx, 1) + bit_price(&m, S_ISREPG1 + ctx, r != 1);
					if (r != 1) rep_head[r] += bit_price(&m, S_ISREPG2 + ctx, r != 2);
				}
			}
			const uint32_t match_head = bit_price(&m, S_ISMATCH + (ctx << 4), 1) + bit_price(&m, S_ISREP + ctx, 0);
			const size_t count = opt_match_list(&ix, i, max_occ, list, OPT_LIST);
			size_t e = 0;
			for (size_t l = 2; l <= maxl; l++) {
				for (unsigned r = 0; r < 4; r++)
					if (rl[r] >= l) opt_relax(nodes, j + l, c0 + rep_head[r] + replenp[l], u, mk(T_LONG_REP, r, (unsigned)l));
				while (e < count && list[e].len < l) e++;
				if (e == count) continue;
				/* distance price from the static tables: pos slot, then pos coder / direct bits + align */
				const unsigned dist = list[e].dist, lctx = l - 2 < 3 ? (unsigned)l - 2 : 3;
				uint32_t dp;
				if (dist < 4) {
					dp = slotp[lctx][dist];
				} else {
					unsigned nlow = bit_length(dist) - 2, low = dist & ((1u << nlow) - 1), high = dist >> nlow;
					unsigned pslot = nlow * 2 + high;
					dp = slotp[lctx][pslot];
					if (pslot < 14) dp += tree_rev_price(&m, S_POSCODER + (high << nlow) - pslot, nlow, low);
					else dp += ((nlow - 4) << 11) + alignp[low & 15];
				}
				opt_relax(nodes, j + l, c0 + match_head + lenp[l] + dp, u, mk(T_MATCH, dist, (unsigned)l));
			}
		}
		/* commit: the packets of the cheapest path, then the exact model through them */
		for (size_t j = B; j > 0; j -= nodes[j].pk.len) slab[p + j - nodes[j].pk.len] = nodes[j].pk;
		while (m.pos < p + B) code_packet(&m, &s, slab[m.pos]);
	}
	free(nodes);
	index_free(&ix);
}

