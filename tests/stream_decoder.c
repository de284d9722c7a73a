/*
 * TEST INFRASTRUCTURE ONLY - the CPU decoder that pins mg_decode_stream (tests/test_stream_resume.py compiles it
 * into a temporary directory and loads it with ctypes; the product never links it).
 *
 * It is built from the oracle port's own model: the whole port is included, so the slot map (S_*), Model,
 * next_ctx and the rep shifting are the ones code_packet uses, and this file only adds code_packet run backwards.
 */
#include "../oracle/mg_oracle.c"

/* the codes of MG_EINVAL / MG_ESLAB (include/megalania_cuda.h) */
#define MGO_EINVAL (-1)
#define MGO_ESLAB (-4)

/* LZMA-alone stream of data[0..n) -> slab (n slots): the inverse of mgo_encode_slab.  Header: properties byte 0
 * (lc = lp = pb = 0), size field n or all ones (then the stream must end with the end marker, exactly at n), at
 * least 13 + 5 bytes, else MGO_EINVAL.  Payload: every packet must reproduce data[] inside [0, n), the stream must be
 * consumed exactly and the range decoder's code end at 0, else MGO_ESLAB.  The packet that starts at a position goes
 * to that slot; every other slot is LITERAL / 0 / 1. */
int cpu_decode_stream(const uint8_t* data, size_t n, const uint8_t* stream, size_t len, MgoPacket* slab);

/* ---- stream -> slab: code_packet run backwards ------------------------------------------ */
/* An LZMA-alone stream at lc = lp = pb = 0 codes exactly this model; decoding it gives the slab that encodes
 * to it.  The range decoder mirrors the encoder above step for step (normalise after every bit), so a
 * well-formed stream ends with every byte consumed and code == 0.  Every decoded byte is checked against
 * data[], which is why no output buffer is needed.  Returns 0, MGO_EINVAL (header) or MGO_ESLAB (payload). */
typedef struct {
	const uint8_t* in;
	size_t len, at;
	uint32_t range, code;
	int short_read;
} RangeDecoder;

static void rd_shift(RangeDecoder* d)
{
	d->range <<= 8;
	if (d->at >= d->len) {
		d->short_read = 1;
		d->code <<= 8;
		return;
	}
	d->code = (d->code << 8) | d->in[d->at++];
}

static unsigned decode_bit(Model* m, RangeDecoder* d, unsigned slot)
{
	unsigned v = m->p[slot];
	uint32_t bound = (d->range >> 11) * v;
	unsigned bit;
	if (d->code < bound) {
		d->range = bound;
		bit = 0;
		v += (2048 - v) >> 5;
	} else {
		d->code -= bound;
		d->range -= bound;
		bit = 1;
		v -= v >> 5;
	}
	m->p[slot] = (uint16_t)v;
	while ((d->range & 0xFF000000u) == 0) rd_shift(d);
	return bit;
}

static unsigned decode_direct(RangeDecoder* d, unsigned nbits)
{
	unsigned value = 0;
	while (nbits--) {
		d->range >>= 1;
		unsigned bit = d->code >= d->range;
		if (bit) d->code -= d->range;
		value = (value << 1) | bit;
		if ((d->range & 0xFF000000u) == 0) rd_shift(d);
	}
	return value;
}

static unsigned decode_tree(Model* m, RangeDecoder* d, unsigned base, unsigned nbits)
{
	unsigned node = 1;
	for (unsigned i = 0; i < nbits; i++) node = (node << 1) | decode_bit(m, d, base + node);
	return node - (1u << nbits);
}

static unsigned decode_tree_rev(Model* m, RangeDecoder* d, unsigned base, unsigned nbits)
{
	unsigned node = 1, value = 0;
	for (unsigned i = 0; i < nbits; i++) {
		unsigned bit = decode_bit(m, d, base + node);
		node = (node << 1) | bit;
		value |= bit << i;
	}
	return value;
}

static unsigned decode_length(Model* m, RangeDecoder* d, unsigned base)
{
	if (!decode_bit(m, d, base + LEN_CHOICE1)) return 2 + decode_tree(m, d, base + LEN_LOW, 3);
	if (!decode_bit(m, d, base + LEN_CHOICE2)) return 10 + decode_tree(m, d, base + LEN_MID, 3);
	return 18 + decode_tree(m, d, base + LEN_HIGH, 8);
}

static uint32_t decode_distance(Model* m, RangeDecoder* d, unsigned len)
{
	unsigned lctx = len - 2;
	if (lctx > 3) lctx = 3;
	unsigned pslot = decode_tree(m, d, S_POSSLOT + lctx * 64, 6);
	if (pslot < 4) return pslot;
	unsigned nlow = (pslot >> 1) - 1;
	uint32_t dist = (uint32_t)(2 | (pslot & 1)) << nlow;
	if (pslot < 14) return dist + decode_tree_rev(m, d, S_POSCODER + dist - pslot, nlow);
	dist += decode_direct(d, nlow - 4) << 4;
	return dist + decode_tree_rev(m, d, S_ALIGN, 4);
}

/* 1 if data[pos .. pos+len) equals data[pos-dist-1 ..] and lies inside [0, n) */
static int copy_ok(const Model* m, uint64_t dist, size_t len)
{
	if (m->pos < dist + 1 || m->pos + len > m->n) return 0;
	return memcmp(m->data + m->pos, m->data + m->pos - dist - 1, len) == 0;
}

int cpu_decode_stream(const uint8_t* data, size_t n, const uint8_t* stream, size_t len, MgoPacket* slab)
{
	if (len < 13 + 5 || stream[0] != 0) return MGO_EINVAL;
	uint64_t size = 0;
	for (int i = 0; i < 8; i++) size |= (uint64_t)stream[5 + i] << (8 * i);
	const int known = size != ~0ull;
	if (known && size != n) return MGO_EINVAL;
	RangeDecoder d = { stream, len, 13, 0xFFFFFFFFu, 0, 0 };
	if (d.in[d.at++] != 0) return MGO_ESLAB;
	for (int i = 0; i < 4; i++) d.code = (d.code << 8) | d.in[d.at++];
	Model m;
	model_init(&m, data, n);
	for (size_t i = 0; i < n; i++) slab[i] = mk(T_LITERAL, 0, 1);
	for (;;) {
		if (known && m.pos == n) break;
		if (d.short_read) return MGO_ESLAB;
		unsigned ctx = m.ctx;
		MgoPacket pk;
		if (!decode_bit(&m, &d, S_ISMATCH + (ctx << 4))) {
			if (m.pos >= n) return MGO_ESLAB;
			/* the coded tree: a matched literal while the decoded bits agree with the match byte (code_packet) */
			int matched = ctx >= 7;
			if (matched && m.pos < (size_t)m.rep[0] + 1) return MGO_ESLAB;
			unsigned mbyte = matched ? m.data[m.pos - m.rep[0] - 1] : 0;
			unsigned node = 1; /* lc = 0: one literal table, S_LIT */
			for (int i = 7; i >= 0; i--) {
				unsigned slot = node;
				unsigned mbit = (mbyte >> i) & 1;
				if (matched) slot += (1 + mbit) << 8;
				unsigned bit = decode_bit(&m, &d, S_LIT + slot);
				if (matched) matched = mbit == bit;
				node = (node << 1) | bit;
			}
			if ((node & 0xff) != m.data[m.pos]) return MGO_ESLAB;
			pk = mk(T_LITERAL, 0, 1);
		} else if (!decode_bit(&m, &d, S_ISREP + ctx)) {
			unsigned l = decode_length(&m, &d, S_LEN);
			uint32_t dist = decode_distance(&m, &d, l);
			if (dist == 0xFFFFFFFFu) { /* end marker: only where the size is unknown, and only at n */
				if (known || m.pos != n) return MGO_ESLAB;
				break;
			}
			if (!copy_ok(&m, dist, l)) return MGO_ESLAB;
			m.rep[3] = m.rep[2];
			m.rep[2] = m.rep[1];
			m.rep[1] = m.rep[0];
			m.rep[0] = dist;
			pk = mk(T_MATCH, dist, l);
		} else if (!decode_bit(&m, &d, S_ISREPG0 + ctx)) {
			if (!decode_bit(&m, &d, S_ISREP0LONG + (ctx << 4))) {
				if (!copy_ok(&m, m.rep[0], 1)) return MGO_ESLAB;
				pk = mk(T_SHORT_REP, 0, 1);
			} else {
				unsigned l = decode_length(&m, &d, S_REPLEN);
				if (!copy_ok(&m, m.rep[0], l)) return MGO_ESLAB;
				pk = mk(T_LONG_REP, 0, l);
			}
		} else {
			unsigned idx = 1;
			if (decode_bit(&m, &d, S_ISREPG1 + ctx)) idx = decode_bit(&m, &d, S_ISREPG2 + ctx) ? 3 : 2;
			unsigned l = decode_length(&m, &d, S_REPLEN);
			if (!copy_ok(&m, m.rep[idx], l)) return MGO_ESLAB;
			uint32_t dd = m.rep[idx];
			for (unsigned i = idx; i > 0; i--) m.rep[i] = m.rep[i - 1];
			m.rep[0] = dd;
			pk = mk(T_LONG_REP, idx, l);
		}
		slab[m.pos] = pk;
		m.ctx = (uint8_t)next_ctx(ctx, pk.type);
		m.pos += pk.len;
	}
	if (d.short_read || d.at != len || d.code != 0) return MGO_ESLAB;
	return 0;
}
