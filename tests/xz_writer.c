/*
 * TEST INFRASTRUCTURE ONLY - the CPU .xz writer that pins mg_encode_slab_xz (tests/test_xz_output.py compiles it into
 * a temporary directory and loads it with ctypes; the product never links it).
 *
 * It is built from the oracle port: the whole port is included, so Model, Sink, code_packet and rc_shift_low are the
 * ones the port's cost and LZMA-alone bytes use, and this file only adds the semantics of include/megalania_cuda.h
 * mg_encode_slab_xz, written sequentially: the cut candidates and the chunk plan priced with the port's cost sink,
 * each chunk range-coded by a fresh port coder from the port's model at the chunk's start, and the container.  The
 * device stream must equal it byte for byte.
 */
#include "../oracle/mg_oracle.c"

/* The .xz stream of the slab: its length (written only while it fits cap), 0 when a chunk would code to more than
 * 65536 bytes.  chunk_bytes 0 = 61440.  bounds (may be NULL): the chunk starts and n, *chunks of them + 1. */
size_t cpu_encode_xz(const uint8_t* data, size_t n, const MgoPacket* slab, uint32_t chunk_bytes, uint8_t* out, size_t cap,
                     uint32_t* bounds, size_t bounds_cap, size_t* chunks);
/* Cut candidates: positions and the cost of everything before them (0 first, n last); returns the count. */
size_t cpu_xz_candidates(const uint8_t* data, size_t n, const MgoPacket* slab, uint32_t* pos, uint64_t* cost, size_t cap);

#define XZ_GRANULE 4096
#define LZMA2_MAX_U (1u << 21)
#define LZMA2_MAX_C (1u << 16)

size_t cpu_xz_candidates(const uint8_t* data, size_t n, const MgoPacket* slab, uint32_t* pos, uint64_t* cost, size_t cap)
{
	Model m;
	Sink s;
	model_init(&m, data, n);
	sink_init(&s, SINK_COST);
	size_t count = 0, next = XZ_GRANULE;
	if (count < cap) {
		pos[count] = 0;
		cost[count] = 0;
	}
	count++;
	while (m.pos < n) {
		code_packet(&m, &s, slab[m.pos]);
		if (m.pos >= next && m.pos < n) { /* the first packet boundary at or after a multiple of the granule */
			if (count < cap) {
				pos[count] = (uint32_t)m.pos;
				cost[count] = s.cost;
			}
			count++;
			next = (m.pos / XZ_GRANULE + 1) * XZ_GRANULE;
		}
	}
	if (count < cap) {
		pos[count] = (uint32_t)n;
		cost[count] = s.cost;
	}
	return count + 1;
}

typedef struct {
	uint8_t* out;
	size_t cap, len;
} Buf;

static void put(Buf* b, uint8_t x)
{
	if (b->len < b->cap) b->out[b->len] = x;
	b->len++;
}

static void put_le(Buf* b, uint64_t x, int bytes)
{
	for (int i = 0; i < bytes; i++) put(b, (uint8_t)(x >> (8 * i)));
}

static void put_varint(Buf* b, uint64_t x)
{
	while (x >= 0x80) {
		put(b, (uint8_t)(x | 0x80));
		x >>= 7;
	}
	put(b, (uint8_t)x);
}

static uint32_t crc32_of(const uint8_t* p, size_t len)
{
	uint32_t c = 0xffffffffu;
	for (size_t i = 0; i < len; i++) {
		c ^= p[i];
		for (int k = 0; k < 8; k++) c = (c >> 1) ^ (0xEDB88320u & (0u - (c & 1u)));
	}
	return ~c;
}

static uint64_t crc64_of(const uint8_t* p, size_t len)
{
	uint64_t c = ~0ull;
	for (size_t i = 0; i < len; i++) {
		c ^= p[i];
		for (int k = 0; k < 8; k++) c = (c >> 1) ^ (0xC96C5795D7870F42ull & (0ull - (c & 1ull)));
	}
	return ~c;
}

/* the CRC32 of bytes already written (the buffer is large enough: the caller sizes it from a first pass) */
static uint32_t crc32_from(const Buf* b, size_t from) { return b->len <= b->cap ? crc32_of(b->out + from, b->len - from) : 0; }

size_t cpu_encode_xz(const uint8_t* data, size_t n, const MgoPacket* slab, uint32_t chunk_bytes, uint8_t* out, size_t cap,
                     uint32_t* bounds, size_t bounds_cap, size_t* chunks)
{
	if (chunk_bytes == 0) chunk_bytes = 61440;
	/* candidates and the chunk plan */
	size_t ncut = cpu_xz_candidates(data, n, slab, NULL, NULL, 0);
	uint32_t* cpos = malloc(sizeof(uint32_t) * ncut);
	uint64_t* ccost = malloc(sizeof(uint64_t) * ncut);
	cpu_xz_candidates(data, n, slab, cpos, ccost, ncut);
	const uint64_t budget = (uint64_t)chunk_bytes * 8 * 2048;
	uint32_t* start = malloc(sizeof(uint32_t) * (ncut + 1));
	size_t nchunk = 0;
	for (size_t s = 0; s + 1 < ncut;) {
		size_t e = s + 1;
		while (e + 1 < ncut && ccost[e + 1] - ccost[s] <= budget && cpos[e + 1] - cpos[s] <= LZMA2_MAX_U) e++;
		start[nchunk++] = cpos[s];
		s = e;
	}
	start[nchunk] = (uint32_t)n;
	if (chunks) *chunks = nchunk;
	if (bounds)
		for (size_t c = 0; c <= nchunk && c < bounds_cap; c++) bounds[c] = start[c];

	Buf b = {out, cap, 0};
	const uint8_t flags[2] = {0x00, 0x04};
	put(&b, 0xFD), put(&b, '7'), put(&b, 'z'), put(&b, 'X'), put(&b, 'Z'), put(&b, 0x00);
	put(&b, flags[0]), put(&b, flags[1]);
	put_le(&b, crc32_of(flags, 2), 4);
	/* block header: 12 bytes (size byte 12 / 4 - 1 = 2), no size fields, one filter: LZMA2, dictionary >= max(n, 4 KiB) */
	const size_t block = b.len;
	unsigned dict = 0;
	while (dict < 40 && ((uint64_t)(2u | (dict & 1u)) << (dict / 2 + 11)) < n) dict++;
	put(&b, 2), put(&b, 0x00), put(&b, 0x21), put(&b, 0x01), put(&b, (uint8_t)dict);
	put(&b, 0), put(&b, 0), put(&b, 0);
	put_le(&b, crc32_from(&b, block), 4);
	/* chunks: the port's model runs on through all of them, each gets a fresh range coder */
	Model m;
	model_init(&m, data, n);
	uint8_t* payload = malloc(LZMA2_MAX_C + 16);
	size_t ok = 1;
	for (size_t c = 0; c < nchunk; c++) {
		Sink s;
		sink_init(&s, SINK_RC);
		s.out = payload;
		s.out_cap = LZMA2_MAX_C;
		while (m.pos < start[c + 1]) code_packet(&m, &s, slab[m.pos]);
		for (int i = 0; i < 5; i++) rc_shift_low(&s);
		if (s.out_len > LZMA2_MAX_C) {
			ok = 0;
			break;
		}
		const uint32_t u = start[c + 1] - start[c] - 1, z = (uint32_t)s.out_len - 1;
		put(&b, (uint8_t)((c == 0 ? 0xE0u : 0x80u) | (u >> 16)));
		put(&b, (uint8_t)(u >> 8)), put(&b, (uint8_t)u);
		put(&b, (uint8_t)(z >> 8)), put(&b, (uint8_t)z);
		if (c == 0) put(&b, 0x00); /* properties: lc = lp = pb = 0 */
		for (size_t i = 0; i < s.out_len; i++) put(&b, payload[i]);
	}
	put(&b, 0x00);
	const uint64_t unpadded = b.len - block + 8;
	while ((b.len - block) & 3) put(&b, 0);
	put_le(&b, crc64_of(data, n), 8);
	const size_t index = b.len;
	put(&b, 0x00);
	put_varint(&b, 1);
	put_varint(&b, unpadded);
	put_varint(&b, n);
	while ((b.len - index) & 3) put(&b, 0);
	put_le(&b, crc32_from(&b, index), 4);
	const uint32_t backward = (uint32_t)((b.len - index) / 4 - 1);
	uint8_t tail[6] = {(uint8_t)backward, (uint8_t)(backward >> 8), (uint8_t)(backward >> 16), (uint8_t)(backward >> 24),
	                   flags[0], flags[1]};
	put_le(&b, crc32_of(tail, 6), 4);
	for (int i = 0; i < 6; i++) put(&b, tail[i]);
	put(&b, 'Y'), put(&b, 'Z');
	free(payload);
	free(start);
	free(cpos);
	free(ccost);
	return ok ? b.len : 0;
}
