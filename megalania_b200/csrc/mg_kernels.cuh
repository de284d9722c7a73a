// Kernels of the annealing hot path (sm_100a).  One warp = one model = one chain / slab / query.
#pragma once
#include "mg_device.cuh"
#include "mg_finder.cuh"

namespace mg {

// One CTA of 26 warps per SM: 26 models + the transition tables (48 KB, see mg_device.cuh) fill the 227 KB of
// shared memory.  The walk is bound by shared-memory wavefronts; whole windows of plain literals are priced from
// per-lane queues built once per input (walk_windows()).
#ifndef MG_WARPS_PER_CTA
#define MG_WARPS_PER_CTA 26
#endif
constexpr int WARPS_PER_CTA = MG_WARPS_PER_CTA;
constexpr int CTA_THREADS = WARPS_PER_CTA * 32;
constexpr uint32_t RECIP_ENTRIES = 288;
// Kernel experiments (tools/variants.sh): 0 = the product; bit 0 = literal queues off (every literal takes the
// single-step path); bit 1 = walk_windows() keeps the next window's type/length word in a register (round-2 form up
// to 27e4c2c) instead of staging it by cp.async.
#ifndef MG_WALK_VARIANT
#define MG_WALK_VARIANT 0
#endif

struct ChainStats {
	unsigned long long evals, attempts, accepted, new_best, packets, bits, slab_bytes, ck_bytes, finds, candidates,
	    edits, overflows, rejoined, find_cycles, chain_cycles, chunks, gave_up;
};

struct ChainState {
	uint64_t rng;
	uint64_t cur_cost;
	uint64_t best_cost;
	uint64_t slab_cost;   // exact cost of the current slab (cur_cost may be 0 = "accept the first proposal")
	uint32_t live_count;
	uint32_t err;
	uint32_t eval_index;  // successful evaluations since the chain's slab was last set
	uint32_t journal_count;     // edits accepted since the best slab last equalled the current slab
	uint32_t journal_overflow;  // != 0: the journal is incomplete, the next new best copies the whole slab
	// A proposal suspended at a checkpoint crossing when the launch's packet budget ran out (see
	// AnnealArgs::suspend).  Its model is the record it had just written into the non-live buffer
	// of slot susp_slot-1, its edits so far sit in the chain's accept/reject buffer.
	uint32_t susp_slot;      // 0 = nothing suspended
	uint32_t susp_j0;        // first checkpoint index the proposal rewrites
	uint32_t susp_stored, susp_count, susp_overflow;  // EditLog counters
	uint32_t pad;
};
constexpr uint32_t JOURNAL_CAP = 1024;

// ---- the accept/reject buffer of one proposal (replaces packet_slab_undo_stack) -------------------
struct Edit {
	uint32_t pos;
	uint32_t pad;
	uint64_t pk;
};

struct EditLog {
	Edit* e;
	uint32_t cap;
	uint32_t stored;    // physical entries
	uint32_t count;     // logical edits (what the reference's undo stack would hold)
	uint32_t dup_pos;   // position whose entry may be rewritten (pos+1 of a shrink), or ~0
	uint32_t dup_index;
	bool overflow;
};

// Dynamic shared memory of one CTA.  A warp's block starts on a 128-byte boundary with its record, so that the
// record's rows are bank rows (slot map in mg_device.cuh).
struct alignas(128) WarpShared {
	Record rec;
	FindScratch fs;
	uint64_t bar;
	ChainStats stats;    // counters of the running launch (kept out of the register file; lane 0 only)
};
struct alignas(128) CtaShared {
	uint32_t trans[TRANS_WORDS];
	uint32_t recip[RECIP_ENTRIES];
	uint4 lane_tab[32];    // match_lane_const() per lane
	WarpShared warp[WARPS_PER_CTA];
};
static_assert(offsetof(WarpShared, rec) == 0 && sizeof(Record) % 128 == 0, "record rows must be bank rows");
static_assert(offsetof(CtaShared, warp) % 128 == 0, "record alignment");
static_assert(sizeof(CtaShared) <= 232448, "one CTA must fit the 227 KB of shared memory");

__device__ __forceinline__ WarpShared* warp_block(CtaShared* sh, int warp) { return &sh->warp[warp]; }

// One literal queue per 32-byte window of the input, built once per context (litq_build_kernel): for each lane the
// up to QUEUE_ROUNDS table steps it owes the window when all 32 slots hold plain literals and the automaton is in
// state 0.  Layout [window][3 blocks][32 lanes] x 16 bytes (eight entries per lane and block; the third block is
// only read for the few windows in which some lane owes more than 16 steps); entry = u16:
//   bits 0-11   byte offset of the probability in the record (lane L only ever names slots in bank L)
//   bit  12     lane 0, entry 0 only: the third block is in use
//   bits 13-15  transition-table section (one step: bit; two steps on the slot: 2 + first bit << 1 + second bit)
// Entries a lane does not need name its spare slot (value 0) in section 0: table entry 0 is a zero-price fixed point.
// A window some lane would need more rounds for has 0xffff in lane 0's first entry: it takes the single-step path.
constexpr uint32_t QUEUE_UNUSABLE = 0xffffu, QUEUE_MORE = 0x1000u, QUEUE_BLOCKS = 3, QUEUE_MAX_ROUNDS = 8 * QUEUE_BLOCKS;

struct Tables {
	const uint32_t* trans;   // [TRANS_WORDS] stored probability after | price << 16 (price: reference generate_table.py:7-9)
	const uint32_t* recip;   // [RECIP_ENTRIES]
	const uint4* litq;       // [windows][64] literal queues, or null
};

__device__ __forceinline__ void cta_tables_load(CtaShared* sh, const Tables& t)
{
	for (int i = threadIdx.x; i < (int)TRANS_WORDS; i += blockDim.x) sh->trans[i] = t.trans[i];
	for (int i = threadIdx.x; i < (int)RECIP_ENTRIES; i += blockDim.x) sh->recip[i] = t.recip[i];
	if (threadIdx.x < 32) {
		const LaneConst c = match_lane_const((int)threadIdx.x);
		sh->lane_tab[threadIdx.x] = make_uint4(c.shb, c.mask2, c.base, c.sel);
	}
	if ((threadIdx.x & 31) == 0) mbar_init(&warp_block(sh, threadIdx.x >> 5)->bar, 1);
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	__syncthreads();
}

// Error bits a walk can raise
constexpr uint32_t ERR_BAD_PACKET = 1, ERR_NOT_BOUNDARY = 2, ERR_OUTPUT_FULL = 4;

// Memory-safety check of a packet about to be priced at model m (the reference asserts /
// reads out of bounds instead; src/lzma_packet_encoder.c:186-190).
__device__ __forceinline__ bool packet_ok(const Model& m, uint32_t n, uint32_t type, uint32_t len, uint32_t dist)
{
	if (len == 0 || len > n - m.pos) return false;
	switch (type) {
	case T_LITERAL: return len == 1;
	case T_SHORT_REP: return len == 1 && m.rep0 < m.pos;
	case T_MATCH: return len >= 2 && len <= MAX_MATCH && dist < m.pos;
	case T_LONG_REP: return len >= 2 && len <= MAX_MATCH && dist < 4 && model_rep(m, dist) < m.pos;
	default: return false;
	}
}

// Running totals of one walk
struct Tally {
	uint64_t total;  // uniform: cost flushed so far
	uint32_t acc;    // per lane: cost since the last flush
	uint32_t bits;  // modelled bits in excess of 9 per packet (two's complement)
};

__device__ __forceinline__ void tally_flush(Tally& t)
{
	t.total += __reduce_add_sync(FULL, t.acc);
	t.acc = 0;
}

// memcmp(data+pos-d-1, data+pos, len) == 0 across the warp (src/packet_slab_neighbour.c:74-80)
__device__ __forceinline__ bool rep_matches(int lane, const uint8_t* __restrict__ data, uint32_t pos, uint32_t d,
                                            uint32_t len)
{
	bool same = true;
	const uint8_t* a = data + pos;
	const uint8_t* b = data + (pos - d - 1);
	for (uint32_t i = lane; i < len; i += 32) same = same && a[i] == b[i];
	return __all_sync(FULL, same);
}


__device__ __forceinline__ void log_put(int lane, EditLog& lg, uint32_t pos, uint64_t pk)
{
	lg.count++;
	if (pos == lg.dup_pos) {
		if (lane == 0) lg.e[lg.dup_index].pk = pk;
		return;
	}
	if (lg.stored >= lg.cap) {
		lg.overflow = true;
		return;
	}
	if (lane == 0) {
		lg.e[lg.stored].pos = pos;
		lg.e[lg.stored].pk = pk;
	}
	lg.stored++;
}

// ---- the walk ----------------------------------------------------------------------------------------
// Everything a walking warp needs besides its registers.  Lane roles in the single-literal path:
// lane 0 owns is_match[ctx], lanes 1..8 own literal-tree depth 0..7, lanes 9..31 sit it out.
struct WalkEnv {
	int lane;
	SmemU16 probs;        // the model's probabilities
	SmemU32 trans;        // the CTA's transition table
	SmemU32 recip;        // the CTA's reciprocal table
	SmemU32 reps;         // rec->rep[4]
	uint16_t* probs_ptr;  // generic pointer to the same probabilities (bulk compares only)
	Record* rec;
	const uint64_t* __restrict__ slab;
	const uint8_t* __restrict__ data;
	const uint32_t* __restrict__ abs_dist;  // region merges: the distance a LONG_REP slot stood for in its owner chain, or null
	const uint4* __restrict__ litq;         // the context's literal queues, or null
	uint32_t n;
	uint32_t trans_addr;  // shared address of trans[]
	uint32_t lane_tab_addr;  // shared address of this lane's match_lane_const() entry
	uint32_t ev_addr;        // shared address of the warp's staging area (literal queue, MATCH descriptors, next window)
	uint32_t stage_addr;     // shared address of the next window's staging area
	// single-literal path (slot map in mg_device.cuh): with u = ((b >> lit_sh) & lit_mask) ^ lit_x the lane's
	// probability for data byte b lives at lit_addr + u + (u & lit_hm)  (+ 2 * ctx on lane 0); in matched mode a
	// tree lane whose prefix agrees with the match byte uses litv_addr + 2 * (b >> lit_psh) + 512 * match bit
	uint32_t lit_addr, lit_sh, lit_mask, lit_x, lit_hm;
	uint32_t litv_addr, lit_psh;
	uint32_t bit_shl;     // b << bit_shl puts the lane's data bit at bit 13 (the table's section bit)
	uint32_t bitmask;     // 0x2000 on tree lanes
	uint32_t ctxmask;     // ~0 on lane 0
	bool lit_active;      // lanes 0..8
};

__device__ __forceinline__ WalkEnv make_env(int lane, WarpShared* ws, const CtaShared* sh, const uint64_t* slab,
                                            const uint8_t* data, uint32_t n, const uint4* litq)
{
	WalkEnv e;
	e.lane = lane;
	// Two opaque base addresses, everything else a compile-time offset from them: left to itself the
	// compiler re-derives each shared address from the generic pointer (S2R SR_CgaCtaId + LEA + IMAD)
	// wherever it is short of registers, which was ~10 % of the instructions of a non-literal packet.
	uint32_t cta_base = smem_u32(sh), warp_base = smem_u32(ws);
	asm volatile("" : "+r"(cta_base), "+r"(warp_base));
	e.probs.a = warp_base + (uint32_t)offsetof(WarpShared, rec) + (uint32_t)offsetof(Record, probs);
	e.trans.a = cta_base + (uint32_t)offsetof(CtaShared, trans);
	e.recip.a = cta_base + (uint32_t)offsetof(CtaShared, recip);
	e.reps.a = warp_base + (uint32_t)offsetof(WarpShared, rec) + (uint32_t)offsetof(Record, rep);
	e.probs_ptr = ws->rec.probs;
	e.rec = &ws->rec;
	e.slab = slab;
	e.data = data;
	e.abs_dist = nullptr;
	e.litq = (MG_WALK_VARIANT & 1) ? nullptr : litq;
	e.n = n;
	e.trans_addr = e.trans.a;
	e.lane_tab_addr = cta_base + (uint32_t)offsetof(CtaShared, lane_tab) + 16u * (uint32_t)lane;
	e.ev_addr = warp_base + (uint32_t)offsetof(WarpShared, fs) + (uint32_t)offsetof(FindScratch, len_price);
	e.stage_addr = e.ev_addr + STAGE_OFFSET;
	const bool tree = lane >= 1 && lane <= 8;
	const uint32_t d = tree ? (uint32_t)lane - 1 : 0;
	// byte offsets, see lit0_slot(): depth <= 3 one slot per word (4 * node), depth 4 the same with the XOR,
	// depth 5..7 u + (u & hm) with u = 2 * (prefix ^ x)
	uint32_t first = S_DUMMY, sh_ = 8, mask = 0, x = 0, hm = 0;
	if (lane == 0) first = S_ISMATCH;
	else if (tree && d <= 3) { first = S_LIT0 + 2u * (1u << d); sh_ = 6 - d; mask = ((1u << d) - 1u) << 2; }
	else if (tree && d == 4) { first = S_LIT0 + 32; sh_ = 2; mask = 0x3c; x = LITX4 << 2; }
	else if (tree && d == 5) { first = S_LIT0 + 96; sh_ = 2; mask = 0x3e; x = LITX5 << 1; }
	else if (tree && d == 6) { first = S_LIT0 + 160; sh_ = 1; mask = 0x7e; x = LITX6 << 1; hm = 64; }
	else if (tree && d == 7) { first = S_LIT0 + 288; sh_ = 0; mask = 0xfe; x = LITX7 << 1; hm = 0xc0; }
	e.lit_addr = e.probs.a + 2 * first;
	e.lit_sh = sh_;
	e.lit_mask = mask;
	e.lit_x = x;
	e.lit_hm = hm;
	e.litv_addr = e.probs.a + 2 * (S_LITV + (1u << d));
	e.lit_psh = tree ? 8u - d : 8u;
	e.bitmask = tree ? 0x2000u : 0u;
	e.ctxmask = lane == 0 ? 0xffffffffu : 0u;
	e.bit_shl = 6u + d;
	e.lit_active = lane <= 8;
	// Opaque to the compiler on purpose: it otherwise re-derives these constants from threadIdx inside the
	// literal loop instead of keeping them in registers.
	asm volatile("" : "+r"(e.lit_addr), "+r"(e.lit_sh), "+r"(e.lit_mask), "+r"(e.lit_x), "+r"(e.lit_hm), "+r"(e.bit_shl),
	             "+r"(e.bitmask), "+r"(e.ctxmask));
	return e;
}

// MATCH descriptors of the current window: lane i turns ITS slot, if it holds a MATCH that is valid
// at position base+i, into the packed words the MATCH fast path needs (match_desc() with state 0)
// and stores {F, G, amask | direct << 26, dist}; F == 0 marks every other slot.  ~70 instructions
// once per window for all its matches instead of once per match.
__device__ __forceinline__ void window_matches(const WalkEnv& e, Window& w)
{
	__syncwarp();
	// opaque on purpose: the compiler otherwise computes match_desc() speculatively for EVERY window right after
	// the window is decoded (36 instructions per window of plain literals, 8 % of all instructions of the bench)
	uint32_t meta = w.meta;
	asm volatile("" : "+r"(meta));
	const uint32_t len = meta_len(meta), dist = w.dist, pos = w.base + (uint32_t)e.lane;
	const bool ok = meta_type(meta) == T_MATCH && len - 2 <= MAX_MATCH - 2 && pos < e.n && len <= e.n - pos && dist < pos;
	if (__any_sync(FULL, ok)) {
		MatchDesc d = {0, 0, 0, 0};
		if (ok) d = match_desc(0, len, dist);
		sts_v4(e.ev_addr + MATCH_DESC_OFFSET + 16u * (uint32_t)e.lane, d.F, d.G, d.amask | (d.direct << 26), dist);
	}
	w.md_base = w.base;
	__syncwarp();
}

// Per-checkpoint bookkeeping kept beside the records, in DELTA form: cost and packets between the
// previous checkpoint (or the start of the file) and this one.  Deltas stay valid for the
// untouched tail when a proposal stops early (see walker_checkpoint), absolutes would not.
struct CkMeta {
	uint64_t dcost;
	uint32_t dpidx;
	uint32_t pos;
};

// Where checkpoints of the walk go (all null when the walk writes none)
struct CkSink {
	Record* ck;          // indexed by slot-1
	uint32_t* ck_pos;    // optional: absolute positions (top-k queries)
	CkMeta* meta;        // optional
	const uint8_t* live; // anneal: which of the two buffers is current per slot-1 (write the other); null = buffer 0
	uint32_t nck;        // anneal: records per buffer
	uint32_t stride;
	uint32_t next;       // next position that triggers a checkpoint
	uint32_t written;    // count, for stats
	uint32_t last_pidx;  // packet index / cost at the previous checkpoint of this walk
	uint64_t last_cost;
	uint32_t test;       // != 0: compare each crossing with the chain's current checkpoint there
	uint32_t converged;  // slot at which the model re-joined the current slab's trajectory (0 = not)
	uint32_t suspend_pidx;  // WALK_REPAIR: stop at the first checkpoint at or past this packet index (~0 = never)
	long long deadline;     // WALK_REPAIR: ... or at the first checkpoint after this clock64() value (0 = none)
};

// The state a walk keeps in registers.  The rep distances stay in e.rec->rep[] (shared memory):
// only matches touch them, and keeping them out of the register loop keeps the literal path tight.
struct Walker {
	uint32_t pos;
	uint32_t delta;  // pos - packet index: constant across single-byte packets
	uint32_t ctx;
	uint32_t mb;     // data[pos - rep0 - 1], valid whenever ctx >= 7 (fetched right after a non-literal packet)
	Tally t;
	Window w;
};

__device__ __forceinline__ uint32_t walker_pidx(const Walker& k) { return k.pos - k.delta; }

__device__ __forceinline__ Model walker_model(const WalkEnv& e, const Walker& k)
{
	Model m;
	m.pos = k.pos;
	m.pidx = k.pos - k.delta;
	m.ctx = k.ctx;
	m.rep0 = e.reps.get(0);
	m.rep1 = e.reps.get(1);
	m.rep2 = e.reps.get(2);
	m.rep3 = e.reps.get(3);
	return m;
}

// The match byte is fetched on demand: only a literal that directly follows a non-literal packet
// reads it (the automaton is below 7 after any literal, src/lzma_state.c:34-40).
constexpr uint32_t MB_UNKNOWN = 0xffffffffu;
__device__ __forceinline__ uint32_t walker_mb(const WalkEnv& e, Walker& k)
{
	if (k.mb == MB_UNKNOWN) {
		const uint32_t rep0 = e.reps.get(0);
		k.mb = (k.pos < e.n && rep0 < k.pos) ? e.data[k.pos - rep0 - 1] : 0;
	}
	return k.mb;
}

__device__ __forceinline__ void walker_init(const WalkEnv& e, Walker& k)
{
	Model m;
	model_init(e.lane, e.probs, m);
	if (e.lane < 4) e.reps.set(e.lane, 0);
	__syncwarp();
	k.pos = k.delta = k.ctx = k.mb = 0;
	k.t = {0, 0, 0};
	k.w.base = WINDOW_NONE;
	k.w.pf_base = WINDOW_NONE;
	k.w.md_base = WINDOW_NONE;
}

__device__ __forceinline__ void walker_load(const WalkEnv& e, Walker& k, const Record* src, uint64_t* bar, uint32_t& parity)
{
	Model m;
	uint64_t cost;
	record_load(e.lane, e.rec, m, cost, src, bar, parity);
	k.pos = m.pos;
	k.delta = m.pos - m.pidx;
	k.ctx = m.ctx;
	k.t = {cost, 0, 0};
	k.w.base = WINDOW_NONE;
	k.w.pf_base = WINDOW_NONE;
	k.w.md_base = WINDOW_NONE;
	k.mb = MB_UNKNOWN;
}

// Generic (any packet type) price + adapt: the slow path of the walk.
__device__ __forceinline__ void walker_apply(const WalkEnv& e, Walker& k, Model& m, uint32_t type, uint32_t len,
                                             uint32_t dist, uint32_t byte)
{
	const uint32_t mbyte = (type == T_LITERAL && k.ctx >= 7) ? walker_mb(e, k) : 0u;
	k.t.bits += apply_packet(e.lane, e.probs, e.trans, m, type, len, dist, byte, mbyte, k.t.acc) - 9u;
	k.pos = m.pos;
	k.delta = m.pos - m.pidx;
	k.ctx = m.ctx;
	if (type == T_MATCH || type == T_LONG_REP) {
		// every lane holds the same values; each writes them so that it can read them back unsynchronised
		e.reps.set(0, m.rep0);
		e.reps.set(1, m.rep1);
		e.reps.set(2, m.rep2);
		e.reps.set(3, m.rep3);
	}
	__syncwarp();  // lanes are not guaranteed to run in lockstep: order these stores before later reads (pair steps
	               // reach a slot from another lane than the one that wrote it here)
	if (type != T_LITERAL) k.mb = MB_UNKNOWN;
}

__device__ __forceinline__ void walker_store(const WalkEnv& e, const Walker& k, Record* dst)
{
	const Model m = walker_model(e, k);
	record_store(e.lane, e.rec, m, k.t.total, dst);
}

// Is the walking model, at a checkpoint crossing, bit-identical to the checkpoint the chain's
// CURRENT slab left at the same slot (same position, automaton state, rep distances and all
// probabilities)?  If so everything after this point is priced exactly as it was for the current
// slab, and the proposal can stop here: an exact early exit, no approximation.
__device__ __forceinline__ bool walker_rejoined(const WalkEnv& e, const Walker& k, const Record* old, uint32_t old_pos)
{
	if (old_pos != k.pos) return false;
	if (old->ctx != k.ctx || old->rep[0] != e.rec->rep[0] || old->rep[1] != e.rec->rep[1] || old->rep[2] != e.rec->rep[2] ||
	    old->rep[3] != e.rec->rep[3])
		return false;
	const uint32_t* mine = reinterpret_cast<const uint32_t*>(e.probs_ptr);
	const uint32_t* theirs = reinterpret_cast<const uint32_t*>(old->probs);
	constexpr uint32_t WORDS = S_COUNT / 2;
	for (uint32_t base = 0; base < WORDS; base += 32) {  // uniform trip count: the vote needs every lane
		const uint32_t i = base + (uint32_t)e.lane;
		const bool differs = i < WORDS && mine[i] != theirs[i];
		if (__any_sync(FULL, differs)) return false;
	}
	return true;
}

__device__ __forceinline__ void walker_checkpoint(const WalkEnv& e, Walker& k, CkSink& ck)
{
	tally_flush(k.t);
	const uint32_t slot = k.pos / ck.stride;
	const uint32_t cur = ck.live ? ck.live[slot - 1] : 0u;
	const uint32_t buf = ck.live ? cur ^ 1u : 0u;
	bool same = false;
	if (ck.test) same = walker_rejoined(e, k, ck.ck + (size_t)cur * ck.nck + (slot - 1), ck.meta[(size_t)cur * ck.nck + (slot - 1)].pos);
	walker_store(e, k, ck.ck + (size_t)buf * ck.nck + (slot - 1));
	const uint32_t pidx = walker_pidx(k);
	if (e.lane == 0) {
		if (ck.ck_pos) ck.ck_pos[(size_t)buf * ck.nck + (slot - 1)] = k.pos;
		if (ck.meta) {
			CkMeta m;
			m.dcost = k.t.total - ck.last_cost;
			m.dpidx = pidx - ck.last_pidx;
			m.pos = k.pos;
			ck.meta[(size_t)buf * ck.nck + (slot - 1)] = m;
		}
	}
	ck.last_cost = k.t.total;
	ck.last_pidx = pidx;
	ck.next = (slot + 1) * ck.stride;
	ck.written++;
	if (same) ck.converged = slot;
}

// Sum of the deltas of the chain's CURRENT checkpoints 1..upto: absolute packet index and cost at
// checkpoint `upto` (upto = 0: start of file).
__device__ __forceinline__ void ck_absolute(int lane, const CkMeta* meta, const uint8_t* live, uint32_t nck, uint32_t upto,
                                            uint32_t& pidx, uint64_t& cost)
{
	uint32_t p = 0;
	uint64_t c = 0;
	for (uint32_t i = (uint32_t)lane; i < upto; i += 32) {
		const CkMeta m = meta[(size_t)live[i] * nck + i];
		p += m.dpidx;
		c += m.dcost;
	}
	for (int o = 16; o > 0; o >>= 1) {
		p += __shfl_xor_sync(FULL, p, o);
		c += __shfl_xor_sync(FULL, c, o);
	}
	pidx = p;
	cost = c;
}

// ---- windows of 32 plain literals -----------------------------------------------------------------
// Four queue entries of one lane (two words): the probability at each entry's offset takes the one or two steps the
// entry's section names.  The four probability loads go out together and the table loads follow as their inputs
// arrive: a lane's entries on one slot are adjacent in its queue (litq_build_kernel emits slot by slot), so the only
// hazard inside the group is "same slot as the entry before", which takes the probability the entry before produced
// instead of the one loaded.  The stores follow in order, so the last entry of a slot wins.
__device__ __forceinline__ void queue_rounds4(uint32_t v0, uint32_t v1, uint32_t probs_a, uint32_t trans_a, uint32_t& acc)
{
	asm volatile(
	    "{\n\t"
	    ".reg .b32 h0, h1, a0, a1, a2, a3, s0, s1, s2, s3, p0, p1, p2, p3, t0, t1, t2, t3, x;\n\t"
	    ".reg .b16 q0, q1, q2, q3;\n\t"
	    ".reg .pred e1, e2, e3;\n\t"
	    "shr.u32 h0, %1, 16;\n\t"
	    "shr.u32 h1, %2, 16;\n\t"
	    "and.b32 a0, %1, 0x0FFE;\n\t"
	    "and.b32 a1, h0, 0x0FFE;\n\t"
	    "and.b32 a2, %2, 0x0FFE;\n\t"
	    "and.b32 a3, h1, 0x0FFE;\n\t"
	    "add.u32 a0, a0, %3;\n\t"
	    "add.u32 a1, a1, %3;\n\t"
	    "add.u32 a2, a2, %3;\n\t"
	    "add.u32 a3, a3, %3;\n\t"
	    "ld.shared.u16 q0, [a0];\n\t"
	    "ld.shared.u16 q1, [a1];\n\t"
	    "ld.shared.u16 q2, [a2];\n\t"
	    "ld.shared.u16 q3, [a3];\n\t"
	    "and.b32 s0, %1, 0xE000;\n\t"
	    "and.b32 s1, h0, 0xE000;\n\t"
	    "and.b32 s2, %2, 0xE000;\n\t"
	    "and.b32 s3, h1, 0xE000;\n\t"
	    "add.u32 s0, s0, %4;\n\t"
	    "add.u32 s1, s1, %4;\n\t"
	    "add.u32 s2, s2, %4;\n\t"
	    "add.u32 s3, s3, %4;\n\t"
	    "setp.eq.u32 e1, a1, a0;\n\t"
	    "setp.eq.u32 e2, a2, a1;\n\t"
	    "setp.eq.u32 e3, a3, a2;\n\t"
	    "cvt.u32.u16 p0, q0;\n\t"
	    "cvt.u32.u16 p1, q1;\n\t"
	    "cvt.u32.u16 p2, q2;\n\t"
	    "cvt.u32.u16 p3, q3;\n\t"
	    "add.u32 s0, s0, p0;\n\t"
	    "ld.shared.u32 t0, [s0];\n\t"
	    "@e1 and.b32 p1, t0, 0xFFFF;\n\t"
	    "add.u32 s1, s1, p1;\n\t"
	    "ld.shared.u32 t1, [s1];\n\t"
	    "@e2 and.b32 p2, t1, 0xFFFF;\n\t"
	    "add.u32 s2, s2, p2;\n\t"
	    "ld.shared.u32 t2, [s2];\n\t"
	    "@e3 and.b32 p3, t2, 0xFFFF;\n\t"
	    "add.u32 s3, s3, p3;\n\t"
	    "ld.shared.u32 t3, [s3];\n\t"
	    "cvt.u16.u32 q0, t0;\n\t"
	    "cvt.u16.u32 q1, t1;\n\t"
	    "cvt.u16.u32 q2, t2;\n\t"
	    "cvt.u16.u32 q3, t3;\n\t"
	    "st.shared.u16 [a0], q0;\n\t"
	    "st.shared.u16 [a1], q1;\n\t"
	    "st.shared.u16 [a2], q2;\n\t"
	    "st.shared.u16 [a3], q3;\n\t"
	    "shr.u32 t0, t0, 16;\n\t"
	    "shr.u32 t1, t1, 16;\n\t"
	    "shr.u32 t2, t2, 16;\n\t"
	    "shr.u32 t3, t3, 16;\n\t"
	    "add.u32 t0, t0, t1;\n\t"
	    "add.u32 t2, t2, t3;\n\t"
	    "add.u32 %0, %0, t0;\n\t"
	    "add.u32 %0, %0, t2;\n\t"
	    "}"
	    : "+r"(acc)
	    : "r"(v0), "r"(v1), "r"(probs_a), "r"(trans_a)
	    : "memory");
}

// Prices whole windows of 32 plain literals (automaton state 0 before and after), starting with the current
// window and carrying on, window after window, for as long as the next one is all plain literals too and ends
// at or before `wend`: lane L performs the table steps of its own queue, all on slots of bank L (slot map in
// mg_device.cuh), so the lanes neither share a bank nor an address and need no ordering among themselves; per
// slot the steps are in input order.  The kernel is bound by instruction issue, so the loop is kept bare: a lane's
// queue entries come straight from global memory into its registers, one window ahead of their use, and all it
// looks at of the next window is the type/length word of its slab slots.  The generic window state (k.w) is
// dropped on the way out: window_seek() reloads it.
// Returns false when the current window has no usable queue (the caller then takes its literals one by one).
__device__ __forceinline__ bool walk_windows(const WalkEnv& e, Walker& k, uint32_t wend)
{
	bool any = false;
	uint32_t acc = k.t.acc;
	const uint32_t pa = e.probs.a, ta = e.trans_addr;
	uint32_t base = k.w.base;
	const uint4* q = e.litq + (size_t)(base >> 5) * (QUEUE_BLOCKS * 32) + (uint32_t)e.lane;
	const uint32_t* slab_hi = reinterpret_cast<const uint32_t*>(e.slab) + 1;  // type << 16 | len of slot i at [2 * i]
	// The next window's type/length words travel global -> shared memory by cp.async into the lane's own slot of
	// the staging area (the place window_prefetch() puts them; a copy window_seek() left in flight there carries
	// the same words).  Held in a register the load was sunk by ptxas to the end of the window - the kernel is
	// compiled against a 72-register cap - and every window waited out one HBM round trip there (34 % of all warp
	// samples, profiles/r02_final_anneal_kernel_ncu.txt, line of the __all_sync below).
	const uint32_t hi_stage = e.stage_addr + 8u * (uint32_t)e.lane + 4u;
	uint4 a = __ldcg(q), b = __ldcg(q + 32);
	for (;;) {
		const uint32_t head = __shfl_sync(FULL, a.x, 0) & 0xffffu;
		if (head == QUEUE_UNUSABLE) break;
		const bool more = base + 64u <= wend;  // another whole window may follow
		uint32_t next_hi = 0;
		if (MG_WALK_VARIANT & 2) {
			if (more) next_hi = __ldcg(slab_hi + 2 * (size_t)(base + 32u + (uint32_t)e.lane));
		} else if (more) {
			asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n\tcp.async.commit_group;" ::"r"(hi_stage),
			             "l"(slab_hi + 2 * (size_t)(base + 32u + (uint32_t)e.lane))
			             : "memory");
		}
		queue_rounds4(a.x, a.y, pa, ta, acc);
		queue_rounds4(a.z, a.w, pa, ta, acc);
		if (more) a = __ldcg(q + QUEUE_BLOCKS * 32);
		queue_rounds4(b.x, b.y, pa, ta, acc);
		queue_rounds4(b.z, b.w, pa, ta, acc);
		if (more) b = __ldcg(q + QUEUE_BLOCKS * 32 + 32);
		if (head & QUEUE_MORE) {
			// the rare window in which some lane owes more than 16 steps: eight more from the third block
			const uint4 c = __ldcg(q + 64);
			queue_rounds4(c.x, c.y, pa, ta, acc);
			queue_rounds4(c.z, c.w, pa, ta, acc);
		}
		any = true;
		base += 32u;
		if (!more) break;
		// the per-lane sums are 32 bits wide: a window adds at most 24 x 45 056 to one
		if ((base & 1023u) == 0) {
			k.t.acc = acc;
			tally_flush(k.t);
			acc = 0;
		}
		if (!(MG_WALK_VARIANT & 2)) {
			// the lane reads the word it copied itself: no warp-level ordering needed
			asm volatile("cp.async.wait_group 0;\n\tld.shared.u32 %0, [%1];" : "=r"(next_hi) : "r"(hi_stage) : "memory");
		}
		if (!__all_sync(FULL, next_hi == ((T_LITERAL << 16) | 1u))) break;
		q += QUEUE_BLOCKS * 32;
	}
	if (any) {
		k.pos = base;
		k.t.acc = acc;
		k.w.base = WINDOW_NONE;
		k.w.pf_base = WINDOW_NONE;
		k.w.md_base = WINDOW_NONE;
		__syncwarp();  // other paths reach these slots from other lanes
	}
	return any;
}

enum WalkMode { WALK_PLAIN = 0, WALK_REPAIR_HEAD = 1, WALK_REPAIR = 2 };
enum WalkResult { WALK_DONE = 0, WALK_NEED_FIND = 1, WALK_ERROR = 2, WALK_REJOINED = 3, WALK_SUSPENDED = 4 };

// Prices packets from k.pos until stop_pos bytes or packet index stop_pidx is reached.
//   WALK_PLAIN        the slab as it is (neighbour.c:22-32, main.c:116-118)
//   WALK_REPAIR_HEAD  repair rules for the first three packets after a mutation (neighbour.c:82-98)
//   WALK_REPAIR       repair rules from the fourth packet on: a LITERAL slot can no longer change
//                     there, so literals take the same fast path as in WALK_PLAIN
// Returns WALK_NEED_FIND with `pending` = the failed LONG_REP (index forced to 3, neighbour.c:99-108)
// when the caller has to pick a replacement from the top-k at k.pos.
// k.t.bits only accumulates the EXCESS over 9 bits per packet; see walker_bits().
// MODE is a run-time argument on purpose: the annealing kernel calls this from ONE site for all
// three phases, which keeps its code (and instruction-cache footprint) a third of the size of
// three specialised copies.  A walk that writes no checkpoints passes ck.next = 0xffffffff.
__device__ __forceinline__ uint32_t walk(const uint32_t MODE, const WalkEnv& e, Walker& k, uint32_t stop_pos, uint32_t stop_pidx, CkSink& ck,
                                         EditLog* lg, uint32_t override_pos, uint64_t override_pk, uint64_t& pending,
                                         uint64_t& pending_old, uint32_t& err)
{
	for (;;) {
		if (k.pos >= stop_pos || k.pos - k.delta == stop_pidx) return WALK_DONE;
		if (k.pos >= ck.next) {
			walker_checkpoint(e, k, ck);
			if (ck.converged) return WALK_REJOINED;
			if (MODE == WALK_REPAIR && k.pos < stop_pos &&
			    (k.pos - k.delta >= ck.suspend_pidx || (ck.deadline != 0 && clock64() >= ck.deadline)))
				return WALK_SUSPENDED;
		}
		if (k.pos - k.w.base >= 32u) {
			// the per-lane sums are 32 bits wide: a lane adds at most ~10^5 per packet, so once per KiB of input is plenty
			if (((k.pos ^ k.w.base) >> 10) != 0) tally_flush(k.t);
			window_seek(e.lane, k.w, e.slab, e.data, e.n, k.pos, e.stage_addr);
		}
		uint32_t limit = k.w.base + 32 < stop_pos ? k.w.base + 32 : stop_pos;
		limit = ck.next < limit ? ck.next : limit;
		if (stop_pidx != 0xffffffffu) {
			// the packet index only drifts from the position on multi-byte packets (slow path)
			const uint32_t stop_at = stop_pidx + k.delta;
			limit = stop_at < limit ? stop_at : limit;
		}
		while (k.pos < limit) {
			const uint32_t meta = window_meta(k.w, k.pos);
			if (MODE != WALK_REPAIR_HEAD && (meta & 0xffffu) == META_LITERAL) {
				const uint32_t ctx = k.ctx;
				// ---- a whole window of plain literals: every lane works off its own queue (walk_windows) ----
				if (ctx == 0 && k.pos == k.w.base && k.w.litmask == FULL && limit - k.pos == 32u && e.litq != nullptr) {
					// whole windows may go on up to the nearest of: the stop position, the next checkpoint, the stop packet
					uint32_t wend = stop_pos < ck.next ? stop_pos : ck.next;
					if (stop_pidx != 0xffffffffu) wend = stop_pidx + k.delta < wend ? stop_pidx + k.delta : wend;
					if (walk_windows(e, k, wend)) break;  // the window moved on: recompute the limits
				}
				// ---- one literal: plain (slot classes on lanes 0..8, the lane's slot computed from the data
				// byte) or matched (lzma_packet_encoder.c:123-130: the tree follows the match byte for as long
				// as the prefixes agree) -----------------------------------------------------------------
				const uint32_t byte = (meta >> 16) & 0xff;
				const uint32_t u = ((byte >> e.lit_sh) & e.lit_mask) ^ e.lit_x;
				uint32_t addr = e.lit_addr + u + (u & e.lit_hm) + 2u * (ctx & e.ctxmask);
				if (ctx >= 7) {
					const uint32_t mb = walker_mb(e, k);
					if (e.bitmask != 0 && (mb >> e.lit_psh) == (byte >> e.lit_psh))
						addr = e.litv_addr + 2u * (byte >> e.lit_psh) + 512u * ((mb >> (e.lit_psh - 1)) & 1u);
				}
				k.ctx = ctx < 4 ? 0u : ctx < 10 ? ctx - 3 : ctx - 6;
				if (e.lit_active) {
					const uint32_t tr = lds_u32(e.trans_addr + ((byte << e.bit_shl) & e.bitmask) + lds_u16(addr));
					sts_u16(addr, tr);
					k.t.acc += tr >> 16;
				}
				__syncwarp();  // the window path reaches the same slots from other lanes
				k.pos++;
				continue;
			}
			// ---- a MATCH outside the repair head: repair never touches it (neighbour.c:82-117), so it
			// is priced straight from the slab.  One warp step: F/G/amask are the same on every lane,
			// the lane's four constants turn them into its slot and bit ----------------------------
			if (MODE != WALK_REPAIR_HEAD && meta_type(meta) == T_MATCH) {
				if (k.w.md_base != k.w.base) window_matches(e, k.w);
				const uint4 d = lds_v4(e.ev_addr + MATCH_DESC_OFFSET + 16u * (k.pos - k.w.base));
				if (d.x != 0) {
					const uint32_t len = meta_len(meta), dist = d.w, amask = d.z & 0x3ffffffu;
					uint32_t shb, mask2, base, sel;
					asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
					             : "=r"(shb), "=r"(mask2), "=r"(base), "=r"(sel)
					             : "r"(e.lane_tab_addr));
					const uint32_t nwb = (d.x >> shb) & mask2;
					const uint32_t slot = base + __byte_perm(d.y | k.ctx, 0, sel) + (nwb >> 1);
					if ((amask >> e.lane) & 1u) code_bit(e.probs, e.trans, slot, nwb & 1u, k.t.acc);
					if (e.lane == 0) k.t.acc += (d.z >> 26) << 11;  // src/perplexity_encoder.c:12-17
					k.t.bits += (uint32_t)__popc(amask) - 9u;
					// src/lzma_state.c:59-65, 29-57
					const uint32_t r0 = e.reps.get(0), r1 = e.reps.get(1), r2 = e.reps.get(2);
					e.reps.set(0, dist);
					e.reps.set(1, r0);
					e.reps.set(2, r1);
					e.reps.set(3, r2);
					__syncwarp();
					k.ctx = k.ctx < 7 ? 7 : 10;
					k.pos += len;
					k.delta += len - 1;
					k.mb = MB_UNKNOWN;
					continue;
				}
			}
			// ---- every other packet ---------------------------------------------------------------
			Model m = walker_model(e, k);
			uint32_t type = meta_type(meta), len = meta_len(meta), dist = 0;
			const uint32_t byte = meta_byte(meta) & 0xff;
			if (type == T_MATCH || type == T_LONG_REP) dist = window_dist(k.w, k.pos);
			if (MODE == WALK_REPAIR_HEAD && k.pos == override_pos) {
				type = pk_type(override_pk);
				len = pk_len(override_pk);
				dist = pk_dist(override_pk);
			}
			if (MODE != WALK_PLAIN) {
				const uint64_t old = pk_pack(type, dist, len);
				if (type == T_SHORT_REP || type == T_LITERAL) {
					const uint32_t rep_byte = (m.rep0 < m.pos) ? e.data[m.pos - m.rep0 - 1] : 0x100u;
					if (byte == rep_byte) {
						if (MODE == WALK_REPAIR_HEAD) type = T_SHORT_REP;  // only the first three packets convert
					} else {
						type = T_LITERAL;
					}
					dist = 0;
					len = 1;
				} else if (type == T_LONG_REP) {
					if (len < 2 || len > e.n - m.pos || dist > 3) {
						err = ERR_BAD_PACKET;
						return WALK_ERROR;
					}
					bool good = model_rep(m, dist) < m.pos && rep_matches(e.lane, e.data, m.pos, model_rep(m, dist), len);
					for (uint32_t idx = 0; idx < 4 && !good; idx++) {
						dist = idx;
						good = model_rep(m, dist) < m.pos && rep_matches(e.lane, e.data, m.pos, model_rep(m, dist), len);
					}
					if (!good && e.abs_dist) {
						// a merged slab: the rep distances in front of this region changed, but the distance
						// the packet stood for in its owner chain is known - keep the match, as a MATCH
						const uint32_t d = e.abs_dist[m.pos] - 1u;  // stored + 1; 0 = no entry -> 0xffffffff fails d < pos
						if (d < m.pos && rep_matches(e.lane, e.data, m.pos, d, len)) {
							type = T_MATCH;
							dist = d;
							good = true;
						}
					}
					if (!good) {
						pending = pk_pack(T_LONG_REP, dist, len);
						pending_old = old;
						return WALK_NEED_FIND;
					}
				}
				const uint64_t now = pk_pack(type, dist, len);
				if (now != old) log_put(e.lane, *lg, m.pos, now);
			}
			if (!packet_ok(m, e.n, type, len, dist)) {
				err = ERR_BAD_PACKET;
				return WALK_ERROR;
			}
			walker_apply(e, k, m, type, len, dist, byte);
			break;  // the packet index may have drifted: recompute the limits
		}
	}
}

// modelled bits priced since packet index pidx_from (fast-path literals count 9 each)
__device__ __forceinline__ uint64_t walker_bits(const Walker& k, uint32_t pidx_from)
{
	return (uint64_t)(walker_pidx(k) - pidx_from) * 9 + (int64_t)(int32_t)k.t.bits;
}

// ---- K3a: score whole slabs ---------------------------------------------------------------------
struct ScoreArgs {
	const uint8_t* data;
	uint32_t n;
	const uint64_t* slabs;   // [nslabs][n] packed
	uint32_t nslabs;
	uint32_t stop_pos;       // price [0, stop_pos)
	uint64_t* out_cost;      // [nslabs]
	uint32_t* out_count;     // [nslabs] live packets, may be null
	uint32_t* out_err;       // [nslabs]
	Record* ck;              // [nslabs][nslots-1] or null
	uint32_t* ck_pos;        // [nslabs][nslots-1] or null
	CkMeta* ck_meta;         // [nslabs][nslots-1] or null
	uint32_t stride, nslots;
	uint32_t ck_chain_stride;  // records between consecutive slabs' checkpoint blocks
	Record* final_model;     // [nslabs] model after the walk, or null
	Tables tables;
};

__global__ void __launch_bounds__(CTA_THREADS) score_kernel(ScoreArgs a)
{
	extern __shared__ __align__(128) unsigned char smem_raw[];
	CtaShared* sh = reinterpret_cast<CtaShared*>(smem_raw);
	cta_tables_load(sh, a.tables);
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const uint32_t s = blockIdx.x * WARPS_PER_CTA + warp;
	if (s >= a.nslabs) return;
	WarpShared* ws = warp_block(sh, warp);
	const WalkEnv e = make_env(lane, ws, sh, a.slabs + (size_t)s * a.n, a.data, a.n, a.tables.litq);
	Walker k;
	walker_init(e, k);
	const size_t ckoff = (size_t)s * a.ck_chain_stride;
	CkSink ck;
	ck.ck = a.ck ? a.ck + ckoff : nullptr;
	ck.ck_pos = a.ck_pos ? a.ck_pos + ckoff : nullptr;
	ck.meta = a.ck_meta ? a.ck_meta + ckoff : nullptr;
	ck.live = nullptr;
	ck.nck = 0;
	ck.stride = a.stride;
	ck.next = a.stride;
	ck.written = 0;
	ck.last_pidx = 0;
	ck.last_cost = 0;
	ck.test = 0;
	ck.converged = 0;
	ck.suspend_pidx = 0xffffffffu;
	ck.deadline = 0;
	uint64_t pending = 0, pending_old = 0;
	uint32_t err = 0;
	if (!a.ck) ck.next = 0xffffffffu;
	walk(WALK_PLAIN, e, k, a.stop_pos, 0xffffffffu, ck, nullptr, 0xffffffffu, 0, pending, pending_old, err);
	tally_flush(k.t);
	asm volatile("cp.async.wait_group 0;" ::: "memory");  // the window staged ahead of the walk
	if (!err && k.pos != a.stop_pos) err = ERR_NOT_BOUNDARY;
	if (a.final_model) walker_store(e, k, a.final_model + s);
	if (lane == 0) {
		a.out_cost[s] = k.t.total;
		if (a.out_count) a.out_count[s] = walker_pidx(k);
		a.out_err[s] = err;
	}
}

// ---- K2: top-k queries ---------------------------------------------------------------------------
struct TopkArgs {
	const uint8_t* data;
	uint32_t n;
	const uint32_t* occ_start;
	const uint32_t* occ;
	const uint64_t* slab;  // packed, n slots
	int state_mode;
	const uint32_t* positions;
	uint32_t npos, k;
	const Record* ck;  // mode 1: checkpoints of `slab`
	const uint32_t* ck_pos;
	uint32_t nslots, stride;
	uint64_t* out_pk;      // [npos][k]
	uint32_t* out_price;   // [npos][k]
	int32_t* out_count;    // [npos]
	uint32_t* out_err;     // [npos]
	unsigned long long* candidates;
	FindLimits limits;
	Tables tables;
};

__global__ void __launch_bounds__(CTA_THREADS) topk_kernel(TopkArgs a)
{
	extern __shared__ __align__(128) unsigned char smem_raw[];
	CtaShared* sh = reinterpret_cast<CtaShared*>(smem_raw);
	cta_tables_load(sh, a.tables);
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	WarpShared* ws = warp_block(sh, warp);
	const WalkEnv e = make_env(lane, ws, sh, a.slab, a.data, a.n, a.tables.litq);
	uint32_t parity = 0;
	unsigned long long cand = 0;
	for (uint32_t q = blockIdx.x * WARPS_PER_CTA + warp; q < a.npos; q += gridDim.x * WARPS_PER_CTA) {
		const uint32_t qpos = a.positions[q];
		Walker k;
		uint32_t err = 0;
		if (qpos >= a.n) {
			err = ERR_NOT_BOUNDARY;
		} else if (a.state_mode == 0) {
			walker_init(e, k);
			k.pos = k.delta = qpos;
		} else {
			// last checkpoint at or before the query
			uint32_t below = 0;
			for (uint32_t j = lane; j + 1 < a.nslots; j += 32) below += a.ck_pos[j] <= qpos ? 1u : 0u;
			below = __reduce_add_sync(FULL, below);
			if (below == 0)
				walker_init(e, k);
			else
				walker_load(e, k, a.ck + (below - 1), &ws->bar, parity);
			CkSink ck = {};
			ck.next = 0xffffffffu;
			ck.suspend_pidx = 0xffffffffu;
			ck.deadline = 0;
			uint64_t pending = 0, pending_old = 0;
			walk(WALK_PLAIN, e, k, qpos, 0xffffffffu, ck, nullptr, 0xffffffffu, 0, pending, pending_old, err);
			if (!err && k.pos != qpos) err = ERR_NOT_BOUNDARY;
		}
		uint32_t pops = 0;
		if (!err) {
			pops = warp_find(lane, e.probs, e.trans, e.recip, &ws->fs, a.data, a.n, a.occ_start, a.occ,
			                 walker_model(e, k), a.slab[qpos], a.k, 0, a.limits);
			cand += ws->fs.candidates;
			for (uint32_t i = lane; i < pops; i += 32) {
				const uint32_t en = ws->fs.pop_order[i];
				a.out_pk[(size_t)q * a.k + i] = ws->fs.ent_pk[en];
				a.out_price[(size_t)q * a.k + i] = ws->fs.ent_price[en];
			}
		}
		if (lane == 0) {
			a.out_count[q] = (int32_t)pops;
			a.out_err[q] = err;
		}
		__syncwarp();
	}
	asm volatile("cp.async.wait_group 0;" ::: "memory");
	if (lane == 0 && cand) atomicAdd(a.candidates, cand);
}

// ---- greedy parse (starting slabs) ---------------------------------------------------------------------
// One warp per byte region: from a fresh model at the region's first byte it takes, packet after packet, the
// cheapest candidate per byte of the exact top-k (the last one popped) and prices it, until the region is
// covered; the last packet is cut to the region's end.  With one region and no finder limits this is the
// oracle's greedy slab (mgo_greedy_slab) packet for packet.  Regions parsed side by side do not know each other's
// rep distances: what every LONG_REP stood for is recorded (abs_dist, stored + 1) and the caller sends the stitched
// slab through the forced repair pass of the region merge (mg_anneal_merge_import), which keeps such a packet as a
// MATCH at that distance and re-decides SHORT_REP / LITERAL by the reference's rule.
struct GreedyArgs {
	const uint8_t* data;
	uint32_t n;
	const uint32_t* occ_start;
	const uint32_t* occ;
	Tables tables;
	FindLimits limits;
	uint32_t k;
	const uint32_t* bounds;  // [nregions + 1]
	uint32_t nregions;
	uint64_t* slab;          // [n] packed, pre-filled with literals
	uint32_t* abs_dist;      // [n] zeroed
	uint32_t* err;
};

__global__ void __launch_bounds__(CTA_THREADS) greedy_kernel(GreedyArgs a)
{
	extern __shared__ __align__(128) unsigned char smem_raw[];
	CtaShared* sh = reinterpret_cast<CtaShared*>(smem_raw);
	cta_tables_load(sh, a.tables);
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	WarpShared* ws = warp_block(sh, warp);
	const WalkEnv e = make_env(lane, ws, sh, a.slab, a.data, a.n, nullptr);
	for (uint32_t r = (uint32_t)warp * gridDim.x + blockIdx.x; r < a.nregions; r += gridDim.x * WARPS_PER_CTA) {
		const uint32_t lo = a.bounds[r], hi = a.bounds[r + 1];
		Walker k;
		walker_init(e, k);
		k.pos = k.delta = lo;
		while (k.pos < hi) {
			Model m = walker_model(e, k);
			const uint32_t count = warp_find(lane, e.probs, e.trans, e.recip, &ws->fs, a.data, a.n, a.occ_start, a.occ, m, 0, a.k, 0,
			                                 a.limits);
			uint64_t pk = count ? ws->fs.ent_pk[ws->fs.pop_order[count - 1]] : PK_LITERAL;
			__syncwarp();
			uint32_t type = pk_type(pk), len = pk_len(pk), dist = pk_dist(pk);
			if (len > hi - k.pos) {
				if ((type == T_MATCH || type == T_LONG_REP) && hi - k.pos >= 2) {
					len = hi - k.pos;
				} else {
					type = T_LITERAL;
					len = 1;
					dist = 0;
				}
				pk = pk_pack(type, dist, len);
			}
			if (!packet_ok(m, a.n, type, len, dist)) {
				if (lane == 0) atomicOr(a.err, ERR_BAD_PACKET);
				break;
			}
			if (lane == 0) {
				a.slab[k.pos] = pk;
				if (type == T_LONG_REP) a.abs_dist[k.pos] = model_rep(m, dist) + 1u;
			}
			walker_apply(e, k, m, type, len, dist, a.data[k.pos]);
		}
	}
}

// ---- K3/K4: the annealing loop ---------------------------------------------------------------------


struct TraceRec {
	uint64_t cost;
	uint32_t flags;
	uint32_t undo_count;
};

struct AnnealArgs {
	const uint8_t* data;
	uint32_t n;
	const uint32_t* occ_start;
	const uint32_t* occ;
	Tables tables;
	FindLimits limits;
	uint32_t chains, k, stride, nslots, log_cap, track_best;
	uint64_t* slabs;     // [chains][n]
	uint64_t* bests;     // [chains][n] or null
	Record* ck;          // [chains][2][nslots-1]
	CkMeta* ck_meta;     // [chains][2][nslots-1]
	uint8_t* ck_live;    // [chains][nslots-1] which of the two buffers is current
	Edit* logs;          // [chains][log_cap]
	Edit* journal;       // [chains][JOURNAL_CAP] or null (no best tracking)
	ChainState* state;   // [chains]
	ChainStats* stats;   // [chains]
	TraceRec* trace;     // [chains][trace_cap] or null
	uint32_t trace_cap;
	uint32_t* attempts_out;  // [chains]
	// run parameters
	uint32_t evals, max_attempts, schedule, step, num_iters, first_eval;
	unsigned long long packet_budget;
	unsigned long long cycle_budget;  // SM clocks: chains stop (suspending their proposal) once the launch has run this long
	uint32_t early_exit;  // stop a proposal where its model re-joins the current slab's checkpoints
	const uint32_t* abs_dist; // repair_only after a region merge: see WalkEnv::abs_dist
	const uint32_t* regions;  // [chains][2] or null: a chain only mutates packets that start in its byte range
	uint32_t chain_first;     // the launch covers chains [chain_first, chain_first + chains)
	uint32_t repair_only;     // one forced pass per chain: repair + price the whole slab, commit (after a merge)
	uint32_t suspend;     // packet_budget is exact: a proposal that crosses it is suspended at its next
	                      // checkpoint and carried on by the next launch, so all warps end together
	const float* temps;
};

#ifndef MG_ANNEAL_MIN_CTAS
#define MG_ANNEAL_MIN_CTAS 1
#endif
__global__ void __launch_bounds__(CTA_THREADS, MG_ANNEAL_MIN_CTAS) anneal_kernel(AnnealArgs a)
{
	extern __shared__ __align__(128) unsigned char smem_raw[];
	CtaShared* sh = reinterpret_cast<CtaShared*>(smem_raw);
	cta_tables_load(sh, a.tables);
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	// chains are dealt round-robin over the CTAs, so that a population smaller than a full wave (huge inputs: a
	// 16 MiB chain is 270 MB) still puts warps on every SM
	if ((uint32_t)warp * gridDim.x + blockIdx.x >= a.chains) return;
	const uint32_t c = a.chain_first + (uint32_t)warp * gridDim.x + blockIdx.x;
	WarpShared* ws = warp_block(sh, warp);
	const uint32_t n = a.n, nck = a.nslots - 1;
	const uint32_t reg_lo = a.regions ? a.regions[2 * c] : 0u, reg_hi = a.regions ? a.regions[2 * c + 1] : 0u;
	uint64_t* slab = a.slabs + (size_t)c * n;
	WalkEnv e_init = make_env(lane, ws, sh, slab, a.data, n, a.tables.litq);
	e_init.abs_dist = a.abs_dist;
	// not const: rebuilt after every finder call instead of staying live across it (see the call)
	WalkEnv e = e_init;
	Record* ck_base = a.ck + (size_t)c * 2 * nck;
	CkMeta* ck_meta = a.ck_meta + (size_t)c * 2 * nck;
	uint8_t* ck_live = a.ck_live + (size_t)c * nck;
	ChainState st = a.state[c];
	// the forced pass after a merge draws from a fixed generator: every process that repairs the same
	// merged slab (multi-GPU merges) must make the same picks; the chain's own generator is left alone
	uint64_t rng = a.repair_only ? 0x6D65726765ull : st.rng;
	uint32_t parity = 0;
	// Counters live in shared memory and are touched by lane 0 only: lanes of a warp are not
	// guaranteed to run in lockstep, so a read-modify-write by all of them could count twice.
	ChainStats& cs = ws->stats;
	if (lane == 0) cs = ChainStats{0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
	const long long t_start = clock64();
	unsigned long long packets_done = 0;  // uniform copy of cs.packets for the budget test
	EditLog lg;
	lg.e = a.logs + (size_t)c * a.log_cap;
	lg.cap = a.log_cap;
	const float temp = a.temps ? a.temps[c] : 0.f;

	uint32_t done = 0, attempts = 0;
	const uint32_t first_eval = a.first_eval == 0xffffffffu ? st.eval_index : a.first_eval;
	const long long deadline = a.cycle_budget ? t_start + (long long)a.cycle_budget : 0;
	while (done < a.evals && attempts < a.max_attempts && st.err == 0 &&
	       (a.packet_budget == 0 || packets_done < a.packet_budget) && (deadline == 0 || clock64() < deadline)) {
		attempts++;
		const uint64_t rng_at_start = rng;
		Walker k;
		CkSink ck;
		ck.ck = ck_base;
		ck.ck_pos = nullptr;
		ck.meta = ck_meta;
		ck.live = ck_live;
		ck.nck = nck;
		ck.stride = a.stride;
		ck.written = 0;
		ck.converged = 0;
		uint32_t j0 = 0, target = 0;
		uint32_t phase = 0, mode = WALK_PLAIN;
		const bool resumed = st.susp_slot != 0;
		if (resumed) {
			// ---- carry on the proposal the previous launch suspended (phase 2, at a checkpoint) ----
			const uint32_t slot = st.susp_slot;
			j0 = st.susp_j0;
			lg.stored = st.susp_stored;
			lg.count = st.susp_count;
			lg.overflow = st.susp_overflow != 0;
			lg.dup_pos = 0xffffffffu;  // only the first three repaired packets can rewrite an entry
			lg.dup_index = 0;
			st.susp_slot = 0;
			walker_load(e, k, ck_base + (size_t)(ck_live[slot - 1] ^ 1u) * nck + (slot - 1), &ws->bar, parity);
			if (lane == 0) cs.ck_bytes += sizeof(Record);
			ck.next = (slot + 1) * a.stride;
			ck.last_pidx = walker_pidx(k);
			ck.last_cost = k.t.total;
			ck.test = a.early_exit;
			phase = 2;
			mode = WALK_REPAIR;
		} else {
			lg.stored = lg.count = 0;
			lg.dup_pos = 0xffffffffu;
			lg.dup_index = 0;
			lg.overflow = false;

			// ---- pick the packet to mutate and the checkpoint to start from ------------------
			// neighbour.c:163 draws a packet index; a chain confined to a byte range (cooperative
			// regions, see mg_anneal_merge_regions) draws a byte of its range instead and mutates
			// the first packet that starts at or after it
			const bool by_pos = a.regions != nullptr;
			if (by_pos)
				target = reg_lo + rng31(rng) % (reg_hi - reg_lo);
			else if (!a.repair_only)
				target = rng31(rng) % st.live_count;
			// last checkpoint at or before the target: running sums of the delta records
			uint32_t pidx0 = 0;
			uint64_t cost0 = 0;
			if (!a.repair_only) {
				uint32_t carry_p = 0;
				uint64_t carry_c = 0;
				for (uint32_t base = 0; base < nck; base += 32) {
					const uint32_t i = base + lane;
					CkMeta mt = {0, 0, 0};
					if (i < nck) mt = ck_meta[(size_t)ck_live[i] * nck + i];
					uint32_t p = mt.dpidx;
					uint64_t cc = mt.dcost;
					for (int o = 1; o < 32; o <<= 1) {
						const uint32_t tp = __shfl_up_sync(FULL, p, o);
						const uint64_t tc = __shfl_up_sync(FULL, cc, o);
						if (lane >= o) {
							p += tp;
							cc += tc;
						}
					}
					p += carry_p;
					cc += carry_c;
					const uint32_t cnt = __popc(__ballot_sync(FULL, i < nck && (by_pos ? mt.pos : p) <= target));
					if (cnt) {
						j0 = base + cnt;
						pidx0 = __shfl_sync(FULL, p, (int)cnt - 1);
						cost0 = __shfl_sync(FULL, cc, (int)cnt - 1);
					}
					carry_p = __shfl_sync(FULL, p, 31);
					carry_c = __shfl_sync(FULL, cc, 31);
					if (cnt < 32) break;
				}
			}
			if (j0 == 0) {
				walker_init(e, k);
			} else {
				walker_load(e, k, ck_base + (size_t)ck_live[j0 - 1] * nck + (j0 - 1), &ws->bar, parity);
				// the record's own counters date from the proposal that wrote it; the running sums are current
				k.delta = k.pos - pidx0;
				k.t.total = cost0;
				if (lane == 0) cs.ck_bytes += sizeof(Record);
			}
			ck.next = 0xffffffffu;  // no checkpoints while the prefix is priced
			ck.last_pidx = pidx0;
			ck.last_cost = cost0;
			ck.test = 0;
			if (a.repair_only) {
				// no mutation: the whole slab goes through the repair rules, every checkpoint is rewritten
				ck.next = a.stride;
				phase = 2;
				mode = WALK_REPAIR;
			}
		}
		const uint32_t start_pos = k.pos, start_pidx = walker_pidx(k);
		ck.suspend_pidx = 0xffffffffu;
		ck.deadline = a.suspend ? deadline : 0;
		if (a.suspend && a.packet_budget) {
			const unsigned long long lim = (unsigned long long)start_pidx + (a.packet_budget - packets_done);
			ck.suspend_pidx = lim < 0xffffffffull ? (uint32_t)lim : 0xffffffffu;
		}
		uint64_t pending = 0, pending_old = 0;
		uint32_t err = 0;

		// One proposal = a small state machine around ONE walk call site, ONE finder call site and
		// ONE place that prices a packet chosen outside the walk:
		//   phase 0  price the prefix up to the target packet (neighbour.c:22-32, from the
		//            checkpoint instead of from byte 0), then mutate it (neighbour.c:119-152)
		//   phase 1  repair + price the next three packets (neighbour.c:82-98, count < 4)
		//   phase 2  repair + price the rest, writing fresh checkpoints
		const bool by_pos = a.regions != nullptr;
		uint32_t stop_pidx = (resumed || by_pos || a.repair_only) ? 0xffffffffu : target;
		uint32_t stop_pos = (by_pos && phase == 0) ? target : n;
		uint32_t pos = 0, byte0 = 0;       // the mutated packet's position and data byte
		uint64_t first = 0, newpk = 0, override_pk = 0, excluded = 0;
		uint32_t override_pos = 0xffffffffu;
		uint32_t want_find = 0;            // 1 mutation pick, 2 repair pick
		bool pick_best = false, failed = false, suspended = false, gave_up = false;
		for (;;) {
			const uint32_t res = walk(mode, e, k, stop_pos, stop_pidx, ck, &lg, override_pos, override_pk, pending, pending_old, err);
			if (res == WALK_ERROR) {
				st.err = err;
				break;
			}
			if (res == WALK_REJOINED) break;
			if (res == WALK_SUSPENDED) {
				suspended = true;
				break;
			}
			if (res == WALK_NEED_FIND) {
				pick_best = rng31(rng) % 4 == 0;  // neighbour.c:107
				excluded = pending;
				want_find = 2;
			} else if (phase == 0) {
				if (by_pos && (k.pos >= n || k.pos >= reg_hi)) {
					failed = true;  // no packet starts in the rest of the chain's range: not an evaluation
					break;
				}
				if (k.pos >= n) {
					st.err = ERR_NOT_BOUNDARY;
					break;
				}
				stop_pos = n;
				// ---- mutate ----------------------------------------------------------------------
				pos = k.pos;
				if (pos - k.w.base >= 32u) {
					tally_flush(k.t);
					window_seek(lane, k.w, slab, a.data, n, pos, e.stage_addr);
				}
				const uint32_t meta0 = window_meta(k.w, pos);
				const uint32_t dist0 = window_dist(k.w, pos);
				first = pk_pack(meta_type(meta0), dist0, meta_len(meta0));
				byte0 = meta_byte(meta0) & 0xff;
				want_find = 1;
				excluded = first;
				pick_best = false;
				if (pos + 1 < n && rng31(rng) % 2 == 0) {
					const uint64_t second = slab[pos + 1];
					const uint32_t ft = pk_type(first), flen = pk_len(first);
					const uint32_t stype = pk_type(second), slen = pk_len(second), sdist = pk_dist(second);
					if ((ft == T_LONG_REP || ft == T_MATCH) && flen > 2) {
						newpk = PK_LITERAL;
						override_pos = pos + 1;
						override_pk = pk_pack(ft, pk_dist(first), flen - 1);
						log_put(lane, lg, pos, newpk);
						lg.dup_index = lg.stored;
						log_put(lane, lg, pos + 1, override_pk);
						lg.dup_pos = pos + 1;  // a later repair of this slot rewrites the entry in place
						want_find = 0;
					} else if ((ft == T_LITERAL || ft == T_SHORT_REP) && (stype == T_MATCH || stype == T_LONG_REP)) {
						const int64_t src =
						    (int64_t)pos - (int64_t)(stype == T_LONG_REP ? model_rep(walker_model(e, k), sdist & 3) : sdist);
						if (slen < MAX_MATCH && src > 0 && byte0 == a.data[src - 1]) {
							newpk = pk_pack(stype, sdist, slen + 1);
							log_put(lane, lg, pos, newpk);
							want_find = 0;
						}
					}
				}
				ck.next = (j0 + 1) * a.stride;  // from here on the walk refreshes the checkpoints it passes
			} else if (phase == 1) {
				phase = 2;
				mode = WALK_REPAIR;
				stop_pidx = 0xffffffffu;
				ck.test = a.early_exit;  // from the fourth packet on the walk may re-join the current slab's trajectory
				continue;
			} else {
				break;  // reached the end of the slab
			}

			if (want_find) {
				if (lane == 0) cs.finds++;
				const long long t_find = clock64();
				// in a clock-boxed launch the finder may give a long bucket up - never on the launch's first
				// proposal, so every launch makes progress
				// The finder is not inlined, and the registers it gets are the ones this kernel does not keep live
				// across the call: with the proposal's state left in registers it ran out of local memory (400 B of
				// spill stores, 71 local loads + 56 stores inside its 32-occurrence step).  So the state is parked in
				// local memory around the call - once per find instead of once per step - and the walk's lane
				// constants are rebuilt after it: 188 B of spill stores, 25 + 21 local accesses per step, the
				// finder's share of the warp time 0.31 -> 0.24 (+7.9 % evaluations/s on the bench workload,
				// profiles/r02_parked_ab.log).
				const Model fm = walker_model(e, k);
				struct Parked { Walker k; CkSink ck; EditLog lg; ChainState st; } parked = {k, ck, lg, st};
				asm volatile("" ::"l"(&parked) : "memory");
				const uint32_t count = warp_find(lane, e.probs, e.trans, e.recip, &ws->fs, a.data, n, a.occ_start, a.occ, fm,
				                                 excluded, a.k, (a.suspend && attempts > 1) ? deadline : 0, a.limits);
				asm volatile("" ::"l"(&parked) : "memory");
				k = parked.k;
				ck = parked.ck;
				lg = parked.lg;
				st = parked.st;
				e = make_env(lane, ws, sh, slab, a.data, n, a.tables.litq);
				e.abs_dist = a.abs_dist;
				k.w.md_base = WINDOW_NONE;  // the finder's length tables share the window mirrors' memory
				k.w.pf_base = WINDOW_NONE;  // ... and the staging area of the next window
				if (count == FIND_GAVE_UP) {
					gave_up = true;
					break;
				}
				if (lane == 0) {
					cs.candidates += ws->fs.candidates;
					cs.chunks += ws->fs.chunks;
					cs.find_cycles += (unsigned long long)(clock64() - t_find);
				}
				uint64_t chosen = 0;
				bool have = false;
				if (count != 0) {
					// neighbour.c:48-72
					uint32_t choice = rng31(rng) % count;
					for (int i = 1; i < 8; i++) {
						const uint32_t r = rng31(rng) % count;
						choice = r > choice ? r : choice;
					}
					if (rng31(rng) % 8 == 0 || pick_best) choice = count - 1;
					chosen = ws->fs.ent_pk[ws->fs.pop_order[choice]];
					have = true;
				}
				if (want_find == 1) {
					if (!have) {
						failed = true;  // no alternative at this position: not an evaluation (main.c:81-84)
						break;
					}
					newpk = chosen;
					log_put(lane, lg, pos, newpk);
				} else {
					// repair pick: the slot keeps the forced LONG_REP(3) if the finder is empty
					newpk = have ? chosen : pending;
					if (newpk != pending_old) log_put(lane, lg, k.pos, newpk);
				}
				want_find = 0;
			}

			// ---- price a packet chosen outside the walk: the mutated one or a repair pick --------
			{
				const uint32_t type = pk_type(newpk), len = pk_len(newpk), dist = pk_dist(newpk);
				Model m = walker_model(e, k);
				if (!packet_ok(m, n, type, len, dist)) {
					st.err = ERR_BAD_PACKET;
					break;
				}
				const uint32_t byte = phase == 0 ? byte0 : a.data[k.pos];
				walker_apply(e, k, m, type, len, dist, byte);
			}
			if (phase == 0) {
				phase = 1;
				mode = WALK_REPAIR_HEAD;
				stop_pidx = walker_pidx(k) + 3;
			}
		}
		if (st.err) break;
		tally_flush(k.t);
		packets_done += walker_pidx(k) - start_pidx;
		if (lane == 0) {
			cs.packets += walker_pidx(k) - start_pidx;
			cs.bits += walker_bits(k, start_pidx);
			cs.slab_bytes += (uint64_t)(k.pos - start_pos) * 9;
			cs.ck_bytes += (uint64_t)ck.written * sizeof(Record);
		}
		if (gave_up) {
			// the deadline passed inside the match finder: the proposal is taken back whole (same generator
			// state, nothing committed) and the next launch draws it again
			rng = rng_at_start;
			attempts--;
			if (lane == 0) cs.gave_up++;
			break;
		}
		if (suspended) {
			// out of budget in the middle of the suffix: the checkpoint just written is the resume point
			st.susp_slot = k.pos / a.stride;
			st.susp_j0 = j0;
			st.susp_stored = lg.stored;
			st.susp_count = lg.count;
			st.susp_overflow = lg.overflow ? 1u : 0u;
			attempts--;  // counted by the launch that finishes it
			break;
		}
		if (failed) {
			if (a.trace && attempts <= a.trace_cap && lane == 0) {
				TraceRec r = {0, 0, 0};
				a.trace[(size_t)c * a.trace_cap + attempts - 1] = r;
			}
			continue;
		}
		if (lane == 0) cs.edits += lg.count;
		if (lg.overflow) {
			// accept/reject buffer too small for this proposal: drop it, uncounted
			if (lane == 0) cs.overflows++;
			if (a.trace && attempts <= a.trace_cap && lane == 0) {
				TraceRec r = {0, 0, lg.count};
				a.trace[(size_t)c * a.trace_cap + attempts - 1] = r;
			}
			continue;
		}

		// ---- the proposal's full cost ---------------------------------------------------------
		// A walk that re-joined the current slab's trajectory at checkpoint `converged` prices the
		// rest exactly as the current slab does: its cost and packet count are the current totals
		// minus what the current slab had spent up to that checkpoint.
		uint64_t cost = k.t.total;
		uint32_t live_new = walker_pidx(k);
		uint32_t flip_end = nck;  // checkpoints j0+1 .. flip_end were rewritten by this proposal
		if (ck.converged) {
			uint32_t old_pidx;
			uint64_t old_cost;
			ck_absolute(lane, ck_meta, ck_live, nck, ck.converged, old_pidx, old_cost);
			cost += st.slab_cost - old_cost;
			live_new += st.live_count - old_pidx;
			flip_end = ck.converged;
			if (lane == 0) cs.rejoined++;
		}

		// ---- accept / reject: main.c:86-96 ---------------------------------------------------
		const uint32_t r = rng31(rng);
		bool uphill;
		if (a.schedule == 0) {
			const uint64_t i = (uint64_t)first_eval + done;
			const uint64_t mod = i * i + 1 + (uint64_t)a.step * (uint64_t)a.num_iters / 2;
			const uint64_t x = (uint64_t)r % mod;
			uphill = x * x < (uint64_t)a.num_iters;
		} else {
			const float ex = -__logf(((float)r + 0.5f) * (1.0f / 2147483648.0f));
			uphill = (float)(cost - st.cur_cost) <= temp * ex;
		}
		uint32_t flags = 1;
		if (st.cur_cost == 0 || cost < st.cur_cost || uphill || a.repair_only) {
			flags |= 2;
			st.cur_cost = cost;
			st.slab_cost = cost;
			st.live_count = live_new;
			// commit the accept/reject buffer and the checkpoints written on the way
			__syncwarp();
			for (uint32_t i = lane; i < lg.stored; i += 32) slab[lg.e[i].pos] = lg.e[i].pk;
			for (uint32_t j = j0 + lane; j < flip_end; j += 32) ck_live[j] ^= 1;
			__syncwarp();
			if (lane == 0) cs.accepted++;
			// The best slab is kept in step with the current one through a journal of accepted
			// edits (src/main.c:89-92 copies the whole slab on every new best; early in a run that
			// is nearly every proposal).  Only a journal overflow falls back to a full copy.
			Edit* jl = a.track_best ? a.journal + (size_t)c * JOURNAL_CAP : nullptr;
			if (jl && !st.journal_overflow) {
				if (st.journal_count + lg.stored <= JOURNAL_CAP) {
					for (uint32_t i = lane; i < lg.stored; i += 32) jl[st.journal_count + i] = lg.e[i];
					st.journal_count += lg.stored;
				} else {
					st.journal_overflow = 1;
				}
			}
			if (st.best_cost == 0 || cost < st.best_cost) {
				st.best_cost = cost;
				flags |= 4;
				if (lane == 0) cs.new_best++;
				if (jl) {
					uint64_t* best = a.bests + (size_t)c * n;
					__syncwarp();
					if (st.journal_overflow) {
						if ((((uintptr_t)slab | (uintptr_t)best) & 15) == 0) {
							const uint4* src4 = reinterpret_cast<const uint4*>(slab);
							uint4* dst4 = reinterpret_cast<uint4*>(best);
							const uint32_t n4 = n / 2;
							uint32_t i = lane;
							for (; i + 96 < n4; i += 128) {
								const uint4 v0 = src4[i], v1 = src4[i + 32], v2 = src4[i + 64], v3 = src4[i + 96];
								dst4[i] = v0;
								dst4[i + 32] = v1;
								dst4[i + 64] = v2;
								dst4[i + 96] = v3;
							}
							for (; i < n4; i += 32) dst4[i] = src4[i];
							if ((n & 1) && lane == 0) best[n - 1] = slab[n - 1];
						} else {
							uint32_t i = lane;
							for (; i + 96 < n; i += 128) {
								const uint64_t v0 = slab[i], v1 = slab[i + 32], v2 = slab[i + 64], v3 = slab[i + 96];
								best[i] = v0;
								best[i + 32] = v1;
								best[i + 64] = v2;
								best[i + 96] = v3;
							}
							for (; i < n; i += 32) best[i] = slab[i];
						}
						if (lane == 0) cs.slab_bytes += 16ull * n;
					} else {
						// later entries win: inside a step through match_any, across steps by order
						for (uint32_t base = 0; base < st.journal_count; base += 32) {
							const uint32_t i = base + lane;
							const bool valid = i < st.journal_count;
							const uint32_t jpos = valid ? jl[i].pos : 0xffffff00u + (uint32_t)lane;
							const uint64_t jpk = valid ? jl[i].pk : 0;
							const uint32_t peers = __match_any_sync(FULL, jpos);
							if (valid && (peers >> lane) == 1u) best[jpos] = jpk;
							__syncwarp();
						}
						if (lane == 0) cs.slab_bytes += 24ull * st.journal_count;
					}
					st.journal_count = 0;
					st.journal_overflow = 0;
				}
			}
		}
		if (a.trace && attempts <= a.trace_cap && lane == 0) {
			TraceRec rec = {cost, flags, lg.count};
			a.trace[(size_t)c * a.trace_cap + attempts - 1] = rec;
		}
		done++;
		__syncwarp();
	}

	asm volatile("cp.async.wait_group 0;" ::: "memory");
	if (lane == 0) {
		cs.evals = done;
		cs.attempts = attempts;
		cs.chain_cycles = (unsigned long long)(clock64() - t_start);
		if (!a.repair_only) st.rng = rng;
		st.eval_index = first_eval + done;
		a.state[c] = st;
		a.stats[c] = ws->stats;
		a.attempts_out[c] = attempts;
	}
}

// ---- K5: range coder over one slab (src/range_encoder.c) -------------------------------------------
struct EncodeArgs {
	const uint8_t* data;
	uint32_t n;
	const uint64_t* slab;
	uint8_t* out;
	uint32_t cap;
	uint32_t* out_len;
	uint32_t* out_err;
	uint32_t* out_events;  // events coded (modelled bits + direct-bit groups)
	unsigned long long* out_wait;  // [3] clocks each strand spent waiting for its neighbour (producer, range, low), or null
	Tables tables;
};

struct RangeCoder {
	uint64_t low;
	uint32_t range;
	uint32_t cache;
	uint64_t cache_size;
	uint8_t* out;
	uint32_t cap, len;
};

__device__ __forceinline__ void rc_put(RangeCoder& rc, uint32_t b)
{
	if (rc.len < rc.cap) rc.out[rc.len] = (uint8_t)b;
	rc.len++;
}

// src/range_encoder.c:18-38
__device__ __forceinline__ void rc_shift_low(RangeCoder& rc)
{
	const uint32_t hi = (uint32_t)(rc.low >> 32), lo = (uint32_t)rc.low;
	if (lo < 0xFF000000u || hi != 0) {
		uint32_t first = rc.cache;
		do {
			rc_put(rc, (first + (hi & 0xff)) & 0xff);
			first = 0xff;
		} while (--rc.cache_size != 0);
		rc.cache = (lo >> 24) & 0xff;
	}
	rc.cache_size++;
	rc.low = (uint64_t)(lo << 8);
}

// src/range_encoder.c:47-64
__device__ __forceinline__ void rc_bit(RangeCoder& rc, uint32_t bit, uint32_t prob)
{
	const uint32_t bound = (rc.range >> 11) * prob;
	if (bit) {
		rc.low += bound;
		rc.range -= bound;
	} else {
		rc.range = bound;
	}
	while ((rc.range & 0xFF000000u) == 0) {
		rc.range <<= 8;
		rc_shift_low(rc);
	}
}

// src/range_encoder.c:66-81
__device__ __forceinline__ void rc_direct(RangeCoder& rc, uint32_t bits, uint32_t nbits)
{
	while (nbits) {
		nbits--;
		rc.range >>= 1;
		if ((bits >> nbits) & 1) rc.low += rc.range;
		if ((rc.range & 0xFF000000u) == 0) {
			rc.range <<= 8;
			rc_shift_low(rc);
		}
	}
}

// One CTA of three warps joined by two rings in shared memory - a pipeline of the coder's three strands:
//   warp 0 (producer) walks the slab with the model exactly as the scorer does and appends each packet's
//          (bit, probability) events - in the reference's coding order, direct bits included - to ring A;
//          plain literals (nine events from nine lanes, no cross-lane traffic) take a short path;
//   warp 1, lane 0 (range) runs the one strictly sequential recurrence of the whole path, the range
//          (src/range_encoder.c:47-81): per event range -> range >> 11 -> multiply-add -> normalise, and nothing
//          else.  Events come pre-digested: q = the probability of the coded bit (p or 2048 - p), so that the new
//          range is (range >> 11) * q + (bit ? range & 2047 : 0) for either bit value - one multiply-add, no
//          select.  What the event adds to `low` and whether it shifts go to ring B;
//   warp 2, lane 0 (low) adds up `low`, propagates carries and writes the bytes (src/range_encoder.c:18-45).
//          `low` never feeds back into the range, so this strand only has to keep pace.
// The three warps sit on different schedulers of the SM.  Round 1 ran everything back to back on one warp (1.2 s per
// MiB), the first split (model walk | coder) took 0.39 s; the range chain alone is ~15 dependent cycles per event.
constexpr uint32_t ENC_RING = 8192;   // ring A, events; a packet appends at most 28
constexpr uint32_t ENC_RING_B = 4096; // ring B, (add, shifts) pairs
constexpr uint32_t ENC_DIRECT = 0x80000000u;

struct EncodeShared {
	Record rec;
	uint32_t ring[ENC_RING];
	uint2 ring_b[ENC_RING_B];
	unsigned char stage[STAGE_BYTES];
	uint32_t head;    // events produced so far (producer writes, range reads)
	uint32_t tail;    // events consumed so far
	uint32_t head_b;  // ring B entries produced (range writes, low reads)
	uint32_t tail_b;
	uint32_t done;    // 1 = producer finished, 2 = producer stopped on an error
	uint32_t done_b;  // range strand finished
	uint32_t err;
};

__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p)
{
	uint32_t v;
	asm volatile("ld.acquire.cta.shared.u32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
	return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v)
{
	asm volatile("st.release.cta.shared.u32 [%0], %1;" ::"r"(smem_u32(p)), "r"(v) : "memory");
}

// event word of a modelled bit coded at probability p (of a zero): q | bit << 15
__device__ __forceinline__ uint32_t enc_event(uint32_t p, uint32_t bit) { return (bit ? 2048u - p : p) | (bit << 15); }

// The producer publishes `head` (a fence + a store) once per ENC_PUBLISH events, not per packet.
constexpr uint32_t ENC_PUBLISH = 256;

// The packets of [m.pos, end): encode_kernel from a fresh model (start = null) up to n, encode_chunks_kernel from the
// checkpoint record `start`, TMA-loaded on `bar`.  (The extra block and the copy of `end` keep encode_kernel's
// machine code what it was before the chunk kernel shared this function.)
__device__ __forceinline__ void encode_produce(EncodeShared* sh, const EncodeArgs& a, int lane, const Record* start,
                                               uint32_t end, uint64_t* bar)
{
	Model m;
	const SmemU16 probs{smem_u32(sh->rec.probs)};
	{
		if (start) {
			uint64_t cost;
			uint32_t parity = 0;
			record_load(lane, &sh->rec, m, cost, start, bar, parity);
			// the walk stores probabilities pre-shifted (p << PROB_SHIFT), the range coder keeps plain ones
			for (uint32_t i = (uint32_t)lane; i < S_COUNT; i += 32) probs.set(i, probs.get(i) >> PROB_SHIFT);
			__syncwarp();
		} else {
			model_init(lane, probs, m, 1024);
		}
	}
	Window w;
	w.base = WINDOW_NONE;
	w.pf_base = WINDOW_NONE;
	uint32_t head = 0, published = 0, tail_seen = 0, err = 0;
	unsigned long long waited = 0;
	const uint32_t ring = smem_u32(sh->ring);
	const uint32_t stage = smem_u32(sh->stage);
	// literal lanes: lane 0 is_match, lanes 1..8 tree depth 0..7 (slot map in mg_device.cuh); per-lane constants of
	// the plain tree as in make_env(): slot byte offset = first + u + (u & hm), u = ((b >> sh) & mask) ^ x
	const bool tree = lane >= 1 && lane <= 8;
	const uint32_t depth = tree ? (uint32_t)lane - 1 : 0;
	uint32_t lit_first = 2u * S_DUMMY, lit_sh = 8, lit_mask = 0, lit_x = 0, lit_hm = 0;
	if (lane == 0) lit_first = 2u * S_ISMATCH;
	else if (tree && depth <= 3) { lit_first = 2u * (S_LIT0 + 2u * (1u << depth)); lit_sh = 6 - depth; lit_mask = ((1u << depth) - 1u) << 2; }
	else if (tree && depth == 4) { lit_first = 2u * (S_LIT0 + 32); lit_sh = 2; lit_mask = 0x3c; lit_x = LITX4 << 2; }
	else if (tree && depth == 5) { lit_first = 2u * (S_LIT0 + 96); lit_sh = 2; lit_mask = 0x3e; lit_x = LITX5 << 1; }
	else if (tree && depth == 6) { lit_first = 2u * (S_LIT0 + 160); lit_sh = 1; lit_mask = 0x7e; lit_x = LITX6 << 1; lit_hm = 64; }
	else if (tree && depth == 7) { lit_first = 2u * (S_LIT0 + 288); lit_sh = 0; lit_mask = 0xfe; lit_x = LITX7 << 1; lit_hm = 0xc0; }
	const uint32_t lit_addr = probs.a + lit_first;
	const uint32_t stop = end;
	while (m.pos < stop) {
		// room for a whole window of literals (32 x 9 events; the largest other packet appends 28)?
		if (head + 288 - tail_seen > ENC_RING) {
			const long long t0 = clock64();
			while (head + 288 - tail_seen > ENC_RING) {
				if (published != head) {
					__syncwarp();
					if (lane == 0) st_release_u32(&sh->head, head);
					published = head;
				}
				tail_seen = ld_acquire_u32(&sh->tail);
				if (head + 288 - tail_seen > ENC_RING) __nanosleep(64);
			}
			waited += (unsigned long long)(clock64() - t0);
		}
		window_seek(lane, w, a.slab, a.data, a.n, m.pos, stage);
		const uint32_t meta = window_meta(w, m.pos);
		if ((meta & 0xffffu) == META_LITERAL && m.ctx < 7) {
			// ---- run of plain literals (src/lzma_packet_encoder.c:106-121): every lane follows its own slot
			// class through the run, nine events per literal straight into the ring -----------------------
			const uint32_t idx = m.pos - w.base;
			uint32_t run = (uint32_t)__ffs((int)~(w.litmask >> idx)) - 1u;  // 0xffffffff when every slot up to the window's end is one
			run = run < 32u - idx ? run : 32u - idx;
			run = run < stop - m.pos ? run : stop - m.pos;
			uint32_t cj = m.ctx;
			uint32_t at = head + (uint32_t)lane;
			for (uint32_t i = 0; i < run; i++) {
				const uint32_t b = (__shfl_sync(FULL, w.meta, (int)(idx + i)) >> 16) & 0xffu;
				if (lane <= 8) {
					const uint32_t u = ((b >> lit_sh) & lit_mask) ^ lit_x;
					const uint32_t addr = lit_addr + u + (u & lit_hm) + (lane == 0 ? 2u * cj : 0u);
					const uint32_t bit = tree ? (b >> (7 - depth)) & 1u : 0u;
					const uint32_t p = lds_u16(addr);
					sts_u32(ring + 4u * (at & (ENC_RING - 1)), enc_event(p, bit));
					sts_u16(addr, bit ? p - (p >> 5) : p + ((2048u - p) >> 5));
				}
				at += 9;
				cj = cj < 4 ? 0u : cj - 3;
			}
			m.ctx = cj;
			head += 9 * run;
			m.pos += run;
			m.pidx += run;
		} else {
			const uint32_t type = meta_type(meta), len = meta_len(meta), dist = window_dist(w, m.pos);
			const uint32_t byte = meta_byte(meta) & 0xff;
			if (!packet_ok(m, a.n, type, len, dist)) {
				err = ERR_BAD_PACKET;
				break;
			}
			uint32_t mbyte = 0;
			if (type == T_LITERAL && m.ctx >= 7) mbyte = a.data[m.pos - m.rep0 - 1];
			DistParts dp;
			dp.pslot = dp.nlow = dp.low = dp.rbase = dp.rbits = dp.direct = 0;
			if (type == T_MATCH) dp = dist_parts(dist);
			uint32_t slot = 0, bit = 0;
			const bool active = packet_event(lane, lane_role(lane), type, len, dist, m.ctx, byte, mbyte, dp, slot, bit);
			const uint32_t mask = __ballot_sync(FULL, active);
			// lanes are in coding order; the direct bits of a far match sit before the reverse-tree lanes
			const uint32_t has_direct = dp.direct ? 1u : 0u;
			const uint32_t before_direct = __popc(mask & ((1u << FIRST_REVTREE_LANE) - 1u));
			if (active) {
				const uint32_t p = probs.get(slot);
				const uint32_t rank = __popc(mask & ((1u << lane) - 1u)) + (lane >= FIRST_REVTREE_LANE ? has_direct : 0u);
				sts_u32(ring + 4u * ((head + rank) & (ENC_RING - 1)), enc_event(p, bit));
				probs.set(slot, bit ? p - (p >> 5) : p + ((2048u - p) >> 5));
			}
			if (lane == 0 && has_direct)
				sts_u32(ring + 4u * ((head + before_direct) & (ENC_RING - 1)),
				        ENC_DIRECT | (dp.direct << 26) | ((dist & ((1u << dp.nlow) - 1u)) >> 4));
			head += __popc(mask) + has_direct;
			model_advance(m, type, len, dist);
		}
		__syncwarp();  // every lane's events are in the ring (and its probabilities stored) before anything else
		if (head - published >= ENC_PUBLISH) {
			if (lane == 0) st_release_u32(&sh->head, head);
			published = head;
		}
	}
	asm volatile("cp.async.wait_group 0;" ::: "memory");
	__syncwarp();
	if (lane == 0) {
		sh->err = err;
		if (a.out_wait) a.out_wait[0] = waited;
		st_release_u32(&sh->head, head);
		st_release_u32(&sh->done, err ? 2u : 1u);
	}
}

// ---- the range strand ----
// One modelled bit (src/range_encoder.c:47-64).  With bound = (range >> 11) * p:
//   bit 0: range' = bound,         low unchanged      = (range >> 11) * q                     (q = p)
//   bit 1: range' = range - bound, low += bound       = (range >> 11) * q + (range & 2047)    (q = 2048 - p)
// The state is kept as hi = range >> 11 and the kept low bits of the NEXT event, both selected from the two
// normalisation outcomes in parallel with the test, so that the dependent chain per event is multiply-add ->
// select -> multiply-add.  p stays within [31, 2017] (src/probability_model.c:5-15): one shift always suffices.
struct RangeChain {
	uint32_t range;  // the reference's range (normalised)
	uint32_t hi;     // range >> 11
	uint32_t lk;     // range & (the coming event codes a 1 ? 2047 : 0); only valid between range_event calls that pass keep_next
};

__device__ __forceinline__ uint32_t enc_keep(uint32_t e) { return (e >> 15) ? 2047u : 0u; }

// keep_next = enc_keep(the event after e) when it is known (then ch.lk stays valid), anything otherwise.
// Returns what the event means for `low`: x = the amount added, y = 1 when the coder shifts after it.
__device__ __forceinline__ uint2 range_event(RangeChain& ch, uint32_t e, uint32_t keep_next)
{
	const uint32_t q = e & 0x7fffu;
	const uint32_t next = ch.hi * q + ch.lk;
	uint2 out;
	out.x = (e >> 15) ? ch.range - next : 0u;
	const bool shift = (next & 0xFF000000u) == 0;
	out.y = shift ? 1u : 0u;
	ch.hi = shift ? next >> 3 : next >> 11;
	ch.lk = shift ? ((next & 7u) << 8) & keep_next : next & keep_next;
	ch.range = shift ? next << 8 : next;
	return out;
}

struct RingBWriter {
	uint32_t ring;  // shared address of ring_b
	uint32_t head, published, tail_seen;
	EncodeShared* sh;
	unsigned long long waited;
};

__device__ __forceinline__ void ring_b_room(RingBWriter& wb, uint32_t want)
{
	if (wb.head + want - wb.tail_seen <= ENC_RING_B) return;
	const long long t0 = clock64();
	while (wb.head + want - wb.tail_seen > ENC_RING_B) {
		if (wb.published != wb.head) {
			st_release_u32(&wb.sh->head_b, wb.head);
			wb.published = wb.head;
		}
		wb.tail_seen = ld_acquire_u32(&wb.sh->tail_b);
	}
	wb.waited += (unsigned long long)(clock64() - t0);
}

__device__ __forceinline__ void ring_b_put(RingBWriter& wb, uint2 v)
{
	asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(wb.ring + 8u * (wb.head & (ENC_RING_B - 1))), "r"(v.x), "r"(v.y) : "memory");
	wb.head++;
}

// any event, nothing known about its neighbours (src/range_encoder.c:66-81 for the direct bits)
__device__ __forceinline__ void range_any(RangeChain& ch, RingBWriter& wb, uint32_t e)
{
	if (e & ENC_DIRECT) {
		uint32_t range = ch.range, nbits = (e >> 26) & 31u;
		const uint32_t bits = e & 0x3ffffffu;
		ring_b_room(wb, nbits);
		while (nbits) {
			nbits--;
			range >>= 1;
			uint2 out;
			out.x = ((bits >> nbits) & 1u) ? range : 0u;
			out.y = 0;
			if ((range & 0xFF000000u) == 0) {
				range <<= 8;
				out.y = 1;
			}
			ring_b_put(wb, out);
		}
		ch.range = range;
		ch.hi = range >> 11;
	} else {
		ch.lk = ch.range & enc_keep(e);
		ring_b_put(wb, range_event(ch, e, 0));
	}
}

__device__ __forceinline__ void encode_range(EncodeShared* sh, const EncodeArgs& a)
{
	RangeChain ch = {0xFFFFFFFFu, 0xFFFFFFFFu >> 11, 0};
	RingBWriter wb = {smem_u32(sh->ring_b), 0, 0, 0, sh, 0};
	uint32_t tail = 0;
	unsigned long long starved = 0;
	const uint32_t ring = smem_u32(sh->ring);
	for (;;) {
		uint32_t head = ld_acquire_u32(&sh->head);
		if (head == tail) {
			if (ld_acquire_u32(&sh->done) == 0) {
				const long long t0 = clock64();
				__nanosleep(32);
				starved += (unsigned long long)(clock64() - t0);
				continue;
			}
			head = ld_acquire_u32(&sh->head);  // published before `done`
			if (head == tail) break;
		}
		// a bounded batch, so that the producer sees ring A drain (and the low strand ring B fill) while a long
		// backlog is coded
		if (head - tail > ENC_RING / 8) head = tail + ENC_RING / 8;
		while (tail != head && (tail & 3u) != 0) {
			ring_b_room(wb, 1);
			range_any(ch, wb, lds_u32(ring + 4u * (tail & (ENC_RING - 1))));
			tail++;
		}
		// groups of four events per 16-byte load, the next group in flight while this one is coded
		if (head - tail >= 4) {
			uint4 v = lds_v4(ring + 4u * (tail & (ENC_RING - 1)));
			while (head - tail >= 4) {
				const uint4 cur = v;
				v = lds_v4(ring + 4u * ((tail + 4) & (ENC_RING - 1)));  // may run past head: never used then
				tail += 4;
				ring_b_room(wb, 4);
				if ((cur.x | cur.y | cur.z | cur.w) & ENC_DIRECT) {
					range_any(ch, wb, cur.x);
					range_any(ch, wb, cur.y);
					range_any(ch, wb, cur.z);
					range_any(ch, wb, cur.w);
				} else {
					ch.lk = ch.range & enc_keep(cur.x);
					const uint2 o0 = range_event(ch, cur.x, enc_keep(cur.y));
					const uint2 o1 = range_event(ch, cur.y, enc_keep(cur.z));
					const uint2 o2 = range_event(ch, cur.z, enc_keep(cur.w));
					const uint2 o3 = range_event(ch, cur.w, 0);
					// four entries = two 16-byte stores (ring B never wraps inside a group: its head stays a multiple
					// of 2 only if no direct bits came before - so store entry by entry unless aligned)
					if ((wb.head & 1u) == 0) {
						const uint32_t at0 = wb.ring + 8u * (wb.head & (ENC_RING_B - 1));
						const uint32_t at1 = wb.ring + 8u * ((wb.head + 2) & (ENC_RING_B - 1));
						sts_v4(at0, o0.x, o0.y, o1.x, o1.y);
						sts_v4(at1, o2.x, o2.y, o3.x, o3.y);
						wb.head += 4;
					} else {
						ring_b_put(wb, o0);
						ring_b_put(wb, o1);
						ring_b_put(wb, o2);
						ring_b_put(wb, o3);
					}
				}
			}
		}
		while (tail != head) {
			ring_b_room(wb, 1);
			range_any(ch, wb, lds_u32(ring + 4u * (tail & (ENC_RING - 1))));
			tail++;
		}
		st_release_u32(&sh->tail, tail);
		st_release_u32(&sh->head_b, wb.head);
		wb.published = wb.head;
	}
	if (a.out_wait) a.out_wait[1] = starved + wb.waited;
	st_release_u32(&sh->head_b, wb.head);
	st_release_u32(&sh->done_b, 1u);
}

// ---- the low strand: low += what each event added, shift when it shifted (src/range_encoder.c:18-45) ----
// A whole warp takes 32 ring-B entries per step, one per lane.  `low` only changes what is written at a SHIFT, so
// the adds between two shifts are summed first - a segmented scan across the lanes (segments end at the lanes
// that shift; the sum of a segment is below 2^32: the coder's range bounds everything added between two
// normalisations) - and lane 0 then performs one `low += sum; shift` per shift of the step, about four per 32 entries.
__device__ __forceinline__ void encode_low(EncodeShared* sh, const EncodeArgs& a, int lane)
{
	RangeCoder rc = {0, 0xFFFFFFFFu, 0, 1, a.out, a.cap, 0};  // lane 0's copy is the coder
	uint32_t tail = 0, pending = 0;  // pending: adds since the last shift (uniform)
	unsigned long long starved = 0;
	const uint32_t ring = smem_u32(sh->ring_b);
	for (;;) {
		uint32_t head = ld_acquire_u32(&sh->head_b);
		if (head == tail) {
			if (ld_acquire_u32(&sh->done_b) == 0) {
				const long long t0 = clock64();
				__nanosleep(32);
				starved += (unsigned long long)(clock64() - t0);
				continue;
			}
			head = ld_acquire_u32(&sh->head_b);
			if (head == tail) break;
		}
		if (head - tail > ENC_RING_B / 4) head = tail + ENC_RING_B / 4;
		while (tail != head) {
			const uint32_t cnt = head - tail < 32u ? head - tail : 32u;
			uint32_t add = 0, shifts = 0;
			if ((uint32_t)lane < cnt)
				asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(add), "=r"(shifts) : "r"(ring + 8u * ((tail + (uint32_t)lane) & (ENC_RING_B - 1))) : "memory");
			tail += cnt;
			const uint32_t m = __ballot_sync(FULL, shifts != 0);
			const uint32_t seg = (uint32_t)__popc(m & ((1u << lane) - 1u));  // shifts before this entry
			// inclusive segmented sum: a lane that shifts ends up with everything added since the shift before it
			uint32_t x = add;
#pragma unroll
			for (int d = 1; d < 32; d <<= 1) {
				const uint32_t y = __shfl_up_sync(FULL, x, d), sg = __shfl_up_sync(FULL, seg, d);
				if (lane >= d && sg == seg) x += y;
			}
			// what follows the step's last shift carries over to the next step
			const uint32_t nshift = (uint32_t)__popc(m);
			const uint32_t trailing = __reduce_add_sync(FULL, seg == nshift ? add : 0u);
			uint32_t todo = m;
			bool first = true;
			while (todo) {
				const int who = __ffs((int)todo) - 1;
				todo &= todo - 1;
				const uint32_t sum = __shfl_sync(FULL, x, who);
				if (lane == 0) {
					rc.low += (uint64_t)sum + (first ? pending : 0u);
					rc_shift_low(rc);
				}
				first = false;
			}
			pending = (nshift ? 0u : pending) + trailing;
		}
		if (lane == 0) st_release_u32(&sh->tail_b, tail);
		__syncwarp();
	}
	if (lane == 0) {
		rc.low += pending;
		for (int i = 0; i < 5; i++) rc_shift_low(rc);  // src/range_encoder.c:40-45
		const uint32_t err = sh->err;
		*a.out_len = rc.len;
		*a.out_err = err | (rc.len > rc.cap ? ERR_OUTPUT_FULL : 0);
		*a.out_events = ld_acquire_u32(&sh->tail);
		if (a.out_wait) a.out_wait[2] = starved;
	}
}

__global__ void __launch_bounds__(96) encode_kernel(EncodeArgs a)
{
	extern __shared__ __align__(128) unsigned char smem_raw[];
	EncodeShared& sh = *reinterpret_cast<EncodeShared*>(smem_raw);
	if (threadIdx.x == 0) {
		sh.head = sh.tail = sh.head_b = sh.tail_b = sh.done = sh.done_b = sh.err = 0;
	}
	__syncthreads();
	if (threadIdx.x < 32)
		encode_produce(&sh, a, (int)threadIdx.x, nullptr, a.n, nullptr);
	else if (threadIdx.x == 32)
		encode_range(&sh, a);
	else if (threadIdx.x >= 64)
		encode_low(&sh, a, (int)threadIdx.x - 64);
}

// ---- K8: the chunks of an LZMA2 stream, one CTA each ------------------------------------------------------
// An LZMA2 chunk that resets nothing keeps the probabilities, automaton state and rep distances of the chunk before
// it and restarts only the range coder.  So once the model at each chunk's start is known - a checkpoint record of
// the plan walk (score_kernel) - every chunk is an independent LZMA-alone payload: encode_kernel's three strands
// over [bounds[c], bounds[c + 1]), started from that record, with a fresh coder that flushes at the chunk's end.
constexpr uint32_t NO_RECORD = 0xffffffffu;
struct ChunkArgs {
	EncodeArgs enc;             // data, n, slab; out = [chunks][enc.cap] bytes; out_len, out_err, out_events = [chunks]
	const Record* ck;           // the plan walk's checkpoint records
	const uint32_t* bounds;     // [chunks + 1]: chunk c codes [bounds[c], bounds[c + 1]), all packet boundaries
	const uint32_t* start_rec;  // [chunks]: the record holding the model at bounds[c], NO_RECORD = a fresh model
};
constexpr size_t CHUNK_BAR_OFFSET = (sizeof(EncodeShared) + 7) & ~(size_t)7;
constexpr size_t CHUNK_SMEM = CHUNK_BAR_OFFSET + sizeof(uint64_t);

__global__ void __launch_bounds__(96) encode_chunks_kernel(ChunkArgs c)
{
	extern __shared__ __align__(128) unsigned char smem_raw[];
	EncodeShared& sh = *reinterpret_cast<EncodeShared*>(smem_raw);
	uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + CHUNK_BAR_OFFSET);
	const uint32_t chunk = blockIdx.x;
	EncodeArgs a = c.enc;
	a.out += (size_t)chunk * a.cap;
	a.out_len += chunk;
	a.out_err += chunk;
	a.out_events += chunk;
	a.out_wait = nullptr;
	if (threadIdx.x == 0) {
		sh.head = sh.tail = sh.head_b = sh.tail_b = sh.done = sh.done_b = sh.err = 0;
		mbar_init(bar, 1);
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
	}
	__syncthreads();
	if (threadIdx.x < 32) {
		const uint32_t r = c.start_rec[chunk];
		encode_produce(&sh, a, (int)threadIdx.x, r == NO_RECORD ? nullptr : c.ck + r, c.bounds[chunk + 1], bar);
	} else if (threadIdx.x == 32) {
		encode_range(&sh, a);
	} else if (threadIdx.x >= 64) {
		encode_low(&sh, a, (int)threadIdx.x - 64);
	}
}

// ---- slab format conversion: host LZMAPacket (12 B) <-> packed u64 ----------------------------------
__global__ void pack_kernel(const uint32_t* __restrict__ raw, uint64_t* __restrict__ packed, size_t count)
{
	for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
		const uint32_t type = raw[i * 3] & 0xff, dist = raw[i * 3 + 1], len = raw[i * 3 + 2] & 0xffff;
		packed[i] = pk_pack(type, dist, len);
	}
}

__global__ void unpack_kernel(const uint64_t* __restrict__ packed, uint32_t* __restrict__ raw, size_t count)
{
	for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
		const uint64_t p = packed[i];
		raw[i * 3] = pk_type(p);
		raw[i * 3 + 1] = pk_dist(p);
		raw[i * 3 + 2] = pk_len(p);
	}
}

__global__ void fill_literal_kernel(uint64_t* __restrict__ packed, size_t count)
{
	for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x)
		packed[i] = PK_LITERAL;
}

// Copies one block of `words` 16-byte words to `copies` destinations `stride` words apart (slab,
// checkpoint and index replication when many chains start from the same slab): one launch
// instead of one cudaMemcpyAsync per chain.
__global__ void replicate_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, size_t words, size_t stride,
                                 uint32_t copies)
{
	for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < words; i += (size_t)gridDim.x * blockDim.x) {
		const uint4 v = src[i];
		for (uint32_t c = 0; c < copies; c++) dst[(size_t)c * stride + i] = v;
	}
}

// Cooperative regions, pass A: for every LONG_REP slot on the live path of region r's owner chain, the
// absolute distance it stands for there (rep distances only: no probabilities, one thread per region,
// started from the owner's last checkpoint at or before the region).
__global__ void region_abs_reps_kernel(const uint64_t* __restrict__ slabs, uint32_t n, const uint32_t* __restrict__ bounds,
                                       const uint32_t* __restrict__ owners, uint32_t nregions, const Record* __restrict__ ck,
                                       const CkMeta* __restrict__ ck_meta, const uint8_t* __restrict__ ck_live, uint32_t nck,
                                       uint32_t has_ck, uint32_t stride, uint32_t* __restrict__ abs_dist)
{
	const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
	if (r >= nregions) return;
	const uint32_t c = owners[r], lo = bounds[r], hi = bounds[r + 1];
	if (c == 0xffffffffu) return;  // owned by another process (multi-GPU merges)
	const uint64_t* slab = slabs + (size_t)c * n;
	uint32_t pos = 0, rep[4] = {0, 0, 0, 0};
	if (has_ck) {
		uint32_t j = lo / stride;
		if (j > nck) j = nck;
		while (j > 0) {
			const uint32_t live = ck_live[(size_t)c * nck + (j - 1)];
			if (ck_meta[((size_t)c * 2 + live) * nck + (j - 1)].pos <= lo) {
				const Record* rec = ck + ((size_t)c * 2 + live) * nck + (j - 1);
				pos = rec->pos;
				for (int i = 0; i < 4; i++) rep[i] = rec->rep[i];
				break;
			}
			j--;
		}
	}
	while (pos < hi) {
		const uint64_t pk = slab[pos];
		const uint32_t type = pk_type(pk), len = pk_len(pk), dist = pk_dist(pk);
		if (type == T_MATCH) {
			rep[3] = rep[2];
			rep[2] = rep[1];
			rep[1] = rep[0];
			rep[0] = dist;
		} else if (type == T_LONG_REP) {
			const uint32_t idx = dist & 3, d = rep[idx];
			if (pos >= lo) abs_dist[pos] = d + 1;  // 0 = no entry (the parts of several processes are summed)
			for (uint32_t i = idx; i > 0; i--) rep[i] = rep[i - 1];  // src/lzma_state.c:67-81
			rep[0] = d;
		}
		pos += len ? len : 1;
	}
}

// Cooperative regions: dst[i] = slab of chain owners[r] at i, for i in region r = [bounds[r], bounds[r+1]).
__global__ void merge_regions_kernel(const uint64_t* __restrict__ slabs, uint32_t n, const uint32_t* __restrict__ bounds,
                                     const uint32_t* __restrict__ owners, uint32_t nregions, uint64_t* __restrict__ dst)
{
	for (uint32_t r = blockIdx.x; r < nregions; r += gridDim.x) {
		if (owners[r] == 0xffffffffu) continue;  // owned by another process: its slots stay 0
		const uint64_t* src = slabs + (size_t)owners[r] * n;
		for (uint32_t i = bounds[r] + threadIdx.x; i < bounds[r + 1]; i += blockDim.x) dst[i] = src[i];
	}
}

// Every slot of a slab a chain may walk must be decodable on its own terms
// (type, length, extent, absolute match distance).
__global__ void validate_kernel(const uint64_t* __restrict__ packed, uint32_t n, uint32_t* bad)
{
	for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
		const uint64_t p = packed[i];
		const uint32_t type = pk_type(p), len = pk_len(p), dist = pk_dist(p);
		bool ok = len >= 1 && len <= n - i;
		if (type == T_LITERAL || type == T_SHORT_REP) ok = ok && len == 1;
		else if (type == T_MATCH) ok = ok && len >= 2 && len <= MAX_MATCH && dist < i;
		else if (type == T_LONG_REP) ok = ok && len >= 2 && len <= MAX_MATCH && dist < 4;
		else ok = false;
		if (!ok) atomicAdd(bad, 1u);
	}
}

// ---- literal queues (walk_windows) --------------------------------------------------------------------
// One warp per 32-byte window of the input.  Lane L collects, slot by slot, the bits the window's 32 plain
// literals send to the slots of bank L (is_match[0] on lane 0: 32 zero bits), pairs them up (two steps on one
// slot = one two-step table section) and writes its entries; lanes with nothing left to do name their spare
// slot.  Steps on different slots commute, steps on one slot keep the input order: the model after the queue
// is the model after the 32 literals (src/lzma_packet_encoder.c:106-121, src/probability_model.c:5-15).
__global__ void __launch_bounds__(256) litq_build_kernel(const uint8_t* __restrict__ data, uint32_t n, uint32_t nwin, uint4* __restrict__ out)
{
	const int lane = threadIdx.x & 31;
	const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	if (w >= nwin) return;
	const uint32_t base = w * 32u;
	const uint32_t b = data[base + (uint32_t)lane];  // windows are whole: base + 32 <= n
	const uint32_t spare = 2u * (2u * (uint32_t)lane + 1u);  // row 0, odd slot of this bank
	uint32_t ent[QUEUE_MAX_ROUNDS];
	uint32_t count = 0;
#pragma unroll
	for (uint32_t i = 0; i < QUEUE_MAX_ROUNDS; i++) ent[i] = spare;
	auto put = [&](uint32_t off, uint32_t section) {
#pragma unroll
		for (uint32_t i = 0; i < QUEUE_MAX_ROUNDS; i++)
			if (i == count) ent[i] = off | (section << 13);
		count++;
	};
	// the bits the window sends to one slot (mask of window positions, bit i of `bits` = the data bit of
	// position i), in input order, two at a time
	auto emit = [&](uint32_t off, uint32_t members, uint32_t bits) {
		while (members) {
			const uint32_t i0 = (uint32_t)__ffs((int)members) - 1u;
			members &= members - 1;
			const uint32_t b0 = (bits >> i0) & 1u;
			if (members) {
				const uint32_t i1 = (uint32_t)__ffs((int)members) - 1u;
				members &= members - 1;
				put(off, 2u + (b0 << 1) + ((bits >> i1) & 1u));
			} else {
				put(off, b0);
			}
		}
	};
	if (lane == 0) emit(2u * S_ISMATCH, FULL, 0);
	for (uint32_t d = 0; d < 8; d++) {
		const uint32_t prefix = b >> (8 - d);
		const uint32_t slot = S_LIT0 + lit0_slot(d, prefix);
		const uint32_t bits = __ballot_sync(FULL, (b >> (7 - d)) & 1u);
		// every distinct slot of this depth, handled by the lane that owns its bank
		uint32_t todo = FULL;
		while (todo) {
			const int leader = __ffs((int)todo) - 1;
			const uint32_t s = __shfl_sync(FULL, slot, leader);
			const uint32_t members = __ballot_sync(FULL, slot == s);
			todo &= ~members;
			if ((int)((s >> 1) & 31u) == lane) emit(2u * s, members, bits);
		}
	}
	const uint32_t most = __reduce_max_sync(FULL, count);
	if (lane == 0) {
		if (most > QUEUE_MAX_ROUNDS) ent[0] = QUEUE_UNUSABLE;
		else if (most > QUEUE_ROUNDS) ent[0] |= QUEUE_MORE;
	}
	uint4 lo, hi, ex;
	lo.x = ent[0] | ent[1] << 16;
	lo.y = ent[2] | ent[3] << 16;
	lo.z = ent[4] | ent[5] << 16;
	lo.w = ent[6] | ent[7] << 16;
	hi.x = ent[8] | ent[9] << 16;
	hi.y = ent[10] | ent[11] << 16;
	hi.z = ent[12] | ent[13] << 16;
	hi.w = ent[14] | ent[15] << 16;
	ex.x = ent[16] | ent[17] << 16;
	ex.y = ent[18] | ent[19] << 16;
	ex.z = ent[20] | ent[21] << 16;
	ex.w = ent[22] | ent[23] << 16;
	out[(size_t)w * QUEUE_BLOCKS * 32 + (uint32_t)lane] = lo;
	out[(size_t)w * QUEUE_BLOCKS * 32 + 32 + (uint32_t)lane] = hi;
	out[(size_t)w * QUEUE_BLOCKS * 32 + 64 + (uint32_t)lane] = ex;
	(void)n;
}

// ---- K1: bigram index (src/substring_enumerator.c:26-47) ---------------------------------------------
// Stable counting sort of positions 0..n-2 by (data[i], data[i+1]).  Each warp owns a contiguous
// range of positions and a private histogram row, so the scatter needs no atomics and stays
// in ascending position order inside a bucket.
constexpr uint32_t INDEX_KEYS = 65536;

__device__ __forceinline__ void index_walk(const uint8_t* __restrict__ data, uint32_t n, uint32_t* row, uint32_t begin,
                                           uint32_t end, const uint32_t* start, uint32_t* occ)
{
	const int lane = threadIdx.x & 31;
	const uint32_t lt = (1u << lane) - 1;
	for (uint32_t base = begin; base < end; base += 32) {
		const uint32_t i = base + lane;
		const bool in = i < end;
		const uint32_t key = in ? ((uint32_t)data[i] << 8 | data[i + 1]) : 0xffffffffu;
		const uint32_t peers = __match_any_sync(FULL, key);
		const uint32_t rank = __popc(peers & lt);
		uint32_t slot = 0;
		if (in && rank == 0) {
			slot = row[key];
			row[key] = slot + __popc(peers);
		}
		slot = __shfl_sync(FULL, slot, __ffs(peers) - 1);
		if (in && occ) occ[start[key] + slot + rank] = i;
		__syncwarp();
	}
	(void)n;
}

__global__ void index_count_kernel(const uint8_t* __restrict__ data, uint32_t n, uint32_t* rows, uint32_t per_warp)
{
	const uint32_t wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const uint32_t begin = wid * per_warp;
	const uint32_t total = n - 1;
	if (begin >= total) return;
	const uint32_t end = begin + per_warp < total ? begin + per_warp : total;
	index_walk(data, n, rows + (size_t)wid * INDEX_KEYS, begin, end, nullptr, nullptr);
}

// rows[w][key] -> exclusive prefix over w; totals[key] = bucket size
__global__ void index_prefix_kernel(uint32_t* rows, uint32_t nwarps, uint32_t* totals)
{
	const uint32_t key = blockIdx.x * blockDim.x + threadIdx.x;
	if (key >= INDEX_KEYS) return;
	uint32_t run = 0;
	for (uint32_t w = 0; w < nwarps; w++) {
		const uint32_t c = rows[(size_t)w * INDEX_KEYS + key];
		rows[(size_t)w * INDEX_KEYS + key] = run;
		run += c;
	}
	totals[key] = run;
}

// start[key] = exclusive scan of totals, start[65536] = n-1.  One block of 1024 threads.
__global__ void __launch_bounds__(1024) index_scan_kernel(const uint32_t* totals, uint32_t* start)
{
	__shared__ uint32_t part[1024];
	const uint32_t tid = threadIdx.x;
	uint32_t local[64];
	uint32_t sum = 0;
	for (int i = 0; i < 64; i++) {
		local[i] = sum;
		sum += totals[tid * 64 + i];
	}
	part[tid] = sum;
	__syncthreads();
	for (uint32_t off = 1; off < 1024; off <<= 1) {
		uint32_t v = tid >= off ? part[tid - off] : 0;
		__syncthreads();
		part[tid] += v;
		__syncthreads();
	}
	const uint32_t base = part[tid] - sum;
	for (int i = 0; i < 64; i++) start[tid * 64 + i] = base + local[i];
	if (tid == 1023) start[INDEX_KEYS] = part[1023];
}

__global__ void index_scatter_kernel(const uint8_t* __restrict__ data, uint32_t n, uint32_t* rows, uint32_t per_warp,
                                     const uint32_t* start, uint32_t* occ)
{
	const uint32_t wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	const uint32_t begin = wid * per_warp;
	const uint32_t total = n - 1;
	if (begin >= total) return;
	const uint32_t end = begin + per_warp < total ? begin + per_warp : total;
	index_walk(data, n, rows + (size_t)wid * INDEX_KEYS, begin, end, start, occ);
}

// ---- K6: LZMA-alone payload -> slab (the range coder of K5 run backwards) ---------------------------------
// Range decoding is one dependent chain, so one warp: lane 0 decodes, the warp checks a match's bytes against the
// resident input 32 at a time.  The model is the reference's plain one (src/lzma_state.h:15-55, the order
// export_model maps to) with plain probabilities: the walk's bank-owned slot map and transition tables serve
// lane-parallel pricing, which a decoder has no use for.  Every decoded byte is compared with the input instead of
// being written, so a stream either decodes to exactly this input or is rejected with the position it failed at.
constexpr uint32_t DS_LIT = 0, DS_LEN = 768, DS_REPLEN = DS_LEN + 514, DS_POSSLOT = DS_REPLEN + 514;
constexpr uint32_t DS_ALIGN = DS_POSSLOT + 256, DS_POSCODER = DS_ALIGN + 16, DS_ISMATCH = DS_POSCODER + 115;
constexpr uint32_t DS_ISREP = DS_ISMATCH + 192, DS_ISREPG0 = DS_ISREP + 12, DS_ISREPG1 = DS_ISREPG0 + 12;
constexpr uint32_t DS_ISREPG2 = DS_ISREPG1 + 12, DS_ISREP0LONG = DS_ISREPG2 + 12, DS_TOTAL = DS_ISREP0LONG + 192;
constexpr uint32_t DL_CHOICE2 = 1, DL_LOW = 2, DL_MID = 2 + 128, DL_HIGH = 2 + 256;  // one length coder, pos_state 0
static_assert(DS_TOTAL == 2615, "the decoder's model is the reference's");

// what stopped the decoder (DecodeStatus.err); 0 = the stream is this input's
enum : uint32_t {
	DEC_OK = 0,
	DEC_FIRST_BYTE = 1,  // the range coder's first byte is not 0
	DEC_LITERAL = 2,     // a literal differs from the input
	DEC_SOURCE = 3,      // a match or rep reaches before position 0
	DEC_PAST_END = 4,    // a packet runs past the input's end (or a packet where only the end marker may stand)
	DEC_COPY = 5,        // a match or rep copies bytes that differ from the input
	DEC_MARKER = 6,      // an end marker before the input's end, or in a stream whose size is known
	DEC_SHORT = 7,       // the stream ends before the input does
	DEC_TRAILING = 8,    // bytes left over after the last packet
	DEC_CODE = 9         // the range decoder's code is not 0 at the end
};

struct DecodeStatus {
	uint32_t err;
	uint32_t pos;                 // position of the packet that failed (n when the end checks failed)
	unsigned long long events;    // modelled bits + direct-bit groups decoded
	unsigned long long consumed;  // payload bytes read
};

struct DecodeArgs {
	const uint8_t* data;     // the context's input (n + 32 bytes, zero padded)
	uint32_t n;
	const uint8_t* stream;   // the payload: everything after the 13-byte header
	unsigned long long len;  // its length
	uint32_t known_size;     // 1: stop at n; 0: the end marker must stand at n
	uint64_t* slab;          // n packed slots, filled with PK_LITERAL beforehand
	DecodeStatus* status;
};

constexpr uint32_t DEC_BUF = 16384;   // payload bytes staged in shared memory
constexpr uint32_t DEC_MARGIN = 256;  // restage when fewer are left: a packet reads at most 48 (one per bit, <= 48 bits)

struct RangeDecoder {
	uint16_t* probs;
	const uint8_t* buf;           // staged payload [base, base + DEC_BUF)
	unsigned long long base, at, len;
	uint32_t range, code;
	uint32_t short_read;
	unsigned long long events;
};

__device__ __forceinline__ void rd_shift(RangeDecoder& d)
{
	d.range <<= 8;
	uint32_t b = 0;
	if (d.at < d.len && d.at - d.base < DEC_BUF) b = d.buf[d.at++ - d.base];
	else d.short_read = 1;
	d.code = (d.code << 8) | b;
}

// src/range_encoder.c:47-64 and src/probability_model.c:5-15, backwards
__device__ __forceinline__ uint32_t rd_bit(RangeDecoder& d, uint32_t slot)
{
	uint32_t v = d.probs[slot];
	const uint32_t bound = (d.range >> 11) * v;
	uint32_t bit;
	if (d.code < bound) {
		d.range = bound;
		v += (2048u - v) >> 5;
		bit = 0;
	} else {
		d.code -= bound;
		d.range -= bound;
		v -= v >> 5;
		bit = 1;
	}
	d.probs[slot] = (uint16_t)v;
	d.events++;
	if ((d.range & 0xFF000000u) == 0) rd_shift(d);  // p stays within [31, 2017]: one shift always suffices
	return bit;
}

// src/range_encoder.c:66-81, backwards
__device__ __forceinline__ uint32_t rd_direct(RangeDecoder& d, uint32_t nbits)
{
	uint32_t value = 0;
	d.events++;
	while (nbits--) {
		d.range >>= 1;
		const uint32_t bit = d.code >= d.range ? 1u : 0u;
		if (bit) d.code -= d.range;
		value = (value << 1) | bit;
		if ((d.range & 0xFF000000u) == 0) rd_shift(d);
	}
	return value;
}

__device__ __forceinline__ uint32_t rd_tree(RangeDecoder& d, uint32_t base, uint32_t nbits)
{
	uint32_t node = 1;
	for (uint32_t i = 0; i < nbits; i++) node = (node << 1) | rd_bit(d, base + node);
	return node - (1u << nbits);
}

__device__ __forceinline__ uint32_t rd_tree_rev(RangeDecoder& d, uint32_t base, uint32_t nbits)
{
	uint32_t node = 1, value = 0;
	for (uint32_t i = 0; i < nbits; i++) {
		const uint32_t bit = rd_bit(d, base + node);
		node = (node << 1) | bit;
		value |= bit << i;
	}
	return value;
}

// src/lzma_packet_encoder.c:42-63
__device__ __forceinline__ uint32_t rd_length(RangeDecoder& d, uint32_t base)
{
	if (!rd_bit(d, base)) return 2 + rd_tree(d, base + DL_LOW, 3);
	if (!rd_bit(d, base + DL_CHOICE2)) return 10 + rd_tree(d, base + DL_MID, 3);
	return 18 + rd_tree(d, base + DL_HIGH, 8);
}

// src/lzma_packet_encoder.c:71-104: distance - 1 (0xffffffff = the end marker)
__device__ __forceinline__ uint32_t rd_distance(RangeDecoder& d, uint32_t len)
{
	const uint32_t lctx = len - 2 < 3 ? len - 2 : 3;
	const uint32_t pslot = rd_tree(d, DS_POSSLOT + lctx * 64, 6);
	if (pslot < 4) return pslot;
	const uint32_t nlow = (pslot >> 1) - 1;
	const uint32_t dist = (2u | (pslot & 1u)) << nlow;
	if (pslot < 14) return dist + rd_tree_rev(d, DS_POSCODER + dist - pslot, nlow);
	const uint32_t mid = rd_direct(d, nlow - 4) << 4;
	return dist + mid + rd_tree_rev(d, DS_ALIGN, 4);
}

__global__ void __launch_bounds__(32) decode_kernel(DecodeArgs a)
{
	__shared__ uint16_t probs[DS_TOTAL];
	__shared__ __align__(16) uint8_t buf[DEC_BUF];
	const uint32_t lane = threadIdx.x;
	for (uint32_t i = lane; i < DS_TOTAL; i += 32) probs[i] = 1024;  // src/probability.h:7
	RangeDecoder d;
	d.probs = probs;
	d.buf = buf;
	d.base = 0;
	d.at = 0;
	d.len = a.len;
	d.range = 0xFFFFFFFFu;
	d.code = 0;
	d.short_read = 0;
	d.events = 0;
	const unsigned long long first = a.len < DEC_BUF ? a.len : DEC_BUF;
	for (uint32_t i = lane; i < first; i += 32) buf[i] = a.stream[i];
	__syncwarp();
	uint32_t err = DEC_OK, pos = 0;
	// lane 0's decoder state: the automaton and the rep distances (src/lzma_state.c)
	uint32_t ctx = 0, rep0 = 0, rep1 = 0, rep2 = 0, rep3 = 0;
	if (lane == 0) {
		if (a.len < 5) {
			err = DEC_SHORT;
		} else if (buf[0] != 0) {
			err = DEC_FIRST_BYTE;
		} else {
			for (int i = 1; i < 5; i++) d.code = (d.code << 8) | buf[i];
			d.at = 5;
		}
	}
	err = __shfl_sync(FULL, err, 0);
	while (err == DEC_OK) {
		if (a.known_size && pos == a.n) break;
		// restage the payload when the next packet could read past the staged bytes
		const unsigned long long at = __shfl_sync(FULL, d.at, 0);
		if (at + DEC_MARGIN > d.base + DEC_BUF && d.base + DEC_BUF < a.len) {
			__syncwarp();
			const unsigned long long left = a.len - at;
			const uint32_t count = left < DEC_BUF ? (uint32_t)left : DEC_BUF;
			for (uint32_t i = lane; i < count; i += 32) buf[i] = a.stream[at + i];
			d.base = at;
			__syncwarp();
		}
		uint32_t type = T_LITERAL, len = 1, dist = 0, src = 0, marker = 0;  // src: distance - 1 of the bytes a copy reads
		if (lane == 0) {
			if (d.short_read) {
				err = DEC_SHORT;
			} else if (!rd_bit(d, DS_ISMATCH + (ctx << 4))) {
				// src/lzma_packet_encoder.c:106-136: the matched tree while the decoded bits agree with the match byte
				if (pos >= a.n) {
					err = DEC_PAST_END;
				} else {
					bool matched = ctx >= 7;
					const uint32_t mbyte = matched && pos > rep0 ? a.data[pos - rep0 - 1] : 0u;
					uint32_t node = 1;
					for (int i = 7; i >= 0; i--) {
						const uint32_t mbit = (mbyte >> i) & 1u;
						const uint32_t slot = matched ? node + ((1u + mbit) << 8) : node;
						const uint32_t bit = rd_bit(d, DS_LIT + slot);
						matched = matched && mbit == bit;
						node = (node << 1) | bit;
					}
					if ((node & 0xffu) != a.data[pos]) err = DEC_LITERAL;
				}
			} else if (!rd_bit(d, DS_ISREP + ctx)) {
				len = rd_length(d, DS_LEN);
				dist = rd_distance(d, len);
				if (dist == 0xFFFFFFFFu) {
					if (a.known_size || pos != a.n) err = DEC_MARKER;
					marker = 1;
				} else {
					type = T_MATCH;
					src = dist;
				}
			} else if (!rd_bit(d, DS_ISREPG0 + ctx)) {
				src = rep0;
				if (!rd_bit(d, DS_ISREP0LONG + (ctx << 4))) {
					type = T_SHORT_REP;
				} else {
					type = T_LONG_REP;
					len = rd_length(d, DS_REPLEN);
				}
			} else {
				dist = 1;
				if (rd_bit(d, DS_ISREPG1 + ctx)) dist = rd_bit(d, DS_ISREPG2 + ctx) ? 3 : 2;
				type = T_LONG_REP;
				len = rd_length(d, DS_REPLEN);
				src = dist == 1 ? rep1 : dist == 2 ? rep2 : rep3;
			}
			if (err == DEC_OK && !marker && type != T_LITERAL) {
				if ((unsigned long long)pos < (unsigned long long)src + 1) err = DEC_SOURCE;
				else if ((unsigned long long)pos + len > a.n) err = DEC_PAST_END;
			}
			if (err == DEC_OK && !marker) {
				// src/lzma_state.c:29-81: the automaton and the rep distances
				if (type == T_MATCH) {
					rep3 = rep2;
					rep2 = rep1;
					rep1 = rep0;
					rep0 = dist;
				} else if (type == T_LONG_REP && dist != 0) {
					if (dist == 3) rep3 = rep2;
					if (dist >= 2) rep2 = rep1;
					rep1 = rep0;
					rep0 = src;
				}
				ctx = type == T_LITERAL ? (ctx < 4 ? 0u : ctx < 10 ? ctx - 3 : ctx - 6)
				    : type == T_MATCH   ? (ctx < 7 ? 7u : 10u)
				    : type == T_SHORT_REP ? (ctx < 7 ? 9u : 11u)
				                          : (ctx < 7 ? 8u : 11u);
			}
		}
		err = __shfl_sync(FULL, err, 0);
		marker = __shfl_sync(FULL, marker, 0);
		if (err != DEC_OK || marker) break;
		type = __shfl_sync(FULL, type, 0);
		len = __shfl_sync(FULL, len, 0);
		src = __shfl_sync(FULL, src, 0);
		if (type != T_LITERAL) {
			// the copied bytes must be the input's, 32 per step
			bool differ = false;
			for (uint32_t i = lane; i < len; i += 32) differ |= a.data[pos + i] != a.data[pos - src - 1 + i];
			if (__any_sync(FULL, differ)) {
				err = DEC_COPY;
				break;
			}
		}
		if (lane == 0) a.slab[pos] = pk_pack(type, dist, len);
		pos += len;
	}
	if (lane == 0) {
		if (err == DEC_OK) {
			if (d.short_read) err = DEC_SHORT;
			else if (d.at != a.len) err = DEC_TRAILING;
			else if (d.code != 0) err = DEC_CODE;
		}
		a.status->err = err;
		a.status->pos = pos;
		a.status->events = d.events;
		a.status->consumed = d.at;
	}
}

// ---- shortest-path parse (starting slabs, mg_anneal_optimal_init) ------------------------------------------
// Semantics in include/megalania_cuda.h; tests/optimal_parse.c is the same parse with one region, written
// sequentially.  Two kernels: the match list of every position (fully parallel), then one warp per region that
// relaxes the nodes of a block in ascending order and commits the cheapest path.  The model is the reference's plain
// one in shared memory (the DS_ slot map of K6): the parse reads it to build static price tables once per block and
// adapts it once per committed packet, so the walk's lane-parallel layout would buy nothing here.
constexpr uint32_t OPT_BLOCK = 4096;  // nodes per block (prices are those of the model at the block's start)
constexpr uint32_t OPT_LIST = 32;     // match-list entries per position
constexpr uint32_t OPT_INF = 0xffffffffu;

// Match list of position i: walk the bigram bucket from the nearest earlier occurrence backwards (max_occ at most),
// keep an entry only when it is longer than every earlier one, stop at min(273, n - i) bytes or at OPT_LIST entries.
// One warp per position: 32 occurrences per step, their lengths byte by byte in the lanes, then the running maximum
// over the lanes in walk order decides which become entries.
struct MatchListArgs {
	const uint8_t* data;
	uint32_t n;
	const uint32_t* occ_start;
	const uint32_t* occ;
	uint32_t max_occ;
	uint2* lists;     // [n][OPT_LIST] (len, distance - 1)
	uint8_t* counts;  // [n]
};

__global__ void __launch_bounds__(256) matchlist_kernel(MatchListArgs a)
{
	const uint32_t lane = threadIdx.x & 31;
	const uint32_t warps = gridDim.x * (blockDim.x >> 5);
	for (uint32_t i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < a.n; i += warps) {
		uint32_t count = 0;
		if (i != 0 && i + 1 < a.n) {
			const uint32_t key = (uint32_t)a.data[i] << 8 | a.data[i + 1];
			const uint32_t first = a.occ_start[key];
			uint32_t lo = first, hi = a.occ_start[key + 1];
			while (lo < hi) {  // the first occurrence at or after i (uniform: every lane searches alike)
				const uint32_t mid = lo + (hi - lo) / 2;
				if (a.occ[mid] < i) lo = mid + 1;
				else hi = mid;
			}
			const uint32_t limit = a.n - i < 273 ? a.n - i : 273;
			uint32_t best = 0, visited = 0, at = lo;
			while (at > first && visited < a.max_occ && count < OPT_LIST && best < limit) {
				uint32_t step = at - first < 32 ? at - first : 32;
				if (a.max_occ - visited < step) step = a.max_occ - visited;
				uint32_t len = 0, o = 0;
				if (lane < step) {
					o = a.occ[at - 1 - lane];
					len = 2;
					while (len < limit && a.data[i + len] == a.data[o + len]) len++;
				}
				uint32_t run = len;  // inclusive running maximum in walk order
				for (uint32_t d = 1; d < 32; d <<= 1) {
					const uint32_t v = __shfl_up_sync(FULL, run, d);
					if (lane >= d && v > run) run = v;
				}
				uint32_t before = __shfl_up_sync(FULL, run, 1);
				if (lane == 0) before = 0;
				const bool keep = len > (before > best ? before : best);
				const uint32_t mask = __ballot_sync(FULL, keep);
				const uint32_t rank = count + __popc(mask & ((1u << lane) - 1u));
				if (keep && rank < OPT_LIST) a.lists[(size_t)i * OPT_LIST + rank] = make_uint2(len, i - o - 1);
				count += __popc(mask);
				if (count > OPT_LIST) count = OPT_LIST;
				const uint32_t top = __shfl_sync(FULL, run, 31);
				if (top > best) best = top;
				visited += step;
				at -= step;
			}
		}
		if (lane == 0) a.counts[i] = (uint8_t)count;
	}
}

struct OptimalArgs {
	const uint8_t* data;
	uint32_t n;
	const uint32_t* trans;    // the context's transition tables: section 0 holds the price of bit 0 at every p
	const uint2* lists;       // matchlist_kernel's output
	const uint8_t* counts;
	const uint32_t* bounds;   // [nregions + 1]
	uint32_t nregions;
	uint4* nodes;             // [gridDim.x][OPT_BLOCK + 1][2]: (info, dist, rep0, rep1), (rep2, rep3, -, -)
	uint64_t* slab;           // [n] packed, pre-filled with literals
	uint32_t* abs_dist;       // [n] zeroed
	unsigned long long* nodes_relaxed;
};

struct OptShared {
	uint32_t price[2048];     // src/generate_table.py, the price of a bit against probability p
	uint32_t cost[OPT_BLOCK + 1];
	uint32_t lenp[2][274];    // match / rep length prices
	uint32_t slotp[4][64];    // pos-slot prices per length context
	uint32_t alignp[16];
	uint32_t litp[256];       // plain-literal trees (without is_match)
	uint32_t ent_len[OPT_LIST], ent_dist[OPT_LIST], ent_dp[OPT_LIST][4];
	uint16_t probs[DS_TOTAL];
};

__device__ __forceinline__ uint32_t opt_bit(const OptShared& s, uint32_t slot, uint32_t bit)
{
	const uint32_t p = s.probs[slot];
	return s.price[bit ? 2048u - p : p];
}

__device__ __forceinline__ uint32_t opt_tree(const OptShared& s, uint32_t base, uint32_t nbits, uint32_t value)
{
	uint32_t c = 0, node = 1;
	for (uint32_t i = nbits; i-- > 0;) {
		const uint32_t bit = (value >> i) & 1u;
		c += opt_bit(s, base + node, bit);
		node = (node << 1) | bit;
	}
	return c;
}

__device__ __forceinline__ uint32_t opt_tree_rev(const OptShared& s, uint32_t base, uint32_t nbits, uint32_t value)
{
	uint32_t c = 0, node = 1;
	for (uint32_t i = 0; i < nbits; i++) {
		const uint32_t bit = value & 1u;
		c += opt_bit(s, base + node, bit);
		node = (node << 1) | bit;
		value >>= 1;
	}
	return c;
}

__device__ __forceinline__ uint32_t opt_length(const OptShared& s, uint32_t base, uint32_t len)
{
	uint32_t v = len - 2;
	if (v < 8) return opt_bit(s, base, 0) + opt_tree(s, base + DL_LOW, 3, v);
	v -= 8;
	const uint32_t c = opt_bit(s, base, 1);
	if (v < 8) return c + opt_bit(s, base + DL_CHOICE2, 0) + opt_tree(s, base + DL_MID, 3, v);
	return c + opt_bit(s, base + DL_CHOICE2, 1) + opt_tree(s, base + DL_HIGH, 8, v - 8);
}

// adapt one slot (src/probability_model.c:5-15)
__device__ __forceinline__ void opt_code(OptShared& s, uint32_t slot, uint32_t bit)
{
	uint32_t v = s.probs[slot];
	if (bit) v -= v >> 5;
	else v += (2048u - v) >> 5;
	s.probs[slot] = (uint16_t)v;
}

__device__ __forceinline__ void opt_code_tree(OptShared& s, uint32_t base, uint32_t nbits, uint32_t value, bool rev)
{
	uint32_t node = 1;
	for (uint32_t i = 0; i < nbits; i++) {
		const uint32_t bit = rev ? (value >> i) & 1u : (value >> (nbits - 1 - i)) & 1u;
		opt_code(s, base + node, bit);
		node = (node << 1) | bit;
	}
}

__device__ __forceinline__ void opt_code_length(OptShared& s, uint32_t base, uint32_t len)
{
	uint32_t v = len - 2;
	opt_code(s, base, v >= 8);
	if (v < 8) return opt_code_tree(s, base + DL_LOW, 3, v, false);
	opt_code(s, base + DL_CHOICE2, v >= 16);
	if (v < 16) return opt_code_tree(s, base + DL_MID, 3, v - 8, false);
	opt_code_tree(s, base + DL_HIGH, 8, v - 16, false);
}

// the model's part of src/lzma_packet_encoder.c:106-194 for one packet (lane 0 only)
__device__ void opt_code_packet(OptShared& s, const uint8_t* data, uint32_t pos, uint32_t ctx, uint32_t rep0,
                                uint32_t type, uint32_t len, uint32_t dist)
{
	if (type == T_LITERAL) {
		opt_code(s, DS_ISMATCH + (ctx << 4), 0);
		const uint32_t byte = data[pos];
		bool matched = ctx >= 7;
		const uint32_t mbyte = matched ? data[pos - rep0 - 1] : 0u;
		uint32_t node = 1;
		for (int i = 7; i >= 0; i--) {
			const uint32_t bit = (byte >> i) & 1u;
			uint32_t slot = node;
			if (matched) {
				const uint32_t mbit = (mbyte >> i) & 1u;
				slot += (1u + mbit) << 8;
				matched = mbit == bit;
			}
			opt_code(s, DS_LIT + slot, bit);
			node = (node << 1) | bit;
		}
		return;
	}
	opt_code(s, DS_ISMATCH + (ctx << 4), 1);
	opt_code(s, DS_ISREP + ctx, type != T_MATCH);
	if (type == T_MATCH) {
		opt_code_length(s, DS_LEN, len);
		const uint32_t lctx = len - 2 < 3 ? len - 2 : 3;
		if (dist < 4) return opt_code_tree(s, DS_POSSLOT + lctx * 64, 6, dist, false);
		const uint32_t nlow = 30u - (uint32_t)__clz(dist), low = dist & ((1u << nlow) - 1), high = dist >> nlow;
		const uint32_t pslot = nlow * 2 + high;
		opt_code_tree(s, DS_POSSLOT + lctx * 64, 6, pslot, false);
		if (pslot < 14) opt_code_tree(s, DS_POSCODER + (high << nlow) - pslot, nlow, low, true);
		else opt_code_tree(s, DS_ALIGN, 4, low & 15, true);
		return;
	}
	if (type == T_SHORT_REP || dist == 0) {
		opt_code(s, DS_ISREPG0 + ctx, 0);
		opt_code(s, DS_ISREP0LONG + (ctx << 4), type == T_LONG_REP);
	} else {
		opt_code(s, DS_ISREPG0 + ctx, 1);
		opt_code(s, DS_ISREPG1 + ctx, dist != 1);
		if (dist != 1) opt_code(s, DS_ISREPG2 + ctx, dist != 2);
	}
	if (type == T_LONG_REP) opt_code_length(s, DS_REPLEN, len);
}

// node info word: type[7:0] | len[23:8] | ctx after the packet[31:24]
__device__ __forceinline__ uint32_t opt_info(uint32_t type, uint32_t len, uint32_t ctx) { return type | (len << 8) | (ctx << 24); }

// One warp per region, regions dealt over the CTAs.  Per node j (ascending), lane L owns the targets j + l with
// l = L (mod 32): it takes the cheapest of its candidate edges (LITERAL, SHORT_REP for l = 1; LONG_REP 0..3, then
// MATCH otherwise; the first one on a tie) and replaces the target only if that is strictly cheaper.  Being the only
// writer of its targets within the step, it needs no atomics, and the result is the sequential rule.
__global__ void __launch_bounds__(32) optimal_kernel(OptimalArgs a)
{
	__shared__ __align__(16) OptShared s;
	const uint32_t lane = threadIdx.x;
	for (uint32_t i = lane; i < 2048; i += 32) s.price[i] = i ? a.trans[i] >> 16 : 0u;
	uint4* nodes = a.nodes + (size_t)blockIdx.x * (OPT_BLOCK + 1) * 2;
	unsigned long long relaxed = 0;
	for (uint32_t r = blockIdx.x; r < a.nregions; r += gridDim.x) {
		const uint32_t lo = a.bounds[r], hi = a.bounds[r + 1];
		for (uint32_t i = lane; i < DS_TOTAL; i += 32) s.probs[i] = 1024;  // src/probability.h:7
		uint32_t ctx = 0, rep0 = 0, rep1 = 0, rep2 = 0, rep3 = 0;  // the exact model's state (every lane)
		for (uint32_t p = lo; p < hi;) {
			const uint32_t B = hi - p < OPT_BLOCK ? hi - p : OPT_BLOCK;
			__syncwarp();
			// static price tables from the model as it stands at p
			for (uint32_t l = 2 + lane; l <= 273; l += 32) {
				s.lenp[0][l] = opt_length(s, DS_LEN, l);
				s.lenp[1][l] = opt_length(s, DS_REPLEN, l);
			}
			for (uint32_t i = lane; i < 256; i += 32) {
				s.slotp[i >> 6][i & 63] = opt_tree(s, DS_POSSLOT + (i >> 6) * 64, 6, i & 63);
				s.litp[i] = opt_tree(s, DS_LIT, 8, i);
			}
			if (lane < 16) s.alignp[lane] = opt_tree_rev(s, DS_ALIGN, 4, lane);
			for (uint32_t j = lane; j <= B; j += 32) s.cost[j] = j ? OPT_INF : 0u;
			if (lane == 0) {
				nodes[0] = make_uint4(opt_info(T_LITERAL, 1, ctx), 0, rep0, rep1);
				nodes[1] = make_uint4(rep2, rep3, 0, 0);
			}
			__syncwarp();
			for (uint32_t j = 0; j < B; j++) {
				const uint4 na = nodes[2 * j], nb = nodes[2 * j + 1];
				const uint32_t c0 = s.cost[j], uctx = na.x >> 24;
				const uint32_t rep[4] = {na.z, na.w, nb.x, nb.y};
				const uint32_t i = p + j, maxl = B - j < 273 ? B - j : 273;
				// how far each rep distance matches (0 = not legal here), 32 bytes per step
				uint32_t rl[4];
				for (int q = 0; q < 4; q++) {
					rl[q] = 0;
					if (rep[q] < i) {
						rl[q] = maxl;
						for (uint32_t base = 0; base < maxl; base += 32) {
							const uint32_t k = base + lane;
							const bool differ = k < maxl && a.data[i + k] != a.data[i + k - rep[q] - 1];
							const uint32_t bal = __ballot_sync(FULL, differ);
							if (bal) {
								rl[q] = base + __ffs(bal) - 1;
								break;
							}
						}
					}
				}
				// the match list: entry e's distance price for each length context, in shared memory
				const uint32_t count = a.counts[i];
				if (lane < count) {
					const uint2 en = a.lists[(size_t)i * OPT_LIST + lane];
					s.ent_len[lane] = en.x;
					s.ent_dist[lane] = en.y;
					const uint32_t dist = en.y;
					uint32_t extra = 0, pslot = dist;
					if (dist >= 4) {
						const uint32_t nlow = 30u - (uint32_t)__clz(dist), low = dist & ((1u << nlow) - 1), high = dist >> nlow;
						pslot = nlow * 2 + high;
						extra = pslot < 14 ? opt_tree_rev(s, DS_POSCODER + (high << nlow) - pslot, nlow, low)
						                   : ((nlow - 4) << 11) + s.alignp[low & 15];
					}
					for (int c = 0; c < 4; c++) s.ent_dp[lane][c] = s.slotp[c][pslot] + extra;
				}
				__syncwarp();
				const uint32_t is_rep = opt_bit(s, DS_ISMATCH + (uctx << 4), 1) + opt_bit(s, DS_ISREP + uctx, 1);
				uint32_t rep_head[4];
				rep_head[0] = is_rep + opt_bit(s, DS_ISREPG0 + uctx, 0) + opt_bit(s, DS_ISREP0LONG + (uctx << 4), 1);
				const uint32_t g0 = is_rep + opt_bit(s, DS_ISREPG0 + uctx, 1);
				rep_head[1] = g0 + opt_bit(s, DS_ISREPG1 + uctx, 0);
				rep_head[2] = g0 + opt_bit(s, DS_ISREPG1 + uctx, 1) + opt_bit(s, DS_ISREPG2 + uctx, 0);
				rep_head[3] = g0 + opt_bit(s, DS_ISREPG1 + uctx, 1) + opt_bit(s, DS_ISREPG2 + uctx, 1);
				const uint32_t match_head = opt_bit(s, DS_ISMATCH + (uctx << 4), 1) + opt_bit(s, DS_ISREP + uctx, 0);
				uint32_t e = 0;
				for (uint32_t l = lane; l <= maxl; l += 32) {
					if (l == 0) continue;
					uint32_t best = OPT_INF, type = 0, dist = 0;
					if (l == 1) {
						// LITERAL (matched against rep0 after a match or rep), then SHORT_REP
						const uint32_t byte = a.data[i];
						best = opt_bit(s, DS_ISMATCH + (uctx << 4), 0);
						if (uctx < 7) {
							best += s.litp[byte];
						} else {
							const uint32_t mbyte = a.data[i - rep[0] - 1];
							bool matched = true;
							uint32_t node = 1;
							for (int b = 7; b >= 0; b--) {
								const uint32_t bit = (byte >> b) & 1u;
								uint32_t slot = node;
								if (matched) {
									const uint32_t mbit = (mbyte >> b) & 1u;
									slot += (1u + mbit) << 8;
									matched = mbit == bit;
								}
								best += opt_bit(s, DS_LIT + slot, bit);
								node = (node << 1) | bit;
							}
						}
						type = T_LITERAL;
						if (rep[0] < i && byte == a.data[i - rep[0] - 1]) {
							const uint32_t c = is_rep + opt_bit(s, DS_ISREPG0 + uctx, 0) + opt_bit(s, DS_ISREP0LONG + (uctx << 4), 0);
							if (c < best) {
								best = c;
								type = T_SHORT_REP;
							}
						}
					} else {
						for (int q = 0; q < 4; q++) {
							if (rl[q] < l) continue;
							const uint32_t c = rep_head[q] + s.lenp[1][l];
							if (c < best) {
								best = c;
								type = T_LONG_REP;
								dist = (uint32_t)q;
							}
						}
						while (e < count && s.ent_len[e] < l) e++;
						if (e < count) {
							const uint32_t c = match_head + s.lenp[0][l] + s.ent_dp[e][l - 2 < 3 ? l - 2 : 3];
							if (c < best) {
								best = c;
								type = T_MATCH;
								dist = s.ent_dist[e];
							}
						}
					}
					if (best == OPT_INF || c0 + best >= s.cost[j + l]) continue;
					s.cost[j + l] = c0 + best;
					// the target's state: src/lzma_state.c:29-81
					uint32_t r0 = rep[0], r1 = rep[1], r2 = rep[2], r3 = rep[3];
					if (type == T_MATCH) {
						r3 = r2;
						r2 = r1;
						r1 = r0;
						r0 = dist;
					} else if (type == T_LONG_REP) {
						const uint32_t d = rep[dist];
						if (dist > 2) r3 = r2;
						if (dist > 1) r2 = r1;
						if (dist > 0) r1 = r0;
						r0 = d;
					}
					nodes[2 * (j + l)] = make_uint4(opt_info(type, l, next_ctx(uctx, type)), dist, r0, r1);
					nodes[2 * (j + l) + 1] = make_uint4(r2, r3, 0, 0);
				}
				__syncwarp();
			}
			// commit: mark the cheapest path in the slab, then run the exact model through it
			if (lane == 0) {
				for (uint32_t j = B; j > 0;) {
					const uint4 na = nodes[2 * j];
					const uint32_t type = na.x & 0xffu, len = (na.x >> 8) & 0xffffu;
					j -= len;
					a.slab[p + j] = pk_pack(type, na.y, len);
				}
				for (uint32_t q = p; q < p + B;) {
					const uint64_t pk = a.slab[q];
					const uint32_t type = pk_type(pk), len = pk_len(pk), dist = pk_dist(pk);
					opt_code_packet(s, a.data, q, ctx, rep0, type, len, dist);
					if (type == T_MATCH) {
						rep3 = rep2;
						rep2 = rep1;
						rep1 = rep0;
						rep0 = dist;
					} else if (type == T_LONG_REP) {
						const uint32_t d = dist == 0 ? rep0 : dist == 1 ? rep1 : dist == 2 ? rep2 : rep3;
						a.abs_dist[q] = d + 1u;  // what the packet stands for, for the seam repair
						if (dist > 2) rep3 = rep2;
						if (dist > 1) rep2 = rep1;
						if (dist > 0) rep1 = rep0;
						rep0 = d;
					}
					ctx = next_ctx(ctx, type);
					q += len;
				}
			}
			ctx = __shfl_sync(FULL, ctx, 0);
			rep0 = __shfl_sync(FULL, rep0, 0);
			rep1 = __shfl_sync(FULL, rep1, 0);
			rep2 = __shfl_sync(FULL, rep2, 0);
			rep3 = __shfl_sync(FULL, rep3, 0);
			relaxed += B;
			p += B;
		}
	}
	if (lane == 0 && relaxed) atomicAdd(a.nodes_relaxed, relaxed);
}

}  // namespace mg
