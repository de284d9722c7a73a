/* C ABI of the B200 annealing engine (libmegalania_cuda.so).
 *
 * This is the boundary a Megalania host binds instead of its per-bit CPU plug-ins: plain
 * pointers and sizes, opaque handles, no C++ or torch types.  Every call returns 0 on
 * success or a negative MG_E* code; mg_last_error() gives the text for the calling thread.
 * All buffers named "host" are caller-owned host memory; the library owns its device
 * memory and streams.  One host thread per handle.  There is no CPU fallback: without a
 * CUDA device every compute entry point fails with MG_ECUDA.
 *
 * Each entry point states the reference interface it replaces (paths are relative to the
 * reference tree).
 */
#ifndef MEGALANIA_CUDA_H
#define MEGALANIA_CUDA_H

#include <stddef.h>
#include <stdint.h>

#include "output_interface.h"

#if defined(__GNUC__)
#define MG_API __attribute__((visibility("default")))
#else
#define MG_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ---- types shared with the host ------------------------------------------------------ */

/* One slab slot.  Same 12-byte layout and type codes as src/lzma_packet.h:5-17. */
#ifndef MG_HAVE_LZMA_PACKET
#define MG_HAVE_LZMA_PACKET
#define INVALID 0
#define LITERAL 1
#define MATCH 2
#define SHORT_REP 3
#define LONG_REP 4
typedef struct {
	uint8_t type;
	uint32_t dist; /* MATCH: distance-1; LONG_REP: rep index 0..3; else 0 */
	uint16_t len;  /* 1 for LITERAL/SHORT_REP, 2..273 otherwise */
} LZMAPacket;
#endif

/* src/lzma_state.h:58-62.  Only lc = lp = pb = 0 is supported, like the reference. */
#ifndef MG_HAVE_LZMA_PROPERTIES
#define MG_HAVE_LZMA_PROPERTIES
typedef struct {
	uint8_t lc;
	uint8_t lp;
	uint8_t pb;
} LZMAProperties;
#endif

enum {
	MG_OK = 0,
	MG_EINVAL = -1,  /* bad argument (null pointer, size 0, unsupported lc/lp/pb, k out of range) */
	MG_ECUDA = -2,   /* CUDA runtime failure, or no usable device */
	MG_ENOMEM = -3,  /* host or device allocation failed */
	MG_ESLAB = -4,   /* a slab holds an undecodable packet or a query is not on a packet boundary */
	MG_EOUTPUT = -5, /* OutputInterface.write returned false */
	MG_ESTATE = -6   /* call order violated (e.g. run before set_slab) */
};

typedef struct mg_ctx mg_ctx;       /* one input file resident on one GPU */
typedef struct mg_anneal mg_anneal; /* a population of annealing chains over that file */

MG_API const char* mg_last_error(void);
/* Library/ABI version, (major << 16) | minor. */
MG_API uint32_t mg_version(void);

/* Device memory released by the library is kept (per device) for its next request of the same size, so that
 * repeated one-shot calls do not pay cudaMalloc / cudaFree of ~90 GB each time; this hands it all back to the driver
 * (the library also does so by itself when an allocation fails). */
MG_API void mg_pool_trim(void);

/* ---- context ------------------------------------------------------------------------- */

/* Replaces lzma_state_init (src/lzma_state.c:16-27), packet_enumerator_new
 * (src/packet_enumerator.c:20-27 -> substring_enumerator_new, src/substring_enumerator.c:49-78:
 * the bigram index is built on the device) and top_k_packet_finder_new
 * (src/top_k_packet_finder.c:38-58).  Copies data[0..n) to device `device`. */
MG_API int mg_ctx_create(const uint8_t* data, size_t n, LZMAProperties props, int device, mg_ctx** out);
MG_API void mg_ctx_destroy(mg_ctx* ctx);
MG_API size_t mg_ctx_size(const mg_ctx* ctx);
MG_API int mg_ctx_device(const mg_ctx* ctx);
/* Match-finder limits for inputs beyond the reference's reach (SURVEY 8(f) #4).  The reference enumerates EVERY
 * earlier occurrence of the bigram at a position (its window test is commented out, src/substring_enumerator.c:97,
 * its index is O(n), :16-24): on run-heavy data one find walks 10^5..10^7 occurrences.  window = farthest match
 * start in bytes before the position (0 = unlimited), max_occurrences = only the nearest that many earlier
 * occurrences (0 = all).  Both default to 0 = the reference's semantics, which every parity claim is made under;
 * with limits the candidate lists are the reference's lists restricted to the surviving occurrences, in the same
 * order.  Applies to mg_find_topk and to chains created afterwards or already running. */
MG_API int mg_ctx_set_finder_limits(mg_ctx* ctx, size_t window, uint32_t max_occurrences);
/* Chains that fill the device exactly once: SMs x chains per SM (one warp and one model in shared memory each).
 * Populations are best sized in multiples of it. */
MG_API uint32_t mg_ctx_full_wave(const mg_ctx* ctx);
/* The device's SM clock in kHz (cudaDevAttrClockRate; 0 if the driver does not say): what turns a wall-clock step
 * length into mg_anneal_run_params.cycle_budget, which counts SM clocks (clock64()). */
MG_API uint32_t mg_ctx_sm_clock_khz(const mg_ctx* ctx);

/* ---- parity function 2: cost(data, slab) ----------------------------------------------- */

/* Replaces the perplexity back end driven over a whole slab: lzma_encode_packet
 * (src/lzma_packet_encoder.c:169-194) + perplexity_encoder (src/perplexity_encoder.c:6-17),
 * as looped in src/packet_slab_neighbour.c:22-32 and src/main.c:116-118.
 * slabs: nslabs consecutive slabs of n packets each (host).  out_cost[i] is the cost of slab i
 * in 1/2048-bit units, exactly the reference's uint64 total. */
MG_API int mg_score_slabs(mg_ctx* ctx, const LZMAPacket* slabs, size_t nslabs, uint64_t* out_cost);

/* ---- parity function 1: topk(data, state, position, excluded) --------------------------- */

/* Replaces top_k_packet_finder_find / _count / _pop (src/top_k_packet_finder.c:120-138,67-70)
 * over packet_enumerator_for_each (src/packet_enumerator.c:57-74) and
 * substring_enumerator_for_each (src/substring_enumerator.c:85-105).
 *   state_mode 0: freshly initialised model with position forced to positions[q]
 *                 (the recipe of src/main.c:53-57);
 *   state_mode 1: the model reached by pricing slab[0 .. positions[q]); positions[q] must be
 *                 a live packet boundary of the slab (any order).
 * The excluded candidate is slab[positions[q]] (src/top_k_packet_finder.c:99-101).
 * Results per query q: out_counts[q] candidates (<= k) in the reference's pop order, worst
 * first, at out_pops[q*k ..]; out_prices (optional, may be NULL) receives the integer
 * cost/len of each pop.  1 <= k <= 32 (the reference uses 20, src/main.c:49). */
MG_API int mg_find_topk(mg_ctx* ctx, const LZMAPacket* slab, int state_mode, const uint64_t* positions,
                 size_t npos, int k, LZMAPacket* out_pops, uint32_t* out_prices, int32_t* out_counts);

/* Device time (CUDA events around the kernel) and candidates enumerated by the last mg_find_topk on ctx. */
MG_API int mg_find_topk_stats(const mg_ctx* ctx, double* kernel_ms, uint64_t* candidates);

/* ---- parity function 3: bytes(data, slab) ---------------------------------------------- */

/* Replaces the final pass of src/main.c:110-119: lzma_encode_header
 * (src/lzma_header_encoder.c:5-21) + lzma_encode_packet over range_encoder
 * (src/range_encoder.c:18-101).  The range coder runs on the device; the finished stream is
 * handed to `out` (header fields first, then the payload). */
MG_API int mg_encode_slab(mg_ctx* ctx, const LZMAPacket* slab, OutputInterface* out);
/* Same, into a caller buffer; *out_len receives the stream length (may exceed cap: then
 * nothing past cap was written and the call returns MG_EINVAL). */
MG_API int mg_encode_slab_buffer(mg_ctx* ctx, const LZMAPacket* slab, uint8_t* out, size_t cap, size_t* out_len);
/* Device time (CUDA events around the range-coder kernel) and events coded (modelled bits + direct-bit groups)
 * by the last mg_encode_slab / mg_encode_slab_buffer on ctx. */
MG_API int mg_encode_stats(const mg_ctx* ctx, double* kernel_ms, uint64_t* events);

/* ---- stream -> slab: resume from an existing .lzma stream --------------------------------- */

/* Replaces nothing in the reference (it has no way to read its output back).  Decodes an LZMA-alone stream of the
 * context's input - an earlier megalania output, or e.g. liblzma's with lc = lp = pb = 0 - into the slab that encodes
 * to it: the packet that starts at a position goes to that position's slot, every other slot is LITERAL / 0 / 1
 * (packet_slab_new's value).  The range decoder runs on the device (one warp) with this project's model, the range
 * coder of mg_encode_slab run backwards; the result can start a search anywhere a slab can (mg_anneal_set_slab,
 * mg_anneal_oneshot).  stream: host, len bytes; out_slab: host, n packets.
 *   MG_EINVAL: fewer than 13 + 5 bytes; a properties byte other than 0 (the message names the lc / lp / pb found);
 *              a size field that is neither n nor all ones (unknown size).  The dictionary size is ignored.
 *   MG_ESLAB:  the payload is not this input's: the range coder's first byte is not 0; a literal differs from the
 *              input; a match or rep reaches before position 0, runs past n or copies bytes that differ; with the size
 *              unknown, the end marker does not stand exactly at n; the stream ends early, has bytes left over, or the
 *              decoder's code is not 0 at the end.  The message gives the position.  Every read is bounds-checked. */
MG_API int mg_decode_stream(mg_ctx* ctx, const uint8_t* stream, size_t len, LZMAPacket* out_slab);
/* Device time (CUDA events around the decoder kernel) and events decoded (modelled bits + direct-bit groups, the unit
 * of mg_encode_stats) by the last mg_decode_stream on ctx. */
MG_API int mg_decode_stats(const mg_ctx* ctx, double* kernel_ms, uint64_t* events);

/* ---- the annealing loop ---------------------------------------------------------------- */

enum {
	MG_SCHEDULE_REFERENCE = 0, /* src/main.c:86 rule, evaluated in 64-bit integers */
	MG_SCHEDULE_TEMPERATURE = 1 /* Metropolis at a fixed per-chain temperature (tempering) */
};

typedef struct {
	uint32_t chains;            /* independent annealing chains (one warp each) */
	uint32_t top_k;             /* candidates kept per find; reference: 20 */
	uint32_t checkpoint_stride; /* bytes between model checkpoints, >= 512; 0 = default */
	uint32_t edit_log_capacity; /* per-chain accept/reject buffer entries; 0 = default */
	uint32_t track_best;        /* keep a per-chain best slab (src/main.c:89-92) */
	uint32_t trace_capacity;    /* per-chain proposal trace records per run (0 = none) */
	uint64_t seed;              /* chain c draws from splitmix64 seeded by (seed, c) */
} mg_anneal_params;

typedef struct {
	uint32_t evals;        /* successful proposals to run per chain in this call */
	uint32_t max_attempts; /* bound on proposals drawn per chain, 0 = 64*evals + 1024 */
	uint32_t schedule;     /* MG_SCHEDULE_* */
	uint32_t step;         /* reference schedule: `step` of src/main.c:69 */
	uint32_t num_iters;    /* reference schedule: `num_iters` of src/main.c:67 (0 = n) */
	uint32_t first_eval;   /* reference schedule: value of i for the first proposal, or
	                          MG_CONTINUE_EVALS to carry each chain's own count on from its last run */
	const float* temperatures; /* MG_SCHEDULE_TEMPERATURE: host array [chains], 1/2048-bit units */
	uint64_t packet_budget; /* 0 = none; else a chain also stops after the evaluation that brings the
	                           packets it priced in this call to this many (see `suspend` for an exact
	                           budget): a reproducible way to box a step */
	uint32_t no_early_exit; /* != 0: always price a proposal to the end of the slab.  By default a
	                           proposal stops at the first checkpoint where its whole model (every
	                           probability, automaton state, rep distances, position) is bit-identical
	                           to the checkpoint the current slab left there: the rest is priced
	                           exactly as for the current slab, so the full cost is still exact */
	uint32_t suspend;       /* != 0 (with packet_budget and / or cycle_budget): the budget is exact.  A proposal that crosses it is
	                           suspended at the next checkpoint it writes and carried on by the next
	                           mg_anneal_run on the same chains, so every warp ends a step at the same
	                           moment even when one evaluation is a large part of the step (1 MiB slabs).
	                           Trajectories do not depend on where proposals are suspended.  Replacing a
	                           chain's slab (set_slab, swap, broadcast) drops its suspended proposal */
	uint64_t cycle_budget;  /* 0 = none; else SM clocks after which the chains stop: at the end of the evaluation
	                           in flight, or (with suspend) at the next checkpoint it writes; with suspend the
	                           match finder also gives a long bucket up at the deadline and the proposal is
	                           drawn again, from the same generator state, by the next call.  A wall-clock box:
	                           how many evaluations fit is not reproducible, each chain's trajectory still is */
	const uint32_t* regions; /* NULL, or host array [chains][2]: chain c only mutates packets that START in the byte range
	                           [regions[2c], regions[2c+1]) (it still re-prices everything after them).  Instead of
	                           src/packet_slab_neighbour.c:163's uniform packet index the chain draws a byte of
	                           its range and mutates the first packet at or after it.  With all chains started
	                           from one slab this turns the population into a cooperative search: see
	                           mg_anneal_merge_regions */
} mg_anneal_run_params;
#define MG_CONTINUE_EVALS 0xffffffffu

typedef struct {
	uint64_t evals;        /* successful proposals (the headline unit), all chains */
	uint64_t attempts;     /* proposals drawn, including failed ones */
	uint64_t accepted;
	uint64_t new_best;
	uint64_t packets_scored;   /* packets priced, all chains */
	uint64_t bits_scored;      /* modelled bits priced (algorithmic work of the scorer) */
	uint64_t slab_bytes_read;  /* algorithmic HBM bytes: slab slots + data walked */
	uint64_t checkpoint_bytes; /* checkpoint bytes loaded + stored */
	uint64_t finder_calls;
	uint64_t finder_candidates; /* candidates enumerated and priced */
	uint64_t edits;            /* slab edits logged */
	uint64_t log_overflows;    /* proposals abandoned because the edit log was full */
	uint64_t rejoined;         /* proposals that stopped early at a re-joined checkpoint */
	uint64_t finder_cycles;    /* SM clocks spent inside the match finder, summed over chains */
	uint64_t chain_cycles;     /* SM clocks each chain's warp was busy, summed over chains */
	uint64_t finder_chunks;    /* 32-occurrence steps of the match finder */
	uint64_t max_chain_cycles; /* the longest-running chain: chain_cycles / (chains * this) = how evenly the step ended */
	uint64_t finder_gave_up;   /* clock-boxed steps: proposals taken back because the deadline passed inside the match
	                              finder (redrawn by the next call from the same generator state) */
	double kernel_ms;          /* device time of the launch(es), CUDA events */
	uint32_t launches;         /* kernels launched by this call */
} mg_anneal_stats;

typedef struct {
	uint64_t cost;       /* proposal cost, 0 when the proposal failed */
	uint32_t flags;      /* bit0 success, bit1 accepted, bit2 new best */
	uint32_t undo_count; /* edits logged (packet_slab_neighbour_undo_count) */
} mg_trace_rec;

/* Allocates the chains: slab, best slab, double-buffered checkpoints, edit log per chain.
 * Replaces packet_slab_new (src/packet_slab.c:15-35) per chain and packet_slab_undo_stack
 * (src/packet_slab_undo_stack.c). */
MG_API int mg_anneal_create(mg_ctx* ctx, const mg_anneal_params* params, mg_anneal** out);
MG_API void mg_anneal_destroy(mg_anneal* an);
/* Device bytes one chain needs under `params` (for sizing the population). */
MG_API size_t mg_anneal_chain_bytes(const mg_ctx* ctx, const mg_anneal_params* params);

/* Sets the current slab of chains [first, first+count) to `slab` (host, n packets; NULL = all
 * LITERAL as packet_slab_new does), rescoring and checkpointing them.  The chains' current
 * cost becomes the slab cost when adopt_cost != 0, else 0 ("first proposal always accepted",
 * src/main.c:74,87).  Best slabs/costs are reset only when reset_best != 0. */
MG_API int mg_anneal_set_slab(mg_anneal* an, uint32_t first, uint32_t count, const LZMAPacket* slab,
                       int adopt_cost, int reset_best);

/* A starting slab better than the reference's all-literal one (src/packet_slab.c:30-32), built on the device: the
 * input is cut into `nregions` equal byte regions, each parsed greedily from a fresh model - at every packet the
 * cheapest candidate per byte of the exact top-k (src/top_k_packet_finder.c, under the context's finder limits) -
 * and the stitched slab goes through the forced repair pass of the region merge (rep packets whose distances
 * changed at a seam, see mg_anneal_merge_regions).  It becomes the current slab of chain `dst_chain`, priced exactly
 * (*cost_out); mg_anneal_broadcast_chain hands it to the other chains.  nregions = 1 with no finder limits is the
 * oracle's greedy parse packet for packet.  Search strategy on top of the hot path: off unless asked for. */
MG_API int mg_anneal_greedy_init(mg_anneal* an, uint32_t nregions, uint32_t dst_chain, uint64_t* cost_out);

/* A starting slab from a shortest-path parse instead of a greedy one (no reference counterpart; liblzma's optimum
 * parse makes the same approximations).  Regions as in mg_anneal_greedy_init (equal cuts, at least 64 bytes each),
 * each parsed from a fresh model; the context's finder limits do not apply.
 *   Match list of position i (0 < i < n - 1): the bigram bucket of (d[i], d[i+1]) walked from the nearest earlier
 *   occurrence backwards, at most max_occ occurrences (0 = 64), each extended up to min(273, n - i) bytes; an
 *   occurrence becomes an entry (len, distance - 1) only when it is longer than every earlier entry, and the walk
 *   stops at an entry of min(273, n - i) bytes or at 32 entries.  A MATCH of length l uses the first entry with
 *   len >= l (the nearest distance that reaches l).
 *   Parse of one region, one exact adaptive model: blocks of B = min(4096, bytes left) from the current position p.
 *   Prices come from the model as it stands at p.  Node 0 holds cost 0 and the model's automaton state and rep
 *   distances; node j keeps the cheapest packet that reached it and the state after it.  Nodes are relaxed in
 *   ascending j, edges in the order LITERAL (matched against rep0 after a match or rep), SHORT_REP, then for each
 *   length l = 2..min(273, B - j): LONG_REP 0..3 (where that rep matches l bytes), MATCH; a target takes its
 *   cheapest edge (the first on a tie) and only if that is strictly cheaper than what it holds.  The path that
 *   reaches node B is written into the slab and the exact model runs through it; no packet crosses a block's end.
 * The stitched slab goes through the same repair pass as mg_anneal_greedy_init's, which prices it exactly
 * (*cost_out).  nregions = 1 is the CPU parse of the tests packet for packet.  Off unless asked for. */
MG_API int mg_anneal_optimal_init(mg_anneal* an, uint32_t nregions, uint32_t max_occ, uint32_t dst_chain,
                                  uint64_t* cost_out);
/* Device time (CUDA events around the match-list and parse kernels) and nodes relaxed (bytes parsed) by the last
 * mg_anneal_optimal_init on ctx. */
MG_API int mg_optimal_stats(const mg_ctx* ctx, double* kernel_ms, uint64_t* nodes);

/* Cooperative regions.  After region-confined chains (mg_anneal_run_params.regions) have run from a
 * common slab, builds the slab that takes region r = [bounds[r], bounds[r+1]) from chain owners[r]
 * (bounds[0] = 0, bounds[nregions] = n), stores it as the current slab of chain `dst_chain`, repairs the
 * packets the seams broke with the reference's own repair rule (src/packet_slab_neighbour.c:82-117: SHORT_REP
 * and LONG_REP packets whose rep distances changed), prices it exactly and rewrites the chain's checkpoints.
 * *cost_out receives the merged slab's cost: the caller keeps it only if it beats the best single chain. */
MG_API int mg_anneal_merge_regions(mg_anneal* an, uint32_t nregions, const uint32_t* bounds, const uint32_t* owners,
                                   uint32_t dst_chain, uint64_t* cost_out);
/* The same in two halves, for hosts whose regions live on several GPUs.  Export writes this process's part into
 * two caller device buffers: dev_slab (n x 8 B packed slots) and dev_abs (n x 4 B, what each LONG_REP of the
 * owners' regions stands for, + 1), zero wherever owners[r] == MG_NO_OWNER.  Parts of different processes
 * cover disjoint slots, so an element-wise SUM over the processes (ncclAllReduce) is the merged whole; every
 * process then imports it: stores it as dst_chain's slab, repairs the seams, prices it, rewrites the
 * checkpoints - deterministic, so all processes end up with the same slab and the same cost. */
#define MG_NO_OWNER 0xffffffffu
MG_API int mg_anneal_merge_export(mg_anneal* an, uint32_t nregions, const uint32_t* bounds, const uint32_t* owners,
                                  void* dev_slab, void* dev_abs);
MG_API int mg_anneal_merge_import(mg_anneal* an, const void* dev_slab, const void* dev_abs, uint32_t dst_chain,
                                  uint64_t* cost_out);
/* Makes every chain's current slab (with its checkpoints and cost) a copy of chain `src_chain`'s: the restart
 * from the best slab of src/main.c:75-77, without a round trip through the host.  Best slabs are kept. */
MG_API int mg_anneal_broadcast_chain(mg_anneal* an, uint32_t src_chain);

/* Runs `evals` successful proposals on every chain: packet_slab_neighbour_generate
 * (src/packet_slab_neighbour.c:154-173) + the accept/undo/best logic of src/main.c:78-102.
 * Blocks until the device is done; stats may be NULL. */
MG_API int mg_anneal_run(mg_anneal* an, const mg_anneal_run_params* run, mg_anneal_stats* stats);

/* Per-chain costs (host arrays [chains], either may be NULL). */
MG_API int mg_anneal_costs(mg_anneal* an, uint64_t* cur_cost, uint64_t* best_cost);
/* Copies a chain's current (which = 0) or best (which = 1) slab to host, n packets. */
MG_API int mg_anneal_get_slab(mg_anneal* an, uint32_t chain, int which, LZMAPacket* out_slab);
/* Proposal trace of the last run for one chain: up to cap records, *count receives how many
 * proposals the chain drew. */
MG_API int mg_anneal_get_trace(mg_anneal* an, uint32_t chain, mg_trace_rec* out, size_t cap, size_t* count);
/* Replica exchange helpers: swap the slabs of two chains on this device / import a slab into a
 * chain keeping its cost (used by the multi-GPU host after the NCCL exchange). */
MG_API int mg_anneal_swap_chains(mg_anneal* an, uint32_t a, uint32_t b);
/* Device pointer and byte size of a chain's current (0) or best (1) packed slab, for hosts
 * that move slabs between GPUs with NCCL themselves.  The packed format is private; only
 * copy it between mg_anneal objects created over identical data. */
MG_API int mg_anneal_device_slab(mg_anneal* an, uint32_t chain, int which, void** dev_ptr, size_t* bytes);
/* Copies a chain's packed current (0) / best (1) slab into a caller DEVICE buffer of
 * mg_ctx_size()*8 bytes (e.g. a tensor the host then broadcasts with NCCL), and the inverse:
 * replaces a chain's current slab from such a buffer, then rescores and checkpoints it. */
MG_API int mg_anneal_export_slab(mg_anneal* an, uint32_t chain, int which, void* dev_dst);
MG_API int mg_anneal_import_slab(mg_anneal* an, uint32_t chain, const void* dev_src, int adopt_cost);
/* After writing a chain's packed current slab through the pointer above: rescore it. */
MG_API int mg_anneal_refresh_chain(mg_anneal* an, uint32_t chain, int adopt_cost);

/* One-shot convenience = create + set_slab(all literal or `init`) + run + pick the best chain.
 * Replaces src/main.c:64-105 for a fixed evaluation budget.  best_slab_out: host, n packets. */
MG_API int mg_anneal_oneshot(mg_ctx* ctx, const mg_anneal_params* params, const mg_anneal_run_params* run,
                      const LZMAPacket* init, LZMAPacket* best_slab_out, uint64_t* best_cost,
                      mg_anneal_stats* stats);

/* ---- several GPUs: one context (and one host thread or process) per GPU -------------------- */

/* The reference is one thread on one slab; its epochs only talk through `packets_best` (src/main.c:75-77,
 * 89-92).  Here replicas are independent inside mg_anneal_run and meet between runs through NCCL over
 * NVLink.  NCCL is bound at run time (libnccl.so.2): hosts that never call mg_comm_init do not need it. */
#define MG_COMM_ID_BYTES 128
/* ncclGetUniqueId: call on one rank, hand the 128 bytes to the others by any means (pipe, MPI, torchrun store). */
MG_API int mg_comm_unique_id(void* id_out);
/* Collective over all ranks: joins ctx's device to the communicator (ncclCommInitRank). */
MG_API int mg_comm_init(mg_ctx* ctx, int rank, int nranks, const void* nccl_id);
MG_API void mg_comm_destroy(mg_ctx* ctx); /* also done by mg_ctx_destroy */
MG_API int mg_comm_rank(const mg_ctx* ctx);
MG_API int mg_comm_size(const mg_ctx* ctx);
/* Collective: best-slab broadcast.  One all-gather of a 40-byte summary per rank finds the rank holding the
 * cheapest best slab (ties: lowest rank); that rank broadcasts the packed slab - with its model checkpoints when
 * the best slab is the chain's current one, so that receivers install it by copy instead of re-pricing 1 MiB on
 * one warp - and every other rank replaces its worst chain (highest current cost) with it, adopting the cost.
 * Costs stay on the device; the host only reads nranks x 40 bytes.  winner_rank = -1: nobody has a best yet.
 * chain_out (may be NULL): the chain of THIS rank that now holds the winning slab - as its best slab on the winner,
 * as its current slab on every other rank. */
MG_API int mg_comm_exchange_best(mg_anneal* an, int* winner_rank, uint64_t* best_cost, uint32_t* chain_out);
/* Collective: one round of replica exchange (parallel tempering) over the replicas of ALL ranks.  temps: host
 * array [chains] of this rank's temperatures, in and out.  One all-gather of (current cost, temperature) per
 * replica; every rank computes the same swap decisions (mg_temper_decide) and only temperatures move. Works
 * without a communicator too (one rank). */
MG_API int mg_comm_temper_exchange(mg_anneal* an, float* temps, uint32_t round_index, uint64_t seed);
/* The swap rule itself, host only (no device, no communicator): replicas adjacent on the temperature ladder -
 * even pairs on even rounds, odd pairs on odd rounds - swap temperatures with the Metropolis probability
 * min(1, exp((1/T_i - 1/T_j) (C_i - C_j))), decided by a counter-based generator keyed by (seed, round, pair). */
MG_API int mg_temper_decide(const uint64_t* costs, const float* temps, size_t count, uint32_t round_index,
                            uint64_t seed, float* out_temps);
/* Collective: mg_anneal_merge_regions with the regions' owners spread over the ranks (owners[r] = MG_NO_OWNER
 * for regions that live elsewhere): export + ncclAllReduce(sum) + import; every rank ends with the same slab. */
MG_API int mg_comm_merge_regions(mg_anneal* an, uint32_t nregions, const uint32_t* bounds, const uint32_t* owners,
                                 uint32_t dst_chain, uint64_t* cost_out);
/* Collective: rank `root`'s chain src_chain (current slab, its checkpoints and cost) becomes chain dst_chain of every
 * other rank, by copy.  src_chain is only read on root, dst_chain only on the others. */
MG_API int mg_comm_broadcast_chain(mg_anneal* an, int root, uint32_t src_chain, uint32_t dst_chain);
/* Collective: one host value per rank, out[r] = rank r's (out holds mg_comm_size entries). */
MG_API int mg_comm_allgather_u64(mg_ctx* ctx, uint64_t value, uint64_t* out);
MG_API int mg_comm_stats(const mg_ctx* ctx, uint64_t* exchanges, uint64_t* installs_by_copy, uint64_t* installs_by_rescore);

/* ---- debugging aid (used by the parity tests) ------------------------------------------- */

/* Model after pricing slab[0..stop): probabilities in the reference's struct order
 * (src/lzma_state.h:47-55, 2615 entries; slots unreachable at lc=lp=pb=0 stay 1024). */
typedef struct {
	uint16_t probs[2615];
	uint8_t ctx_state;
	uint32_t dists[4];
	uint64_t position;
	uint64_t cost;
} mg_model_dump;
MG_API int mg_debug_model_after_prefix(mg_ctx* ctx, const LZMAPacket* slab, size_t stop, mg_model_dump* out);
/* The device-built bigram index (replaces memoize_bigram_positions, src/substring_enumerator.c:26-47):
 * occ_start[65537] = bucket offsets for key (data[i] << 8) | data[i+1], occ[n-1] = positions 0..n-2 sorted by
 * key, ascending inside a bucket - the order substring_enumerator_for_each walks (src/substring_enumerator.c:85-105). */
MG_API int mg_debug_index(mg_ctx* ctx, uint32_t* occ_start, uint32_t* occ);

#ifdef __cplusplus
}
#endif
#endif
