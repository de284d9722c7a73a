/* megalania: drop-in CLI of the reference (src/main.c) over the B200 annealing engine.
 *
 *   megalania [options] <file>  ->  .lzma on stdout, progress on stderr, exit 255 on usage/IO error
 *
 * The structure of src/main.c:64-119 is kept: `steps` rounds of `epochs` restarts, step 0 from the
 * all-literal slab and later steps from the best slab so far, the reference's acceptance rule,
 * then one range-coder pass over the winning slab through the OutputInterface plug-in.  What
 * changes is the engine: every epoch runs on thousands of chains at once (mg_anneal_run), and
 * the iteration budget is explicit because the stock 3 x 200 x n schedule is O(n^2).
 *
 * --rounds N switches to the cooperative search (mg_anneal_merge_regions): all chains work on ONE
 * slab, each confined to a byte region for --round-ms of SM time, the regions' winners are stitched,
 * repaired, priced exactly and kept if cheaper; region boundaries move every round.
 *
 * --gpus N runs one host thread, one context and one chain population per GPU; the ranks meet between
 * epochs / rounds through the library's NCCL collectives (mg_comm_*): best-slab broadcast in the epoch
 * schedule, region merge by all-reduce in the cooperative one.  No Python, no torch.
 *
 * --resume FILE starts the search from the slab of an .lzma stream of the same input (an earlier output, or
 * liblzma's with lc = lp = pb = 0), decoded on the device by mg_decode_stream, instead of from zero; the run
 * never writes a slab costlier than the one it read.
 *
 * --optimal N starts the rounds from a shortest-path parse of N regions built on the device
 * (mg_anneal_optimal_init) instead of from the all-literal slab.
 *
 * --format xz writes the winning slab as an .xz stream (mg_encode_slab_xz: LZMA2 chunks range-coded side by side on
 * the device) instead of .lzma; only the final write changes.
 */
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include "host_io.h"
#include "megalania_cuda.h"

static void usage(const char* argv0)
{
	fprintf(stderr,
	        "usage: %s [--chains N] [--iters N] [--epochs N] [--steps N] [--seed N] [--device N] [--gpus N] [--top-k N]\n"
	        "          [--rounds N | --time SECONDS] [--round-ms N] [--group N] [--temp T] [--sm-khz N]\n"
	        "          [--window BYTES] [--max-occ N] [--greedy REGIONS | --optimal REGIONS | --resume FILE]\n"
	        "          [--format lzma|xz] filename\n",
	        argv0);
}

typedef struct {
	unsigned chains, iters, epochs, steps, device, top_k, rounds, round_ms, group, temp0, gpus, sm_khz, window, max_occ, greedy, optimal;
	unsigned long long seed;
	const uint8_t* data;
	size_t size;
	const uint8_t* resume; /* --resume: the .lzma stream to start from, NULL = none */
	size_t resume_size;
} Config;

typedef struct {
	const Config* cfg;
	int rank;
	unsigned char nccl_id[MG_COMM_ID_BYTES];
	pthread_barrier_t* barrier;
	unsigned sm_khz;         /* SM clocks per millisecond on this rank's device */
	/* results */
	int status;              /* 0 ok */
	mg_ctx* ctx;
	LZMAPacket* packets_best;
	int have_best;
	uint64_t best_perplexity;
	LZMAPacket* resumed;     /* --resume: the decoded slab and its cost */
	uint64_t resumed_cost;
} Worker;

static int die(const Worker* w, const char* what)
{
	fprintf(stderr, "[gpu %u] %s: %s\n", w->cfg->device + (unsigned)w->rank, what, mg_last_error());
	/* with several GPUs the other ranks are, or soon will be, inside a collective that this rank will never
	 * join: leave as a whole instead of hanging them */
	if (w->cfg->gpus > 1) {
		fflush(stderr);
		_exit(1);
	}
	return -1;
}

/* equal regions with the boundaries rotated by `off` bytes; returns the number of regions written */
static unsigned plan_regions(size_t file_size, unsigned nreg, double off, uint32_t* bounds)
{
	const double size = (double)file_size / nreg;
	unsigned nb = 0;
	bounds[nb++] = 0;
	for (unsigned k = 1; k < nreg; k++) {
		uint32_t cut = (uint32_t)(off + k * size);
		if (cut >= file_size) cut = (uint32_t)file_size - 1;
		if (cut > bounds[nb - 1]) bounds[nb++] = cut;
	}
	bounds[nb] = (uint32_t)file_size;
	return nb;
}

/* ---- cooperative regions (megalania_b200/cooperative.py is the same logic) ---------------------------- */
static int run_rounds(Worker* w, mg_anneal* an)
{
	const Config* c = w->cfg;
	const unsigned chains = c->chains, world = c->gpus, rank = (unsigned)w->rank;
	const size_t file_size = c->size;
	unsigned group = c->group;
	if (group == 0 || group > chains) group = chains;
	/* region r belongs to rank r % world: every rank's regions are spread over the whole file */
	unsigned per_rank = chains / group;
	if (per_rank > file_size / 64 / world) per_rank = (unsigned)(file_size / 64 / world);
	if (per_rank == 0) per_rank = 1;
	const unsigned nreg_max = per_rank * world;
	uint32_t* bounds = malloc(sizeof(uint32_t) * (nreg_max + 1));
	uint32_t* owners = malloc(sizeof(uint32_t) * nreg_max);
	uint32_t* region_of_chain = malloc(sizeof(uint32_t) * chains);
	uint32_t* regions = malloc(sizeof(uint32_t) * 2 * chains);
	float* temps = calloc(chains, sizeof(float));
	uint64_t* cur = malloc(sizeof(uint64_t) * chains);
	uint64_t* all = malloc(sizeof(uint64_t) * world);
	if (!bounds || !owners || !region_of_chain || !regions || !temps || !cur || !all) {
		fprintf(stderr, "out of memory\n");
		return -1;
	}
	if (mg_anneal_set_slab(an, 0, chains, w->resumed, 1, 1)) return die(w, "mg_anneal_set_slab");
	if (c->greedy) {
		/* --greedy N: start from a greedy parse of N regions instead of the all-literal slab; every rank builds
		 * the same slab (the parse draws nothing) */
		uint64_t cost = 0;
		if (mg_anneal_greedy_init(an, c->greedy, 0, &cost)) return die(w, "mg_anneal_greedy_init");
		if (mg_anneal_broadcast_chain(an, 0)) return die(w, "mg_anneal_broadcast_chain");
	}
	if (c->optimal) {
		/* --optimal N: the same from a shortest-path parse of N regions (match lists of the default 64
		 * occurrences; --max-occ limits the annealer's finder only) */
		uint64_t cost = 0;
		if (mg_anneal_optimal_init(an, c->optimal, 0, 0, &cost)) return die(w, "mg_anneal_optimal_init");
		if (mg_anneal_broadcast_chain(an, 0)) return die(w, "mg_anneal_broadcast_chain");
		if (w->rank == 0) fprintf(stderr, "current file size: %f\toptimal parse (%u regions)\n", 18 + cost / 16384.f, c->optimal);
	}
	unsigned long long lcg = c->seed, evals = 0;
	double device_ms = 0;
	for (unsigned r = 0; r < c->rounds; r++) {
		lcg = lcg * 6364136223846793005ull + 1442695040888963407ull; /* same sequence on every rank */
		const double size = (double)file_size / nreg_max;
		const double off = (double)((lcg >> 33) % (unsigned long long)(size < 1 ? 1 : size));
		const unsigned regs = plan_regions(file_size, nreg_max, off, bounds);
		/* this rank's regions, its chains dealt round-robin over them */
		unsigned mine = 0;
		for (unsigned k = rank; k < regs; k += world) mine++;
		for (unsigned ch = 0; ch < chains; ch++) {
			const unsigned k = mine ? rank + (ch % mine) * world : rank % regs;
			region_of_chain[ch] = k;
			regions[2 * ch] = bounds[k];
			regions[2 * ch + 1] = bounds[k + 1];
		}
		mg_anneal_run_params run;
		memset(&run, 0, sizeof(run));
		run.evals = 1000000;
		run.schedule = MG_SCHEDULE_TEMPERATURE;
		for (unsigned ch = 0; ch < chains; ch++) temps[ch] = (float)c->temp0 * (1.f - (float)(r + 1) / (float)c->rounds);
		run.temperatures = temps; /* uphill moves with probability exp(-delta / T); the last round is T = 0 */
		run.first_eval = MG_CONTINUE_EVALS;
		run.cycle_budget = (uint64_t)c->round_ms * (uint64_t)w->sm_khz;
		run.regions = regions;
		mg_anneal_stats stats;
		if (mg_anneal_run(an, &run, &stats)) return die(w, "mg_anneal_run");
		evals += stats.evals;
		device_ms += stats.kernel_ms;
		if (mg_anneal_costs(an, cur, NULL)) return die(w, "mg_anneal_costs");
		unsigned best_chain = 0, worst_chain = 0;
		for (unsigned k = 0; k < regs; k++) owners[k] = MG_NO_OWNER;
		for (unsigned ch = 0; ch < chains; ch++) {
			const unsigned k = region_of_chain[ch];
			if (k % world == rank && (owners[k] == MG_NO_OWNER || cur[ch] < cur[owners[k]])) owners[k] = ch;
			if (cur[ch] < cur[best_chain]) best_chain = ch;
			if (cur[ch] > cur[worst_chain]) worst_chain = ch;
		}
		if (worst_chain == best_chain) worst_chain = (best_chain + 1) % chains;
		uint64_t merged = 0, best_single = cur[best_chain];
		unsigned winner = best_chain, src_rank = rank;
		const char* kept = "best chain";
		if (world > 1) {
			if (mg_comm_merge_regions(an, regs, bounds, owners, worst_chain, &merged)) return die(w, "mg_comm_merge_regions");
			if (mg_comm_allgather_u64(w->ctx, cur[best_chain], all)) return die(w, "mg_comm_allgather_u64");
			for (unsigned k = 0; k < world; k++)
				if (all[k] < best_single || (all[k] == best_single && k < src_rank)) {
					best_single = all[k];
					src_rank = k;
				}
			if (merged <= best_single) {
				winner = worst_chain;
				kept = "merged";
			} else {
				/* a single chain somewhere beats the merge: its slab travels from the rank that owns it */
				if (mg_comm_broadcast_chain(an, (int)src_rank, best_chain, worst_chain)) return die(w, "mg_comm_broadcast_chain");
				winner = rank == src_rank ? best_chain : worst_chain;
			}
		} else if (chains > 1) {
			if (mg_anneal_merge_regions(an, regs, bounds, owners, worst_chain, &merged)) return die(w, "mg_anneal_merge_regions");
			if (merged <= best_single) {
				winner = worst_chain;
				kept = "merged";
			}
		}
		w->best_perplexity = (winner == worst_chain && merged != 0 && merged <= best_single) ? merged : best_single;
		if (mg_anneal_broadcast_chain(an, winner)) return die(w, "mg_anneal_broadcast_chain");
		unsigned long long total_evals = evals;
		if (world > 1) {
			if (mg_comm_allgather_u64(w->ctx, evals, all)) return die(w, "mg_comm_allgather_u64");
			total_evals = 0;
			for (unsigned k = 0; k < world; k++) total_evals += all[k];
		}
		if (rank == 0)
			fprintf(stderr, "current file size: %f\tround: %u/%u - %s, %llu evals, %.0f evals/s\n", 18 + w->best_perplexity / 16384.f,
			        r + 1, c->rounds, kept, total_evals, total_evals / (device_ms / 1e3));
	}
	if (w->resumed && w->resumed_cost <= w->best_perplexity) {
		/* the rounds ended no cheaper than the resumed slab: keep that one */
		memcpy(w->packets_best, w->resumed, sizeof(LZMAPacket) * file_size);
		w->best_perplexity = w->resumed_cost;
	} else if (mg_anneal_get_slab(an, 0, 0, w->packets_best)) {
		return die(w, "mg_anneal_get_slab");
	}
	w->have_best = 1;
	free(bounds);
	free(owners);
	free(region_of_chain);
	free(regions);
	free(temps);
	free(cur);
	free(all);
	return 0;
}

/* ---- the reference's schedule: steps x epochs (src/main.c:69-105) ---------------------------------------- */
static int run_epochs(Worker* w, mg_anneal* an)
{
	const Config* c = w->cfg;
	const unsigned chains = c->chains, world = c->gpus;
	uint64_t* best_costs = malloc(sizeof(uint64_t) * chains);
	uint64_t* all = malloc(sizeof(uint64_t) * world);
	if (!best_costs || !all) {
		fprintf(stderr, "out of memory\n");
		return -1;
	}
	unsigned long long evals = 0;
	double device_ms = 0;
	for (unsigned step = 0; step < c->steps; step++) {
		for (unsigned epoch = 0; epoch < c->epochs; epoch++) {
			/* src/main.c:71-77: fresh slab in step 0, the best so far afterwards; cost 0 means
			 * "first proposal always accepted".  A resumed run starts step 0 from the resumed slab */
			if (mg_anneal_set_slab(an, 0, chains, ((step != 0 || w->resumed) && w->have_best) ? w->packets_best : NULL, 0, 0))
				return die(w, "mg_anneal_set_slab");
			mg_anneal_run_params run;
			memset(&run, 0, sizeof(run));
			run.evals = c->iters;
			run.schedule = MG_SCHEDULE_REFERENCE;
			run.step = step;
			run.num_iters = c->iters;
			mg_anneal_stats stats;
			if (mg_anneal_run(an, &run, &stats)) return die(w, "mg_anneal_run");
			evals += stats.evals;
			device_ms += stats.kernel_ms;
			unsigned long long total_evals = evals;
			if (world > 1) {
				/* the cheapest best slab of all ranks reaches every rank (NCCL broadcast, installed by copy) */
				int winner = -1;
				uint64_t cost = 0;
				uint32_t chain = 0;
				if (mg_comm_exchange_best(an, &winner, &cost, &chain)) return die(w, "mg_comm_exchange_best");
				if (winner >= 0 && cost != 0 && (!w->have_best || cost < w->best_perplexity)) {
					w->best_perplexity = cost;
					if (mg_anneal_get_slab(an, chain, winner == w->rank ? 1 : 0, w->packets_best)) return die(w, "mg_anneal_get_slab");
					w->have_best = 1;
				}
				if (mg_comm_allgather_u64(w->ctx, evals, all)) return die(w, "mg_comm_allgather_u64");
				total_evals = 0;
				for (unsigned k = 0; k < world; k++) total_evals += all[k];
			} else {
				if (mg_anneal_costs(an, NULL, best_costs)) return die(w, "mg_anneal_costs");
				unsigned arg = 0;
				for (unsigned ch = 1; ch < chains; ch++)
					if (best_costs[ch] != 0 && (best_costs[arg] == 0 || best_costs[ch] < best_costs[arg])) arg = ch;
				if (best_costs[arg] != 0 && (!w->have_best || best_costs[arg] < w->best_perplexity)) {
					w->best_perplexity = best_costs[arg];
					if (mg_anneal_get_slab(an, arg, 1, w->packets_best)) return die(w, "mg_anneal_get_slab");
					w->have_best = 1;
				}
			}
			if (w->rank == 0)
				fprintf(stderr, "current file size: %f\tstep: %u\tepoch: %04u - %llu evals, %.0f evals/s\n",
				        18 + w->best_perplexity / 16384.f, step + 1, epoch, total_evals, total_evals / (device_ms / 1e3));
		}
	}
	free(best_costs);
	free(all);
	return 0;
}

/* --resume: every rank decodes the stream on its own context (deterministic: all ranks hold the same slab) and
 * scores it; it becomes the best so far */
static int resume_from_stream(Worker* w)
{
	const Config* c = w->cfg;
	w->resumed = malloc(sizeof(LZMAPacket) * c->size);
	w->packets_best = malloc(sizeof(LZMAPacket) * c->size);
	if (!w->resumed || !w->packets_best) {
		fprintf(stderr, "out of memory\n");
		return -1;
	}
	if (mg_decode_stream(w->ctx, c->resume, c->resume_size, w->resumed)) {
		/* a stream of another input is a usage error on every rank alike: leave before any collective */
		fprintf(stderr, "[gpu %u] mg_decode_stream: %s\n", c->device + (unsigned)w->rank, mg_last_error());
		if (c->gpus > 1) {
			fflush(stderr);
			_exit(255);
		}
		return -1;
	}
	if (mg_score_slabs(w->ctx, w->resumed, 1, &w->resumed_cost)) return die(w, "mg_score_slabs");
	memcpy(w->packets_best, w->resumed, sizeof(LZMAPacket) * c->size);
	w->best_perplexity = w->resumed_cost;
	w->have_best = 1;
	if (w->rank == 0) fprintf(stderr, "current file size: %f\tresumed (%zu-byte stream)\n", 18 + w->resumed_cost / 16384.f, c->resume_size);
	return 0;
}

static void* worker_main(void* arg)
{
	Worker* w = (Worker*)arg;
	const Config* c = w->cfg;
	w->status = -1;
	LZMAProperties properties = { 0, 0, 0 };
	mg_anneal* an = NULL;
	int ok = 0;
	do {
		if (mg_ctx_create(c->data, c->size, properties, (int)c->device + w->rank, &w->ctx)) {
			die(w, "mg_ctx_create");
			break;
		}
		if (c->resume && resume_from_stream(w) != 0) break;
		/* SM clocks per millisecond: the device's own figure (mg_ctx_sm_clock_khz) unless --sm-khz says otherwise;
		 * 1965 MHz (B200) only if the driver reports nothing */
		w->sm_khz = c->sm_khz ? c->sm_khz : mg_ctx_sm_clock_khz(w->ctx);
		if (w->sm_khz == 0) w->sm_khz = 1965000;
		if ((c->window || c->max_occ) && mg_ctx_set_finder_limits(w->ctx, c->window, c->max_occ)) {
			die(w, "mg_ctx_set_finder_limits");
			break;
		}
		if (c->gpus > 1 && mg_comm_init(w->ctx, w->rank, (int)c->gpus, w->nccl_id)) {
			die(w, "mg_comm_init");
			break;
		}
		mg_anneal_params params;
		memset(&params, 0, sizeof(params));
		params.chains = c->chains;
		params.top_k = c->top_k;
		params.track_best = 1;
		params.seed = c->seed + 1000003ull * (unsigned long long)w->rank;
		if (mg_anneal_create(w->ctx, &params, &an)) {
			die(w, "mg_anneal_create");
			break;
		}
		if (!w->packets_best) w->packets_best = malloc(sizeof(LZMAPacket) * c->size);
		if (!w->packets_best) {
			fprintf(stderr, "out of memory\n");
			break;
		}
		if ((c->rounds > 0 ? run_rounds(w, an) : run_epochs(w, an)) != 0) break;
		ok = 1;
	} while (0);
	if (an) mg_anneal_destroy(an);
	if (ok) w->status = 0;
	return NULL;
}

int main(int argc, char** argv)
{
	Config cfg;
	memset(&cfg, 0, sizeof(cfg));
	cfg.chains = 1184;
	cfg.epochs = 2;
	cfg.steps = 3;
	cfg.top_k = 20;
	cfg.round_ms = 250;
	cfg.group = 8;
	cfg.temp0 = 4096;    /* --temp: 1/2048 bit, cooled linearly to 0 */
	cfg.gpus = 1;
	cfg.sm_khz = 0;      /* --sm-khz: SM clock that turns --round-ms into an SM-cycle budget; 0 = ask the device */
	cfg.seed = 1673551;  /* src/main.c:68 */
	unsigned time_s = 0; /* --time: annealing budget in seconds of SM time */
	const char* filename = NULL;
	const char* resume_name = NULL;
	int xz = 0; /* --format: lzma (the reference's, the default) or xz */
	for (int i = 1; i < argc; i++) {
		const char* a = argv[i];
		unsigned* target = NULL;
		if (!strcmp(a, "--chains")) target = &cfg.chains;
		else if (!strcmp(a, "--iters")) target = &cfg.iters;
		else if (!strcmp(a, "--epochs")) target = &cfg.epochs;
		else if (!strcmp(a, "--steps")) target = &cfg.steps;
		else if (!strcmp(a, "--device")) target = &cfg.device;
		else if (!strcmp(a, "--gpus")) target = &cfg.gpus;
		else if (!strcmp(a, "--top-k")) target = &cfg.top_k;
		else if (!strcmp(a, "--rounds")) target = &cfg.rounds;
		else if (!strcmp(a, "--round-ms")) target = &cfg.round_ms;
		else if (!strcmp(a, "--group")) target = &cfg.group;
		else if (!strcmp(a, "--temp")) target = &cfg.temp0;
		else if (!strcmp(a, "--time")) target = &time_s;
		else if (!strcmp(a, "--sm-khz")) target = &cfg.sm_khz;
		else if (!strcmp(a, "--window")) target = &cfg.window;   /* match-finder limits for huge inputs; 0 = the */
		else if (!strcmp(a, "--max-occ")) target = &cfg.max_occ; /* reference's unbounded enumeration */
		else if (!strcmp(a, "--greedy")) target = &cfg.greedy;   /* start the rounds from a greedy parse of N regions */
		else if (!strcmp(a, "--optimal")) target = &cfg.optimal; /* ... or from a shortest-path parse of N regions */
		if (target) {
			if (++i >= argc) { usage(argv[0]); return -1; }
			*target = (unsigned)strtoul(argv[i], NULL, 10);
		} else if (!strcmp(a, "--seed")) {
			if (++i >= argc) { usage(argv[0]); return -1; }
			cfg.seed = strtoull(argv[i], NULL, 10);
		} else if (!strcmp(a, "--resume")) {
			if (++i >= argc) { usage(argv[0]); return -1; }
			resume_name = argv[i];
		} else if (!strcmp(a, "--format")) {
			if (++i >= argc || (strcmp(argv[i], "lzma") && strcmp(argv[i], "xz"))) { usage(argv[0]); return -1; }
			xz = !strcmp(argv[i], "xz");
		} else if (a[0] == '-' && a[1] == '-') {
			usage(argv[0]);
			return -1;
		} else if (filename == NULL) {
			filename = a;
		} else {
			usage(argv[0]);
			return -1;
		}
	}
	if (time_s > 0 && cfg.round_ms > 0) cfg.rounds = (time_s * 1000u + cfg.round_ms - 1) / cfg.round_ms;
	if (filename == NULL || cfg.chains == 0 || cfg.gpus == 0 || cfg.gpus > 64 ||
	    (cfg.rounds == 0 && (cfg.steps == 0 || cfg.epochs == 0)) || (resume_name && cfg.greedy) ||
	    (cfg.optimal && (cfg.greedy || resume_name || cfg.rounds == 0))) {
		usage(argv[0]);
		return -1;
	}

	/* stdout carries the .lzma stream and nothing else: libraries that print there (NCCL's version banner does) are
	 * sent to stderr, the stream goes to a private copy of the original descriptor */
	fflush(stdout);
	const int stream_fd = dup(1);
	FILE* stream_out = stream_fd >= 0 ? fdopen(stream_fd, "wb") : NULL;
	if (!stream_out || dup2(2, 1) < 0) {
		fprintf(stderr, "could not set the output stream up\n");
		return -1;
	}

	InputFile input;
	if (input_file_open(&input, filename) < 0) return -1;
	cfg.data = input.data;
	cfg.size = input.size;
	InputFile resume_file = { NULL, 0 };
	if (resume_name) {
		if (input_file_open(&resume_file, resume_name) < 0) return -1;
		cfg.resume = resume_file.data;
		cfg.resume_size = resume_file.size;
	}
	if (cfg.iters == 0) cfg.iters = cfg.size < 2000 ? (unsigned)cfg.size : 2000;

	Worker* workers = calloc(cfg.gpus, sizeof(Worker));
	pthread_t* threads = calloc(cfg.gpus, sizeof(pthread_t));
	if (!workers || !threads) {
		fprintf(stderr, "out of memory\n");
		return -1;
	}
	unsigned char nccl_id[MG_COMM_ID_BYTES];
	memset(nccl_id, 0, sizeof(nccl_id));
	if (cfg.gpus > 1 && mg_comm_unique_id(nccl_id)) {
		fprintf(stderr, "mg_comm_unique_id: %s\n", mg_last_error());
		return -1;
	}
	for (unsigned r = 0; r < cfg.gpus; r++) {
		workers[r].cfg = &cfg;
		workers[r].rank = (int)r;
		memcpy(workers[r].nccl_id, nccl_id, sizeof(nccl_id));
	}
	if (cfg.gpus == 1) {
		worker_main(&workers[0]);
	} else {
		for (unsigned r = 0; r < cfg.gpus; r++)
			if (pthread_create(&threads[r], NULL, worker_main, &workers[r]) != 0) {
				fprintf(stderr, "could not start a thread for GPU %u\n", cfg.device + r);
				return -1;
			}
		for (unsigned r = 0; r < cfg.gpus; r++) pthread_join(threads[r], NULL);
	}
	for (unsigned r = 0; r < cfg.gpus; r++)
		if (workers[r].status != 0) return -1;

	/* the cheapest slab of all ranks (they agree after an exchange; ties go to the lowest rank) */
	unsigned winner = 0;
	for (unsigned r = 1; r < cfg.gpus; r++)
		if (workers[r].have_best && (!workers[winner].have_best || workers[r].best_perplexity < workers[winner].best_perplexity)) winner = r;
	Worker* win = &workers[winner];
	if (!win->have_best) {
		/* no position had an alternative packet (the reference loops forever here): all literals */
		for (size_t i = 0; i < cfg.size; i++) {
			win->packets_best[i].type = LITERAL;
			win->packets_best[i].dist = 0;
			win->packets_best[i].len = 1;
		}
	}

	OutputInterface output;
	StreamSink sink;
	stream_sink_init(&output, &sink, stream_out);
	if (xz ? mg_encode_slab_xz(win->ctx, win->packets_best, 0, &output) : mg_encode_slab(win->ctx, win->packets_best, &output)) {
		fprintf(stderr, "%s: %s\n", xz ? "mg_encode_slab_xz" : "mg_encode_slab", mg_last_error());
		return -1;
	}
	if (fflush(stream_out) != 0 || sink.failed) {
		fprintf(stderr, "could not write the output stream\n");
		return -1;
	}

	for (unsigned r = 0; r < cfg.gpus; r++) {
		free(workers[r].packets_best);
		free(workers[r].resumed);
		mg_ctx_destroy(workers[r].ctx);
	}
	free(workers);
	free(threads);
	if (resume_name) input_file_close(&resume_file);
	input_file_close(&input);
	return 0;
}
