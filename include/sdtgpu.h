/*
 * sdtgpu.h — C ABI of the B200-native pregraph k-mer hashing path (libsdtgpu.so).
 *
 * The reference (SOAPdenovo-Trans 1.04) has no plugin/FFI interface; its seam for this path is
 * a C function boundary inside one process.  Each entry point below names the reference
 * interface it replaces (paths relative to /root/reference/src).  Everything is extern "C",
 * plain pointers and sizes; no C++/torch types; every call returns 0 or an SDTGPU_E* code and
 * never calls exit() — the C caller turns a non-zero status into the reference's
 * printf + exit(-1) convention (check.c:31-34).
 *
 * Input reads are 2-bit packed in the reference's tight-string convention (seq.c:49-90): four
 * bases per byte, first base in bits 7..6, codes A=0 C=1 T=2 G=3 (inc/def.h:39); read i starts
 * at packed + i*stride_bytes (stride_bytes a multiple of 4, >= ceil(max_read_len/4)), which
 * mirrors the reference's fixed-stride seqBuffer[maxReadNum][maxReadLen] (prlHashReads.c:387-395).
 */
#ifndef SDTGPU_H
#define SDTGPU_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDTGPU_OK        0
#define SDTGPU_EINVAL    1	/* bad argument (K even / out of range, misaligned buffer, ...) */
#define SDTGPU_ECUDA     2	/* CUDA runtime error; see sdtgpu_last_error */
#define SDTGPU_ENOMEM    3	/* host or device allocation failed */
#define SDTGPU_ERANGE    4	/* ordinal / capacity limit exceeded */
#define SDTGPU_ESTATE    5	/* call not valid in the handle's current state */

typedef struct sdtgpu sdtgpu_t;

/* One exported node: the reference's kmer_t (inc/newhash.h:65-77) plus bookkeeping.
 * key[0] is the most significant word (high1), key[3] the least (low2 / the MER31 scalar).
 * rword = r_links | linear<<24 | deleted<<25 | checked<<26 | single<<27 | twin<<28 | inEdge<<30,
 * i.e. the raw bit-field word that follows l_links in kmer_t.  ordinal is the position of the
 * k-mer's first instance in the reference's arrival order (read ordinal * max windows + window). */
typedef struct sdtgpu_node {
	uint64_t key[4];
	uint32_t l_links;
	uint32_t rword;
	uint32_t count;
	uint32_t set;		/* hash_kmer(key) % thrd_num (hashFunction.c:108, prlHashReads.c:81) */
	uint64_t ordinal;
} sdtgpu_node;		/* 56 bytes */

/* Binary-compatible with the reference's KmerSet (inc/newhash.h:79-88).  array points to
 * kmer_t records of node_bytes each (24 for MER31, 32 for MER63, 48 for MER127); array, flags and
 * the struct itself come from malloc/calloc so the reference's free_Sets (newhash.c:498) can
 * release them. */
typedef struct sdtgpu_kmerset {
	void *array;
	uint32_t *flags;
	uint64_t size;
	uint64_t count;
	uint64_t max;
	double load_factor;
	uint64_t iter_ptr;
} sdtgpu_kmerset;

typedef struct sdtgpu_stats {
	uint64_t n_instances;	/* "kmer in reads"  (kmerCounter[0], prlHashReads.c:466,662) */
	uint64_t n_nodes;	/* "nodes allocated" (sum of count_kmerset, prlHashReads.c:657) */
	uint64_t n_removed;	/* "%lld kmer removed" (deLowCov, prlHashReads.c:908) */
	uint64_t n_linear;	/* "%lld linear nodes" (Mark1in1outNode, prlHashReads.c:991) */
	uint64_t capacity;	/* device slots */
	uint64_t n_reads;	/* reads pushed (including those shorter than K+1, which are skipped) */
	uint32_t n_grows;	/* device table re-hashes so far */
	uint32_t device_key_words;	/* 1, 2 or 4 */
} sdtgpu_stats;

/* ---- life cycle.  Replaces the set-up part of prlRead2HashTable (prlHashReads.c:355-426):
 * createFilter, the kmerBuffer/hashBanBuffer/prevc/nextc batch buffers, init_kmerset x thrd_num
 * and creatThrds.  K odd, 13..127 (pregraph.c:38-59).  key_words is the reference build being
 * served (1 = MER31, 2 = MER63, 4 = MER127) and fixes hash_kmer's byte count and the exported
 * kmer_t size; the device key width is ceil(2K/64) words independently of it.
 * capacity_hint = expected distinct k-mers (0: single-pass insert: start small and grow by device re-hash;
 * sliced build: sized from the number of windows pushed).
 * device = CUDA ordinal.  flags: SDTGPU_F_* */
#define SDTGPU_F_NKMER     1u	/* the reference's -n (N_kmer): windows containing N become key 0 without links */
#define SDTGPU_F_SLICED    4u	/* sliced build (the default of the drop-in and of bench.py): pushes turn reads into super-k-mer
				 * records (runs of windows that share a minimizer, bases included) appended to the chain of
				 * their table slice; sdtgpu_sync / finalize / export merge copies, cut the chains into work
				 * items and build each item in shared memory, one CTA per item, into a compact node store.
				 * No random DRAM access.  capacity_hint is optional (0: the reads are logged and the slice
				 * count comes from the number of windows pushed; slices that overflow are split, the store
				 * grows).  Same multiset, same hand-back layout as the single-pass insert. */
int sdtgpu_create (sdtgpu_t **out, int device, int K, int key_words, int max_read_len,
		   uint64_t capacity_hint, unsigned flags);
void sdtgpu_destroy (sdtgpu_t *h);
const char *sdtgpu_last_error (const sdtgpu_t *h);	/* h may be NULL: last create() failure */
int sdtgpu_reset (sdtgpu_t *h);	/* empty the table, keep the allocation */

/* ---- the hot path.  Replaces one `sendWorkSignal(2); sendWorkSignal(1);` flush
 * (prlHashReads.c:466-471, 524-527, 561-564, 603-606, 617-619), i.e. chopKmer4read
 * (prlHashReads.c:164-310) over the batch followed by put_kmerset (newhash.c:411-462) of every
 * window.  lens == NULL means every read has uniform_len bases.  nmask (1 bit per base, bit 7 of
 * byte 0 = base 0, stride_bytes/2 bytes per read) is only read with SDTGPU_F_NKMER and may be NULL.
 * first_read_ordinal = number of reads pushed before this batch in arrival order (needed only
 * for export_kmersets' slot-exact layout; pass the running count).
 * push_reads takes HOST buffers (pageable or pinned) and returns as soon as they have been copied
 * to the device (the caller may reuse them immediately); the copy overlaps the kernels of the
 * previous batch and this batch's kernels run asynchronously (the reference does not overlap
 * parsing with hashing; doing so is allowed because the table is order-free).
 * push_reads_device takes DEVICE pointers (16-byte aligned) and only enqueues kernels. */
int sdtgpu_push_reads (sdtgpu_t *h, const uint8_t *packed, const uint32_t *lens, const uint8_t *nmask,
		       uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes, uint64_t first_read_ordinal);
int sdtgpu_push_reads_device (sdtgpu_t *h, const uint8_t *d_packed, const uint32_t *d_lens, const uint8_t *d_nmask,
			      uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes, uint64_t first_read_ordinal);
int sdtgpu_sync (sdtgpu_t *h);

/* ---- multi-GPU, replicated reads (the default sharding of bench.py and exchange.py).
 * After sdtgpu_set_owner (h, rank, n_ranks) every push inserts only the instances this rank owns
 * (owner = mix(key) -> [0, n_ranks), any owner function gives the same union).  The ranks
 * all-gather their packed reads (28 bytes per 100-bp read over NVLink) and each chops all of them:
 * this is exactly the reference's scheme — every worker scans the whole batch and keeps
 * hash % thrd_num == id (prlHashReads.c:79-88) — and it needs no per-k-mer records at all; chopping
 * is ~20x cheaper than inserting, so the redundant chop costs less than writing, sending and
 * re-reading 16-byte records.  stats.n_instances then counts the instances this rank inserted. */
int sdtgpu_set_owner (sdtgpu_t *h, int rank, int n_ranks);

/* ---- multi-GPU, record exchange (alternative; the caller moves the bins, e.g. NCCL all-to-all).
 * The reference's equivalent is "every worker scans the shared hashBanBuffer and keeps
 * hash % thrd_num == id" (prlHashReads.c:79-88).  bucket_reads_device chops this rank's reads and
 * appends each instance as a record of sdtgpu_record_bytes() (8 * (device_key_words + 1)) to the bin of its owner rank
 * (owner = mix(key) -> [0, n_ranks)); insert_records_device upserts received records.
 * Record layout (little endian u64 words): key words (device_key_words, most significant first),
 * then one meta word = ordinal << 8 | left << 4 | right  (left/right 0..3, or 4 = none).
 * d_bins holds n_ranks bins of bin_capacity records each; d_counts[n_ranks] (u64) must be zeroed
 * by the caller and receives the fill of each bin (a bin that would overflow is reported through
 * SDTGPU_ERANGE at the next sdtgpu_sync).  bucket_reads_device is enqueued on the handle's auxiliary
 * stream (sdtgpu_aux_stream), insert_records_device on the main one, so the send side of round r+1
 * overlaps the inserts of round r; the caller orders the two with events. */
size_t sdtgpu_record_bytes (const sdtgpu_t *h);
int sdtgpu_bucket_reads_device (sdtgpu_t *h, const uint8_t *d_packed, const uint32_t *d_lens, const uint8_t *d_nmask,
				uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes, uint64_t first_read_ordinal,
				int n_ranks, void *d_bins, uint64_t bin_capacity, uint64_t *d_counts);
int sdtgpu_insert_records_device (sdtgpu_t *h, const void *d_records, uint64_t n_records);

/* ---- post-pass.  Replaces deLowCov/thread_delow (prlHashReads.c:844-909; only when
 * deLowKmer > 0), Mark1in1outNode/thread_mark (prlHashReads.c:911-992) and the histogram behind
 * freqStat (prlHashReads.c:994-1023): kmerFreq[i] for i in 0..256, the reference prints 1..255.
 * May be called once per table; push after finalize is SDTGPU_ESTATE. */
int sdtgpu_finalize (sdtgpu_t *h, int deLowKmer, int64_t kmerFreq[257], sdtgpu_stats *stats);
int sdtgpu_get_stats (sdtgpu_t *h, sdtgpu_stats *stats);

/* Order-independent fingerprint of the table (test/verification hook): out[0] = sum over nodes of
 * mix64(key words, count, l_links, r_links) mod 2^64, out[1] = sum of counts, out[2] = set link bits
 * (left in the low, right in the high 32 bits), out[3] = nodes.  Equal multisets give equal
 * fingerprints regardless of insertion order, batching, capacity or sharding across GPUs. */
int sdtgpu_table_checksum (sdtgpu_t *h, uint64_t out[4]);

/* ---- hand-back.  export_nodes copies every node (unordered unless sort_by_ordinal) to host
 * memory; thrd_num fixes node.set.  export_kmersets builds thrd_num reference KmerSets whose
 * (set, slot) layout is exactly what the reference's own init_kmerset(1024,0.77f) + put_kmerset
 * sequence would have produced for the same reads in the same order (newhash.c:160-193,
 * 293-462), which is what node2edge.c:46, cutTipPreGraph.c:1012 and prlRead2path.c:817 consume.
 * sets must point to thrd_num pointers; each receives a malloc'ed sdtgpu_kmerset. */
int sdtgpu_export_count (sdtgpu_t *h, uint64_t *n_nodes);
int sdtgpu_export_nodes (sdtgpu_t *h, int thrd_num, int sort_by_ordinal, sdtgpu_node *out, uint64_t max_nodes, uint64_t *n_nodes);
int sdtgpu_export_kmersets (sdtgpu_t *h, int thrd_num, sdtgpu_kmerset **sets);
/* Per reference set: the largest instance ordinal among ALL instances of the newest batch (owner
 * filtering does not apply), 0 for a set that batch did not touch — the set_last_ordinal input of
 * sdtgpu_build_kmersets when nodes of several GPUs are merged (put_kmerset runs encap_kmerset on
 * every call, newhash.c:415).  SDTGPU_ESTATE if no batch was pushed. */
int sdtgpu_last_ordinals (sdtgpu_t *h, int thrd_num, uint64_t *out);
/* the host half of export_kmersets, usable on nodes merged from several ranks */
int sdtgpu_build_kmersets (const sdtgpu_node *nodes, uint64_t n_nodes, int key_words, int thrd_num,
			   const uint64_t *set_last_ordinal /* [thrd_num] or NULL */, sdtgpu_kmerset **sets);
void sdtgpu_free_kmersets (sdtgpu_kmerset **sets, int thrd_num);

/* ---- lookups in the finished table (the reference's searchKmer / search_kmerset, prlRead2path.c:363, which
 * prlRead2edge and prlRead2Ctg call once per read window).
 * Valid only after sdtgpu_finalize: before it both calls return SDTGPU_ESTATE, and sdtgpu_reset puts the handle
 * back into that state.  The first lookup after finalize builds a read-only index over the table (16 bytes per
 * node; SDTGPU_ENOMEM if it does not fit, SDTGPU_ERANGE for a table of 2^32 - 1 slots or more), which is kept until
 * sdtgpu_reset or sdtgpu_destroy; a lookup after reset, push and finalize sees the new table.
 * Both calls only enqueue work on sdtgpu_stream(h): the hits are valid once that stream has been synchronised.
 * Several GPUs: these two calls answer for the handle's own share of the table only, so a key is FOUND on exactly
 * one rank (the one that owns it) and the others report it as absent.  The routed lookups below send every query to
 * its owner and answer like one table.
 *
 * A hit reports count, l_links and rword exactly as sdtgpu_export_nodes would for the node: links after the -d
 * cutoff of finalize, rword with the linear, deleted and single flags.  A window or key that is not in the table
 * has status SDTGPU_HIT_WINDOW (plus SDTGPU_HIT_RC if it applies) and zero count, l_links and rword. */
typedef struct sdtgpu_hit {
	uint32_t count;		/* as sdtgpu_node */
	uint32_t l_links;	/* as sdtgpu_node */
	uint32_t rword;		/* as sdtgpu_node: r_links | linear | deleted | single */
	uint32_t status;	/* SDTGPU_HIT_* bits; 0 = no such window / malformed key (all fields 0) */
} sdtgpu_hit;		/* 16 bytes */
#define SDTGPU_HIT_WINDOW 1u	/* a real window of the read, or a well-formed query key */
#define SDTGPU_HIT_FOUND  2u	/* its canonical k-mer is in this handle's table */
#define SDTGPU_HIT_RC     4u	/* the query / the window's forward k-mer is the reverse complement of the canonical key */

/* n keys in the sdtgpu_node layout (4 u64 each, key[0] the most significant word, the k-mer in the low 2K bits;
 * 16-byte aligned device memory) -> n hits (16-byte aligned device memory).  Each key is canonicalised as the chop
 * does (KmerSmaller: the smaller of the k-mer and its reverse complement).  A key with any bit set at 2K or above
 * is malformed: status 0, it matches nothing. */
int sdtgpu_lookup_kmers_device (sdtgpu_t *h, const uint64_t *d_keys, uint64_t n, sdtgpu_hit *d_out);
/* Every window of a batch of reads, under the conventions of sdtgpu_push_reads_device: tight-string packing,
 * stride_bytes a multiple of 4, 16-byte aligned device buffers, lens == NULL means uniform_len, reads truncated
 * to max_read_len, reads shorter than K+1 have no windows, nmask read only with SDTGPU_F_NKMER.  The windows are
 * exactly those a push chops; with SDTGPU_F_NKMER a window that holds an N looks up key 0 without
 * SDTGPU_HIT_RC, as it was inserted.  Window j of read r goes to d_out[r * maxwin + j], maxwin = max_read_len - K + 1
 * (the ordinal convention of sdtgpu_node); entries for windows a read does not have are all zero. */
int sdtgpu_lookup_reads_device (sdtgpu_t *h, const uint8_t *d_packed, const uint32_t *d_lens, const uint8_t *d_nmask,
				uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes,
				sdtgpu_hit *d_out /* n_reads x (max_read_len - K + 1) */);

/* ---- routed lookups: several GPUs, each rank with a disjoint share of the table, answer like ONE table.  Each rank
 * passes its own queries; every query travels to the rank that owns its canonical key, is answered there, and the
 * hit comes back into the caller's output in the layout of the two calls above.  The hits are bit-identical to
 * sdtgpu_lookup_kmers_device / sdtgpu_lookup_reads_device on one handle built from all ranks' reads with the same -d
 * (every field of a hit depends only on its own node, and the union of the shares is that table).
 *
 * The owner of a canonical key k is the rank whose share holds it, under the sharding the handle was built with:
 *   sliced build, sdtgpu_skm_set_world (rank, world), world > 1     slice_of_min (minval (k)) / n_local  (the slices
 *        (SDTGPU_ROUTE_SKM)                                         are dealt to the ranks in contiguous ranges)
 *   sliced build, sdtgpu_set_owner (rank, n), n > 1                 slice_of_min (minval (k)) % n
 *        (SDTGPU_ROUTE_SLICED)
 *   single-pass insert, sdtgpu_set_owner (rank, n), n > 1            owner_of (key_hash (k), n), the owner function of
 *        (SDTGPU_ROUTE_HASHED)                                      the replicated-reads sharding and of the record
 *                                                                   exchange (sdtgpu_bucket_reads_device)
 *   neither (SDTGPU_ROUTE_ONE)                                      0: the world is 1
 * minval (k) is the minimizer value the sliced build gives a window: the smallest hashed canonical m-mer among the
 * central m-mers of the k-mer (sdtgpu_lookup_route: m, lo, w), computed from the key alone.  A handle filled by the
 * record exchange must declare its share with sdtgpu_set_owner (rank, world) before it finalizes: bucket_reads_device
 * takes the number of ranks per call, and the handle does not otherwise know it.
 *
 * Three halves, so that any transport can move the buffers (sdtgpu_lookup_*_exchange below drives them over NCCL):
 *   stage     sdtgpu_lookup_stage_kmers / _reads take the arguments and conventions of the two calls above, without
 *             the output.  Each well-formed key or window is canonicalised and goes, as device_key_words u64 words
 *             (most significant first), into the region of its owner: owner r's queries are counts[r] queries from
 *             query starts[r] of *d_queries on, with no gaps (starts, counts: [world]).  Malformed keys and windows a
 *             read does not have stay home.  The handle keeps each staged query's output position and RC bit.
 *   answer    the owner: sdtgpu_lookup_answer_buffer (h, n, &q, &r) gives room for n received queries (q) and their
 *             hits (r); the caller puts the queries there in any order; sdtgpu_lookup_answer (h, n) writes hit i for
 *             query i.
 *   unstage   sdtgpu_lookup_unstage_buffer (h, &back) gives room for the hits of this rank's staged queries, which
 *             the caller puts there in staged order (same starts and counts); sdtgpu_lookup_unstage (h, d_out) writes
 *             them to d_out (n hits for keys, n_reads x maxwin for reads, 16-byte aligned), RC put back, and what
 *             did not travel as the single-GPU call writes it (all zero).
 * All of it only after sdtgpu_finalize (SDTGPU_ESTATE before it and after sdtgpu_reset), at most 64 ranks.  A stage
 * builds the lookup index of this rank's share if it is missing.  Unstage needs a stage (else SDTGPU_ESTATE); a new
 * stage replaces the last one.  n = 0 is legal everywhere.  NULL buffers are SDTGPU_EINVAL before any CUDA call.
 * The buffers belong to the handle, grow only and are kept across calls (each call may move them: take the
 * addresses again); sdtgpu_reset and sdtgpu_destroy free them.  The kernels run on sdtgpu_stream(h) and are timed in
 * class 7 of sdtgpu_phase_times; a stage synchronises that stream once (the counts), the other calls only enqueue. */
#define SDTGPU_ROUTE_ONE    0
#define SDTGPU_ROUTE_SKM    1
#define SDTGPU_ROUTE_SLICED 2
#define SDTGPU_ROUTE_HASHED 3
/* out = { SDTGPU_ROUTE_*, rank, world, K, device_key_words, n_slices, n_local, m, lo, w, deLowKmer of finalize,
 * finalized }; the slice fields are 0 where the sharding does not use them */
int sdtgpu_lookup_route (const sdtgpu_t *h, uint64_t out[12]);
int sdtgpu_lookup_stage_kmers (sdtgpu_t *h, const uint64_t *d_keys, uint64_t n,
			       void **d_queries, uint64_t *starts /* world */, uint64_t *counts /* world */);
int sdtgpu_lookup_stage_reads (sdtgpu_t *h, const uint8_t *d_packed, const uint32_t *d_lens, const uint8_t *d_nmask,
			       uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes,
			       void **d_queries, uint64_t *starts /* world */, uint64_t *counts /* world */);
int sdtgpu_lookup_answer_buffer (sdtgpu_t *h, uint64_t n, void **d_queries, sdtgpu_hit **d_replies);
int sdtgpu_lookup_answer (sdtgpu_t *h, uint64_t n);
int sdtgpu_lookup_unstage_buffer (sdtgpu_t *h, sdtgpu_hit **d_back);
int sdtgpu_lookup_unstage (sdtgpu_t *h, sdtgpu_hit *d_out);

/* ---- edges between junction k-mers (the graph kmer2edges builds, node2edge.c:46, without its pruning), one GPU.
 * A node with canonical key k = b0..b(K-1) is read as (v,+) = k and (v,-) = rc(k).  The out-links of (v,+) are the
 * right counters R[x] > 0 of the finalized table (after -d), successor b1..b(K-1) x canonicalised; those of (v,-) the
 * left counters L[x] > 0, successor rc(x b0..b(K-2)), base appended comp(x) = x ^ 2.  A node is linear when exactly one
 * left and one right counter are non-zero (the linear bit of rword), a vertex when it is neither linear nor deleted.
 *   edge    a walk x0 -> x1 -> ... -> xm (m >= 1) over out-links, x0 and xm vertices, x1 .. x(m-1) linear: one per
 *           (oriented vertex, out-link).  Its sequence has m + K bases.  Of a walk and its reverse complement (the walk
 *           from xm in the other orientation) the one kept is the one whose first (K+1)-mer is <= the reverse
 *           complement of its last (K+1)-mer, as (2K+2)-bit integers; equality means the walk is its own reverse
 *           complement (SDTGPU_EDGE_PALINDROME: it runs through a hairpin and holds its interior nodes twice).
 *   cycle   the linear nodes no edge visits form closed walks (poly-A, a circular transcript, a chain closed by two
 *           hairpins, which is SDTGPU_EDGE_PALINDROME too and holds its nodes twice).  One record each, flag
 *           SDTGPU_EDGE_CYCLE: m k-mers read circularly from a start and strand of the library's choice, m + K - 1 bases.
 *   count_sum  the sum of count over x1 .. x(m-1); for a cycle over all its m k-mers.
 *   link       x0's counter for the first step.
 * The records are numbered by start (table position, orientation + before -, counter index), keeping the kept walks
 * only; the cycles follow the edges.  Two builds of one table give byte-identical buffers.  The sequences are in the
 * reads' tight-string convention (4 bases per byte, first base in bits 7..6); each starts at a multiple of 32 bases,
 * its last word zero-padded.
 *
 * sdtgpu_edges_build: out = { edges (cycles included), palindromic edges (cycles included), cycles, bases, vertices,
 * linear nodes on edges, linear nodes on cycles, dangling links } where a palindrome counts its nodes once, and a dangling
 * link is a non-zero counter whose neighbour is not in the table or a linear node's neighbour without the link back
 * (there are none in a table built by this library: both ends of a (K+1)-mer count the same instances).  ms: device
 * time of the build (CUDA events).  Valid after sdtgpu_finalize (SDTGPU_ESTATE before it and after sdtgpu_reset); a
 * handle that holds one rank's share of a sharded table (sdtgpu_lookup_route case other than SDTGPU_ROUTE_ONE) is
 * SDTGPU_EINVAL; NULL arguments are SDTGPU_EINVAL before any CUDA call; SDTGPU_ENOMEM if the buffers do not fit (about
 * 41 bytes per table slot, 8 per walk start, plus the output).  Builds the lookup index if it is missing; synchronises
 * the handle's stream.
 * sdtgpu_edges_buffers: the device addresses of the last build's records (out[0] of them) and sequences, SDTGPU_ESTATE
 * before a build.  The buffers belong to the handle, grow only and may move at the next build; sdtgpu_reset and
 * sdtgpu_destroy free them. */
typedef struct sdtgpu_edge {
	uint64_t seq;		/* first base in the sequence buffer, counted in bases; a multiple of 32 */
	uint32_t length;	/* m: an edge has m+1 k-mers and m+K bases; a cycle has m k-mers and m+K-1 bases */
	uint32_t flags;		/* SDTGPU_EDGE_PALINDROME, SDTGPU_EDGE_CYCLE */
	uint64_t count_sum;
	uint32_t link;
	uint32_t unused;	/* 0 */
} sdtgpu_edge;		/* 32 bytes */
#define SDTGPU_EDGE_PALINDROME 1u
#define SDTGPU_EDGE_CYCLE      2u
int sdtgpu_edges_build (sdtgpu_t *h, uint64_t out[8], double *ms);
int sdtgpu_edges_buffers (sdtgpu_t *h, const sdtgpu_edge **d_edges, const uint8_t **d_seq);

/* pinned host memory for the caller's batch buffers (the reference's seqBuffer/lenBuffer role,
 * prlHashReads.c:387-395); plain pageable memory also works with push_reads, only slower */
int sdtgpu_host_alloc (void **out, size_t bytes);
void sdtgpu_host_free (void *p);

/* ---- measurement hooks */
void *sdtgpu_stream (sdtgpu_t *h);	/* the cudaStream_t the handle's insert work is enqueued on */
void *sdtgpu_aux_stream (sdtgpu_t *h);	/* second stream: H2D copies of push_reads and bucket_reads_device kernels */
/* device time (ms, CUDA events on the handle's stream) and launch count accumulated by the insert
 * kernels since the last call with reset != 0 */
int sdtgpu_kernel_time (sdtgpu_t *h, int reset, double *insert_ms, uint64_t *insert_launches, uint64_t *all_launches);
/* per kernel class: [0] insert (direct, staged or records), [1] partition count pass, [2] partition scatter pass */
int sdtgpu_kernel_times (sdtgpu_t *h, int reset, double ms[3], uint64_t launches[3]);

/* per kernel class since the last reset: [0] insert (single-pass, staged or records), [1] count
 * (staged path) or super-k-mer emit (sliced build), [2] scatter, [3] record dedupe (sliced build),
 * [4] slice build, [5] scans, [6] slice build, retried work items, [7] lookups (index build and lookup kernels) */
int sdtgpu_phase_times (sdtgpu_t *h, int reset, double ms[8], uint64_t launches[8]);
/* SDTGPU_F_SLICED only: out = { slices, slots per slice image, minimizer length m, m-mers per window,
 * bytes per super-k-mer record, records held, nodes in the store, work items retried by the last build,
 * records left after identical ones were merged (last build), work items of the last build,
 * epochs whose records had to be made a second time since create (the block pool was too small),
 * device buffers (re)allocated since create } */
int sdtgpu_slice_geometry (const sdtgpu_t *h, uint64_t out[12]);

/* debug (library built with -DSDT_BUILD_PROF; zeros otherwise): phase clocks of the slice build kernel,
 * summed over thread 0 of every CTA (SM cycles): [0] prepare, [2] insert, [3] compact, [4] work items, [5] chunks */
int sdtgpu_debug_prof (uint64_t out[8], int reset);

/* ---- super-k-mer exchange: the sliced build on several GPUs, one process per GPU (SDTGPU_F_SLICED).
 * The reference shards k-mers over its threads by hash (prlHashReads.c:79-88); here the table slices
 * (ranges of minimizers) are dealt to the ranks in contiguous ranges, so whole super-k-mer records
 * travel — and only one copy of each per sending rank, with a multiplicity: ~1.5 bytes per k-mer instance
 * instead of a 16-byte record each.  Per epoch, on every rank:
 *   sdtgpu_skm_set_world   once, before the first push: rank and number of ranks (needs capacity_hint =
 *                          expected distinct k-mers PER RANK, the same on all ranks);
 *   sdtgpu_skm_set_ordinal_bound  optional: reads pushed on ALL ranks this epoch (lets the slice images
 *                          keep 32-bit ordinals when they fit);
 *   sdtgpu_push_reads*     this rank's own reads (global first_read_ordinal);
 *   sdtgpu_skm_stage       merges this rank's copies and packs the records by owner: rank r's records
 *                          (of sdtgpu_slice_geometry()[4] bytes) are counts[r] records from record
 *                          starts[r] of *d_records on;
 *   (caller)               all-to-all of counts and records (NCCL) into the buffer that
 *   sdtgpu_skm_import_buffer  returns for the total it is going to receive;
 *   sdtgpu_skm_import      builds this rank's slices from the n_records received.
 * Afterwards finalize / export / stats see this rank's share of the table. */
int sdtgpu_skm_set_world (sdtgpu_t *h, int rank, int world);
int sdtgpu_skm_set_ordinal_bound (sdtgpu_t *h, uint64_t n_reads_all_ranks);
int sdtgpu_skm_stage (sdtgpu_t *h, void **d_records, uint64_t *starts /* world */, uint64_t *counts /* world */);
int sdtgpu_skm_import_buffer (sdtgpu_t *h, uint64_t n_records, void **d_buffer);
int sdtgpu_skm_import (sdtgpu_t *h, uint64_t n_records);

/* ---- the same exchange in ONE call, NCCL inside the library (csrc/sdt_nccl.cu).  NCCL is bound at run time
 * (dlopen of libnccl.so.2), so single-GPU users never load it.  A communicator is made once per process:
 *   rank 0:      sdtgpu_comm_unique_id (id);  hand the 128 bytes to every rank (MPI_Bcast, a file, a socket ...)
 *   every rank:  sdtgpu_comm_create (&c, device, id, rank, world);
 * and per epoch, after sdtgpu_skm_set_world and this rank's pushes:
 *   sdtgpu_skm_exchange (h, c, reads_end, &n_received, &collective_ms)
 * = all-reduce of the ordinal bound (reads_end: one past the largest global read ordinal this rank pushed),
 * sdtgpu_skm_stage, all-gather of the counts, one grouped ncclSend / ncclRecv of the records straight into the
 * import buffer, sdtgpu_skm_import.  collective_ms (may be NULL): device time of counts + records, CUDA events.
 * Collective: every rank of the communicator must make the call. */
#define SDTGPU_COMM_ID_BYTES 128
typedef struct sdtgpu_comm sdtgpu_comm_t;
int sdtgpu_comm_unique_id (uint8_t id[SDTGPU_COMM_ID_BYTES]);
int sdtgpu_comm_create (sdtgpu_comm_t **out, int device, const uint8_t id[SDTGPU_COMM_ID_BYTES], int rank, int world);
int sdtgpu_comm_destroy (sdtgpu_comm_t *c);
const char *sdtgpu_comm_last_error (const sdtgpu_comm_t *c);	/* c may be NULL: last failure without a communicator */
int sdtgpu_skm_exchange (sdtgpu_t *h, sdtgpu_comm_t *c, uint64_t reads_end_this_rank, uint64_t *n_received, double *collective_ms);
/* Routed lookups in ONE collective call each (every rank of the communicator makes it, after finalize; a rank with
 * nothing to ask passes n = 0).  The comm's rank and world must equal the handle's sharding (sdtgpu_lookup_route),
 * else SDTGPU_EINVAL before any collective.  Then the ranks all-gather their sharding descriptors (case, world, K,
 * device key words, n_slices, n_local, m, lo, w, -d of finalize, finalized) and all return SDTGPU_EINVAL if they
 * differ; stage, all-gather of the counts (and of every rank's stage status: if one failed, all return), one grouped
 * ncclSend / ncclRecv of the queries into the owners' answer buffers (the own share is a device-local copy), answer,
 * one grouped send / recv of the hits back, unstage into d_out.  Same inputs and outputs as
 * sdtgpu_lookup_kmers_device / sdtgpu_lookup_reads_device; returns when the hits are in d_out.
 * collective_ms (may be NULL): device time of the collectives that move the lookup's data, i.e. the counts
 * all-gather and the two grouped send / recv (CUDA events); stage, answer and unstage are in class 7 of
 * sdtgpu_phase_times. */
int sdtgpu_lookup_kmers_exchange (sdtgpu_t *h, sdtgpu_comm_t *c, const uint64_t *d_keys, uint64_t n, sdtgpu_hit *d_out,
				  double *collective_ms);
int sdtgpu_lookup_reads_exchange (sdtgpu_t *h, sdtgpu_comm_t *c, const uint8_t *d_packed, const uint32_t *d_lens,
				  const uint8_t *d_nmask, uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes,
				  sdtgpu_hit *d_out, double *collective_ms);

/* ---- synthetic reads on the device (bench/test utility; bit-identical to synth.py).
 * d_tr_bases: uint8 codes of all transcripts; d_starts u64[T]; d_lengths u32[T]; d_cum u64[T]. */
int sdtgpu_synth_reads_device (int device, void *stream, const uint8_t *d_tr_bases, const uint64_t *d_starts,
			       const uint32_t *d_lengths, const uint64_t *d_cum, uint32_t n_transcripts,
			       uint64_t seed, uint64_t first_pair, uint64_t n_pairs, uint32_t read_len,
			       uint32_t stride_bytes, uint8_t *d_packed_out);

/* ---- FASTA/FASTQ files parsed and packed on the GPU (csrc/sdt_parse.cu).  The records, their order and every output
 * byte equal what sdtpack_next (include/sdtpack.h) produces for the same files and options; the batches are in the
 * layout sdtgpu_push_reads_device and sdtgpu_lookup_reads_device take.  The text goes to the device in chunks (pinned
 * staging, parallel pread, cudaMemcpyAsync); every chunk starts at a record boundary, a record longer than a chunk
 * makes the chunk grow, junk lines never do.  Device buffers grow only and are freed by close.
 * path2 == NULL: single-ended.  fastq: 0 FASTA, 1 FASTQ.  chunk_bytes: size of one text upload (0 = 64 MiB;
 * small values are for tests).  SDTGPU_EINVAL if a file cannot be opened (sdtgpu_reader_last_error names it).
 * open touches no CUDA state; the first sdtgpu_reader_next sets the reader up on `device`. */
typedef struct sdtgpu_reader sdtgpu_reader_t;
int sdtgpu_reader_open (sdtgpu_reader_t **out, int device, const char *path1, const char *path2, int fastq,
			uint64_t chunk_bytes);
/* The next min (M, remaining) records of the stream, M = max_reads (pairs: max_reads rounded down to even),
 * written to d_packed / d_lens / d_nmask (16-byte aligned device buffers, nmask only with n_kmer) with the
 * conventions and argument checks of sdtpack_next.  *n_out = 0 at end of input.  The pack kernels are enqueued
 * on `stream` (NULL: the legacy default stream); the call returns once *n_out is known, and the outputs are
 * valid once that stream has reached them.  stride_bytes is at most 6144 (4096 with n_kmer). */
int sdtgpu_reader_next (sdtgpu_reader_t *r, void *stream, int max_read_len, int n_kmer, int reverse,
			uint8_t *d_packed, uint32_t *d_lens, uint8_t *d_nmask, uint64_t max_reads,
			uint32_t stride_bytes, uint64_t *n_out);
/* out = { text bytes copied host to device, records returned, chunks uploaded, device buffer (re)allocations } */
int sdtgpu_reader_stats (const sdtgpu_reader_t *r, uint64_t out[4]);
const char *sdtgpu_reader_last_error (const sdtgpu_reader_t *r);	/* r may be NULL: last open() failure */
void sdtgpu_reader_close (sdtgpu_reader_t *r);

/* One library read by `world` ranks together, each parsing only its own byte range (DESIGN §9.1 "One library, several
 * readers").  The stream is the records sdtpack_next returns; a record's ordinal is its place in it (a pair of n1 and n2
 * records, m = min (n1, n2): record i < m of file 1 is 2i, of file 2 is 2i + 1, record j >= m of the longer file is
 * m + j).  Rank r's range of a file of S bytes is [r S / world, (r + 1) S / world); a line belongs to the range that
 * holds its first byte, a record to the range that holds its header line.  Rank r returns the records of its range of
 * file 1 (single-ended), or (pairs) the pairs i in [min (m, c1_r), min (m, c1_r+1)), c1_r = file-1 records before range
 * r, then the records j >= m of the longer file in its range of that file.  Put in ordinal order, every rank's batches
 * are byte for byte the output of sdtpack_next, and every ordinal comes back once.
 *   open_shard  like open (no CUDA state), plus rank and world; SDTGPU_EINVAL unless 0 <= rank < world <= 1024.
 *   summary     scans this rank's range of each file on the device (sets the reader up on `device`) into 256 opaque
 *               bytes: rank, world, fastq, files, sizes, a fingerprint of each file's first and last 4 KiB, and per
 *               file the first line start of the range, its line starts, the FASTA header rule over them and the
 *               first FASTQ header candidate.  Computed once; later calls return the same bytes.
 *   plan        host arithmetic only, the same on every rank: from every rank's summary (world x 256 bytes, in rank
 *               order) where each range starts and how many records come before it.  SDTGPU_EINVAL if a summary is of
 *               other files, sizes, FASTQ-ness or world, or out of order.  out = { records this rank returns,
 *               records of the library, n1, n2 (0 single-ended) }.
 *   next        as for a plain reader, SDTGPU_ESTATE before plan; one call never returns records across a jump in
 *               ordinals (a rank's pairs, then its records of the longer file).
 *   tell        the ordinal of the next record (nothing left: one past the last one returned); on a plain reader
 *               the records returned so far.  SDTGPU_ESTATE on a shard reader before plan.
 *   plan_exchange (csrc/sdt_nccl.cu)  summary, all-gather of the summaries over the library's communicator (a device
 *               buffer of world x 256 bytes), plan.  Collective; SDTGPU_EINVAL before any collective if the
 *               communicator's rank or world is not the reader's.
 * summary and plan on a plain reader are SDTGPU_ESTATE.  The text bytes of sdtgpu_reader_stats count the summary pass
 * and the seeks too: a rank reads its range twice (summary, parse), at most a chunk past its end, and for the file-2
 * half of its pairs (and its records of the longer file) the text from the start of the range that holds the first of
 * them: a few records when both files lay their records out alike, up to one range otherwise. */
#define SDTGPU_READER_SUMMARY_BYTES 256
int sdtgpu_reader_open_shard (sdtgpu_reader_t **out, int device, const char *path1, const char *path2, int fastq,
			      uint64_t chunk_bytes, int rank, int world);
int sdtgpu_reader_summary (sdtgpu_reader_t *r, uint8_t out[SDTGPU_READER_SUMMARY_BYTES]);
int sdtgpu_reader_plan (sdtgpu_reader_t *r, const uint8_t *summaries, uint64_t out[4]);
int sdtgpu_reader_tell (const sdtgpu_reader_t *r, uint64_t *ordinal);
int sdtgpu_reader_plan_exchange (sdtgpu_reader_t *r, sdtgpu_comm_t *c, uint64_t out[4]);

/* reference helpers restated for host callers (tests bind them) */
uint64_t sdtgpu_hash_kmer (const uint64_t key[4], int key_words);	/* hashFunction.c:108 */
int sdtgpu_version (void);

#ifdef __cplusplus
}
#endif
#endif
