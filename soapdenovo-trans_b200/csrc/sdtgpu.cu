// sdtgpu.cu — C ABI (include/sdtgpu.h) over the sm_100a kernels in sdt_kernels.cuh.
// Host-side plumbing only: streams, staging, capacity management, launches, D2H of results.
// There is NO CPU fallback: every entry point either runs the CUDA path or returns an error.
#include "../../include/sdtgpu.h"
#include "sdt_kernels.cuh"
#include "sdt_skm.cuh"
#include "sdt_merge.cuh"
#include "sdt_build.cuh"
#include "sdt_lookup.cuh"
#include "sdt_route.cuh"
#include "sdt_edges.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <chrono>
#include <string>
#include <vector>

using namespace sdt;

namespace {

thread_local std::string g_create_error;

struct Staging
{
	uint8_t *d_packed = nullptr, *d_mask = nullptr;
	u32 *d_lens = nullptr;
	size_t cap_packed = 0, cap_mask = 0, cap_lens = 0;
	cudaEvent_t free_ev = nullptr;	// recorded on the compute stream after the kernel that read this buffer
	cudaEvent_t ready_ev = nullptr;	// recorded on the copy stream after the H2D copies
};

// one pushed batch in the read log of the open epoch (sliced build); offsets into the log arenas
struct LogSeg
{
	size_t off[3];	// packed, lens, mask
	ReadBatch rb;	// pointers are resolved when the segment is used (the arenas may move)
	u64 upper;	// windows of the batch at most
};

enum { ED_STEP, ED_MARK, ED_A, ED_B, ED_OFF_A, ED_OFF_B, ED_STARTS, ED_SEG, ED_CTR, ED_EDGES, ED_SEQ, ED_N };	// sdtgpu::ed

static constexpr int N_CAT = 8;	// timing classes: 0 insert, 1 count / emit, 2 scatter, 3 dedupe, 4 build, 5 scan, 6 build retries, 7 lookups

}	// namespace

// a set of chains of record blocks (sdt_chain.cuh) with what is derived from it
struct ChainLevel
{
	u32 n_chains = 0, cap_chains = 0;
	u64 *head = nullptr, *boff = nullptr, *seg_sum = nullptr, *d_cursor = nullptr;	// d_cursor: [0] pool cursor, [1] output cursor of the merge, [2] work items, [3] group cursor (inside cta_pool's allocation)
	u32 *bcount = nullptr, *bchain = nullptr, *bseq = nullptr, *blist = nullptr, *recs = nullptr;
	uint2 *cta_pool = nullptr;
	u64 pool_blocks = 0, blocks_upper = 0, blist_cap = 0, pool_high = 0;	// pool_high: the largest pool an epoch has needed
	u32 *out = nullptr;	// the merged records, and the work items of the build that skm_merge_kernel cuts them into
	u64 out_cap = 0;
	SkmWork *items = nullptr;
};

struct sdtgpu
{
	int device = 0, K = 0, key_words = 0, W = 0, max_read_len = 0;
	u32 maxwin = 0;
	unsigned flags = 0;
	void *table = nullptr;
	u64 cap = 0;
	bool grow_mode = false;
	Counters *d_ctr = nullptr;
	Counters *h_ctr = nullptr;	// pinned mirror
	cudaStream_t stream = nullptr, copy_stream = nullptr;
	cudaStream_t launch_stream = nullptr;	// stream the next read kernel goes to (main unless bucketing)
	Staging stage[2];
	int next_stage = 0;
	int sm_count = 0;
	size_t mem_total = 0;	// device memory (cudaMemGetInfo is slow — milliseconds with several processes on a box — so it is only asked when an allocation is about to happen)
	u64 pushed_upper = 0;	// upper bound of instances pushed (host-side arithmetic)
	// the most recent batch stays on the device until the next one arrives: the hand-back needs the
	// per-set last instance ordinal (put_kmerset runs encap_kmerset on every call, newhash.c:415)
	uint8_t *last_packed = nullptr, *last_mask = nullptr;
	u32 *last_lens = nullptr;
	size_t last_cap_packed = 0, last_cap_mask = 0, last_cap_lens = 0;
	ReadBatch last_rb;
	bool have_last = false;
	// lagging snapshot of the node counter, so that the capacity check never has to drain the stream
	u64 *h_nodes_snap = nullptr;	// pinned
	cudaEvent_t snap_ev = nullptr;
	bool snap_pending = false;
	u64 snap_pushed = 0, known_nodes = 0, known_at = 0;
	u64 n_reads = 0;
	u64 ord_end = 0;	// one past the largest instance ordinal pushed since the last reset
	u32 n_grows = 0;
	bool finalized = false;
	int deLowKmer = 0;
	u64 *index = nullptr;	// lookup index over the finalized table (sdt_lookup.cuh): made by the first lookup, freed by reset
	u64 idx_cap = 0;
	// routed lookups (sdt_route.cuh): the buffers grow only and are kept across calls; reset and destroy free them
	u64 *rt_q = nullptr, *rt_tag = nullptr, *rt_aq = nullptr;	// staged queries and their tags, received queries
	Hit *rt_ar = nullptr, *rt_back = nullptr;	// replies of this rank as owner, replies to this rank's staged queries
	size_t rt_cap_q = 0, rt_cap_tag = 0, rt_cap_aq = 0, rt_cap_ar = 0, rt_cap_back = 0;	// bytes
	u64 *rt_cur = nullptr, *rt_hcur = nullptr;	// per-owner counts / cursors of the stage; pinned mirror
	bool rt_staged = false;	// a stage awaits its unstage
	u64 rt_n = 0, rt_out = 0;	// queries staged, entries of the caller's output
	u32 owner_rank = 0, owner_ranks = 1;	// sdtgpu_set_owner
	// edges (sdt_edges.cuh): the buffers grow only and are kept across builds; reset and destroy free them
	void *ed[ED_N] = {};
	size_t ed_cap[ED_N] = {};	// bytes
	bool ed_built = false;
	// sliced build (SDTGPU_F_SLICED): reads of the open epoch are kept in a log and turned into super-k-mer
	// records in the chains of their slices as they arrive; sliced_flush merges copies and builds the slices
	bool sliced = false, table_built = false, epoch_open = false, emitted = false, ord_bound_set = false, chains_dropped = false;
	u64 hint = 0, store_want = 0;
	SkmGeom geom = {};
	void *log_mem[3] = { nullptr, nullptr, nullptr };	// packed, lens, mask arenas
	size_t log_cap[3] = { 0, 0, 0 }, log_used[3] = { 0, 0, 0 };
	std::vector<LogSeg> log;
	ChainLevel lv[3];	// [0] the slices (several GPUs: ALL ranks' slices, the sending side), [1] sub-slices of slices that overflowed, [2] this rank's slices, receiving side
	u64 *d_small = nullptr, *h_small = nullptr;	// [0] records made, [1] node cursor, [2] failed work items, [3] work-item cursor, [4] records after the merge, [5] their windows, [8..] owner regions; pinned mirror
	void *d_failed = nullptr, *d_items = nullptr, *h_failed = nullptr;	// SkmWork lists (h_failed: pinned, the first FAILED_PREFIX of d_failed)
	u64 win_left = 0;	// windows the last merge left
	u32 *rx = nullptr;	// records received from other ranks
	u64 rx_cap = 0;
	u32 skm_world = 1, skm_rank = 0, n_local = 0;	// super-k-mer exchange (sdtgpu_skm_set_world): slices per rank; geom.n_slices = n_local * skm_world
	u64 n_reemit = 0, n_alloc = 0;	// since create: epochs whose records were made a second time (block pool too small); device buffers (re)allocated after the first flush
	u64 n_store = 0, n_records = 0, n_retried = 0, n_merged = 0, n_items = 0;	// nodes in the store after the last build
	bool dirty = false;	// records were emitted since the last build
	u32 n_epochs = 0;
	struct Timed { cudaEvent_t e0, e1; int cat; };
	std::vector<Timed> timing;
	double cat_ms[N_CAT] = { 0 };
	u64 cat_launches[N_CAT] = { 0 };
	std::vector<cudaEvent_t> ev_pool;
	u64 all_launches = 0;
	std::string err;
};

namespace {

#define CK(h, call)                                                                                     \
	do                                                                                              \
	{                                                                                               \
		cudaError_t e_ = (call);                                                                \
		if (e_ != cudaSuccess)                                                                  \
		{                                                                                       \
			char b_[512];                                                                   \
			snprintf (b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString (e_), __FILE__, __LINE__); \
			(h)->err = b_;                                                                  \
			return e_ == cudaErrorMemoryAllocation ? SDTGPU_ENOMEM : SDTGPU_ECUDA;          \
		}                                                                                       \
	} while (0)

size_t slot_bytes (int W) { return W == 4 ? sizeof (Slot4) : 32; }

// Slots for `nodes` expected distinct keys: load 0.5 when that fits in 60 GiB, otherwise as sparse
// as 60 GiB allows but never denser than 0.85.  Random access over a table larger than 64 GiB is
// 4x slower on B200 (36 G -> 9.8 G cold-line requests/s at 128 GiB, tools/randacc_bench.cu,
// profiles/r1_randacc_bench.txt), so staying under that size beats a lower load factor.
u64 pick_capacity (u64 nodes, size_t slot)
{
	const u64 fast = (60ull << 30) / slot;
	const u64 sparse = nodes * 2, dense = (u64) ((double) nodes / 0.85) + 1;
	return std::max<u64> (1024, std::max (dense, std::min (sparse, fast)));
}

int fail (sdtgpu *h, int code, const char *msg)
{
	h->err = msg;
	return code;
}

template <int W> void launch_init (sdtgpu *h, void *table, u64 cap)
{
	const u64 want = (cap + BLOCK - 1) / BLOCK;
	const unsigned grid = (unsigned) std::min<u64> (want, (u64) h->sm_count * 16);
	init_table_kernel<W><<<grid, BLOCK, 0, h->stream>>> (static_cast<typename SlotOf<W>::type *> (table), cap);
	h->all_launches++;
}

int init_table (sdtgpu *h, void *table, u64 cap)
{
	switch (h->W)
	{
	case 1: launch_init<1> (h, table, cap); break;
	case 2: launch_init<2> (h, table, cap); break;
	default: launch_init<4> (h, table, cap); break;
	}
	CK (h, cudaGetLastError ());
	return SDTGPU_OK;
}

template <int W> void launch_rehash (sdtgpu *h, void *old, u64 old_cap, void *neu, u64 cap)
{
	typedef typename SlotOf<W>::type S;
	const unsigned grid = (unsigned) std::min<u64> ((old_cap + BLOCK - 1) / BLOCK, (u64) h->sm_count * 16);
	rehash_kernel<W><<<grid, BLOCK, 0, h->stream>>> (static_cast<const S *> (old), old_cap, static_cast<S *> (neu), cap);
	h->all_launches++;
}

int read_counters (sdtgpu *h)
{
	CK (h, cudaMemcpyAsync (h->h_ctr, h->d_ctr, sizeof (Counters), cudaMemcpyDeviceToHost, h->stream));
	CK (h, cudaStreamSynchronize (h->stream));
	return SDTGPU_OK;
}

// Keep the load factor bounded before `incoming` more instances are inserted.  The table never
// fills beyond max_load even if every incoming instance were a new key.  With a capacity hint the
// table is sized once (load <= 0.5 at the hinted count); without one it starts small and grows by
// device re-hash, like the reference's encap_kmerset (newhash.c:293-409).  The check uses a
// lagging snapshot of the device's node counter (copied asynchronously after every launch), so
// the steady state costs no stream synchronisation.
int ensure_capacity (sdtgpu *h, u64 incoming)
{
	const double max_load = 0.90;
	if (h->snap_pending && cudaEventQuery (h->snap_ev) == cudaSuccess)
	{
		h->snap_pending = false;
		h->known_nodes = *h->h_nodes_snap;
		h->known_at = h->snap_pushed;
	}
	const u64 bound = h->known_nodes + (h->pushed_upper - h->known_at);	// >= nodes in the table now
	if ((double) (bound + incoming) <= max_load * (double) h->cap)
		return SDTGPU_OK;
	int rc = read_counters (h);
	if (rc)
		return rc;
	const u64 nodes = h->h_ctr->n_nodes;
	h->known_nodes = nodes;
	h->known_at = h->pushed_upper;
	h->snap_pending = false;
	if ((double) (nodes + incoming) <= max_load * (double) h->cap)
		return SDTGPU_OK;
	u64 new_cap = std::max<u64> (h->cap + h->cap / 2, pick_capacity (nodes + incoming, slot_bytes (h->W)));
	void *neu = nullptr;
	CK (h, cudaMalloc (&neu, new_cap * slot_bytes (h->W)));
	rc = init_table (h, neu, new_cap);
	if (rc)
		return rc;
	switch (h->W)
	{
	case 1: launch_rehash<1> (h, h->table, h->cap, neu, new_cap); break;
	case 2: launch_rehash<2> (h, h->table, h->cap, neu, new_cap); break;
	default: launch_rehash<4> (h, h->table, h->cap, neu, new_cap); break;
	}
	CK (h, cudaGetLastError ());
	CK (h, cudaStreamSynchronize (h->stream));
	CK (h, cudaFree (h->table));
	h->table = neu;
	h->cap = new_cap;
	h->n_grows++;
	return SDTGPU_OK;
}

int snapshot_nodes (sdtgpu *h)
{
	if (h->snap_pending)
		return SDTGPU_OK;
	CK (h, cudaMemcpyAsync (h->h_nodes_snap, &h->d_ctr->n_nodes, sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
	CK (h, cudaEventRecord (h->snap_ev, h->stream));
	h->snap_pending = true;
	h->snap_pushed = h->pushed_upper;
	return SDTGPU_OK;
}

cudaEvent_t get_event (sdtgpu *h)
{
	if (!h->ev_pool.empty ())
	{
		cudaEvent_t e = h->ev_pool.back ();
		h->ev_pool.pop_back ();
		return e;
	}
	cudaEvent_t e = nullptr;
	cudaEventCreate (&e);
	return e;
}

u32 pick_tile_reads (u32 stride_bytes)
{
	u32 t = (16384u / stride_bytes) & ~3u;
	return std::max (4u, std::min ((u32) MAX_TILE_READS, t));
}

size_t insert_smem_bytes (const ReadBatch &rb, bool nmode, size_t hist_bins)
{
	const size_t sw = rb.stride_bytes / 4, mw = nmode ? (rb.mask_stride + 3) / 4 : 0;
	return 4 * (2 * TILE_PAD + rb.tile_reads * sw + rb.tile_reads + 4 + rb.tile_reads * mw + hist_bins);
}

template <int W, bool NMODE, int MODE> int launch_insert_t (sdtgpu *h, const ReadBatch &rb, const Bins &bins, const Lookup &lk)
{
	typedef typename SlotOf<W>::type S;
	auto kern = insert_reads_kernel<W, NMODE, MODE>;
	const size_t smem = insert_smem_bytes (rb, NMODE, MODE == 1 ? 3 * (size_t) bins.n_ranks + 4 : (MODE == 4 ? 2 * (size_t) bins.n_ranks + 2 : (MODE == 5 ? 2 * (size_t) rb.queue_cap * (W + 1) + 2 : 0)));
	if (smem > 48 * 1024)
		CK (h, cudaFuncSetAttribute (kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	int occ = 0;
	CK (h, cudaOccupancyMaxActiveBlocksPerMultiprocessor (&occ, kern, BLOCK, smem));
	if (occ < 1)
		return fail (h, SDTGPU_EINVAL, "read stride too large for one shared-memory tile");
	const u64 n_tiles = (rb.n_reads + rb.tile_reads - 1) / rb.tile_reads;
	const unsigned grid = (unsigned) std::min<u64> (n_tiles, (u64) h->sm_count * occ);
	cudaStream_t ls = h->launch_stream ? h->launch_stream : h->stream;
	cudaEvent_t e0 = get_event (h), e1 = get_event (h);
	CK (h, cudaEventRecord (e0, ls));
	kern<<<grid, BLOCK, smem, ls>>> (static_cast<S *> (h->table), h->cap, rb, bins, h->d_ctr, lk);
	CK (h, cudaGetLastError ());
	CK (h, cudaEventRecord (e1, ls));
	h->timing.push_back ({ e0, e1, (MODE == 0 || MODE == 5) ? 0 : (MODE == 6 ? 7 : 2) });
	h->all_launches++;
	return SDTGPU_OK;
}

template <int MODE> int launch_insert (sdtgpu *h, const ReadBatch &rb, const Bins &bins, const Lookup &lk = Lookup ())
{
	const bool nmode = (h->flags & SDTGPU_F_NKMER) && rb.nmask;
	switch (h->W)
	{
	case 1: return nmode ? launch_insert_t<1, true, MODE> (h, rb, bins, lk) : launch_insert_t<1, false, MODE> (h, rb, bins, lk);
	case 2: return nmode ? launch_insert_t<2, true, MODE> (h, rb, bins, lk) : launch_insert_t<2, false, MODE> (h, rb, bins, lk);
	default: return nmode ? launch_insert_t<4, true, MODE> (h, rb, bins, lk) : launch_insert_t<4, false, MODE> (h, rb, bins, lk);
	}
}

// a batch of device reads, validated (pushes and lookups)
int make_batch (sdtgpu *h, ReadBatch &rb, const uint8_t *d_packed, const u32 *d_lens, const uint8_t *d_nmask,
		u64 n_reads, u32 uniform_len, u32 stride_bytes, u64 first_read_ordinal)
{
	if (stride_bytes == 0 || (stride_bytes & 3) || (u64) stride_bytes * 4 < (u64) h->max_read_len)
		return fail (h, SDTGPU_EINVAL, "stride_bytes must be a multiple of 4 and hold max_read_len bases");
	if (((uintptr_t) d_packed & 15) || ((uintptr_t) d_lens & 3))
		return fail (h, SDTGPU_EINVAL, "device read buffers must be 16-byte aligned");
	if (!d_lens && uniform_len == 0 && n_reads)
		return fail (h, SDTGPU_EINVAL, "lens == NULL needs uniform_len");
	rb.packed = d_packed;
	rb.lens = d_lens;
	rb.nmask = (h->flags & SDTGPU_F_NKMER) ? d_nmask : nullptr;
	rb.n_reads = n_reads;
	rb.first_read_ordinal = first_read_ordinal;
	rb.uniform_len = uniform_len;
	rb.stride_bytes = stride_bytes;
	rb.mask_stride = stride_bytes / 2;	// 1 bit per base for stride_bytes * 4 bases
	rb.tile_reads = pick_tile_reads (stride_bytes);
	rb.K = h->K;
	rb.max_read_len = (u32) h->max_read_len;
	rb.maxwin = h->maxwin;
	// chunk of windows chopped per drain: the queue's capacity on one GPU; with owner filtering only
	// ~1/n of a chunk is owned, so chop 3n/4 capacities' worth (overflow is inserted in place)
	rb.queue_cap = QUEUE_CAP;
	rb.queue_windows = h->owner_ranks > 1 ? std::min<u32> (QUEUE_CAP * h->owner_ranks * 3 / 4, 16384) : QUEUE_CAP;
	rb.owner_rank = h->owner_rank;
	rb.owner_ranks = h->owner_ranks;
	return SDTGPU_OK;
}

// a batch that goes into the table: only before finalize, and its instance ordinals must fit the slot
int make_push_batch (sdtgpu *h, ReadBatch &rb, const uint8_t *d_packed, const u32 *d_lens, const uint8_t *d_nmask,
		     u64 n_reads, u32 uniform_len, u32 stride_bytes, u64 first_read_ordinal)
{
	if (h->finalized)
		return fail (h, SDTGPU_ESTATE, "push after finalize");
	int rc = make_batch (h, rb, d_packed, d_lens, d_nmask, n_reads, uniform_len, stride_bytes, first_read_ordinal);
	if (rc)
		return rc;
	const u64 ord_limit = ORD40_NONE;	// the slot keeps 40 bits of ordinal
	if ((first_read_ordinal + n_reads) >= ord_limit / h->maxwin)
		return fail (h, SDTGPU_ERANGE, "instance ordinal would overflow the slot's ordinal field");
	h->ord_end = std::max<u64> (h->ord_end, (first_read_ordinal + n_reads) * h->maxwin);
	return SDTGPU_OK;
}

u64 instances_upper (const sdtgpu *h, u64 n_reads, u32 uniform_len, bool have_lens)
{
	const u32 len = have_lens ? (u32) h->max_read_len : std::min (uniform_len, (u32) h->max_read_len);
	return len >= (u32) h->K + 1 ? n_reads * (u64) (len - h->K + 1) : 0;
}

int ensure_stage (sdtgpu *h, Staging &s, size_t packed, size_t lens, size_t mask)
{
	if (packed > s.cap_packed)
	{
		if (s.d_packed)
			CK (h, cudaFree (s.d_packed));
		s.cap_packed = packed + packed / 4 + 4096;
		CK (h, cudaMalloc (&s.d_packed, s.cap_packed));
	}
	if (lens > s.cap_lens)
	{
		if (s.d_lens)
			CK (h, cudaFree (s.d_lens));
		s.cap_lens = lens + lens / 4 + 4096;
		CK (h, cudaMalloc (&s.d_lens, s.cap_lens));
	}
	if (mask > s.cap_mask)
	{
		if (s.d_mask)
			CK (h, cudaFree (s.d_mask));
		s.cap_mask = mask + mask / 4 + 4096;
		CK (h, cudaMalloc (&s.d_mask, s.cap_mask));
	}
	return SDTGPU_OK;
}

int h_crc[256];
bool h_crc_ready = false;

void crc_table_host ()
{
	if (h_crc_ready)
		return;
	for (unsigned n = 0; n < 256; n++)
	{
		unsigned c = n;
		for (int k = 0; k < 8; k++)
			c = (c & 1) ? (0xEDB88320u ^ (c >> 1)) : (c >> 1);
		h_crc[n] = (int) c;
	}
	h_crc_ready = true;
}

template <int W>
__global__ void __launch_bounds__ (BLOCK)
export_kernel (const typename SlotOf<W>::type *table, u64 cap, int key_words, int thrd_num, int deLowKmer,
	       sdtgpu_node *out, u64 max_nodes, Counters *ctr)
{
	for (u64 base = blockIdx.x * (u64) BLOCK; base < cap; base += (u64) gridDim.x * BLOCK)
	{
		const u64 i = base + threadIdx.x;
		const bool occ = i < cap && SlotIO<W>::occupied (table + i);
		const unsigned m = __ballot_sync (0xFFFFFFFFu, occ);
		if (!m)
			continue;
		const int lane = threadIdx.x & 31;
		u64 pos = 0;
		if (lane == 0)
			pos = atomicAdd (&ctr->export_cursor, (u64) __popc (m));
		pos = __shfl_sync (0xFFFFFFFFu, pos, 0) + __popc (m & ((1u << lane) - 1u));
		if (!occ || pos >= max_nodes)
			continue;
		Key<W> k;
		u32 L, R, count;
		u64 ord;
		SlotIO<W>::get (table + i, k, L, R, count, ord);
		sdtgpu_node n;
#pragma unroll
		for (int q = 0; q < 4; q++)
			n.key[q] = q < 4 - W ? 0 : k.w[q - (4 - W)];
		n.l_links = L;
		n.rword = node_rword (L, R, count, deLowKmer);
		n.count = count;
		n.set = hash_kmer_impl (n.key, key_words, c_crc) % (u32) thrd_num;
		n.ordinal = ord;
		out[pos] = n;
	}
}

// device copy of the newest batch (device-to-device, a few hundred microseconds per 100 MB)
int retain_last_batch (sdtgpu *h, const ReadBatch &rb)
{
	const size_t pb = (size_t) rb.n_reads * rb.stride_bytes, lb = rb.lens ? (size_t) rb.n_reads * 4 : 0;
	const size_t mb = rb.nmask ? (size_t) rb.n_reads * rb.mask_stride : 0;
	auto fit = [&](void **p, size_t &cap, size_t need) -> cudaError_t {
		if (need <= cap)
			return cudaSuccess;
		if (*p)
			cudaFree (*p);
		*p = nullptr;
		cap = need + need / 4 + 4096;
		return cudaMalloc (p, cap);
	};
	CK (h, fit ((void **) &h->last_packed, h->last_cap_packed, pb));
	CK (h, fit ((void **) &h->last_lens, h->last_cap_lens, lb));
	CK (h, fit ((void **) &h->last_mask, h->last_cap_mask, mb));
	CK (h, cudaMemcpyAsync (h->last_packed, rb.packed, pb, cudaMemcpyDeviceToDevice, h->stream));
	if (lb)
		CK (h, cudaMemcpyAsync (h->last_lens, rb.lens, lb, cudaMemcpyDeviceToDevice, h->stream));
	if (mb)
		CK (h, cudaMemcpyAsync (h->last_mask, rb.nmask, mb, cudaMemcpyDeviceToDevice, h->stream));
	h->last_rb = rb;
	h->last_rb.packed = h->last_packed;
	h->last_rb.lens = lb ? h->last_lens : nullptr;
	h->last_rb.nmask = mb ? h->last_mask : nullptr;
	h->have_last = true;
	return SDTGPU_OK;
}

ReadBatch log_batch (const sdtgpu *h, const LogSeg &s);

// per reference set: (largest instance ordinal + 1) within the retained batch (sliced build: the whole epoch), 0 if none
int set_last_ordinals (sdtgpu *h, int thrd_num, std::vector<u64> &last)
{
	last.assign (thrd_num, 0);
	if (!h->have_last || thrd_num > 1024)
		return SDTGPU_OK;
	u64 *d_last = nullptr;
	CK (h, cudaMalloc (&d_last, thrd_num * sizeof (u64)));
	CK (h, cudaMemsetAsync (d_last, 0, thrd_num * sizeof (u64), h->stream));
	Bins b;
	b.records = nullptr;
	b.counts = d_last;
	b.capacity = (u64) h->key_words;
	b.n_ranks = (u32) thrd_num;
	int rc = SDTGPU_OK;
	if (h->sliced && !h->log.empty ())
	{	// the sliced build keeps every batch of the epoch: the last instance of a set is looked for in all of
		// them (a final batch of a few reads need not touch every set)
		for (size_t i = 0; i < h->log.size () && !rc; i++)
			rc = launch_insert<4> (h, log_batch (h, h->log[i]), b);
	}
	else
		rc = launch_insert<4> (h, h->last_rb, b);
	cudaError_t e = cudaSuccess;
	if (!rc)
	{
		e = cudaMemcpyAsync (last.data (), d_last, thrd_num * sizeof (u64), cudaMemcpyDeviceToHost, h->stream);
		if (e == cudaSuccess)
			e = cudaStreamSynchronize (h->stream);
	}
	cudaFree (d_last);
	if (rc)
		return rc;
	CK (h, e);
	return SDTGPU_OK;
}

int sliced_flush (sdtgpu *h);

// everything pushed is in the table (the sliced build does its work here; the single-pass insert has nothing pending)
int flush_epoch (sdtgpu *h)
{
	return h->sliced ? sliced_flush (h) : SDTGPU_OK;
}

// ---- sliced build over super-k-mers (sdt_skm.cuh, sdt_chain.cuh, sdt_merge.cuh, sdt_build.cuh) ------------
struct TimedLaunch
{	// CUDA events around one launch on the handle's stream, filed under a timing class
	sdtgpu *h;
	cudaEvent_t e0, e1;
	int cat;
	TimedLaunch (sdtgpu *h_, int cat_) : h (h_), e0 (get_event (h_)), e1 (get_event (h_)), cat (cat_) { cudaEventRecord (e0, h->stream); }
	~TimedLaunch ()
	{
		cudaEventRecord (e1, h->stream);
		h->timing.push_back ({ e0, e1, cat });
		h->all_launches++;
	}
};

// SDTGPU_TRACE=1: wall clock of the host-side steps of a flush (drains the stream at every mark)
struct Trace
{
	sdtgpu *h;
	bool on;
	std::chrono::steady_clock::time_point t0;
	Trace (sdtgpu *h_) : h (h_), on (getenv ("SDTGPU_TRACE") != nullptr), t0 (std::chrono::steady_clock::now ()) { }
	void mark (const char *what)
	{
		if (!on)
			return;
		cudaStreamSynchronize (h->stream);
		const auto t1 = std::chrono::steady_clock::now ();
		size_t fr = 0, tot = 0;
		if (atoi (getenv ("SDTGPU_TRACE")) > 1)
			cudaMemGetInfo (&fr, &tot);
		fprintf (stderr, "[sdtgpu] %-28s %8.3f ms   (%.1f GB free)\n", what, std::chrono::duration<double, std::milli> (t1 - t0).count (), fr / 1e9);
		t0 = std::chrono::steady_clock::now ();
	}
};

u32 env_u32 (const char *name, u32 dflt)
{
	const char *e = getenv (name);
	return e && atoll (e) > 0 ? (u32) atoll (e) : dflt;
}

// distinct k-mers to expect from `instances` windows when the caller gave no hint: at sequencing depth the
// distinct k-mers are dominated by error k-mers (a window is error-free with probability 0.99^K at the 1 %
// substitution rate of short reads), never more than the windows themselves.  Only the slice count and the first
// size of the node store come from this; slices that overflow are split and the store grows (sliced_flush).
u64 estimate_distinct (u64 instances, int K)
{
	const double e = (double) instances * (1.0 - pow (0.99, (double) K)) * 1.05 + 65536.0;
	return (u64) std::min ((double) instances + 1024.0, e);
}

// Geometry from the expected distinct count: slices whose images run at ~half load on average
// (minimizer slices are lumpier than hashed k-mers: sd ~14 % of the mean at 1150 keys per slice)
int skm_setup (sdtgpu *h, u64 hint)
{
	SkmGeom g;
	// default: what fits one CTA per SM (227 KB) beside the staging areas: 72 / 84 / 100 bytes per slot for 1- / 2- / 4-word keys
	const u32 dflt = skm_build2_max_slots (h->W);
	g.slice_slots = env_u32 ("SDTGPU_SLICE_SLOTS", dflt);
	if (g.slice_slots < 32 || g.slice_slots > dflt)
		return fail (h, SDTGPU_EINVAL, "SDTGPU_SLICE_SLOTS out of range");
	for (;; g.slice_slots--)
	{	// the largest prime below: the image is probed by double hashing (skm_find2)
		bool prime = true;
		for (u32 d = 2; d * d <= g.slice_slots && prime; d++)
			prime = g.slice_slots % d != 0;
		if (prime)
			break;
	}
	// a chain (the k-mers of one range of minimizers) is sized to a fraction of an image: skm_merge_kernel packs
	// consecutive chains into work items up to an image's worth of windows, which evens out how lumpy chains are
	// (K <= 31 with a hint: a chain is about an image's worth — 2 % faster on C2 than packing small chains;
	// without a hint the chains are made small, so that a guess that is too low by 4x still gives items that fit)
	double load = h->W == 1 ? (h->hint ? 0.45 : 0.3) : (h->W == 2 ? 0.12 : 0.2);	// (long k-mers: nearly every window is a k-mer of its own and chains are lumpy)
	if (const char *e = getenv ("SDTGPU_SLICE_LOAD"))
		if (atof (e) > 0.01 && atof (e) < 0.95)
			load = atof (e);
	const u64 n = std::max<u64> (1, (u64) std::ceil ((double) std::max<u64> (hint, 1) / ((double) g.slice_slots * load)));
	if (n > (1ull << 28))
		return fail (h, SDTGPU_ERANGE, "capacity_hint too large for the sliced build");
	g.n_slices = (u32) n;
	g.m = env_u32 ("SDTGPU_MINIMIZER", h->K >= 21 ? 15u : (u32) std::max (7, h->K - 6));
	if (g.m > 15 || (int) g.m > h->K - 2 || g.m < 5)
		return fail (h, SDTGPU_EINVAL, "SDTGPU_MINIMIZER out of range");
	g.wfull = (u32) h->K - g.m + 1;
	g.lo = g.wfull > 24 && !getenv ("SDTGPU_FULL_WINDOW") ? 4 * ((g.wfull - 17) / 8) : 0;	// the central 17 .. 24 m-mers of a long window
	g.w = g.wfull - 2 * g.lo;
	g.nmax = h->W == 1 ? 32 : 64;
	g.recw = h->W == 1 ? 8 : (h->W == 2 ? 12 : 16);
	g.npos = (u32) h->max_read_len - g.m + 1;
	g.npad = (std::max (g.npos, g.npos - g.wfull + 1 + 6) + 3) & ~3u;
	g.tile_reads = std::max (4u, std::min (64u, (8192u / g.npad) & ~3u));
	g.slice_a = slice_of_min_host (mmer_hash (0), g.n_slices);
	if (g.npad * g.tile_reads > 60000 || h->max_read_len > 60000)
		return fail (h, SDTGPU_ERANGE, "max_read_len too large for the sliced build");
	h->geom = g;
	h->store_want = hint + hint / 8 + 65536;	// node store: compact, one slot per distinct k-mer
	return SDTGPU_OK;
}

static constexpr u32 MAX_FAILED = 1u << 21;
static constexpr u32 MAX_CTAS = 148 * 16 + 64;	// CTAs that keep a block range between launches (SkmChains::cta_pool)

int grow_device (sdtgpu *h, void **mem, size_t *cap, size_t keep, size_t need, const char *what = "buffer", bool slack = false)
{	// *mem holds `keep` live bytes; make room for `need`.  slack: a buffer whose need varies a little from epoch to
	// epoch on the same input (sub-slices, received records: which items overflow depends on the order records
	// arrive in) gets an eighth more the first time, so that the next epoch does not allocate again
	if (need <= *cap)
		return SDTGPU_OK;
	size_t ncap = std::max (*cap + *cap / 2, need + (slack ? need / 8 : 0) + (4u << 20));
	void *neu = nullptr;
	h->n_alloc++;
	if (!keep && *mem)
	{	// nothing to keep: the old buffer goes first
		CK (h, cudaStreamSynchronize (h->stream));
		CK (h, cudaFree (*mem));
		*mem = nullptr;
		*cap = 0;
	}
	if (cudaMalloc (&neu, ncap) != cudaSuccess)
	{	// no room for the head room: exactly what is needed
		cudaGetLastError ();
		ncap = need;
		if (cudaMalloc (&neu, ncap) != cudaSuccess)
		{
			size_t fr = 0, tot = 0;
			cudaGetLastError ();
			cudaMemGetInfo (&fr, &tot);
			char b[256];
			snprintf (b, sizeof b, "device allocation of %.2f GB for the %s failed (it holds %.2f GB now; %.2f of %.2f GB free)", need / 1e9, what, *cap / 1e9, fr / 1e9, tot / 1e9);
			h->err = b;
			return SDTGPU_ENOMEM;
		}
	}
	if (keep)
		CK (h, cudaMemcpyAsync (neu, *mem, keep, cudaMemcpyDeviceToDevice, h->stream));
	CK (h, cudaStreamSynchronize (h->stream));
	if (*mem)
		CK (h, cudaFree (*mem));
	*mem = neu;
	*cap = ncap;
	return SDTGPU_OK;
}

// ---- a set of chains (the slices, or the sub-slices of slices that overflowed) with its block pool
void level_free (ChainLevel &L)
{
	cudaFree (L.head); cudaFree (L.bcount); cudaFree (L.boff); cudaFree (L.seg_sum); cudaFree (L.cta_pool);
	cudaFree (L.bchain); cudaFree (L.bseq); cudaFree (L.blist); cudaFree (L.recs);
	cudaFree (L.items); cudaFree (L.out);
	L = ChainLevel ();
}

SkmChains level_chains (const sdtgpu *h, const ChainLevel &L)
{
	SkmChains c;
	c.head = reinterpret_cast<unsigned long long *> (L.head);
	c.bcount = L.bcount;
	c.bchain = L.bchain;
	c.bseq = L.bseq;
	c.recs = L.recs;
	c.pool_cursor = reinterpret_cast<unsigned long long *> (L.d_cursor);
	c.cta_pool = L.cta_pool;
	c.ctr = h->d_ctr;
	c.pool_blocks = L.pool_blocks;
	c.n_chains = L.n_chains;
	c.recw = h->geom.recw;
	return c;
}

// chains: heads point at their first blocks, nothing linked, the pool cursor behind the first blocks
int level_reset (sdtgpu *h, ChainLevel &L)
{
	if (!L.n_chains)
		return SDTGPU_OK;
	chain_init_kernel<<<std::min<u32> ((L.n_chains + 255) / 256, (u32) h->sm_count * 8), 256, 0, h->stream>>> (reinterpret_cast<unsigned long long *> (L.head), L.bcount, L.n_chains,
														   reinterpret_cast<unsigned long long *> (L.d_cursor));
	CK (h, cudaGetLastError ());
	h->all_launches++;
	if (L.pool_blocks)
		CK (h, cudaMemsetAsync (L.bchain, 0xFF, L.pool_blocks * sizeof (u32), h->stream));
	CK (h, cudaMemsetAsync (L.cta_pool, 0, MAX_CTAS * sizeof (uint2), h->stream));
	L.blocks_upper = L.n_chains;
	return SDTGPU_OK;
}

int level_create (sdtgpu *h, ChainLevel &L, u32 n_chains)
{
	if (n_chains > L.cap_chains)
	{	// (the pool, the block list and the merged runs are kept: they do not depend on the number of chains)
		cudaFree (L.head); cudaFree (L.bcount); cudaFree (L.boff); cudaFree (L.seg_sum); cudaFree (L.cta_pool); cudaFree (L.items);
		L.head = L.boff = L.seg_sum = nullptr;
		L.bcount = nullptr;
		L.cta_pool = nullptr;
		L.items = nullptr;
		L.cap_chains = 0;
		const u32 cap = n_chains + n_chains / 4 + 64;
		const u32 nseg = (cap + SCAN_SEG - 1) / SCAN_SEG;
		CK (h, cudaMalloc (&L.head, (size_t) cap * sizeof (u64)));
		CK (h, cudaMalloc (&L.bcount, (size_t) cap * sizeof (u32)));
		CK (h, cudaMalloc (&L.boff, ((size_t) cap + 1) * sizeof (u64)));
		CK (h, cudaMalloc (&L.seg_sum, (size_t) nseg * sizeof (u64)));
		CK (h, cudaMalloc (&L.items, (size_t) cap * sizeof (SkmWork)));
		CK (h, cudaMalloc (&L.cta_pool, MAX_CTAS * sizeof (uint2) + 4 * sizeof (u64)));
		L.d_cursor = reinterpret_cast<u64 *> (L.cta_pool + MAX_CTAS);
		L.cap_chains = cap;
	}
	L.n_chains = n_chains;
	return level_reset (h, L);
}

// room for `blocks` blocks in the pool (what is there is kept)
int level_reserve (sdtgpu *h, ChainLevel &L, u64 blocks)
{
	L.pool_high = std::max (L.pool_high, blocks);
	if (blocks <= L.pool_blocks)
		return SDTGPU_OK;
	if (L.pool_blocks == 0)
	{	// a pool that was given up for the node store comes back at its full size, in one piece — and if the store
		// of the last epoch is in its way, the store goes (it is rebuilt by the next flush anyway)
		blocks = L.pool_high;
		size_t fr = 0, tot = 0;
		cudaMemGetInfo (&fr, &tot);
		if (h->table && (double) fr < (double) blocks * CH_BLK * h->geom.recw * 4.4 + (1u << 30))
		{
			CK (h, cudaStreamSynchronize (h->stream));
			CK (h, cudaFree (h->table));
			h->table = nullptr;
			h->cap = 0;
			h->n_store = 0;
			h->table_built = false;
		}
	}
	if (blocks >= 0xFFFFFFF0ull)
		return fail (h, SDTGPU_ERANGE, "too many record blocks");
	int rc;
	const size_t bb = (size_t) CH_BLK * h->geom.recw * 4;
	const u64 old = L.pool_blocks;
	size_t cap_r = old * bb, cap_c = old * 4, cap_s = old * 4;
	const bool slack = &L != &h->lv[0];	// (the slices' own pool is sized by a formula of the reads pushed: it does not wander)
	if ((rc = grow_device (h, (void **) &L.recs, &cap_r, old * bb, blocks * bb, "record pool", slack)))
		return rc;
	const u64 neu = cap_r / bb;
	if ((rc = grow_device (h, (void **) &L.bchain, &cap_c, old * 4, neu * 4)) || (rc = grow_device (h, (void **) &L.bseq, &cap_s, old * 4, neu * 4)))
		return rc;
	CK (h, cudaMemsetAsync (L.bchain + old, 0xFF, (neu - old) * sizeof (u32), h->stream));
	L.pool_blocks = neu;
	return SDTGPU_OK;
}

ReadBatch log_batch (const sdtgpu *h, const LogSeg &s)
{
	ReadBatch rb = s.rb;
	rb.packed = static_cast<const uint8_t *> (h->log_mem[0]) + s.off[0];
	rb.lens = s.rb.lens ? reinterpret_cast<const u32 *> (static_cast<const uint8_t *> (h->log_mem[1]) + s.off[1]) : nullptr;
	rb.nmask = s.rb.nmask ? static_cast<const uint8_t *> (h->log_mem[2]) + s.off[2] : nullptr;
	return rb;
}

template <int W, bool NMODE> int launch_emit_t (sdtgpu *h, ReadBatch rb)
{
	const SkmGeom &g = h->geom;
	rb.tile_reads = g.tile_reads;
	auto kern = skm_emit_kernel<W, NMODE>;
	const size_t smem = 4 * (tile_words (rb, NMODE) + 2 * (size_t) g.tile_reads * g.npad + 16 + (size_t) g.tile_reads * ((g.npos - g.wfull + 1 + EMIT_SEG - 1) / EMIT_SEG) + 4);
	if (smem > 48 * 1024)
		CK (h, cudaFuncSetAttribute (kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	int occ = 0;
	CK (h, cudaOccupancyMaxActiveBlocksPerMultiprocessor (&occ, kern, EMIT_NT, smem));
	if (occ < 1)
		return fail (h, SDTGPU_EINVAL, "read stride too large for one shared-memory tile");
	const u64 n_tiles = (rb.n_reads + rb.tile_reads - 1) / rb.tile_reads;
	const unsigned grid = (unsigned) std::min<u64> (n_tiles, std::min<u64> ((u64) h->sm_count * occ, MAX_CTAS));
	{
		TimedLaunch tl (h, 1);
		kern<<<grid, EMIT_NT, smem, h->stream>>> (rb, g, level_chains (h, h->lv[0]), reinterpret_cast<unsigned long long *> (h->d_small));
	}
	CK (h, cudaGetLastError ());
	return SDTGPU_OK;
}

int launch_emit (sdtgpu *h, const ReadBatch &rb)
{
	const bool nmode = (h->flags & SDTGPU_F_NKMER) && rb.nmask;
	switch (h->W)
	{
	case 1: return nmode ? launch_emit_t<1, true> (h, rb) : launch_emit_t<1, false> (h, rb);
	case 2: return nmode ? launch_emit_t<2, true> (h, rb) : launch_emit_t<2, false> (h, rb);
	default: return nmode ? launch_emit_t<4, true> (h, rb) : launch_emit_t<4, false> (h, rb);
	}
}

// blocks a batch of `upper` windows from `n_reads` reads may fill: random minimizers start a new run every
// (w + 1) / 2 windows and every read ends one (C2: 0.124 records per window measured; K = 63: 0.076; K = 127 on
// 150 bp: 0.069), plus what the CTAs hold back; if a batch needs more the kernels say so and the epoch is emitted again
u64 batch_blocks (const sdtgpu *h, u64 upper, u64 n_reads)
{
	u64 rec = (u64) ((double) upper * 2.2 / (h->geom.w + 1.0)) + n_reads + n_reads / 5 + 4096;
	if (getenv ("SDTGPU_REC_DIV"))	// tests: a pool that is too small
		rec = upper / env_u32 ("SDTGPU_REC_DIV", 3) + n_reads / 8 + 4096;
	return rec / CH_BLK + rec / (16 * CH_BLK) + 64;
}

int emit_segment (sdtgpu *h, const LogSeg &s)
{
	int rc;
	ChainLevel &L = h->lv[0];
	const u64 hold = (u64) std::min<u64> ((u64) h->sm_count * 8, MAX_CTAS) * CH_SB;	// what the CTAs may sit on
	L.blocks_upper += batch_blocks (h, s.upper, s.rb.n_reads);
	if ((rc = level_reserve (h, L, L.blocks_upper + hold)))
		return rc;
	return launch_emit (h, log_batch (h, s));
}

// the geometry is fixed when the first records are made: from the hint, or (no hint) from what has been pushed
int skm_open_epoch (sdtgpu *h)
{
	int rc;
	if (h->epoch_open)
		return SDTGPU_OK;
	u64 hint = h->hint;
	if (!hint)
		hint = estimate_distinct (h->pushed_upper, h->K);
	if ((rc = skm_setup (h, hint)))
		return rc;
	h->geom.send_group = 1;
	if (h->skm_world > 1)
	{	// the sending side keeps `world` consecutive slices in one chain (chains as long as on one GPU: the merge in front
		// of the exchange costs what it costs there); the records carry their slice
		const u32 grp = h->skm_world;
		h->n_local = (h->geom.n_slices + grp - 1) / grp * grp;
		if ((u64) h->n_local * h->skm_world > (1ull << 28))
			return fail (h, SDTGPU_ERANGE, "too many slices");
		h->geom.n_slices = h->n_local * h->skm_world;
		h->geom.slice_a = slice_of_min_host (mmer_hash (0), h->geom.n_slices);
		h->geom.send_group = getenv ("SDTGPU_NO_SEND_GROUP") ? 1 : grp;
	}
	const u32 n_chains0 = h->geom.n_slices / h->geom.send_group;
	if (h->lv[0].n_chains != n_chains0)	// (else: same geometry as the last epoch, whose chains sdtgpu_reset has emptied)
	{
		if ((rc = level_create (h, h->lv[0], n_chains0)))
			return rc;
	}
	else if ((rc = level_reset (h, h->lv[0])))
		return rc;
	h->epoch_open = true;
	return SDTGPU_OK;
}


template <int W, bool ORD32> int launch_build2_t (sdtgpu *h, const u32 *rec, const SkmWork *items, u32 n_items, const u64 *n_items_dev, int cat)
{
	typedef typename SlotOf<W>::type S;
	const SkmGeom &g = h->geom;
	auto kern = skm_build2_kernel<W, ORD32>;
	const size_t smem = skm_build2_smem (W, g.slice_slots, ORD32);
	CK (h, cudaFuncSetAttribute (kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	const unsigned grid = (unsigned) std::min<u64> (std::max<u64> (n_items, 1), (u64) h->sm_count);
	unsigned long long *small = reinterpret_cast<unsigned long long *> (h->d_small);
	CK (h, cudaMemsetAsync (small + 3, 0, sizeof (u64), h->stream));	// work-item cursor
	{
		TimedLaunch tl (h, cat);
		kern<<<grid, BUILD_NT, smem, h->stream>>> (static_cast<S *> (h->table), h->cap, small + 1, g, h->K, rec, items, n_items, reinterpret_cast<const unsigned long long *> (n_items_dev), small + 3,
							   static_cast<SkmWork *> (h->d_failed), reinterpret_cast<u32 *> (small + 2), MAX_FAILED, h->d_ctr);
	}
	CK (h, cudaGetLastError ());
	return SDTGPU_OK;
}

int launch_build (sdtgpu *h, const u32 *rec, const SkmWork *items, u32 n_items, int cat, const u64 *n_items_dev = nullptr)
{	// 32-bit ordinals in the slice images when every instance ordinal pushed so far fits (several GPUs: the caller says so)
	const bool ord32 = h->ord_end < 0xFFFFFFFFull && !getenv ("SDTGPU_ORD64");
	switch (h->W)
	{
	case 1: return ord32 ? launch_build2_t<1, true> (h, rec, items, n_items, n_items_dev, cat) : launch_build2_t<1, false> (h, rec, items, n_items, n_items_dev, cat);
	case 2: return ord32 ? launch_build2_t<2, true> (h, rec, items, n_items, n_items_dev, cat) : launch_build2_t<2, false> (h, rec, items, n_items, n_items_dev, cat);
	default: return ord32 ? launch_build2_t<4, true> (h, rec, items, n_items, n_items_dev, cat) : launch_build2_t<4, false> (h, rec, items, n_items, n_items_dev, cat);
	}
}

// the blocks of every chain in order (scan of the blocks per chain, one pass over the linked blocks)
int level_list (sdtgpu *h, ChainLevel &L, u64 *n_blocks)
{
	int rc;
	const u32 nseg = (L.n_chains + SCAN_SEG - 1) / SCAN_SEG;
	{
		TimedLaunch tl (h, 5);
		slice_scan_sums_kernel<<<nseg, SCAN_NT, 0, h->stream>>> (L.bcount, L.n_chains, L.seg_sum);
		slice_scan_kernel<<<nseg, SCAN_NT, 0, h->stream>>> (L.bcount, L.n_chains, L.seg_sum, L.boff, nullptr);
		h->all_launches++;
	}
	CK (h, cudaGetLastError ());
	// (no look at the counts: the list is given room for every block of the pool, the kernel reads the cursor itself)
	const u64 linked = L.pool_blocks > L.n_chains ? L.pool_blocks - L.n_chains : 0, cursor = L.pool_blocks;
	size_t cap_b = L.blist_cap * 4;
	if ((rc = grow_device (h, (void **) &L.blist, &cap_b, 0, std::max<u64> (linked, 1) * 4, "block list", &L != &h->lv[0])))
		return rc;
	L.blist_cap = cap_b / 4;
	if (cursor > L.n_chains)
	{
		TimedLaunch tl (h, 5);
		chain_list_kernel<<<(unsigned) std::min<u64> ((cursor - L.n_chains + 255) / 256, (u64) h->sm_count * 16), 256, 0, h->stream>>> (
			L.bchain, L.bseq, L.boff, L.n_chains, reinterpret_cast<unsigned long long *> (L.d_cursor), L.pool_blocks, L.blist);
	}
	CK (h, cudaGetLastError ());
	*n_blocks = L.n_chains + linked;
	return SDTGPU_OK;
}

template <int W, bool HAS_MULT> int launch_merge_t (sdtgpu *h, ChainLevel &L, u64 /* n_rec: the kernel forms its groups from the chains' own counts */, u32 per_owner, const u64 *region, u64 *rcur)
{
	auto kern = skm_merge_kernel<W, HAS_MULT>;
	const size_t smem = skm_merge_smem<W> ();
	CK (h, cudaFuncSetAttribute (kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	int occ = 0;
	CK (h, cudaOccupancyMaxActiveBlocksPerMultiprocessor (&occ, kern, MG_NT, smem));
	if (occ < 1)
		return fail (h, SDTGPU_ECUDA, "skm_merge_kernel does not fit");
	// (the kernel forms the groups itself: as many consecutive chains as fit a chunk.  One GPU: a CTA takes a contiguous
	// range of chains; sending side: pieces of MG_PIECE chains of an owner, round robin)
	const u32 span = per_owner ? per_owner : L.n_chains;
	const u64 n_pieces = (u64) ((span + MG_PIECE - 1) / MG_PIECE) * (per_owner ? (L.n_chains + per_owner - 1) / per_owner : 1);
	const unsigned grid = (unsigned) std::min<u64> (std::max<u64> (per_owner ? n_pieces : L.n_chains, 1), (u64) h->sm_count * occ);
	unsigned long long *small = reinterpret_cast<unsigned long long *> (h->d_small);
	CK (h, cudaMemsetAsync (small + 4, 0, 2 * sizeof (u64), h->stream));	// surviving records, their windows
	CK (h, cudaMemsetAsync (L.d_cursor + 1, 0, 3 * sizeof (u64), h->stream));	// output cursor, work items, group cursor
	double load = 0.95;	// windows per work item / slots of an image: an item has at most as many distinct k-mers as windows
	if (const char *e = getenv ("SDTGPU_ITEM_LOAD"))
		if (atof (e) > 0.05 && atof (e) < 4.0)
			load = atof (e);
	MergeOut mo;
	mo.out = L.out;
	mo.out_cursor = reinterpret_cast<unsigned long long *> (L.d_cursor + 1);
	mo.out_cap = L.out_cap;
	mo.items = L.items;
	mo.n_items = reinterpret_cast<unsigned long long *> (L.d_cursor + 2);
	mo.max_items = L.cap_chains;
	mo.n_kept = small + 4;
	mo.budget = std::max (1u, (u32) (load * h->geom.slice_slots));
	mo.oversize = std::max (mo.budget, 8 * h->geom.slice_slots);	// (a hot locus has many windows but few distinct k-mers: the build finds out)
	mo.per_owner = per_owner;
	mo.tagged = h->geom.send_group > 1;
	mo.region = region;
	mo.rcur = reinterpret_cast<unsigned long long *> (rcur);
	{
		TimedLaunch tl (h, 3);
		kern<<<grid, MG_NT, smem, h->stream>>> (level_chains (h, L), L.boff, L.blist, mo);
	}
	CK (h, cudaGetLastError ());
	return SDTGPU_OK;
}

int launch_merge (sdtgpu *h, ChainLevel &L, bool has_mult, u64 n_rec, u32 per_owner = 0, const u64 *region = nullptr, u64 *rcur = nullptr)
{
	switch (h->W)
	{
	case 1: return has_mult ? launch_merge_t<1, true> (h, L, n_rec, per_owner, region, rcur) : launch_merge_t<1, false> (h, L, n_rec, per_owner, region, rcur);
	case 2: return has_mult ? launch_merge_t<2, true> (h, L, n_rec, per_owner, region, rcur) : launch_merge_t<2, false> (h, L, n_rec, per_owner, region, rcur);
	default: return has_mult ? launch_merge_t<4, true> (h, L, n_rec, per_owner, region, rcur) : launch_merge_t<4, false> (h, L, n_rec, per_owner, region, rcur);
	}
}

int launch_split (sdtgpu *h, ChainLevel &sub, const u32 *rec, const SkmSplit *chunks, u32 n_chunks)
{
	const unsigned grid = (unsigned) std::min<u64> (n_chunks, std::min<u64> ((u64) h->sm_count * 8, MAX_CTAS));
	TimedLaunch tl (h, 6);
	const SkmChains c = level_chains (h, sub);
	switch (h->W)
	{
	case 1: skm_split_kernel<1><<<grid, SP_NT, 0, h->stream>>> (c, rec, chunks, n_chunks, h->K); break;
	case 2: skm_split_kernel<2><<<grid, SP_NT, 0, h->stream>>> (c, rec, chunks, n_chunks, h->K); break;
	default: skm_split_kernel<4><<<grid, SP_NT, 0, h->stream>>> (c, rec, chunks, n_chunks, h->K); break;
	}
	CK (h, cudaGetLastError ());
	return SDTGPU_OK;
}

// every segment of the read log through skm_emit_kernel again, into a pool that holds `records` records
int skm_emit_all (sdtgpu *h, u64 records)
{
	int rc;
	h->n_reemit++;
	ChainLevel &L = h->lv[0];
	const u64 hold = (u64) std::min<u64> ((u64) h->sm_count * 8, MAX_CTAS) * CH_SB;
	if ((rc = level_reset (h, L)))
		return rc;
	if ((rc = level_reserve (h, L, L.n_chains + records / CH_BLK + records / (8 * CH_BLK) + hold + 4096)))
		return rc;
	CK (h, cudaMemsetAsync (h->d_small, 0, sizeof (u64), h->stream));
	CK (h, cudaMemsetAsync (&h->d_ctr->overflow, 0, sizeof (u64), h->stream));
	for (const LogSeg &s : h->log)
		if ((rc = launch_emit (h, log_batch (h, s))))
			return rc;
	L.blocks_upper = L.pool_blocks - hold;
	return SDTGPU_OK;
}

// part 1 of a flush: all records are in their chains (emitting the read log again if the block pool ran out)
int skm_collect (sdtgpu *h, u64 *n_rec, bool wait = true)
{
	int rc;
	if (!h->emitted)
	{	// no hint: the reads were only logged so far; now their number is known and fixes the geometry
		if ((rc = skm_open_epoch (h)))
			return rc;
		for (const LogSeg &s : h->log)
			if ((rc = emit_segment (h, s)))
				return rc;
		h->emitted = true;
	}
	if (!wait)
		return SDTGPU_OK;
	for (int attempt = 0;; attempt++)
	{
		CK (h, cudaMemcpyAsync (h->h_small, h->d_small, sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaMemcpyAsync (h->h_small + 3, &h->d_ctr->overflow, sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaStreamSynchronize (h->stream));
		if (h->chains_dropped)
		{	// the last flush gave the chains' memory to the node store: everything is emitted again
			h->chains_dropped = false;
			if (h->table)
				CK (h, cudaFree (h->table));
			h->table = nullptr;
			h->cap = 0;
			if ((rc = skm_emit_all (h, h->h_small[0])))
				return rc;
			continue;
		}
		if (!(h->h_small[3] & OVF_RECORDS))
			break;
		if (attempt == 2)
			return fail (h, SDTGPU_ERANGE, "record pool overflow persists");
		if ((rc = skm_emit_all (h, h->h_small[0])))
			return rc;
	}
	*n_rec = h->h_small[0];
	return SDTGPU_OK;
}

int ensure_store (sdtgpu *h, u64 slots)
{
	if (slots <= h->cap && h->table)
		return SDTGPU_OK;
	if (h->table)
		CK (h, cudaFree (h->table));
	h->table = nullptr;
	h->cap = 0;
	h->n_alloc++;
	CK (h, cudaMalloc (&h->table, slots * slot_bytes (h->W)));
	h->cap = slots;
	return SDTGPU_OK;
}

static constexpr int STORE_FULL = -100;	// internal: the node store ran out; the top level enlarges it and builds again
static constexpr int RECORDS_FULL = -101;	// internal: the block pool ran out while the records were made; the flush emits them again

// part 2: the chains of level L -> contiguous runs (copies merged) -> node store
int skm_build_level (sdtgpu *h, ChainLevel &L, bool has_mult, u64 n_rec, u64 n_est, bool top);

// Everything pushed since the last reset becomes the node store.  Records persist until sdtgpu_reset, so a
// later push followed by another flush rebuilds the store from all of them.
int sliced_flush (sdtgpu *h)
{
	int rc;
	if (h->table_built && !h->dirty)
		return SDTGPU_OK;
	h->n_store = 0;
	if (h->log.empty ())
	{
		h->table_built = true;
		h->dirty = false;
		return SDTGPU_OK;
	}
	if (h->skm_world > 1)
		return fail (h, SDTGPU_ESTATE, "super-k-mer exchange: reads were pushed but sdtgpu_skm_stage / sdtgpu_skm_import have not run");
	Trace tr (h);
	ChainLevel &L = h->lv[0];
	for (int attempt = 0;; attempt++)
	{
		u64 n_rec = 0;
		if (!h->emitted && (rc = skm_collect (h, &n_rec, false)))	// (no hint: the records are made now)
			return rc;
		// How many records there are is only needed as a bound (room for the merged runs): the pool's size will do,
		// and nobody has to wait for the kernels to ask them — unless memory is short or something went wrong before
		const bool look = attempt > 0 || h->chains_dropped || (double) L.pool_blocks * CH_BLK * h->geom.recw * 4 > 0.1 * (double) h->mem_total || getenv ("SDTGPU_SLOW_FLUSH");
		if (look)
		{
			if ((rc = skm_collect (h, &n_rec, true)))
				return rc;
			tr.mark ("collect (emit done)");
		}
		else
			n_rec = L.pool_blocks * CH_BLK;
		const u64 n_est = look ? n_rec : (h->n_records ? h->n_records : n_rec - n_rec / 8);
		rc = skm_build_level (h, L, false, n_rec, n_est, true);
		if (rc != RECORDS_FULL || attempt == 2)
			break;
		CK (h, cudaMemsetAsync (&h->d_ctr->overflow, 0, sizeof (u64), h->stream));	// (the pool ran out: the second round looks, and emits again)
	}
	if (rc == RECORDS_FULL)
		return fail (h, SDTGPU_ERANGE, "record pool overflow persists");
	h->n_records = h->h_small[0];
	tr.mark ("build level 0 (total)");
	return rc;
}


// the work items of level L -> node store; items that overflow an image are retried in pieces or, far
// beyond an image, cut into sub-slices
static constexpr u32 FAILED_PREFIX = 4096;	// failed work items that are fetched together with the counters (pinned: h_failed)

int skm_build_runs (sdtgpu *h, ChainLevel &L, u32 n_items, bool top, const u64 *n_items_dev = nullptr)
{
	int rc;
	const SkmGeom g = h->geom;
	unsigned long long *small = reinterpret_cast<unsigned long long *> (h->d_small);
	Trace tr (h);
	if (n_items && (rc = launch_build (h, L.out, L.items, n_items, top ? 4 : 6, n_items_dev)))
		return rc;
	tr.mark ("  build all items");
	std::vector<SkmWork> items, failed;
	std::vector<SkmSplit> splits;
	u64 Q = 0, sub_windows = 0;
	for (u32 depth = 0;; depth++)
	{
		// one look at the device: node cursor, failed items (count and the first of them), overflow flags, and what
		// the merge counted (records and windows left, work items) if nobody has looked yet
		CK (h, cudaMemcpyAsync (h->h_small + 1, small + 1, 2 * sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaMemcpyAsync (h->h_small + 3, &h->d_ctr->overflow, sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaMemcpyAsync (h->h_small + 4, small + 4, 2 * sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaMemcpyAsync (h->h_small + 6, L.d_cursor + 2, sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaMemcpyAsync (h->h_small, small, sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaMemcpyAsync (h->h_failed, h->d_failed, FAILED_PREFIX * sizeof (SkmWork), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaStreamSynchronize (h->stream));
		if (depth == 0)
		{
			if (h->h_small[6] > L.cap_chains)
				return fail (h, SDTGPU_ERANGE, "work item list overflow");
			if (top)
			{
				h->n_merged = h->h_small[4];
				h->n_items = h->h_small[6];
				h->win_left = h->h_small[5];
			}
		}
		if (h->h_small[3] & OVF_RECORDS)
			return RECORDS_FULL;
		if (h->h_small[3] & OVF_STORE)
			return STORE_FULL;
		const u32 n_failed = (u32) h->h_small[2];
		if (n_failed == 0)
			break;
		if ((h->h_small[3] & OVF_FAILED) || n_failed > MAX_FAILED || depth == 10)
			return fail (h, SDTGPU_ERANGE, "too many work items overflowed their images");
		failed.resize (n_failed);
		memcpy (failed.data (), h->h_failed, std::min (n_failed, FAILED_PREFIX) * sizeof (SkmWork));
		if (n_failed > FAILED_PREFIX)
			CK (h, cudaMemcpy (failed.data () + FAILED_PREFIX, static_cast<const SkmWork *> (h->d_failed) + FAILED_PREFIX, (n_failed - FAILED_PREFIX) * sizeof (SkmWork), cudaMemcpyDeviceToHost));
		h->n_retried += n_failed;
		CK (h, cudaMemsetAsync (small + 2, 0, sizeof (u64), h->stream));
		// A failed item holds more distinct k-mers than an image takes (it is a single chain with more windows than
		// the budget of an item, or a piece of one).  Few pieces (<= 4) are retried in place, each piece scanning
		// the item's records for its keys (hash % R == r: a window that is not the piece's costs a roll and a hash,
		// about a third of an insert); an item that needs more — a highly expressed locus — is cut into
		// sub-slices in one pass (skm_split_kernel), top level only.  Distinct k-mers of an item: more than an image
		// took if it was tried, about 0.55 of its windows (C2: 0.48); pieces that still overflow are split again.
		items.clear ();
		for (const SkmWork &f : failed)
		{
			const u32 R0 = std::max (f.R, 1u);
			const double est = std::max (f.R ? (double) g.slice_slots : 0.0, 0.6 * (double) f.wsum) / R0;
			const u32 q = (u32) std::min (1048576.0, std::max (2.0, std::ceil (est / (0.7 * g.slice_slots))));
			if (top && f.R <= 1 && q > 4 && !getenv ("SDTGPU_NO_SPLIT"))
			{
				for (u64 lo = 0; lo < std::max<u64> (f.nrec, 1); lo += 8192)
					splits.push_back ({ f.r0 + lo, (u32) std::min<u64> (f.nrec - lo, 8192), q, (u32) Q, lo ? 0u : f.wsum });
				Q += q;
				sub_windows += f.wsum;
				continue;
			}
			const u32 qq = std::min (q, 4096u);
			for (u32 i = 0; i < qq; i++)
				items.push_back ({ f.r0, f.nrec, f.wsum, f.r + R0 * i, R0 * qq });
		}
		if (items.size () > MAX_FAILED || Q > (1ull << 27) || splits.size () * sizeof (SkmSplit) > (size_t) MAX_FAILED * sizeof (SkmWork))
			return fail (h, SDTGPU_ERANGE, "too many work items overflowed their images");
		if (items.empty ())
			break;
		CK (h, cudaMemcpyAsync (h->d_items, items.data (), items.size () * sizeof (SkmWork), cudaMemcpyHostToDevice, h->stream));
		if ((rc = launch_build (h, L.out, static_cast<const SkmWork *> (h->d_items), (u32) items.size (), 6)))
			return rc;
		CK (h, cudaStreamSynchronize (h->stream));	// `items` is pageable host memory
		tr.mark ("  retry pieces");
	}
	if (!splits.empty ())
	{	// the highly expressed loci: sub-slices by k-mer hash, then merged and built like slices — as many of them
		// at a time as the memory that is left takes (a sub-record per window, twice: chains and merged runs)
		ChainLevel &S = h->lv[1];
		const size_t recb = 4 * (size_t) g.recw;
		const u64 hold = (u64) std::min<u64> ((u64) h->sm_count * 8, MAX_CTAS) * 8 * 256;
		size_t a = 0;
		size_t fr = 0, tot = h->mem_total;
		// (the free memory is asked for only if what the sub-slices hold from earlier epochs is not enough for everything at once)
		const bool all_fits = S.pool_blocks >= Q + sub_windows / CH_BLK + sub_windows / (4 * CH_BLK) + hold + 4096 && S.out_cap >= sub_windows && S.cap_chains >= Q;
		if (!all_fits)
			cudaMemGetInfo (&fr, &tot);
		while (a < splits.size ())
		{
			if (a)
				cudaMemGetInfo (&fr, &tot);	// (a further batch: only when memory is short)
			const double room = (double) fr + (double) S.pool_blocks * CH_BLK * recb + (double) S.out_cap * recb - (2.0 * hold * CH_BLK * recb + (2u << 30));
			const u64 max_win = all_fits ? ~0ull : (u64) std::max (1e6, std::min (room, 0.08 * (double) tot) / (2.6 * recb));	// (never more than 8 % of the memory: it stays allocated)
			size_t b = a;
			u64 win = 0, q0 = splits[a].qbase, q1 = q0;
			while (b < splits.size () && (b == a || win + splits[b].pad <= max_win || splits[b].qbase == splits[b - 1].qbase))
			{	// (pad: windows of the item, on its first piece; the pieces of an item stay together)
				win += splits[b].pad;
				q1 = splits[b].qbase + splits[b].q;
				b++;
			}
			for (size_t k = a; k < b; k++)
				splits[k].qbase -= (u32) q0;
			if ((rc = level_create (h, S, (u32) (q1 - q0))))
				return rc;
			if ((rc = level_reserve (h, S, (q1 - q0) + win / CH_BLK + win / (4 * CH_BLK) + hold + 4096)))
				return rc;
			CK (h, cudaMemcpyAsync (h->d_items, splits.data () + a, (b - a) * sizeof (SkmSplit), cudaMemcpyHostToDevice, h->stream));
			if ((rc = launch_split (h, S, L.out, static_cast<const SkmSplit *> (h->d_items), (u32) (b - a))))
				return rc;
			CK (h, cudaMemcpyAsync (h->h_small + 3, &h->d_ctr->overflow, sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
			CK (h, cudaStreamSynchronize (h->stream));	// `splits` is pageable host memory; d_items is reused below
			if (h->h_small[3] & OVF_RECORDS)
				return fail (h, SDTGPU_ERANGE, "sub-slice pool overflow");
			if (tr.on)
				fprintf (stderr, "[sdtgpu]   split: %zu pieces of %zu, %llu sub-slices, %llu windows\n", b - a, splits.size (), (unsigned long long) (q1 - q0), (unsigned long long) win);
			tr.mark ("  split");
			if ((rc = skm_build_level (h, S, true, win, win, false)))
				return rc;
			tr.mark ("  sub-slices");
			a = b;
		}
	}
	return SDTGPU_OK;
}

int skm_build_level (sdtgpu *h, ChainLevel &L, bool has_mult, u64 n_rec, u64 n_est, bool top)
{	// n_rec: records in the chains at most (room for the merged runs); n_est: about how many there are
	int rc;
	const SkmGeom g = h->geom;
	unsigned long long *small = reinterpret_cast<unsigned long long *> (h->d_small);
	u64 n_blocks = 0;
	Trace tr (h);
	if ((rc = level_list (h, L, &n_blocks)))
		return rc;
	tr.mark (" list");
	{	// the merged runs: at most as many records as went in
		const size_t rec = 4 * (size_t) g.recw;
		size_t cap_b = L.out_cap * rec;
		if ((rc = grow_device (h, (void **) &L.out, &cap_b, 0, std::max<u64> (n_rec, 1) * rec, "merged records", &L != &h->lv[0])))
			return rc;
		L.out_cap = cap_b / rec;
	}
	if ((rc = launch_merge (h, L, has_mult, n_est)))
		return rc;
	// the build takes the number of work items from the device: the host does not wait for the merge
	if (!top)
		return skm_build_runs (h, L, L.cap_chains, false, L.d_cursor + 2);
	u64 win_upper = ~0ull;
	if (!h->table || h->cap < h->store_want)
	{	// the node store has to be sized: by what the merge left (every node needs a window of its own)
		CK (h, cudaMemcpyAsync (h->h_small + 4, small + 4, 2 * sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaStreamSynchronize (h->stream));
		tr.mark (" merge");
		win_upper = h->h_small[5] + 1024;
	}
	const u32 n_items = L.cap_chains;
	for (int attempt = 0;; attempt++)
	{	// the store is rebuilt from all records: node cursor, failed-item count and the two counters start over.
		// Its size: the hint's (or the estimate's) worth, never more than the windows the merge left
		// (the windows the merge leaves vary a little from epoch to epoch on the same input — which copies meet in a
		// chunk depends on the order records arrive in — and a store sized to the window would be freed and allocated
		// again, 18 GB of it, whenever an epoch leaves a few more: 3 % of head room)
		u64 want = h->cap;
		if (win_upper != ~0ull && (!h->table || std::min<u64> (h->store_want, win_upper) > h->cap))
			want = std::min<u64> (h->store_want, win_upper + win_upper / 32 + 65536);
		if (want > h->cap || !h->table)
		{	// no room for the node store beside the chains?  The chains are not needed any more (their records are
			// merged): they go, and a later flush of this epoch emits the read log again
			size_t fr = 0, tot = 0;
			cudaMemGetInfo (&fr, &tot);
			const double need_store = want > h->cap || !h->table ? (double) want * slot_bytes (h->W) - (double) h->cap * slot_bytes (h->W) : 0.0;
			if ((double) fr < need_store + 0.15 * (double) tot && L.recs)	// (15 % of the memory stays free for sub-slices)
			{
				cudaFree (L.recs); cudaFree (L.bchain); cudaFree (L.bseq); cudaFree (L.blist);
				L.recs = L.bchain = L.bseq = L.blist = nullptr;
				L.pool_blocks = L.blist_cap = 0;
				h->chains_dropped = true;
				cudaMemGetInfo (&fr, &tot);
			}
			// never more than the memory takes (15 % of it stays free for sub-slices): if that store runs out, so be it
			const double room = (double) fr + (double) h->cap * slot_bytes (h->W) - 0.15 * (double) tot;
			if (room > 0 && (double) want * slot_bytes (h->W) > room)
				want = std::max<u64> ((u64) (room / slot_bytes (h->W)), std::min<u64> (h->cap, want));
		}
		if ((rc = ensure_store (h, want)))
			return rc;
		CK (h, cudaMemsetAsync (small + 1, 0, 2 * sizeof (u64), h->stream));
		CK (h, cudaMemsetAsync (&h->d_ctr->n_nodes, 0, 2 * sizeof (u64), h->stream));	// n_nodes, n_instances
		h->n_retried = 0;
		rc = skm_build_runs (h, L, n_items, true, L.d_cursor + 2);
		if (rc != STORE_FULL)
			break;
		win_upper = h->win_left + 1024;	// (skm_build_runs has looked)
		if (attempt == 1 || h->cap >= win_upper)
			return fail (h, SDTGPU_ERANGE, "node store exhausted");
		h->store_want = win_upper;	// the estimate was too low: a store that cannot run out, and once more
		CK (h, cudaMemsetAsync (&h->d_ctr->overflow, 0, sizeof (u64), h->stream));
	}
	if (rc)
		return rc;
	CK (h, cudaMemcpyAsync (h->h_small + 1, small + 1, sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
	CK (h, cudaStreamSynchronize (h->stream));
	h->n_store = h->h_small[1];
	h->table_built = true;
	h->dirty = false;
	h->n_epochs++;
	return SDTGPU_OK;
}

// one batch: into the read log (kept for re-emission and the hand-back) and through skm_emit_kernel
int sliced_push (sdtgpu *h, const ReadBatch &rb, u64 upper)
{
	int rc;
	auto up16 = [](size_t x) { return (x + 15) & ~(size_t) 15; };
	const size_t bytes[3] = { up16 ((size_t) rb.n_reads * rb.stride_bytes), rb.lens ? up16 ((size_t) rb.n_reads * 4) : 0,
				  rb.nmask ? up16 ((size_t) rb.n_reads * rb.mask_stride) : 0 };
	const void *src[3] = { rb.packed, rb.lens, rb.nmask };
	const size_t exact[3] = { (size_t) rb.n_reads * rb.stride_bytes, (size_t) rb.n_reads * 4, (size_t) rb.n_reads * rb.mask_stride };
	LogSeg s;
	s.rb = rb;
	s.upper = upper;
	for (int i = 0; i < 3; i++)
	{
		s.off[i] = h->log_used[i];
		if (!bytes[i])
			continue;
		if ((rc = grow_device (h, &h->log_mem[i], &h->log_cap[i], h->log_used[i], h->log_used[i] + bytes[i], "read log")))
			return rc;
		CK (h, cudaMemcpyAsync (static_cast<uint8_t *> (h->log_mem[i]) + s.off[i], src[i], exact[i], cudaMemcpyDeviceToDevice, h->stream));
		h->log_used[i] += bytes[i];
	}
	h->log.push_back (s);
	h->pushed_upper += upper;
	h->dirty = true;
	if (!h->hint && !h->epoch_open)
		return SDTGPU_OK;	// no hint: the geometry waits for the end of the epoch (skm_collect)
	if (h->chains_dropped)
		return SDTGPU_OK;	// the next flush emits the whole read log again
	if ((rc = skm_open_epoch (h)))
		return rc;
	h->emitted = true;
	return emit_segment (h, h->log.back ());
}

u64 iter_slots (const sdtgpu *h) { return h->sliced ? h->n_store : h->cap; }

static_assert (sizeof (Hit) == sizeof (sdtgpu_hit) && SDTGPU_HIT_WINDOW == HIT_WINDOW && SDTGPU_HIT_FOUND == HIT_FOUND && SDTGPU_HIT_RC == HIT_RC, "sdtgpu_hit");

void free_index (sdtgpu *h)
{
	cudaFree (h->index);
	h->index = nullptr;
	h->idx_cap = 0;
}

// The lookup index of the finalized table (sdt_lookup.cuh), made by the first lookup: one entry per node at load
// <= 0.5, 16 bytes per node.  It is not made at finalize, so that a table nobody looks up costs nothing more.
int ensure_index (sdtgpu *h)
{
	if (h->index)
		return SDTGPU_OK;
	const u64 slots = iter_slots (h);
	if (slots >= 0xFFFFFFFFull)
		return fail (h, SDTGPU_ERANGE, "lookup index: the table has 2^32 - 1 slots or more (entries hold 32-bit positions)");
	int rc = read_counters (h);
	if (rc)
		return rc;
	const u64 cap = std::max<u64> (1024, 2 * h->h_ctr->n_nodes);
	if (cudaMalloc (&h->index, cap * sizeof (u64)) != cudaSuccess)
	{
		cudaGetLastError ();
		h->index = nullptr;
		char b[160];
		snprintf (b, sizeof b, "device allocation of %.2f GB for the lookup index failed", cap * sizeof (u64) / 1e9);
		return fail (h, SDTGPU_ENOMEM, b);
	}
	h->idx_cap = cap;
	cudaError_t e;
	{
		TimedLaunch tl (h, 7);
		e = cudaMemsetAsync (h->index, 0xFF, cap * sizeof (u64), h->stream);
		const unsigned grid = (unsigned) std::min<u64> ((slots + BLOCK - 1) / BLOCK, (u64) h->sm_count * 16);
		if (e == cudaSuccess && grid)
		{
			switch (h->W)
			{
			case 1: index_build_kernel<1><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot1 *> (h->table), slots, h->index, cap); break;
			case 2: index_build_kernel<2><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot2 *> (h->table), slots, h->index, cap); break;
			default: index_build_kernel<4><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot4 *> (h->table), slots, h->index, cap); break;
			}
			e = cudaGetLastError ();
		}
	}
	if (e != cudaSuccess)
		free_index (h);
	CK (h, e);
	return SDTGPU_OK;
}

// what both lookups check first: a finalized table, and a hit buffer that takes 16-byte stores
int lookup_prologue (sdtgpu *h, const void *d_out)
{
	CK (h, cudaSetDevice (h->device));
	if (!h->finalized)
		return fail (h, SDTGPU_ESTATE, "lookup before sdtgpu_finalize");
	if ((uintptr_t) d_out & 15)
		return fail (h, SDTGPU_EINVAL, "the hit buffer must be 16-byte aligned");
	return SDTGPU_OK;
}

Lookup make_lookup (const sdtgpu *h, sdtgpu_hit *d_out)
{
	Lookup lk;
	lk.index = h->index;
	lk.idx_cap = h->idx_cap;
	lk.out = reinterpret_cast<Hit *> (d_out);
	lk.deLowKmer = h->deLowKmer;
	return lk;
}

// ---- routed lookups (sdt_route.cuh): how this handle's keys are sharded, as the insert side does it
Route make_route (const sdtgpu *h)
{
	Route rt = {};
	rt.kind = ROUTE_ONE;
	rt.world = 1;
	rt.K = h->K;
	if (h->sliced && h->skm_world > 1)
	{
		rt.kind = ROUTE_SKM;
		rt.world = h->skm_world;
		rt.n_local = h->n_local;
	}
	else if (h->owner_ranks > 1)
	{
		rt.kind = h->sliced ? ROUTE_SLICED : ROUTE_HASHED;
		rt.world = h->owner_ranks;
	}
	if (rt.kind == ROUTE_SKM || rt.kind == ROUTE_SLICED)
	{
		rt.n_slices = h->geom.n_slices;
		rt.m = h->geom.m;
		rt.lo = h->geom.lo;
		rt.w = h->geom.w;
	}
	return rt;
}

void free_route (sdtgpu *h)
{
	cudaFree (h->rt_q); cudaFree (h->rt_tag); cudaFree (h->rt_aq); cudaFree (h->rt_ar); cudaFree (h->rt_back);
	h->rt_q = h->rt_tag = h->rt_aq = nullptr;
	h->rt_ar = h->rt_back = nullptr;
	h->rt_cap_q = h->rt_cap_tag = h->rt_cap_aq = h->rt_cap_ar = h->rt_cap_back = 0;
	h->rt_staged = false;
}

void free_edges (sdtgpu *h)
{
	for (int i = 0; i < ED_N; i++)
	{
		cudaFree (h->ed[i]);
		h->ed[i] = nullptr;
		h->ed_cap[i] = 0;
	}
	h->ed_built = false;
}

// a finalized table, at most ROUTE_MAX_WORLD ranks, the small count buffers, and the index: a rank that stages
// also answers, and building the index here lets a routed lookup fail before any query travels
int route_prologue (sdtgpu *h)
{
	int rc = lookup_prologue (h, nullptr);
	if (rc)
		return rc;
	if (make_route (h).world > ROUTE_MAX_WORLD)
		return fail (h, SDTGPU_EINVAL, "routed lookups: at most 64 ranks");
	if (!h->rt_cur)
	{
		CK (h, cudaMalloc (&h->rt_cur, ROUTE_MAX_WORLD * sizeof (u64)));
		CK (h, cudaMallocHost (&h->rt_hcur, ROUTE_MAX_WORLD * sizeof (u64)));
	}
	return ensure_index (h);
}

// The two passes of a stage around the host's scan of `world` counts.  launch (scatter, stage) enqueues one pass
// on the handle's stream.  n_out: entries of the caller's output (what unstage writes).
template <class F> int route_stage (sdtgpu *h, u64 n_out, F launch, void **d_queries, uint64_t *starts, uint64_t *counts)
{
	int rc;
	const u32 world = make_route (h).world;
	h->rt_staged = false;
	Stage st = { nullptr, nullptr, reinterpret_cast<unsigned long long *> (h->rt_cur) };
	CK (h, cudaMemsetAsync (h->rt_cur, 0, world * sizeof (u64), h->stream));
	if ((rc = launch (false, st)))
		return rc;
	CK (h, cudaMemcpyAsync (h->rt_hcur, h->rt_cur, world * sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
	CK (h, cudaStreamSynchronize (h->stream));
	u64 total = 0;
	for (u32 r = 0; r < world; r++)
	{
		starts[r] = total;
		counts[r] = h->rt_hcur[r];
		h->rt_hcur[r] = total;
		total += counts[r];
	}
	const size_t qb = 8 * (size_t) h->W;
	if ((rc = grow_device (h, (void **) &h->rt_q, &h->rt_cap_q, 0, std::max<u64> (total, 1) * qb, "staged lookups"))
	    || (rc = grow_device (h, (void **) &h->rt_tag, &h->rt_cap_tag, 0, std::max<u64> (total, 1) * sizeof (u64), "staged lookups")))
		return rc;
	if (total)
	{
		CK (h, cudaMemcpyAsync (h->rt_cur, h->rt_hcur, world * sizeof (u64), cudaMemcpyHostToDevice, h->stream));
		st.q = h->rt_q;
		st.tag = h->rt_tag;
		if ((rc = launch (true, st)))
			return rc;
	}
	h->rt_staged = true;
	h->rt_n = total;
	h->rt_out = n_out;
	*d_queries = h->rt_q;
	return SDTGPU_OK;
}

template <int W, bool SCATTER> void launch_route_kmers_t (sdtgpu *h, const u64 *keys, u64 n, const Route &rt, const Stage &st)
{
	const unsigned grid = (unsigned) std::min<u64> ((n + BLOCK - 1) / BLOCK, (u64) h->sm_count * 16);
	TimedLaunch tl (h, 7);
	route_kmers_kernel<W, SCATTER><<<grid, BLOCK, 0, h->stream>>> (keys, n, rt, st);
}

template <int W, bool NMODE, bool SCATTER> int launch_route_reads_t (sdtgpu *h, const ReadBatch &rb, const Route &rt, const Stage &st)
{
	auto kern = route_reads_kernel<W, NMODE, SCATTER>;
	const size_t smem = 4 * tile_words (rb, NMODE);
	if (smem > 48 * 1024)
		CK (h, cudaFuncSetAttribute (kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
	int occ = 0;
	CK (h, cudaOccupancyMaxActiveBlocksPerMultiprocessor (&occ, kern, BLOCK, smem));
	if (occ < 1)
		return fail (h, SDTGPU_EINVAL, "read stride too large for one shared-memory tile");
	const u64 n_tiles = (rb.n_reads + rb.tile_reads - 1) / rb.tile_reads;
	const unsigned grid = (unsigned) std::min<u64> (n_tiles, (u64) h->sm_count * occ);
	TimedLaunch tl (h, 7);
	kern<<<grid, BLOCK, smem, h->stream>>> (rb, rt, st);
	return SDTGPU_OK;
}

template <int W, bool NMODE> int launch_route_reads_w (sdtgpu *h, const ReadBatch &rb, const Route &rt, bool scatter, const Stage &st)
{
	return scatter ? launch_route_reads_t<W, NMODE, true> (h, rb, rt, st) : launch_route_reads_t<W, NMODE, false> (h, rb, rt, st);
}

// ---- edges (sdt_edges.cuh)
static_assert (sizeof (EdgeRec) == sizeof (sdtgpu_edge) && sizeof (EdgeRec) == 32 && SDTGPU_EDGE_PALINDROME == EDGE_PALINDROME
	       && SDTGPU_EDGE_CYCLE == EDGE_CYCLE, "sdtgpu_edge");

int edge_grow (sdtgpu *h, int i, size_t need, size_t keep = 0)
{
	return grow_device (h, &h->ed[i], &h->ed_cap[i], keep, std::max<size_t> (need, 64), "edge graph");
}

// CUDA events around the groups of launches between two host reads of a size: the device time of a build
struct EdgeSpans
{
	sdtgpu *h;
	std::vector<cudaEvent_t> ev;
	explicit EdgeSpans (sdtgpu *h_) : h (h_) { }
	void mark () { ev.push_back (get_event (h)); cudaEventRecord (ev.back (), h->stream); }
	double ms () const
	{
		double t = 0;
		for (size_t i = 0; i + 1 < ev.size (); i += 2)
		{
			float f = 0;
			cudaEventElapsedTime (&f, ev[i], ev[i + 1]);
			t += f;
		}
		return t;
	}
	~EdgeSpans () { for (auto e : ev) h->ev_pool.push_back (e); }
};

template <int W> int edges_build_t (sdtgpu *h, uint64_t out[8], double *ms)
{
	typedef typename SlotOf<W>::type S;
	const S *tab = static_cast<const S *> (h->table);
	const u64 slots = iter_slots (h);
	int rc = read_counters (h);
	if (rc)
		return rc;
	EdgeGraph g = {};
	g.index = h->index;
	g.idx_cap = h->idx_cap;
	g.slots = slots;
	g.K = h->K;
	g.deLowKmer = h->deLowKmer;
	g.max_m = 2 * h->h_ctr->n_linear + 2;	// a palindromic edge holds its nodes twice
	auto bind = [&] () {
		g.step = static_cast<Step *> (h->ed[ED_STEP]);
		g.mark = static_cast<unsigned char *> (h->ed[ED_MARK]);
		g.a = static_cast<u32 *> (h->ed[ED_A]);
		g.b = static_cast<u32 *> (h->ed[ED_B]);
		g.off_a = static_cast<const u64 *> (h->ed[ED_OFF_A]);
		g.off_b = static_cast<const u64 *> (h->ed[ED_OFF_B]);
		g.starts = static_cast<u64 *> (h->ed[ED_STARTS]);
		g.edges = static_cast<EdgeRec *> (h->ed[ED_EDGES]);
		g.seq = static_cast<u64 *> (h->ed[ED_SEQ]);
		g.ctr = static_cast<u64 *> (h->ed[ED_CTR]);
	};
	auto grid = [&] (u64 n) { return (unsigned) std::min<u64> ((n + BLOCK - 1) / BLOCK, (u64) h->sm_count * 16); };
	auto nseg = [] (u64 n) { return (u32) std::max<u64> (1, (n + SCAN_SEG - 1) / SCAN_SEG); };
	auto scan = [&] (const u32 *in, u64 n, int off) {
		u64 *seg = static_cast<u64 *> (h->ed[ED_SEG]), *o = static_cast<u64 *> (h->ed[off]);
		slice_scan_sums_kernel<<<nseg (n), SCAN_NT, 0, h->stream>>> (in, (u32) n, seg);
		slice_scan_kernel<<<nseg (n), SCAN_NT, 0, h->stream>>> (in, (u32) n, seg, o, nullptr);
	};
	auto total = [&] (int off, u64 n, u64 &v) -> int {
		CK (h, cudaGetLastError ());
		CK (h, cudaMemcpyAsync (&v, static_cast<u64 *> (h->ed[off]) + n, sizeof v, cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaStreamSynchronize (h->stream));
		return SDTGPU_OK;
	};
	h->ed_built = false;
	if ((rc = edge_grow (h, ED_STEP, slots * sizeof (Step))) || (rc = edge_grow (h, ED_MARK, slots))
	    || (rc = edge_grow (h, ED_A, slots * 4)) || (rc = edge_grow (h, ED_OFF_A, (slots + 1) * 8))
	    || (rc = edge_grow (h, ED_SEG, nseg (slots) * 8)) || (rc = edge_grow (h, ED_CTR, 8 * sizeof (u64))))
		return rc;
	bind ();
	EdgeSpans sp (h);
	// 1. steps of the linear nodes, walk starts of the vertices
	sp.mark ();
	CK (h, cudaMemsetAsync (g.ctr, 0, 8 * sizeof (u64), h->stream));
	if (slots)
		edge_links_kernel<W><<<grid (slots), BLOCK, 0, h->stream>>> (tab, g);
	scan (g.a, slots, ED_OFF_A);
	sp.mark ();
	u64 n_starts = 0;
	if ((rc = total (ED_OFF_A, slots, n_starts)))
		return rc;
	if (n_starts >= NO_POS)
		return fail (h, SDTGPU_ERANGE, "edges: 2^32 - 1 walk starts or more");
	if ((rc = edge_grow (h, ED_STARTS, n_starts * 8)))
		return rc;
	bind ();
	sp.mark ();
	if (n_starts)
		edge_starts_kernel<W><<<grid (slots), BLOCK, 0, h->stream>>> (tab, g);
	sp.mark ();
	CK (h, cudaGetLastError ());
	// 2. every walk to its end: which strand is kept, and its length
	const u64 n2 = std::max (slots, n_starts);
	if ((rc = edge_grow (h, ED_A, n2 * 4)) || (rc = edge_grow (h, ED_B, n2 * 4)) || (rc = edge_grow (h, ED_OFF_A, (n2 + 1) * 8))
	    || (rc = edge_grow (h, ED_OFF_B, (n2 + 1) * 8)) || (rc = edge_grow (h, ED_SEG, nseg (n2) * 8)))
		return rc;
	bind ();
	g.n_starts = n_starts;
	sp.mark ();
	if (n_starts)
		edge_walk_kernel<W, 0><<<grid (n_starts), BLOCK, 0, h->stream>>> (tab, g);
	scan (g.a, n_starts, ED_OFF_A);
	scan (g.b, n_starts, ED_OFF_B);
	CK (h, cudaMemsetAsync (g.mark, 0, std::max<u64> (slots, 1), h->stream));
	sp.mark ();
	u64 n_edges = 0, n_words = 0;
	if ((rc = total (ED_OFF_A, n_starts, n_edges)) || (rc = total (ED_OFF_B, n_starts, n_words)))
		return rc;
	if ((rc = edge_grow (h, ED_EDGES, n_edges * sizeof (EdgeRec))) || (rc = edge_grow (h, ED_SEQ, n_words * 8)))
		return rc;
	bind ();
	// 3. the kept walks write their edges and mark their nodes; the linear nodes left elect one leader per cycle
	sp.mark ();
	if (n_starts)
		edge_walk_kernel<W, 1><<<grid (n_starts), BLOCK, 0, h->stream>>> (tab, g);
	if (slots)
		edge_cycle_kernel<W, 0><<<grid (slots), BLOCK, 0, h->stream>>> (tab, g);
	scan (g.a, slots, ED_OFF_A);
	scan (g.b, slots, ED_OFF_B);
	sp.mark ();
	u64 n_cycles = 0, n_cwords = 0;
	if ((rc = total (ED_OFF_A, slots, n_cycles)) || (rc = total (ED_OFF_B, slots, n_cwords)))
		return rc;
	if ((rc = edge_grow (h, ED_EDGES, (n_edges + n_cycles) * sizeof (EdgeRec), n_edges * sizeof (EdgeRec)))
	    || (rc = edge_grow (h, ED_SEQ, (n_words + n_cwords) * 8, n_words * 8)))
		return rc;
	bind ();
	g.edge0 = n_edges;
	g.unit0 = n_words;
	// 4. the leaders write their cycles after the edges
	sp.mark ();
	if (slots)
		edge_cycle_kernel<W, 1><<<grid (slots), BLOCK, 0, h->stream>>> (tab, g);
	sp.mark ();
	CK (h, cudaGetLastError ());
	u64 c[8];
	CK (h, cudaMemcpyAsync (c, g.ctr, sizeof c, cudaMemcpyDeviceToHost, h->stream));
	CK (h, cudaStreamSynchronize (h->stream));
	out[0] = n_edges + n_cycles;
	for (int i = 1; i < 8; i++)
		out[i] = c[i];
	*ms = sp.ms ();
	h->ed_built = true;
	return SDTGPU_OK;
}

}	// namespace

// =================================================================================================
extern "C" {

int sdtgpu_version (void) { return 1; }

uint64_t sdtgpu_hash_kmer (const uint64_t key[4], int key_words)
{
	crc_table_host ();
	return hash_kmer_impl (key, key_words, h_crc);
}

const char *sdtgpu_last_error (const sdtgpu_t *h) { return h ? h->err.c_str () : g_create_error.c_str (); }

int sdtgpu_create (sdtgpu_t **out, int device, int K, int key_words, int max_read_len, uint64_t capacity_hint, unsigned flags)
{
	if (!out)
		return SDTGPU_EINVAL;
	*out = nullptr;
	if (flags & ~(SDTGPU_F_NKMER | SDTGPU_F_SLICED))
	{
		g_create_error = "unknown flag (the experimental partitioned insert of round 1, flag 2, was measured slower and removed)";
		return SDTGPU_EINVAL;
	}
	if ((key_words != 1 && key_words != 2 && key_words != 4) || !(K & 1) || K < 13 || K > 32 * key_words - 1)
	{
		g_create_error = "K must be odd, 13 <= K <= 32*key_words-1, key_words in {1,2,4} (pregraph.c:38-59)";
		return SDTGPU_EINVAL;
	}
	if (max_read_len < K + 1)
	{
		g_create_error = "max_read_len must be at least K+1";
		return SDTGPU_EINVAL;
	}
	int n_dev = 0;
	cudaError_t e = cudaGetDeviceCount (&n_dev);
	if (e != cudaSuccess || device < 0 || device >= n_dev)
	{
		g_create_error = std::string ("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString (e) : "bad ordinal");
		return SDTGPU_ECUDA;
	}
	sdtgpu *h = new sdtgpu ();
	h->device = device; h->K = K; h->key_words = key_words; h->max_read_len = max_read_len; h->flags = flags;
	h->W = K <= 31 ? 1 : (K <= 63 ? 2 : 4);
	h->sliced = (flags & SDTGPU_F_SLICED) != 0;
	h->maxwin = (u32) (max_read_len - K + 1);
	auto bail = [&](int rc) { g_create_error = h->err; sdtgpu_destroy (h); return rc; };
	auto body = [&]() -> int {
		CK (h, cudaSetDevice (device));
		cudaDeviceProp prop;
		CK (h, cudaGetDeviceProperties (&prop, device));
		h->sm_count = prop.multiProcessorCount;
		h->mem_total = prop.totalGlobalMem;
		CK (h, cudaStreamCreateWithFlags (&h->stream, cudaStreamNonBlocking));
		CK (h, cudaStreamCreateWithFlags (&h->copy_stream, cudaStreamNonBlocking));
		for (auto &s : h->stage)
		{
			CK (h, cudaEventCreateWithFlags (&s.free_ev, cudaEventDisableTiming));
			CK (h, cudaEventCreateWithFlags (&s.ready_ev, cudaEventDisableTiming));
		}
		CK (h, cudaMalloc (&h->d_ctr, sizeof (Counters)));
		CK (h, cudaMemsetAsync (h->d_ctr, 0, sizeof (Counters), h->stream));
		CK (h, cudaMallocHost (&h->h_nodes_snap, 8 * sizeof (u64)));
		CK (h, cudaEventCreateWithFlags (&h->snap_ev, cudaEventDisableTiming));
		CK (h, cudaMallocHost (&h->h_ctr, sizeof (Counters)));
		memset (h->h_ctr, 0, sizeof (Counters));
		crc_table_host ();
		CK (h, cudaMemcpyToSymbol (c_crc, h_crc, sizeof h_crc));
		h->grow_mode = capacity_hint == 0;
		h->cap = capacity_hint ? pick_capacity (capacity_hint, slot_bytes (h->W)) : (1ull << 20);
		int rc;
		if (h->sliced)
		{	// the geometry is fixed when the first records are made (skm_open_epoch), the node store is sized after the merge
			h->hint = capacity_hint;
			h->cap = 0;
			CK (h, cudaMalloc (&h->d_small, 160 * sizeof (u64)));
			CK (h, cudaMalloc (&h->d_failed, (size_t) MAX_FAILED * sizeof (SkmWork)));
			CK (h, cudaMalloc (&h->d_items, (size_t) MAX_FAILED * sizeof (SkmWork)));
			CK (h, cudaMallocHost (&h->h_small, 160 * sizeof (u64)));
			CK (h, cudaMallocHost (&h->h_failed, 4096 * sizeof (SkmWork)));
			CK (h, cudaMemsetAsync (h->d_small, 0, 160 * sizeof (u64), h->stream));
			CK (h, cudaStreamSynchronize (h->stream));
			if (capacity_hint && (rc = skm_open_epoch (h)))	// (reports a bad geometry at create time)
				return rc;
			return SDTGPU_OK;
		}
		CK (h, cudaMalloc (&h->table, h->cap * slot_bytes (h->W)));
		rc = init_table (h, h->table, h->cap);
		if (rc)
			return rc;
		CK (h, cudaStreamSynchronize (h->stream));
		return SDTGPU_OK;
	};
	int rc = body ();
	if (rc)
		return bail (rc);
	*out = h;
	return SDTGPU_OK;
}

void sdtgpu_destroy (sdtgpu_t *h)
{
	if (!h)
		return;
	cudaSetDevice (h->device);
	if (h->stream)
		cudaStreamSynchronize (h->stream);
	if (h->copy_stream)
		cudaStreamSynchronize (h->copy_stream);
	for (auto &s : h->stage)
	{
		cudaFree (s.d_packed); cudaFree (s.d_lens); cudaFree (s.d_mask);
		if (s.free_ev) cudaEventDestroy (s.free_ev);
		if (s.ready_ev) cudaEventDestroy (s.ready_ev);
	}
	for (auto &p : h->timing) { cudaEventDestroy (p.e0); cudaEventDestroy (p.e1); }
	cudaFree (h->last_packed); cudaFree (h->last_mask); cudaFree (h->last_lens);
	for (auto e : h->ev_pool) cudaEventDestroy (e);
	for (void *m : h->log_mem) cudaFree (m);
	for (auto &L : h->lv)
		level_free (L);
	cudaFree (h->d_small); cudaFree (h->d_failed); cudaFree (h->d_items); cudaFree (h->rx);
	if (h->h_small) cudaFreeHost (h->h_small);
	if (h->h_failed) cudaFreeHost (h->h_failed);
	cudaFree (h->table);
	cudaFree (h->index);
	free_route (h);
	free_edges (h);
	cudaFree (h->rt_cur);
	if (h->rt_hcur) cudaFreeHost (h->rt_hcur);
	cudaFree (h->d_ctr);
	if (h->h_ctr) cudaFreeHost (h->h_ctr);
	if (h->h_nodes_snap) cudaFreeHost (h->h_nodes_snap);
	if (h->snap_ev) cudaEventDestroy (h->snap_ev);
	if (h->stream) cudaStreamDestroy (h->stream);
	if (h->copy_stream) cudaStreamDestroy (h->copy_stream);
	delete h;
}

int sdtgpu_reset (sdtgpu_t *h)
{
	if (!h)
		return SDTGPU_EINVAL;
	CK (h, cudaSetDevice (h->device));
	Trace tr (h);
	if (h->index || h->rt_q || h->rt_aq || h->rt_back || h->ed[ED_STEP])
	{
		CK (h, cudaStreamSynchronize (h->stream));	// (a lookup may still be reading them)
		free_index (h);
		free_route (h);
		free_edges (h);
	}
	h->rt_staged = false;
	CK (h, cudaMemsetAsync (h->d_ctr, 0, sizeof (Counters), h->stream));
	tr.mark ("reset: counters");
	if (h->sliced)
	{	// records, their per-slice counts and the read log go; the store is rewritten by the next build
		CK (h, cudaMemsetAsync (h->d_small, 0, 8 * sizeof (u64), h->stream));
		if (h->hint && h->epoch_open)
		{
			int rc = level_reset (h, h->lv[0]);
			if (rc)
				return rc;
		}
		else
			h->epoch_open = false;	// no hint: the next epoch's geometry comes from what is pushed then (skm_open_epoch empties the chains)
		h->emitted = false;
		h->chains_dropped = false;
		{	// a node store that takes a large part of the memory would be in the way of the next epoch's records
			if (h->table && (double) h->cap * slot_bytes (h->W) > 0.45 * (double) h->mem_total)
			{
				CK (h, cudaStreamSynchronize (h->stream));
				CK (h, cudaFree (h->table));
				h->table = nullptr;
				h->cap = 0;
			}
		}
		tr.mark ("reset: chains");
		h->ord_bound_set = false;
		h->log.clear ();
		h->log_used[0] = h->log_used[1] = h->log_used[2] = 0;
		h->n_store = 0;
		h->table_built = false;
		h->dirty = false;
	}
	else
	{
		int rc = init_table (h, h->table, h->cap);
		if (rc)
			return rc;
	}
	h->pushed_upper = 0; h->n_reads = 0; h->ord_end = 0; h->finalized = false; h->deLowKmer = 0;
	if (h->snap_pending)
		CK (h, cudaEventSynchronize (h->snap_ev));
	h->snap_pending = false;
	h->known_nodes = h->known_at = h->snap_pushed = 0;
	tr.mark ("reset: rest");
	return SDTGPU_OK;
}

void *sdtgpu_stream (sdtgpu_t *h) { return h ? (void *) h->stream : nullptr; }
void *sdtgpu_aux_stream (sdtgpu_t *h) { return h ? (void *) h->copy_stream : nullptr; }

int sdtgpu_sync (sdtgpu_t *h)
{
	if (!h)
		return SDTGPU_EINVAL;
	CK (h, cudaSetDevice (h->device));
	CK (h, cudaStreamSynchronize (h->copy_stream));
	int rc = flush_epoch (h);
	if (rc)
		return rc;
	CK (h, cudaStreamSynchronize (h->stream));
	return SDTGPU_OK;
}

int sdtgpu_push_reads_device (sdtgpu_t *h, const uint8_t *d_packed, const uint32_t *d_lens, const uint8_t *d_nmask,
			      uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes, uint64_t first_read_ordinal)
{
	if (!h)
		return SDTGPU_EINVAL;
	CK (h, cudaSetDevice (h->device));
	ReadBatch rb;
	int rc = make_push_batch (h, rb, d_packed, d_lens, d_nmask, n_reads, uniform_len, stride_bytes, first_read_ordinal);
	if (rc || n_reads == 0)
		return rc;
	h->n_reads += n_reads;
	if ((rc = retain_last_batch (h, rb)))
		return rc;
	if (h->sliced)
	{
		u64 upper = instances_upper (h, n_reads, uniform_len, d_lens != nullptr);
		if (h->owner_ranks > 1)
			upper = upper / h->owner_ranks + upper / (2 * h->owner_ranks) + 1024;
		return sliced_push (h, rb, upper);	// (with owner filtering the record area is simply sized generously)
	}
	{	// single pass: every window goes straight to its (random) slot
		u64 upper = instances_upper (h, n_reads, uniform_len, d_lens != nullptr);
		if (h->owner_ranks > 1)	// owners are a uniform hash of the key: this rank keeps ~1/n (allow 1.5x)
			upper = upper / h->owner_ranks + upper / (2 * h->owner_ranks) + 1024;
		rc = ensure_capacity (h, upper);
		if (rc)
			return rc;
		h->pushed_upper += upper;
		// MODE 5 (chop into a shared-memory queue, then upsert with full warps) is the default also on one
		// GPU: +3.5 % on C2 over upserting straight from the chop loop (MODE 0, SDTGPU_NO_QUEUE=1 for A/B)
		rc = getenv ("SDTGPU_NO_QUEUE") && h->owner_ranks <= 1 ? launch_insert<0> (h, rb, Bins ()) : launch_insert<5> (h, rb, Bins ());
		return rc ? rc : snapshot_nodes (h);
	}
}

int sdtgpu_push_reads (sdtgpu_t *h, const uint8_t *packed, const uint32_t *lens, const uint8_t *nmask,
		       uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes, uint64_t first_read_ordinal)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (n_reads == 0)
		return SDTGPU_OK;
	if (!packed)
		return fail (h, SDTGPU_EINVAL, "packed == NULL");
	CK (h, cudaSetDevice (h->device));
	const bool nmode = (h->flags & SDTGPU_F_NKMER) && nmask;
	Staging &s = h->stage[h->next_stage];
	h->next_stage ^= 1;
	const size_t pbytes = (size_t) n_reads * stride_bytes, lbytes = lens ? (size_t) n_reads * 4 : 0;
	const size_t mstride = stride_bytes / 2, mbytes = nmode ? (size_t) n_reads * mstride : 0;
	// the kernel that last read this staging buffer must be done before it is overwritten
	CK (h, cudaStreamWaitEvent (h->copy_stream, s.free_ev, 0));
	if (pbytes > s.cap_packed || lbytes > s.cap_lens || mbytes > s.cap_mask)
	{
		CK (h, cudaEventSynchronize (s.free_ev));
		int rc = ensure_stage (h, s, pbytes, lbytes, mbytes);
		if (rc)
			return rc;
	}
	CK (h, cudaMemcpyAsync (s.d_packed, packed, pbytes, cudaMemcpyHostToDevice, h->copy_stream));
	if (lens)
		CK (h, cudaMemcpyAsync (s.d_lens, lens, lbytes, cudaMemcpyHostToDevice, h->copy_stream));
	if (nmode)
		CK (h, cudaMemcpyAsync (s.d_mask, nmask, mbytes, cudaMemcpyHostToDevice, h->copy_stream));
	CK (h, cudaEventRecord (s.ready_ev, h->copy_stream));
	CK (h, cudaStreamWaitEvent (h->stream, s.ready_ev, 0));
	CK (h, cudaEventSynchronize (s.ready_ev));	// the caller's buffers are free again when we return
	int rc = sdtgpu_push_reads_device (h, s.d_packed, lens ? s.d_lens : nullptr, nmode ? s.d_mask : nullptr,
					   n_reads, uniform_len, stride_bytes, first_read_ordinal);
	CK (h, cudaEventRecord (s.free_ev, h->stream));
	return rc;
}

int sdtgpu_set_owner (sdtgpu_t *h, int rank, int n_ranks)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (n_ranks < 1 || rank < 0 || rank >= n_ranks)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_set_owner: need 0 <= rank < n_ranks");
	if (h->sliced && !h->log.empty ())
		return fail (h, SDTGPU_ESTATE, "sdtgpu_set_owner must precede the pushes of an epoch");
	h->owner_rank = (u32) rank;
	h->owner_ranks = (u32) n_ranks;
	return SDTGPU_OK;
}

// ---- super-k-mer exchange (multi-GPU sliced build): the slices are dealt to the ranks in contiguous
// ranges; a rank turns ITS reads into records (chains over ALL slices), merges its own copies, hands each
// owner's records to the caller's all-to-all, and builds its own slices from what it receives.
int sdtgpu_skm_set_world (sdtgpu_t *h, int rank, int world)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (!h->sliced)
		return fail (h, SDTGPU_ESTATE, "sdtgpu_skm_set_world needs SDTGPU_F_SLICED");
	if (world < 1 || world > 64 || rank < 0 || rank >= world)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_skm_set_world: need 0 <= rank < world <= 64");
	if (!h->log.empty ())
		return fail (h, SDTGPU_ESTATE, "sdtgpu_skm_set_world must precede the pushes of an epoch");
	if (!h->hint)
		return fail (h, SDTGPU_ESTATE, "the super-k-mer exchange needs capacity_hint (every rank must cut the minimizer space the same way)");
	CK (h, cudaSetDevice (h->device));
	if (h->epoch_open && ((u32) world != h->skm_world || (u32) rank != h->skm_rank))
	{
		h->epoch_open = false;
		level_free (h->lv[0]);
	}
	h->skm_world = (u32) world;
	h->skm_rank = (u32) rank;
	return skm_open_epoch (h);	// the geometry is known from here on (sdtgpu_slice_geometry)
}

int sdtgpu_skm_set_ordinal_bound (sdtgpu_t *h, uint64_t n_reads_all_ranks)
{
	if (!h)
		return SDTGPU_EINVAL;
	h->ord_end = std::max<u64> (h->ord_end, n_reads_all_ranks * h->maxwin);
	h->ord_bound_set = true;
	return SDTGPU_OK;
}

int sdtgpu_skm_stage (sdtgpu_t *h, void **d_records, uint64_t *starts, uint64_t *counts)
{
	int rc;
	if (!h || !d_records || !starts || !counts)
		return SDTGPU_EINVAL;
	if (!h->sliced)
		return fail (h, SDTGPU_ESTATE, "sdtgpu_skm_stage needs SDTGPU_F_SLICED");
	CK (h, cudaSetDevice (h->device));
	if ((rc = skm_open_epoch (h)))
		return rc;
	ChainLevel &L = h->lv[0];
	const u32 world = h->skm_world, per_owner = world > 1 ? h->n_local / h->geom.send_group : L.n_chains;
	u64 n_rec = 0;
	h->emitted = true;	// (a rank without reads still takes part)
	Trace tr (h);
	if ((rc = skm_collect (h, &n_rec)))
		return rc;
	tr.mark ("stage: collect");
	h->n_records = n_rec;
	u64 n_blocks = 0;
	if ((rc = level_list (h, L, &n_blocks)))
		return rc;
	tr.mark ("stage: list");
	// records per owner (an upper bound of what survives the merge) -> where each owner's region starts
	u64 *d_reg = h->d_small + 8;	// [world] region starts, [world] cursors
	chain_owner_count_kernel<<<world, 256, 0, h->stream>>> (level_chains (h, L), per_owner, reinterpret_cast<unsigned long long *> (d_reg));
	CK (h, cudaGetLastError ());
	h->all_launches++;
	CK (h, cudaMemcpyAsync (h->h_small + 8, d_reg, world * sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
	CK (h, cudaStreamSynchronize (h->stream));
	u64 run = 0;
	for (u32 r = 0; r < world; r++)
	{
		const u64 c = h->h_small[8 + r];
		starts[r] = run;
		h->h_small[8 + r] = run;
		h->h_small[8 + world + r] = 0;
		run += c;
	}
	CK (h, cudaMemcpyAsync (d_reg, h->h_small + 8, 2 * world * sizeof (u64), cudaMemcpyHostToDevice, h->stream));
	{
		const size_t rec = 4 * (size_t) h->geom.recw;
		size_t cap_b = L.out_cap * rec;
		if ((rc = grow_device (h, (void **) &L.out, &cap_b, 0, std::max<u64> (run, 1) * rec)))
			return rc;
		L.out_cap = cap_b / rec;
	}
	tr.mark ("stage: owner regions");
	if ((rc = launch_merge (h, L, false, n_rec, per_owner, d_reg, d_reg + world)))
		return rc;
	CK (h, cudaMemcpyAsync (h->h_small + 8 + world, d_reg + world, world * sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
	CK (h, cudaStreamSynchronize (h->stream));
	tr.mark ("stage: merge by owner");
	for (u32 r = 0; r < world; r++)
		counts[r] = h->h_small[8 + world + r];
	*d_records = L.out;
	return SDTGPU_OK;
}

int sdtgpu_skm_import_buffer (sdtgpu_t *h, uint64_t n_records, void **d_buffer)
{
	int rc;
	if (!h || !d_buffer)
		return SDTGPU_EINVAL;
	if (!h->sliced)
		return fail (h, SDTGPU_ESTATE, "sdtgpu_skm_import_buffer needs SDTGPU_F_SLICED");
	CK (h, cudaSetDevice (h->device));
	const size_t rec = 4 * (size_t) h->geom.recw;
	size_t cap_b = h->rx_cap * rec;
	if ((rc = grow_device (h, (void **) &h->rx, &cap_b, 0, std::max<u64> (n_records, 1) * rec, "receive buffer", true)))
		return rc;
	h->rx_cap = cap_b / rec;
	*d_buffer = h->rx;
	return SDTGPU_OK;
}

int sdtgpu_skm_import (sdtgpu_t *h, uint64_t n_records)
{
	int rc;
	if (!h)
		return SDTGPU_EINVAL;
	if (!h->sliced)
		return fail (h, SDTGPU_ESTATE, "sdtgpu_skm_import needs SDTGPU_F_SLICED");
	if (n_records > h->rx_cap)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_skm_import: more records than sdtgpu_skm_import_buffer made room for");
	CK (h, cudaSetDevice (h->device));
	if ((rc = skm_open_epoch (h)))
		return rc;
	const u32 n_local = h->skm_world > 1 ? h->n_local : h->geom.n_slices;
	ChainLevel &R = h->lv[2];
	Trace tr (h);
	if ((rc = level_create (h, R, n_local)))
		return rc;
	tr.mark ("import: chains reset");
	const u64 hold = (u64) std::min<u64> ((u64) h->sm_count * 8, MAX_CTAS) * CH_SB;
	for (int attempt = 0;; attempt++)
	{
		const u64 slack = attempt ? n_records / CH_BLK : n_records / (8 * CH_BLK);	// (blocks the CTAs drop when they refill their ranges)
		if ((rc = level_reserve (h, R, n_local + n_records / CH_BLK + slack + hold + 4096)))
			return rc;
		if (n_records)
		{
			const unsigned grid = (unsigned) std::min<u64> ((n_records + AP_TILE - 1) / AP_TILE, std::min<u64> ((u64) h->sm_count * 8, MAX_CTAS));
			TimedLaunch tl (h, 2);
			const SkmChains c = level_chains (h, R);
			const u32 lo = h->skm_rank * n_local;
			if (h->geom.recw == 8)
				skm_append_kernel<8><<<grid, AP_NT, 0, h->stream>>> (c, h->rx, n_records, lo);
			else if (h->geom.recw == 12)
				skm_append_kernel<12><<<grid, AP_NT, 0, h->stream>>> (c, h->rx, n_records, lo);
			else
				skm_append_kernel<16><<<grid, AP_NT, 0, h->stream>>> (c, h->rx, n_records, lo);
		}
		CK (h, cudaGetLastError ());
		CK (h, cudaMemcpyAsync (h->h_small + 3, &h->d_ctr->overflow, sizeof (u64), cudaMemcpyDeviceToHost, h->stream));
		CK (h, cudaStreamSynchronize (h->stream));
		if (h->h_small[3] & OVF_FOREIGN)
			return fail (h, SDTGPU_EINVAL, "super-k-mer exchange: a received record belongs to another rank's slices");
		tr.mark ("import: append");
		if (!(h->h_small[3] & OVF_RECORDS))
			break;
		if (attempt == 1)
			return fail (h, SDTGPU_ERANGE, "record pool overflow persists (import)");
		CK (h, cudaMemsetAsync (&h->d_ctr->overflow, 0, sizeof (u64), h->stream));
		if ((rc = level_reset (h, R)))
			return rc;
	}
	h->n_store = 0;
	if (!h->ord_bound_set && h->skm_world > 1)
		h->ord_end = ~0ull;	// records of other ranks' reads: their ordinals are not bounded by what this rank pushed
	return skm_build_level (h, R, true, n_records, n_records, true);
}

size_t sdtgpu_record_bytes (const sdtgpu_t *h) { return h ? 8 * (size_t) (h->W + 1) : 0; }

int sdtgpu_bucket_reads_device (sdtgpu_t *h, const uint8_t *d_packed, const uint32_t *d_lens, const uint8_t *d_nmask,
				uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes, uint64_t first_read_ordinal,
				int n_ranks, void *d_bins, uint64_t bin_capacity, uint64_t *d_counts)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (n_ranks < 1 || !d_bins || !d_counts || ((uintptr_t) d_bins & 15))
		return fail (h, SDTGPU_EINVAL, "bad bins");
	CK (h, cudaSetDevice (h->device));
	ReadBatch rb;
	int rc = make_push_batch (h, rb, d_packed, d_lens, d_nmask, n_reads, uniform_len, stride_bytes, first_read_ordinal);
	if (rc || n_reads == 0)
		return rc;
	Bins b;
	b.records = static_cast<u64 *> (d_bins);
	b.counts = reinterpret_cast<u64 *> (d_counts);
	b.capacity = bin_capacity;
	b.n_ranks = (u32) n_ranks;
	h->n_reads += n_reads;
	h->launch_stream = h->copy_stream;	// the send side runs on the auxiliary stream so that it
	rc = launch_insert<1> (h, rb, b);	// overlaps the inserts of the previous round
	h->launch_stream = nullptr;
	return rc;
}

int sdtgpu_insert_records_device (sdtgpu_t *h, const void *d_records, uint64_t n_records)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (h->finalized)
		return fail (h, SDTGPU_ESTATE, "insert after finalize");
	if (n_records == 0)
		return SDTGPU_OK;
	if (h->sliced)
		return fail (h, SDTGPU_ESTATE, "insert_records_device is not available with SDTGPU_F_SLICED");
	if (!d_records || ((uintptr_t) d_records & (h->W == 1 ? 15 : 7)))
		return fail (h, SDTGPU_EINVAL, "records must be aligned device memory (16 bytes for 1-word keys, else 8)");
	CK (h, cudaSetDevice (h->device));
	int rc = flush_epoch (h);
	if (rc)
		return rc;
	rc = ensure_capacity (h, n_records);
	if (rc)
		return rc;
	h->pushed_upper += n_records;
	const unsigned grid = (unsigned) std::min<u64> ((n_records + BLOCK - 1) / BLOCK, (u64) h->sm_count * 8);
	cudaEvent_t e0 = get_event (h), e1 = get_event (h);
	CK (h, cudaEventRecord (e0, h->stream));
	const u64 *rec = static_cast<const u64 *> (d_records);
	switch (h->W)
	{
	case 1: insert_records_kernel<1><<<grid, BLOCK, 0, h->stream>>> (static_cast<Slot1 *> (h->table), h->cap, rec, n_records, h->d_ctr); break;
	case 2: insert_records_kernel<2><<<grid, BLOCK, 0, h->stream>>> (static_cast<Slot2 *> (h->table), h->cap, rec, n_records, h->d_ctr); break;
	default: insert_records_kernel<4><<<grid, BLOCK, 0, h->stream>>> (static_cast<Slot4 *> (h->table), h->cap, rec, n_records, h->d_ctr); break;
	}
	CK (h, cudaGetLastError ());
	CK (h, cudaEventRecord (e1, h->stream));
	h->timing.push_back ({ e0, e1, 0 });
	h->all_launches++;
	return snapshot_nodes (h);
}

static void fill_stats (sdtgpu *h, sdtgpu_stats *st)
{
	st->n_instances = h->h_ctr->n_instances;
	st->n_nodes = h->h_ctr->n_nodes;
	st->n_removed = h->h_ctr->n_removed;
	st->n_linear = h->h_ctr->n_linear;
	st->capacity = h->cap;
	st->n_reads = h->n_reads;
	st->n_grows = h->n_grows;
	st->device_key_words = (u32) h->W;
}

int sdtgpu_get_stats (sdtgpu_t *h, sdtgpu_stats *stats)
{
	if (!h || !stats)
		return SDTGPU_EINVAL;
	CK (h, cudaSetDevice (h->device));
	int rc = flush_epoch (h);
	if (rc)
		return rc;
	rc = read_counters (h);
	if (rc)
		return rc;
	fill_stats (h, stats);
	if (h->h_ctr->overflow && !h->sliced)
		return fail (h, SDTGPU_ERANGE, "a record bin overflowed");
	return SDTGPU_OK;
}

int sdtgpu_finalize (sdtgpu_t *h, int deLowKmer, int64_t kmerFreq[257], sdtgpu_stats *stats)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (h->finalized)
		return fail (h, SDTGPU_ESTATE, "finalize called twice");
	if (deLowKmer < 0 || deLowKmer > 127)
		return fail (h, SDTGPU_EINVAL, "deLowKmer is a char in the reference (0..127)");
	CK (h, cudaSetDevice (h->device));
	CK (h, cudaStreamSynchronize (h->copy_stream));
	int frc = flush_epoch (h);
	if (frc)
		return frc;
	const u64 slots = iter_slots (h);	// the whole table, or the node store of the sliced build
	const unsigned grid = (unsigned) std::min<u64> ((slots + BLOCK - 1) / BLOCK, (u64) h->sm_count * 8);
	if (grid)
		switch (h->W)
		{
		case 1: finalize_kernel<1><<<grid, BLOCK, 0, h->stream>>> (static_cast<Slot1 *> (h->table), slots, deLowKmer, h->d_ctr); break;
		case 2: finalize_kernel<2><<<grid, BLOCK, 0, h->stream>>> (static_cast<Slot2 *> (h->table), slots, deLowKmer, h->d_ctr); break;
		default: finalize_kernel<4><<<grid, BLOCK, 0, h->stream>>> (static_cast<Slot4 *> (h->table), slots, deLowKmer, h->d_ctr); break;
		}
	CK (h, cudaGetLastError ());
	h->all_launches++;
	h->finalized = true;
	h->deLowKmer = deLowKmer;
	int rc = read_counters (h);
	if (rc)
		return rc;
	if (h->h_ctr->overflow && !h->sliced)
		return fail (h, SDTGPU_ERANGE, "a record bin overflowed");
	if (kmerFreq)
		for (int i = 0; i < 257; i++)
			kmerFreq[i] = (int64_t) h->h_ctr->freq[i];
	if (stats)
		fill_stats (h, stats);
	return SDTGPU_OK;
}

int sdtgpu_export_count (sdtgpu_t *h, uint64_t *n_nodes)
{
	if (!h || !n_nodes)
		return SDTGPU_EINVAL;
	CK (h, cudaSetDevice (h->device));
	int rc = flush_epoch (h);
	if (rc)
		return rc;
	rc = read_counters (h);
	if (rc)
		return rc;
	*n_nodes = h->h_ctr->n_nodes;
	return SDTGPU_OK;
}

int sdtgpu_export_nodes (sdtgpu_t *h, int thrd_num, int sort_by_ordinal, sdtgpu_node *out, uint64_t max_nodes, uint64_t *n_nodes)
{
	if (!h || !out || !n_nodes || thrd_num < 1)
		return SDTGPU_EINVAL;
	CK (h, cudaSetDevice (h->device));
	int rc = flush_epoch (h);
	if (rc)
		return rc;
	rc = read_counters (h);
	if (rc)
		return rc;
	const u64 n = h->h_ctr->n_nodes;
	*n_nodes = n;
	if (n > max_nodes)
		return fail (h, SDTGPU_ERANGE, "export buffer too small");
	if (n == 0)
		return SDTGPU_OK;
	sdtgpu_node *d_out = nullptr;
	CK (h, cudaMalloc (&d_out, n * sizeof (sdtgpu_node)));
	CK (h, cudaMemsetAsync (&h->d_ctr->export_cursor, 0, sizeof (u64), h->stream));
	const u64 slots = iter_slots (h);
	const unsigned grid = (unsigned) std::min<u64> ((slots + BLOCK - 1) / BLOCK, (u64) h->sm_count * 8);
	switch (h->W)
	{
	case 1: export_kernel<1><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot1 *> (h->table), slots, h->key_words, thrd_num, h->deLowKmer, d_out, n, h->d_ctr); break;
	case 2: export_kernel<2><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot2 *> (h->table), slots, h->key_words, thrd_num, h->deLowKmer, d_out, n, h->d_ctr); break;
	default: export_kernel<4><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot4 *> (h->table), slots, h->key_words, thrd_num, h->deLowKmer, d_out, n, h->d_ctr); break;
	}
	h->all_launches++;
	cudaError_t e = cudaGetLastError ();
	if (e == cudaSuccess)
		e = cudaMemcpyAsync (out, d_out, n * sizeof (sdtgpu_node), cudaMemcpyDeviceToHost, h->stream);
	if (e == cudaSuccess)
		e = cudaStreamSynchronize (h->stream);
	cudaFree (d_out);
	CK (h, e);
	if (sort_by_ordinal)
		std::sort (out, out + n, [](const sdtgpu_node &a, const sdtgpu_node &b) {
			return a.set != b.set ? a.set < b.set : a.ordinal < b.ordinal;
		});
	return SDTGPU_OK;
}

int sdtgpu_export_kmersets (sdtgpu_t *h, int thrd_num, sdtgpu_kmerset **sets)
{
	if (!h || !sets || thrd_num < 1)
		return SDTGPU_EINVAL;
	uint64_t n = 0;
	int rc = sdtgpu_export_count (h, &n);
	if (rc)
		return rc;
	sdtgpu_node *nodes = (sdtgpu_node *) malloc (std::max<uint64_t> (n, 1) * sizeof (sdtgpu_node));
	if (!nodes)
		return fail (h, SDTGPU_ENOMEM, "host allocation for export failed");
	rc = sdtgpu_export_nodes (h, thrd_num, 0, nodes, n, &n);
	std::vector<u64> last;
	if (!rc)
		rc = set_last_ordinals (h, thrd_num, last);
	if (!rc)
	{
		// last[s] = (largest instance ordinal of set s in the newest batch) + 1, or 0 when that batch
		// had no instance of s.  In the latter case a later instance than the set's newest key can only
		// have come from an older batch; every batch of >= a few hundred reads touches every set, so a
		// set that the newest batch missed is assumed to have ended with its newest key.
		std::vector<uint64_t> last_ord (thrd_num, 0);
		for (int t = 0; t < thrd_num; t++)
			last_ord[t] = last[t] ? last[t] - 1 : 0;
		rc = sdtgpu_build_kmersets (nodes, n, h->key_words, thrd_num, h->have_last ? last_ord.data () : nullptr, sets);
		if (rc)
			h->err = "sdtgpu_build_kmersets failed";
	}
	free (nodes);
	return rc;
}

int sdtgpu_last_ordinals (sdtgpu_t *h, int thrd_num, uint64_t *out)
{
	if (!h || !out || thrd_num < 1)
		return SDTGPU_EINVAL;
	CK (h, cudaSetDevice (h->device));
	int rc = flush_epoch (h);
	if (rc)
		return rc;
	std::vector<u64> last;
	rc = set_last_ordinals (h, thrd_num, last);
	if (rc)
		return rc;
	for (int t = 0; t < thrd_num; t++)
		out[t] = last[t] ? last[t] - 1 : 0;
	return h->have_last ? SDTGPU_OK : SDTGPU_ESTATE;
}

int sdtgpu_table_checksum (sdtgpu_t *h, uint64_t out[4])
{
	if (!h || !out)
		return SDTGPU_EINVAL;
	CK (h, cudaSetDevice (h->device));
	int rc = flush_epoch (h);
	if (rc)
		return rc;
	u64 *d = nullptr;
	CK (h, cudaMalloc (&d, 4 * sizeof (u64)));
	CK (h, cudaMemsetAsync (d, 0, 4 * sizeof (u64), h->stream));
	const u64 slots = iter_slots (h);
	const unsigned grid = (unsigned) std::min<u64> ((slots + BLOCK - 1) / BLOCK, (u64) h->sm_count * 8);
	if (grid)
		switch (h->W)
		{
		case 1: checksum_kernel<1><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot1 *> (h->table), slots, d); break;
		case 2: checksum_kernel<2><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot2 *> (h->table), slots, d); break;
		default: checksum_kernel<4><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot4 *> (h->table), slots, d); break;
		}
	h->all_launches++;
	cudaError_t e = cudaGetLastError ();
	if (e == cudaSuccess)
		e = cudaMemcpyAsync (out, d, 4 * sizeof (u64), cudaMemcpyDeviceToHost, h->stream);
	if (e == cudaSuccess)
		e = cudaStreamSynchronize (h->stream);
	cudaFree (d);
	CK (h, e);
	return SDTGPU_OK;
}

int sdtgpu_lookup_kmers_device (sdtgpu_t *h, const uint64_t *d_keys, uint64_t n, sdtgpu_hit *d_out)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (n && (!d_keys || !d_out))
		return fail (h, SDTGPU_EINVAL, "sdtgpu_lookup_kmers_device: NULL buffer");
	int rc = lookup_prologue (h, d_out);
	if (rc)
		return rc;
	if ((uintptr_t) d_keys & 15)
		return fail (h, SDTGPU_EINVAL, "the key buffer must be 16-byte aligned");
	if (n == 0)
		return SDTGPU_OK;
	if ((rc = ensure_index (h)))
		return rc;
	const Lookup lk = make_lookup (h, d_out);
	const unsigned grid = (unsigned) std::min<u64> ((n + BLOCK - 1) / BLOCK, (u64) h->sm_count * 16);
	{
		TimedLaunch tl (h, 7);
		switch (h->W)
		{
		case 1: lookup_kmers_kernel<1><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot1 *> (h->table), lk, reinterpret_cast<const u64 *> (d_keys), n, h->K); break;
		case 2: lookup_kmers_kernel<2><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot2 *> (h->table), lk, reinterpret_cast<const u64 *> (d_keys), n, h->K); break;
		default: lookup_kmers_kernel<4><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot4 *> (h->table), lk, reinterpret_cast<const u64 *> (d_keys), n, h->K); break;
		}
	}
	CK (h, cudaGetLastError ());
	return SDTGPU_OK;
}

int sdtgpu_lookup_reads_device (sdtgpu_t *h, const uint8_t *d_packed, const uint32_t *d_lens, const uint8_t *d_nmask,
				uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes, sdtgpu_hit *d_out)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (n_reads && (!d_packed || !d_out))
		return fail (h, SDTGPU_EINVAL, "sdtgpu_lookup_reads_device: NULL buffer");
	int rc = lookup_prologue (h, d_out);
	if (rc)
		return rc;
	ReadBatch rb;
	if ((rc = make_batch (h, rb, d_packed, d_lens, d_nmask, n_reads, uniform_len, stride_bytes, 0)))
		return rc;
	if (n_reads == 0)
		return SDTGPU_OK;
	if ((rc = ensure_index (h)))
		return rc;
	// windows a read does not have are never written by the kernel: zero them first, unless every read has them all
	if (d_lens || std::min (uniform_len, (u32) h->max_read_len) != (u32) h->max_read_len)
		CK (h, cudaMemsetAsync (d_out, 0, n_reads * h->maxwin * sizeof (sdtgpu_hit), h->stream));
	return launch_insert<6> (h, rb, Bins (), make_lookup (h, d_out));
}

int sdtgpu_lookup_route (const sdtgpu_t *h, uint64_t out[12])
{
	if (!h || !out)
		return SDTGPU_EINVAL;
	const Route rt = make_route (h);
	const u32 rank = rt.kind == ROUTE_SKM ? h->skm_rank : (rt.kind == ROUTE_ONE ? 0 : h->owner_rank);
	const uint64_t v[12] = { rt.kind, rank, rt.world, (u64) h->K, (u64) h->W, rt.n_slices, rt.n_local, rt.m, rt.lo, rt.w,
				 (u64) h->deLowKmer, h->finalized ? 1u : 0u };
	memcpy (out, v, sizeof v);
	return SDTGPU_OK;
}

int sdtgpu_lookup_stage_kmers (sdtgpu_t *h, const uint64_t *d_keys, uint64_t n, void **d_queries, uint64_t *starts, uint64_t *counts)
{
	if (!h)
		return SDTGPU_EINVAL;
	if ((n && !d_keys) || !d_queries || !starts || !counts)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_lookup_stage_kmers: NULL buffer");
	int rc = route_prologue (h);
	if (rc)
		return rc;
	if ((uintptr_t) d_keys & 15)
		return fail (h, SDTGPU_EINVAL, "the key buffer must be 16-byte aligned");
	const Route rt = make_route (h);
	const u64 *keys = reinterpret_cast<const u64 *> (d_keys);
	auto launch = [&](bool scatter, const Stage &st) -> int {
		if (n == 0)
			return SDTGPU_OK;
		switch (h->W)
		{
		case 1: scatter ? launch_route_kmers_t<1, true> (h, keys, n, rt, st) : launch_route_kmers_t<1, false> (h, keys, n, rt, st); break;
		case 2: scatter ? launch_route_kmers_t<2, true> (h, keys, n, rt, st) : launch_route_kmers_t<2, false> (h, keys, n, rt, st); break;
		default: scatter ? launch_route_kmers_t<4, true> (h, keys, n, rt, st) : launch_route_kmers_t<4, false> (h, keys, n, rt, st); break;
		}
		CK (h, cudaGetLastError ());
		return SDTGPU_OK;
	};
	return route_stage (h, n, launch, d_queries, starts, counts);
}

int sdtgpu_lookup_stage_reads (sdtgpu_t *h, const uint8_t *d_packed, const uint32_t *d_lens, const uint8_t *d_nmask,
			       uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes,
			       void **d_queries, uint64_t *starts, uint64_t *counts)
{
	if (!h)
		return SDTGPU_EINVAL;
	if ((n_reads && !d_packed) || !d_queries || !starts || !counts)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_lookup_stage_reads: NULL buffer");
	int rc = route_prologue (h);
	if (rc)
		return rc;
	ReadBatch rb;
	if ((rc = make_batch (h, rb, d_packed, d_lens, d_nmask, n_reads, uniform_len, stride_bytes, 0)))
		return rc;
	const Route rt = make_route (h);
	const bool nmode = (h->flags & SDTGPU_F_NKMER) && rb.nmask;
	auto launch = [&](bool scatter, const Stage &st) -> int {
		if (n_reads == 0)
			return SDTGPU_OK;
		int r;
		switch (h->W)
		{
		case 1: r = nmode ? launch_route_reads_w<1, true> (h, rb, rt, scatter, st) : launch_route_reads_w<1, false> (h, rb, rt, scatter, st); break;
		case 2: r = nmode ? launch_route_reads_w<2, true> (h, rb, rt, scatter, st) : launch_route_reads_w<2, false> (h, rb, rt, scatter, st); break;
		default: r = nmode ? launch_route_reads_w<4, true> (h, rb, rt, scatter, st) : launch_route_reads_w<4, false> (h, rb, rt, scatter, st); break;
		}
		if (r)
			return r;
		CK (h, cudaGetLastError ());
		return SDTGPU_OK;
	};
	return route_stage (h, n_reads * h->maxwin, launch, d_queries, starts, counts);
}

int sdtgpu_lookup_answer_buffer (sdtgpu_t *h, uint64_t n, void **d_queries, sdtgpu_hit **d_replies)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (!d_queries || !d_replies)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_lookup_answer_buffer: NULL buffer");
	int rc = lookup_prologue (h, nullptr);
	if (rc)
		return rc;
	if ((rc = grow_device (h, (void **) &h->rt_aq, &h->rt_cap_aq, 0, std::max<u64> (n, 1) * 8 * h->W, "received lookups"))
	    || (rc = grow_device (h, (void **) &h->rt_ar, &h->rt_cap_ar, 0, std::max<u64> (n, 1) * sizeof (Hit), "lookup replies")))
		return rc;
	*d_queries = h->rt_aq;
	*d_replies = reinterpret_cast<sdtgpu_hit *> (h->rt_ar);
	return SDTGPU_OK;
}

int sdtgpu_lookup_answer (sdtgpu_t *h, uint64_t n)
{
	if (!h)
		return SDTGPU_EINVAL;
	int rc = lookup_prologue (h, nullptr);
	if (rc)
		return rc;
	if (n > h->rt_cap_aq / (8 * h->W) || n > h->rt_cap_ar / sizeof (Hit))
		return fail (h, SDTGPU_EINVAL, "sdtgpu_lookup_answer: more queries than sdtgpu_lookup_answer_buffer made room for");
	if (n == 0)
		return SDTGPU_OK;
	if ((rc = ensure_index (h)))
		return rc;
	const Lookup lk = make_lookup (h, reinterpret_cast<sdtgpu_hit *> (h->rt_ar));
	const unsigned grid = (unsigned) std::min<u64> ((n + BLOCK - 1) / BLOCK, (u64) h->sm_count * 16);
	{
		TimedLaunch tl (h, 7);
		switch (h->W)
		{
		case 1: route_answer_kernel<1><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot1 *> (h->table), lk, h->rt_aq, n); break;
		case 2: route_answer_kernel<2><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot2 *> (h->table), lk, h->rt_aq, n); break;
		default: route_answer_kernel<4><<<grid, BLOCK, 0, h->stream>>> (static_cast<const Slot4 *> (h->table), lk, h->rt_aq, n); break;
		}
	}
	CK (h, cudaGetLastError ());
	return SDTGPU_OK;
}

int sdtgpu_lookup_unstage_buffer (sdtgpu_t *h, sdtgpu_hit **d_back)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (!d_back)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_lookup_unstage_buffer: NULL buffer");
	int rc = lookup_prologue (h, nullptr);
	if (rc)
		return rc;
	if (!h->rt_staged)
		return fail (h, SDTGPU_ESTATE, "sdtgpu_lookup_unstage_buffer without a stage");
	if ((rc = grow_device (h, (void **) &h->rt_back, &h->rt_cap_back, 0, std::max<u64> (h->rt_n, 1) * sizeof (Hit), "lookup replies")))
		return rc;
	*d_back = reinterpret_cast<sdtgpu_hit *> (h->rt_back);
	return SDTGPU_OK;
}

int sdtgpu_lookup_unstage (sdtgpu_t *h, sdtgpu_hit *d_out)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (!d_out && (!h->rt_staged || h->rt_out))
		return fail (h, SDTGPU_EINVAL, "sdtgpu_lookup_unstage: NULL buffer");
	int rc = lookup_prologue (h, d_out);
	if (rc)
		return rc;
	if (!h->rt_staged)
		return fail (h, SDTGPU_ESTATE, "sdtgpu_lookup_unstage without a stage");
	if (h->rt_n > h->rt_cap_back / sizeof (Hit))
		return fail (h, SDTGPU_ESTATE, "sdtgpu_lookup_unstage: the replies need sdtgpu_lookup_unstage_buffer first");
	h->rt_staged = false;
	if (h->rt_n < h->rt_out)	// malformed keys, windows a read does not have: all zero, as the single-GPU lookup writes them
		CK (h, cudaMemsetAsync (d_out, 0, h->rt_out * sizeof (sdtgpu_hit), h->stream));
	if (h->rt_n)
	{
		const unsigned grid = (unsigned) std::min<u64> ((h->rt_n + BLOCK - 1) / BLOCK, (u64) h->sm_count * 16);
		TimedLaunch tl (h, 7);
		route_unstage_kernel<<<grid, BLOCK, 0, h->stream>>> (h->rt_back, h->rt_tag, h->rt_n, reinterpret_cast<Hit *> (d_out));
	}
	CK (h, cudaGetLastError ());
	return SDTGPU_OK;
}

int sdtgpu_edges_build (sdtgpu_t *h, uint64_t out[8], double *ms)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (!out || !ms)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_edges_build: NULL output");
	if (make_route (h).kind != ROUTE_ONE)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_edges_build: the handle holds one rank's share of a sharded table");
	int rc = lookup_prologue (h, nullptr);
	if (rc)
		return rc;
	if ((rc = ensure_index (h)))
		return rc;
	switch (h->W)
	{
	case 1: return edges_build_t<1> (h, out, ms);
	case 2: return edges_build_t<2> (h, out, ms);
	default: return edges_build_t<4> (h, out, ms);
	}
}

int sdtgpu_edges_buffers (sdtgpu_t *h, const sdtgpu_edge **d_edges, const uint8_t **d_seq)
{
	if (!h)
		return SDTGPU_EINVAL;
	if (!d_edges || !d_seq)
		return fail (h, SDTGPU_EINVAL, "sdtgpu_edges_buffers: NULL output");
	if (!h->ed_built)
		return fail (h, SDTGPU_ESTATE, "sdtgpu_edges_buffers before sdtgpu_edges_build");
	*d_edges = static_cast<const sdtgpu_edge *> (h->ed[ED_EDGES]);
	*d_seq = static_cast<const uint8_t *> (h->ed[ED_SEQ]);
	return SDTGPU_OK;
}

int sdtgpu_host_alloc (void **out, size_t bytes)
{
	if (!out)
		return SDTGPU_EINVAL;
	*out = nullptr;
	return cudaMallocHost (out, bytes ? bytes : 1) == cudaSuccess ? SDTGPU_OK : SDTGPU_ENOMEM;
}

void sdtgpu_host_free (void *p)
{
	if (p)
		cudaFreeHost (p);
}

static int collect_times (sdtgpu *h)
{
	CK (h, cudaSetDevice (h->device));
	CK (h, cudaStreamSynchronize (h->copy_stream));
	CK (h, cudaStreamSynchronize (h->stream));
	for (auto &p : h->timing)
	{
		float ms = 0;
		CK (h, cudaEventElapsedTime (&ms, p.e0, p.e1));
		h->cat_ms[p.cat] += ms;
		h->cat_launches[p.cat]++;
		h->ev_pool.push_back (p.e0);
		h->ev_pool.push_back (p.e1);
	}
	h->timing.clear ();
	return SDTGPU_OK;
}

int sdtgpu_kernel_time (sdtgpu_t *h, int reset, double *insert_ms, uint64_t *insert_launches, uint64_t *all_launches)
{
	if (!h)
		return SDTGPU_EINVAL;
	int rc = collect_times (h);
	if (rc)
		return rc;
	if (insert_ms) *insert_ms = h->cat_ms[0];
	if (insert_launches) *insert_launches = h->cat_launches[0];
	if (all_launches) *all_launches = h->all_launches;
	if (reset)
	{
		for (int i = 0; i < N_CAT; i++) { h->cat_ms[i] = 0; h->cat_launches[i] = 0; }
		h->all_launches = 0;
	}
	return SDTGPU_OK;
}

int sdtgpu_kernel_times (sdtgpu_t *h, int reset, double ms[3], uint64_t launches[3])
{
	if (!h)
		return SDTGPU_EINVAL;
	int rc = collect_times (h);
	if (rc)
		return rc;
	for (int i = 0; i < 3; i++)
	{
		if (ms) ms[i] = h->cat_ms[i];
		if (launches) launches[i] = h->cat_launches[i];
	}
	if (reset)
	{
		for (int i = 0; i < N_CAT; i++) { h->cat_ms[i] = 0; h->cat_launches[i] = 0; }
		h->all_launches = 0;
	}
	return SDTGPU_OK;
}

int sdtgpu_phase_times (sdtgpu_t *h, int reset, double ms[8], uint64_t launches[8])
{
	if (!h)
		return SDTGPU_EINVAL;
	int rc = collect_times (h);
	if (rc)
		return rc;
	for (int i = 0; i < N_CAT; i++)
	{
		if (ms) ms[i] = h->cat_ms[i];
		if (launches) launches[i] = h->cat_launches[i];
	}
	if (reset)
	{
		for (int i = 0; i < N_CAT; i++) { h->cat_ms[i] = 0; h->cat_launches[i] = 0; }
		h->all_launches = 0;
	}
	return SDTGPU_OK;
}

int sdtgpu_debug_prof (uint64_t out[8], int reset)
{
#ifdef SDT_BUILD_PROF
	unsigned long long v[8];
	if (cudaMemcpyFromSymbol (v, g_build_prof, sizeof v) != cudaSuccess)
		return SDTGPU_ECUDA;
	for (int i = 0; i < 8; i++)
		out[i] = v[i];
	if (reset)
	{
		memset (v, 0, sizeof v);
		cudaMemcpyToSymbol (g_build_prof, v, sizeof v);
	}
	return SDTGPU_OK;
#else
	for (int i = 0; i < 8; i++)
		out[i] = 0;
	(void) reset;
	return SDTGPU_OK;
#endif
}

int sdtgpu_slice_geometry (const sdtgpu_t *h, uint64_t out[12])
{
	if (!h || !out)
		return SDTGPU_EINVAL;
	if (!h->sliced)
		return SDTGPU_ESTATE;
	out[0] = h->geom.n_slices; out[1] = h->geom.slice_slots; out[2] = h->geom.m; out[3] = h->geom.w;
	out[4] = 4 * (uint64_t) h->geom.recw; out[5] = h->n_records; out[6] = h->n_store; out[7] = h->n_retried;
	out[8] = h->n_merged; out[9] = h->n_items; out[10] = h->n_reemit; out[11] = h->n_alloc;
	return SDTGPU_OK;
}

}	// extern "C"
