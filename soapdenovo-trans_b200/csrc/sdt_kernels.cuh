// sdt_kernels.cuh — the sm_100a kernels of the pregraph hashing path.
//
//   insert_reads_kernel<W, NMODE, MODE>
//       chop (prlHashReads.c:164-310) fused with put_kmerset (newhash.c:411-462): persistent CTAs
//       stage tiles of 2-bit packed reads into shared memory with 16-byte vector loads and walk the
//       tile's flattened (read, offset) windows.  What happens to a window depends on MODE:
//         5  the default insert: windows are chopped into a shared-memory queue of (key, meta)
//            records, optionally filtered by owner rank (replicated-reads multi-GPU sharding), and
//            the queue is drained with every lane issuing an upsert;
//         0  upsert straight from the chop loop (kept for A/B, SDTGPU_NO_QUEUE=1);
//         1  send side of the record exchange: records into per-owner bins;
//         4  per reference set, the largest instance ordinal of the batch (hand-back helper);
//         6  lookup: each window's canonical key in the finalized table's index (sdt_lookup.cuh), one
//            sdtgpu_hit per window at read * maxwin + window.
//   insert_records_kernel  receive side of the record exchange.
//   init / rehash / finalize / export / checksum kernels: table maintenance, the post-pass
//       (thread_delow prlHashReads.c:844-887, thread_mark :911-967) and verification.
#pragma once
#include "sdt_device.cuh"
#include "sdt_lookup.cuh"

namespace sdt {

static constexpr int TILE_PAD = 8;	// u32 words of padding on both sides of the staged tile
static constexpr int BLOCK = 256;
static constexpr int MAX_TILE_READS = 256;
static constexpr u32 QUEUE_CAP = 1024;	// records in the owned-instance queue (MODE 5); tuned on C2: 512..1536 equal, 3072+ slower

struct ReadBatch
{
	const uint8_t *packed;	// n_reads x stride_bytes, tight-string packed
	const u32 *lens;	// or nullptr: uniform_len
	const uint8_t *nmask;	// or nullptr; n_reads x mask_stride bytes, 1 bit per base
	u64 n_reads;
	u64 first_read_ordinal;
	u32 uniform_len, stride_bytes, mask_stride;
	u32 tile_reads;		// reads per shared-memory tile (multiple of 4, <= MAX_TILE_READS)
	int K;
	u32 max_read_len, maxwin;	// maxwin = max_read_len - K + 1 (ordinal = read * maxwin + window)
	u32 queue_windows, queue_cap;	// MODE 5: windows chopped per drain of the owned-instance queue; its capacity (records)
	u32 owner_rank, owner_ranks;	// owner_ranks > 1: insert only instances whose owner_of (mix(key)) == owner_rank
};

struct Counters
{
	u64 n_nodes;		// distinct keys in the table
	u64 n_instances;	// windows processed ("kmer in reads")
	u64 overflow;		// reserved
	u64 n_removed, n_linear;	// finalize
	u64 export_cursor;
	u64 pad[2];
	unsigned long long freq[257];	// kmerFreq histogram (thread_mark, prlHashReads.c:946-954)
};

struct Bins
{
	u64 *records;		// MODE 1: n_ranks x capacity x (W + 1) u64
	u64 *counts;		// per bin: fill (MODE 1), last ordinal + 1 (MODE 4)
	u64 capacity;		// MODE 1: records per bin; MODE 4: key_words of the reference build
	u32 n_ranks;		// bins: owner ranks (MODE 1), reference sets (MODE 4)
};

__device__ __forceinline__ u32 bswap32 (u32 x) { return __byte_perm (x, 0, 0x0123); }

__device__ __forceinline__ uint4 ldg_stream (const uint4 *p)
{
	uint4 v;
	asm volatile ("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
	return v;
}

// ---- hash_kmer restated (hashFunction.c:83-122): CRC-32 table arithmetic carried in a signed int
// (arithmetic >> 8), over the raw bytes of the reference's Kmer object (8 * key_words bytes, words
// in declaration order, each little endian), masked to 24 bits.  Its only use in the reference is
// owner set = hash % thrd_num (prlHashReads.c:81); here it is needed at hand-back time only.
__constant__ int c_crc[256];

__host__ __device__ inline u32 hash_kmer_impl (const uint64_t *key, int key_words, const int *tab)
{
	int crc = ~0;
	for (int w = 4 - key_words; w < 4; w++)
		for (int b = 0; b < 8; b++)
		{
			const int byte = (int) (signed char) (unsigned char) (key[w] >> (8 * b));
			crc = tab[(crc ^ byte) & 0xff] ^ (crc >> 8);
		}
	crc = ~crc;
	return (u32) crc & 0x00ffffffu;
}

// one window -> canonical key and the link bases in the stored orientation (SURVEY.md §8a-2);
// *flipped (if given): the canonical key is the reverse complement of the window's forward k-mer
template <int W, bool NMODE>
__device__ __forceinline__ void chop_window (const u32 *rd, const u32 *mk, int len, int j, int K,
					     Key<W> &key, u32 &left, u32 &right, bool *flipped = nullptr)
{
	Key<W> f, rc;
	extract_fwd<W> (rd, j + K, K, f);
	revcomp<W> (f, K, rc);
	u32 prev = 4, next = 4;
	if (j > 0)
		prev = base_at (rd, j - 1);
	if (j + K < len)
		next = base_at (rd, j + K);
	if constexpr (NMODE)
	{	// -n: a window that holds an N becomes key 0 without links; an N neighbour is no link
		bool bad = false;
		for (int q = j >> 5; q <= (j + K - 1) >> 5; q++)
		{
			u32 m = mk[q];
			const int lo = q << 5;
			if (j > lo)
				m &= 0xFFFFFFFFu >> (j - lo);
			if (j + K < lo + 32)
				m &= 0xFFFFFFFFu << (lo + 32 - (j + K));
			bad |= (m != 0);
		}
		if (j > 0 && ((mk[(j - 1) >> 5] >> (31 - ((j - 1) & 31))) & 1))
			prev = 4;
		if (j + K < len && ((mk[(j + K) >> 5] >> (31 - ((j + K) & 31))) & 1))
			next = 4;
		if (bad)
		{
#pragma unroll
			for (int i = 0; i < W; i++)
				key.w[i] = 0;
			left = right = 4;
			if (flipped)
				*flipped = false;
			return;
		}
	}
	const bool fwd = key_less<W> (f, rc);
	if (flipped)
		*flipped = !fwd;
	if (fwd)
	{
		key = f;
		left = prev;
		right = next;
	}
	else
	{
		key = rc;
		left = next < 4 ? (next ^ 2u) : 4u;
		right = prev < 4 ? (prev ^ 2u) : 4u;
	}
}

template <int W> __device__ __forceinline__ void store_record (u64 *rec, const Key<W> &key, u32 left, u32 right, u64 ord)
{
	const u64 meta = (ord << 8) | (left << 4) | right;
	if constexpr (W == 1)
		*reinterpret_cast<ulonglong2 *> (rec) = make_ulonglong2 (key.w[0], meta);
	else
	{
#pragma unroll
		for (int i = 0; i < W; i++)
			rec[i] = key.w[i];
		rec[W] = meta;
	}
}

template <int W> __device__ __forceinline__ void load_record (const u64 *rec, Key<W> &key, u64 &meta)
{
	if constexpr (W == 1)
	{
		const ulonglong2 v = *reinterpret_cast<const ulonglong2 *> (rec);
		key.w[0] = v.x;
		meta = v.y;
	}
	else
	{
#pragma unroll
		for (int q = 0; q < W; q++)
			key.w[q] = rec[q];
		meta = rec[W];
	}
}

// Note on the per-tile __syncthreads(): ncu attributes ~35 % of warp stall samples to it, but a
// warp-autonomous variant (each warp staging its own 32-read tile, no block barrier at all) measured
// 4 % SLOWER on C2 (13.5 vs 14.1 G instances/s): the kernel is bound by L2 request rate to cold
// lines, warps parked at the barrier are not what limits it.
template <int W, bool NMODE, int MODE>
__global__ void __launch_bounds__ (BLOCK)
insert_reads_kernel (typename SlotOf<W>::type *table, u64 cap, ReadBatch rb, Bins bins, Counters *ctr, Lookup lk)
{
	extern __shared__ __align__(16) u32 smem[];
	const int tid = threadIdx.x;
	const u32 sw = rb.stride_bytes >> 2;			// u32 words per read
	const u32 mw = NMODE ? ((rb.mask_stride + 3) >> 2) : 0;	// mask words per read
	u32 *tile = smem + TILE_PAD;
	u32 *prefix = smem + TILE_PAD + rb.tile_reads * sw + TILE_PAD;	// tile_reads + 1 entries
	u32 *mtile = prefix + rb.tile_reads + 4;
	u32 *hist = mtile + rb.tile_reads * mw;	// MODE 1: bins.n_ranks counters + u64 bases behind them
	u64 *base = reinterpret_cast<u64 *> (hist + ((bins.n_ranks + 1) & ~1u));
	__shared__ u32 warp_sums[BLOCK / 32];
	const u64 n_tiles = (rb.n_reads + rb.tile_reads - 1) / rb.tile_reads;
	const int K = rb.K;
	u32 created = 0;
	u64 instances = 0, owned = 0;
	__shared__ u32 q_count;
	u64 *queue = reinterpret_cast<u64 *> (hist);	// MODE 5: QUEUE_WINDOWS records of (W + 1) u64
	if (MODE == 5 && tid == 0)
		q_count = 0;

	if (tid < TILE_PAD)
	{
		smem[tid] = 0;
		smem[TILE_PAD + rb.tile_reads * sw + tid] = 0;
	}
	if (MODE == 4)
		for (u32 b = tid; b < 2 * bins.n_ranks; b += BLOCK)
			hist[b] = 0;
	else if (MODE != 0)
		for (u32 b = tid; b < bins.n_ranks; b += BLOCK)
			hist[b] = 0;

	for (u64 t = blockIdx.x; t < n_tiles; t += gridDim.x)
	{
		const u64 r0 = t * rb.tile_reads;
		const u32 nr = (u32) min ((u64) rb.tile_reads, rb.n_reads - r0);
		// ---- stage the tile: coalesced 16-byte loads, byte-swapped so that base order == bit order
		{
			const u32 words = nr * sw;
			const uint4 *src = reinterpret_cast<const uint4 *> (rb.packed + r0 * rb.stride_bytes);
			const u32 nvec = words >> 2;
			for (u32 v = tid; v < nvec; v += BLOCK)
			{
				uint4 x = ldg_stream (src + v);
				tile[4 * v + 0] = bswap32 (x.x);
				tile[4 * v + 1] = bswap32 (x.y);
				tile[4 * v + 2] = bswap32 (x.z);
				tile[4 * v + 3] = bswap32 (x.w);
			}
			const u32 *src32 = reinterpret_cast<const u32 *> (src);
			for (u32 v = 4 * nvec + tid; v < words; v += BLOCK)
				tile[v] = bswap32 (__ldg (src32 + v));
			if constexpr (NMODE)
			{
				const uint8_t *msrc = rb.nmask + r0 * rb.mask_stride;
				for (u32 v = tid; v < nr * mw; v += BLOCK)
				{
					const u32 rr = v / mw, q = v - rr * mw;
					u32 x = 0;
					for (u32 b = 0; b < 4; b++)
					{
						const u32 byte = 4 * q + b;
						if (byte < rb.mask_stride)
							x |= (u32) msrc[(u64) rr * rb.mask_stride + byte] << (24 - 8 * b);
					}
					mtile[v] = x;
				}
			}
		}
		// ---- windows per read -> exclusive prefix (the reference's indexArray, prlHashReads.c:516-518)
		u32 total;
		const bool uniform = (rb.lens == nullptr);
		u32 nwin_u = 0;
		if (uniform)
		{
			const u32 len = min (rb.uniform_len, rb.max_read_len);
			nwin_u = len >= (u32) K + 1 ? len - K + 1 : 0;	// reads shorter than K+1 are skipped (:507)
			total = nwin_u * nr;
		}
		else
		{
			u32 c = 0;
			if ((u32) tid < nr)
			{
				const u32 len = min (rb.lens[r0 + tid], rb.max_read_len);
				c = len >= (u32) K + 1 ? len - K + 1 : 0;
			}
			u32 x = c;
#pragma unroll
			for (int d = 1; d < 32; d <<= 1)
			{
				const u32 y = __shfl_up_sync (0xFFFFFFFFu, x, d);
				if ((tid & 31) >= d)
					x += y;
			}
			if ((tid & 31) == 31)
				warp_sums[tid >> 5] = x;
			__syncthreads ();
			u32 off = 0;
			for (int w = 0; w < (tid >> 5); w++)
				off += warp_sums[w];
			if ((u32) tid < rb.tile_reads)
				prefix[tid] = off + x - c;
			if (tid == BLOCK - 1)
				prefix[rb.tile_reads] = off + x;
			__syncthreads ();
			total = prefix[rb.tile_reads];
		}
		__syncthreads ();
		instances += (tid == 0) ? total : 0;

		// MODE 1 walks the tile twice: sweep 0 counts the tile's records per bin, ONE global atomic per
		// non-empty bin then reserves their space, sweep 1 writes the records (chopping twice is cheap;
		// a contended global cursor atomic per warp was 3x slower, profiles/r1_multi_gpu.md)
		for (u32 chunk0 = 0; chunk0 < total; chunk0 += (MODE == 5 ? rb.queue_windows : total))
		{
		const u32 chunk1 = MODE == 5 ? min (total, chunk0 + rb.queue_windows) : total;
		for (int sweep = (MODE == 1 ? 0 : 1); sweep < 2; sweep++)
		{
		for (u32 w = chunk0 + tid; w < chunk1; w += BLOCK)
		{
			u32 r, j, len;
			if (uniform)
			{
				r = w / nwin_u;
				j = w - r * nwin_u;
				len = nwin_u + K - 1;
			}
			else
			{	// largest r with prefix[r] <= w
				u32 lo = 0, hi = nr - 1;
				while (lo < hi)
				{
					const u32 mid = (lo + hi + 1) >> 1;
					if (prefix[mid] <= w)
						lo = mid;
					else
						hi = mid - 1;
				}
				r = lo;
				j = w - prefix[r];
				len = prefix[r + 1] - prefix[r] + K - 1;
			}
			Key<W> key;
			u32 left, right;
			bool flipped;
			chop_window<W, NMODE> (tile + r * sw, NMODE ? (mtile + r * mw) : nullptr, (int) len, (int) j, K, key, left, right, MODE == 6 ? &flipped : nullptr);
			const u64 ord = (rb.first_read_ordinal + r0 + r) * rb.maxwin + j;
			if (MODE == 6)
				store_hit (lk.out + (r0 + r) * (u64) rb.maxwin + j, index_probe<W> (table, lk, key, flipped ? HIT_RC : 0u));
			else if (MODE == 0)
				created += Table<W>::upsert (table, cap, key, left, right, ord);
			else if (MODE == 5)
			{	// replicated-reads sharding: every rank chops every read and keeps the k-mers it owns (the
				// reference's own scheme, prlHashReads.c:79-88, with GPUs in place of threads).  Owned
				// instances are first compacted into a shared-memory queue so that the upserts below run
				// with full warps (filtering in place left 1 lane in n_ranks busy per memory round trip).
				if (rb.owner_ranks <= 1 || owner_of (key_hash<W> (key), rb.owner_ranks) == rb.owner_rank)
				{
					const u32 pos = atomicAdd (&q_count, 1u);
					if (pos < rb.queue_cap)
						store_record<W> (queue + (u64) pos * (W + 1), key, left, right, ord);
					else	// more owned instances in this chunk than expected (skewed owners): insert in place
						created += Table<W>::upsert (table, cap, key, left, right, ord);
				}
			}
			else if (MODE == 1)
			{	// send side of the exchange: bin = owner rank, fixed capacity per bin
				const u32 b = owner_of (key_hash<W> (key), bins.n_ranks);
				if (sweep == 0)
					atomicAdd (&hist[b], 1u);
				else
				{
					const u64 pos = base[b] + atomicAdd (&hist[b], 1u);
					if (pos < bins.capacity)	// else: the host sees counts[b] > capacity and reports it
						store_record<W> (bins.records + ((u64) b * bins.capacity + pos) * (W + 1), key, left, right, ord);
				}
			}
			else if (MODE == 4)
			{	// per reference set: the largest instance ordinal (bins.n_ranks = thrd_num, bins.capacity = key_words)
				uint64_t k4[4] = { 0, 0, 0, 0 };
#pragma unroll
				for (int q = 0; q < W; q++)
					k4[4 - W + q] = key.w[q];
				const u32 set = hash_kmer_impl (k4, (int) bins.capacity, c_crc) % bins.n_ranks;
				u64 *smax = reinterpret_cast<u64 *> (hist);
				if (ord + 1 > smax[set])
					atomicMax (&smax[set], ord + 1);	// stored +1 so that 0 means "no instance"
			}
		}
		if (MODE == 1)
		{
			__syncthreads ();
			if (sweep == 0)
			{
				for (u32 b = tid; b < bins.n_ranks; b += BLOCK)
				{
					const u32 c = hist[b];
					if (c)
					{
						base[b] = atomicAdd (bins.counts + b, (u64) c);
						hist[b] = 0;
					}
				}
				__syncthreads ();
			}
			else
				for (u32 b = tid; b < bins.n_ranks; b += BLOCK)
					hist[b] = 0;
		}
		}
		if (MODE == 5)
		{	// drain the queue of owned instances with every lane busy
			__syncthreads ();
			const u32 nq_all = q_count, nq = min (nq_all, rb.queue_cap);
			__syncthreads ();
			if (tid == 0)
			{
				q_count = 0;
				owned += nq_all;
			}
			for (u32 i = tid; i < nq; i += BLOCK)
			{
				Key<W> key;
				u64 meta;
				load_record<W> (queue + (u64) i * (W + 1), key, meta);
				created += Table<W>::upsert (table, cap, key, (u32) (meta >> 4) & 15u, (u32) meta & 15u, meta >> 8);
			}
			__syncthreads ();
		}
		}
		__syncthreads ();	// the tile is overwritten by the next iteration
	}
	if (MODE == 4)
	{
		__syncthreads ();
		const u64 *smax = reinterpret_cast<const u64 *> (hist);
		for (u32 b = tid; b < bins.n_ranks; b += BLOCK)
			if (smax[b])
				atomicMax (bins.counts + b, smax[b]);
	}
	// ---- counters: one atomic per warp
#pragma unroll
	for (int d = 16; d > 0; d >>= 1)
		created += __shfl_down_sync (0xFFFFFFFFu, created, d);
	if ((tid & 31) == 0 && created)
		atomicAdd (&ctr->n_nodes, (u64) created);
	// instances are counted by the rank that inserts them
	if (MODE == 0 && tid == 0 && instances)
		atomicAdd (&ctr->n_instances, instances);
	if (MODE == 5 && tid == 0 && owned)
		atomicAdd (&ctr->n_instances, owned);
}

template <int W>
__global__ void __launch_bounds__ (BLOCK)
insert_records_kernel (typename SlotOf<W>::type *table, u64 cap, const u64 *records, u64 n, Counters *ctr)
{
	u32 created = 0;
	for (u64 i = blockIdx.x * (u64) BLOCK + threadIdx.x; i < n; i += (u64) gridDim.x * BLOCK)
	{
		Key<W> key;
		u64 meta;
		const u64 *rec = records + i * (W + 1);
		if constexpr (W == 1)
		{
			const ulonglong2 v = *reinterpret_cast<const ulonglong2 *> (rec);
			key.w[0] = v.x;
			meta = v.y;
		}
		else
		{
#pragma unroll
			for (int q = 0; q < W; q++)
				key.w[q] = rec[q];
			meta = rec[W];
		}
		created += Table<W>::upsert (table, cap, key, (u32) (meta >> 4) & 15u, (u32) meta & 15u, meta >> 8);
	}
#pragma unroll
	for (int d = 16; d > 0; d >>= 1)
		created += __shfl_down_sync (0xFFFFFFFFu, created, d);
	if ((threadIdx.x & 31) == 0)
	{
		if (created)
			atomicAdd (&ctr->n_nodes, (u64) created);
	}
	if (blockIdx.x == 0 && threadIdx.x == 0)
		atomicAdd (&ctr->n_instances, n);
}

// ------------------------------------------------------------------------------------------------
// slot accessors shared by init / rehash / finalize / export
template <int W> struct SlotIO
{
	typedef typename SlotOf<W>::type S;
	static __device__ __forceinline__ void init (S *s)
	{
		uint4 *q = reinterpret_cast<uint4 *> (s);
		const uint4 ones = make_uint4 (~0u, ~0u, ~0u, ~0u);
		const uint4 pay = make_uint4 ((u32) PAYLOAD0_INIT, (u32) (PAYLOAD0_INIT >> 32), 0, 0);
		if constexpr (W == 4)
		{
			q[0] = ones; q[1] = ones; q[2] = pay; q[3] = make_uint4 (0, 0, 0, 0);
		}
		else
		{
			q[0] = ones; q[1] = pay;
		}
	}
	static __device__ __forceinline__ const u64 *keyp (const S *s) { return reinterpret_cast<const u64 *> (s); }
	static __device__ __forceinline__ bool occupied (const S *s)
	{
		if constexpr (W == 1)
			return keyp (s)[0] != EMPTY64;
		else
			return !(keyp (s)[0] == EMPTY64 && keyp (s)[1] == EMPTY64);
	}
	static __device__ __forceinline__ void get (const S *s, Key<W> &k, u32 &L, u32 &R, u32 &count, u64 &ord)
	{
#pragma unroll
		for (int i = 0; i < W; i++)
			k.w[i] = keyp (s)[i];
		L = (u32) (s->p.ordL & 0xFFFFFF); R = s->p.R & 0xFFFFFF; count = s->p.count; ord = s->p.ordL >> 24;
	}
	static __device__ __forceinline__ void set_links (S *s, u32 L, u32 R) { s->p.ordL = (s->p.ordL & ~0xFFFFFFull) | L; s->p.R = R; }
	// rehash only: keys are unique there, so claiming the first 8 / 16 bytes is enough
	static __device__ __forceinline__ bool claim (S *s, const Key<W> &k)
	{
		if constexpr (W == 1)
			return atomicCAS (reinterpret_cast<u64 *> (s), EMPTY64, k.w[0]) == EMPTY64;
		else
		{
			u64 a, b;
			return cas128 (s, EMPTY64, EMPTY64, k.w[0], k.w[1], a, b);
		}
	}
	static __device__ __forceinline__ void put (S *s, const Key<W> &k, u32 L, u32 R, u32 count, u64 ord)
	{
		if constexpr (W == 4)
		{
			s->key[2] = k.w[2]; s->key[3] = k.w[3];
		}
		s->p.ordL = (ord << 24) | L; s->p.R = R; s->p.count = count;
	}
};

template <int W>
__global__ void __launch_bounds__ (BLOCK)
init_table_kernel (typename SlotOf<W>::type *table, u64 cap)
{
	for (u64 i = blockIdx.x * (u64) BLOCK + threadIdx.x; i < cap; i += (u64) gridDim.x * BLOCK)
		SlotIO<W>::init (table + i);
}

// move every node of `old` into the (larger, empty) table `neu`
template <int W>
__global__ void __launch_bounds__ (BLOCK)
rehash_kernel (const typename SlotOf<W>::type *old, u64 old_cap, typename SlotOf<W>::type *neu, u64 cap)
{
	for (u64 i = blockIdx.x * (u64) BLOCK + threadIdx.x; i < old_cap; i += (u64) gridDim.x * BLOCK)
	{
		if (!SlotIO<W>::occupied (old + i))
			continue;
		Key<W> k;
		u32 L, R, count;
		u64 ord;
		SlotIO<W>::get (old + i, k, L, R, count, ord);
		u64 idx = slot_of (key_hash<W> (k), cap);
		while (!SlotIO<W>::claim (neu + idx, k))
			if (++idx == cap)
				idx = 0;
		SlotIO<W>::put (neu + idx, k, L, R, count, ord);
	}
}

// thread_delow (prlHashReads.c:844-887) + thread_mark (:911-967) in one streaming pass
template <int W>
__global__ void __launch_bounds__ (BLOCK)
finalize_kernel (typename SlotOf<W>::type *table, u64 cap, int deLowKmer, Counters *ctr)
{
	__shared__ u32 hist[257];
	__shared__ u32 s_removed, s_linear;
	for (int i = threadIdx.x; i < 257; i += BLOCK)
		hist[i] = 0;
	if (threadIdx.x == 0)
		s_removed = s_linear = 0;
	__syncthreads ();
	for (u64 i = blockIdx.x * (u64) BLOCK + threadIdx.x; i < cap; i += (u64) gridDim.x * BLOCK)
	{
		if (!SlotIO<W>::occupied (table + i))
			continue;
		Key<W> k;
		u32 L, R, count;
		u64 ord;
		SlotIO<W>::get (table + i, k, L, R, count, ord);
		if (deLowKmer > 0)
		{
			u32 nL = L, nR = R;
#pragma unroll
			for (int b = 0; b < 4; b++)
			{
				const u32 cl = (L >> (6 * b)) & 63, cr = (R >> (6 * b)) & 63;
				if (cl > 0 && cl <= (u32) deLowKmer)
					nL &= ~(63u << (6 * b));
				if (cr > 0 && cr <= (u32) deLowKmer)
					nR &= ~(63u << (6 * b));
			}
			if (nL != L || nR != R)
				SlotIO<W>::set_links (table + i, nL, nR);
			L = nL;
			R = nR;
			if (L == 0 && R == 0)
				atomicAdd (&s_removed, 1u);
		}
		u32 in_num = 0, out_num = 0, l_cvg = 0, r_cvg = 0;
#pragma unroll
		for (int b = 0; b < 4; b++)
		{
			const u32 cl = (L >> (6 * b)) & 63, cr = (R >> (6 * b)) & 63;
			in_num += cl > 0; l_cvg += cl;
			out_num += cr > 0; r_cvg += cr;
		}
		atomicAdd (&hist[count == 1 ? 1 : max (l_cvg, r_cvg)], 1u);	// single == (count == 1)
		if (in_num == 1 && out_num == 1)
			atomicAdd (&s_linear, 1u);
	}
	__syncthreads ();
	for (int i = threadIdx.x; i < 257; i += BLOCK)
		if (hist[i])
			atomicAdd (&ctr->freq[i], (unsigned long long) hist[i]);
	if (threadIdx.x == 0)
	{
		if (s_removed)
			atomicAdd (&ctr->n_removed, (u64) s_removed);
		if (s_linear)
			atomicAdd (&ctr->n_linear, (u64) s_linear);
	}
}

// Order-independent fingerprint of the table: sums over all nodes of a 64-bit mix of
// (key, count, l_links, r_links) and of a few plain totals.  Any two runs that hold the same
// multiset of nodes — whatever the insertion order, batching, capacity or sharding — agree on it;
// the oracle computes the same sums on the CPU (oracle.table_checksum).
template <int W>
__global__ void __launch_bounds__ (BLOCK)
checksum_kernel (const typename SlotOf<W>::type *table, u64 cap, u64 *out /* [4] */)
{
	u64 h = 0, c = 0, l = 0, n = 0;
	for (u64 i = blockIdx.x * (u64) BLOCK + threadIdx.x; i < cap; i += (u64) gridDim.x * BLOCK)
	{
		if (!SlotIO<W>::occupied (table + i))
			continue;
		Key<W> k;
		u32 L, R, count;
		u64 ord;
		SlotIO<W>::get (table + i, k, L, R, count, ord);
		u64 x = 0x9E3779B97F4A7C15ull;
#pragma unroll
		for (int q = 0; q < W; q++)
			x = fmix64 (x ^ k.w[q]);
		x = fmix64 (x ^ (((u64) count << 32) | L));
		x = fmix64 (x ^ R);
		h += x;
		c += count;
		l += (u64) __popc (L) + ((u64) __popc (R) << 32);
		n += 1;
	}
#pragma unroll
	for (int d = 16; d > 0; d >>= 1)
	{
		h += __shfl_down_sync (0xFFFFFFFFu, h, d);
		c += __shfl_down_sync (0xFFFFFFFFu, c, d);
		l += __shfl_down_sync (0xFFFFFFFFu, l, d);
		n += __shfl_down_sync (0xFFFFFFFFu, n, d);
	}
	if ((threadIdx.x & 31) == 0)
	{
		atomicAdd (out + 0, h);
		atomicAdd (out + 1, c);
		atomicAdd (out + 2, l);
		atomicAdd (out + 3, n);
	}
}

}	// namespace sdt
