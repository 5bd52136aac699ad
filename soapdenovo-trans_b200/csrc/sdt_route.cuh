// sdt_route.cuh — lookups routed to the rank that owns each k-mer (sdtgpu_lookup_stage_* / _answer / _unstage).
//
// On several GPUs every rank holds a disjoint share of the table.  A routed lookup stages each query in the region
// of the rank that owns its canonical key, the owner answers it with index_probe (sdt_lookup.cuh) and the reply
// goes back to the position the single-GPU lookup would have written.  The owner must be computed exactly as the
// insert side shards the keys; the three shardings are restated here in one device function, route_owner:
//
//   ROUTE_SKM     sliced build, super-k-mer exchange (sdtgpu_skm_set_world): slices are dealt in contiguous
//                 ranges, slice / n_local (sdtgpu_skm_import, lo = skm_rank * n_local)
//   ROUTE_SLICED  sliced build, sdtgpu_set_owner: slice % world (skm_emit_kernel, step 3)
//   ROUTE_HASHED  single-pass insert, sdtgpu_set_owner (replicated reads) or the record exchange: owner_of (key_hash)
//                 (insert_reads_kernel MODE 5 and MODE 1)
//   ROUTE_ONE     one GPU: everything is rank 0's
//
// The slice of a canonical key is slice_of_min of its minimizer value: the smallest mmer_hash (min (f, rc (f)))
// over the central w m-mers of the key, positions lo .. lo + w - 1 (skm_emit_kernel, steps 1-2).  It is computed
// from the key's words alone, so it serves keys that never were a window; the set of m-mers is the same for a
// k-mer and its reverse complement.  Key 0 gives mmer_hash (0), which is where the emit kernel puts -n N-windows.
//
// Staging runs in two passes over the queries, both block-aggregated: count per owner, then (after the host has
// turned the counts into region starts) scatter with one global cursor atomic per owner and block-sized chunk.
// The reads kernel shares the read tile of the sliced build (tile_setup / tile_stage / tile_locate, the same
// staging and flattening insert_reads_kernel does) and chop_window, so the windows staged are exactly the windows
// a push inserts.
#pragma once
#include "sdt_skm.cuh"
#include "sdt_lookup.cuh"

namespace sdt {

enum : u32 { ROUTE_ONE = 0, ROUTE_SKM = 1, ROUTE_SLICED = 2, ROUTE_HASHED = 3 };	// SDTGPU_ROUTE_*
static constexpr u32 ROUTE_MAX_WORLD = 64;
static constexpr u64 ROUTE_RC = 1ull << 63;	// in a staged query's tag: the query is the reverse complement of its key

struct Route
{
	u32 kind, world;
	u32 n_slices, n_local;	// sliced builds
	u32 m, lo, w;		// minimizer length, first and number of the central m-mers of a window
	int K;
};

// what the staging kernels write: query words (W per query) and tags (output position | ROUTE_RC) in the owners'
// regions; cursor[r] runs from region r's start (scatter pass) or counts (count pass)
struct Stage
{
	u64 *q, *tag;
	unsigned long long *cursor;
};

// bits [s, s + 2m) of a key (bit 0 = the least significant bit of the last word), m <= 15
template <int W> __device__ __forceinline__ u32 key_bits (const Key<W> &k, u32 s, u32 m)
{
	const u32 q = s >> 6, off = s & 63;	// word from the bottom, bit in it
	u64 lo = 0, hi = 0;
#pragma unroll
	for (int i = 0; i < W; i++)
	{	// (selects, not an indexed load: the key stays in registers)
		if ((u32) (W - 1 - i) == q)
			lo = k.w[i];
		if ((u32) (W - 1 - i) == q + 1)
			hi = k.w[i];
	}
	const u64 v = off ? (lo >> off) | (hi << (64 - off)) : lo;
	return (u32) v & ((1u << (2 * m)) - 1u);
}

// the minimizer value skm_emit_kernel gives the window whose canonical key is k
template <int W> __device__ __forceinline__ u32 key_minval (const Key<W> &k, const Route &rt)
{
	const u32 msh = 32 - 2 * rt.m;
	u32 mv = 0xFFFFFFFFu;
	for (u32 p = rt.lo; p < rt.lo + rt.w; p++)
	{	// m-mer p: bases p .. p + m - 1 of the k-mer, whose first base is at bits 2 (K - 1) + 1 .. 2 (K - 1)
		const u32 f = key_bits<W> (k, 2 * ((u32) rt.K - rt.m - p), rt.m);
		u32 c = __brev (f ^ 0xAAAAAAAAu);	// (as skm_emit_kernel: complement, reverse the 2-bit groups)
		c = (((c >> 1) & 0x55555555u) | ((c & 0x55555555u) << 1)) >> msh;
		mv = min (mv, mmer_hash (min (f, c)));
	}
	return mv;
}

// the rank whose table holds the canonical key k
template <int W> __device__ __forceinline__ u32 route_owner (const Key<W> &k, const Route &rt)
{
	switch (rt.kind)
	{
	case ROUTE_SKM: return slice_of_min (key_minval<W> (k, rt), rt.n_slices) / rt.n_local;
	case ROUTE_SLICED: return slice_of_min (key_minval<W> (k, rt), rt.n_slices) % rt.world;
	case ROUTE_HASHED: return owner_of (key_hash<W> (k), rt.world);
	default: return 0;
	}
}

// One block-sized chunk of queries: SCATTER = false adds each owner's count to s_cnt; SCATTER = true reserves the
// chunk's places with one global atomic per owner and writes the queries.  Every thread of the block calls it.
template <int W, bool SCATTER>
__device__ __forceinline__ void stage_chunk (const Stage &st, u32 *s_cnt, unsigned long long *s_base, u32 world,
					     bool valid, u32 owner, const Key<W> &key, u64 tag)
{
	u32 local = 0;
	if (valid)
		local = atomicAdd (&s_cnt[owner], 1u);
	if constexpr (SCATTER)
	{
		__syncthreads ();
		if (threadIdx.x < world)
		{
			const u32 c = s_cnt[threadIdx.x];
			if (c)
				s_base[threadIdx.x] = atomicAdd (st.cursor + threadIdx.x, (unsigned long long) c);
			s_cnt[threadIdx.x] = 0;
		}
		__syncthreads ();
		if (valid)
		{
			const u64 pos = s_base[owner] + local;
#pragma unroll
			for (int i = 0; i < W; i++)
				st.q[pos * W + i] = key.w[i];
			st.tag[pos] = tag;
		}
		__syncthreads ();	// s_base is rewritten by the next chunk
	}
}

template <bool SCATTER> __device__ __forceinline__ void stage_flush (const Stage &st, u32 *s_cnt, u32 world)
{	// count pass: the block's counts to the global ones
	if constexpr (!SCATTER)
	{
		__syncthreads ();
		if (threadIdx.x < world && s_cnt[threadIdx.x])
			atomicAdd (st.cursor + threadIdx.x, (unsigned long long) s_cnt[threadIdx.x]);
	}
}

// keys in the sdtgpu_node layout: validated and canonicalised as lookup_kmers_kernel does; malformed keys stay home
template <int W, bool SCATTER>
__global__ void __launch_bounds__ (BLOCK)
route_kmers_kernel (const u64 *keys, u64 n, Route rt, Stage st)
{
	__shared__ u32 s_cnt[ROUTE_MAX_WORLD];
	__shared__ unsigned long long s_base[ROUTE_MAX_WORLD];
	if (threadIdx.x < ROUTE_MAX_WORLD)
		s_cnt[threadIdx.x] = 0;
	__syncthreads ();
	for (u64 i0 = blockIdx.x * (u64) BLOCK; i0 < n; i0 += (u64) gridDim.x * BLOCK)
	{
		const u64 i = i0 + threadIdx.x;
		bool ok = i < n;
		Key<W> key;
		u32 owner = 0;
		u64 tag = i;
		if (ok)
		{
			const ulonglong2 lo = *reinterpret_cast<const ulonglong2 *> (keys + 4 * i);
			const ulonglong2 hi = *reinterpret_cast<const ulonglong2 *> (keys + 4 * i + 2);
			const u64 q[4] = { lo.x, lo.y, hi.x, hi.y };
#pragma unroll
			for (int w = 0; w < 4; w++)
			{	// word w holds bits 64 (3 - w) .. 64 (3 - w) + 63 of the key; bits at 2K and above must be clear
				const int bits = 2 * rt.K - 64 * (3 - w);
				if (bits <= 0)
					ok &= q[w] == 0;
				else if (bits < 64)
					ok &= (q[w] >> bits) == 0;
			}
			Key<W> f, rc;
#pragma unroll
			for (int w = 0; w < W; w++)
				f.w[w] = q[4 - W + w];
			revcomp<W> (f, rt.K, rc);
			const bool fwd = key_less<W> (f, rc);
			key = fwd ? f : rc;
			tag |= fwd ? 0 : ROUTE_RC;
			if (ok)
				owner = route_owner<W> (key, rt);
		}
		stage_chunk<W, SCATTER> (st, s_cnt, s_base, rt.world, ok, owner, key, tag);
	}
	stage_flush<SCATTER> (st, s_cnt, rt.world);
}

// every window of a batch of reads (the conventions of insert_reads_kernel); window j of read r has output position
// r * maxwin + j
template <int W, bool NMODE, bool SCATTER>
__global__ void __launch_bounds__ (BLOCK)
route_reads_kernel (ReadBatch rb, Route rt, Stage st)
{
	extern __shared__ __align__(16) u32 smem[];
	__shared__ u32 warp_sums[BLOCK / 32];
	__shared__ u32 s_cnt[ROUTE_MAX_WORLD];
	__shared__ unsigned long long s_base[ROUTE_MAX_WORLD];
	const u32 tid = threadIdx.x;
	if (tid < ROUTE_MAX_WORLD)
		s_cnt[tid] = 0;
	ReadTile<NMODE> tl;
	tile_setup<NMODE> (tl, smem, rb);
	const u64 n_tiles = (rb.n_reads + rb.tile_reads - 1) / rb.tile_reads;
	for (u64 t = blockIdx.x; t < n_tiles; t += gridDim.x)
	{
		tile_stage<NMODE, BLOCK> (tl, rb, t, warp_sums);
		for (u32 w0 = 0; w0 < tl.total; w0 += BLOCK)
		{
			const u32 w = w0 + tid;
			const bool valid = w < tl.total;
			Key<W> key;
			u32 owner = 0;
			u64 tag = 0;
			if (valid)
			{
				u32 r, j, len, left, right;
				bool flipped;
				tile_locate<NMODE> (tl, rb.K, w, r, j, len);
				chop_window<W, NMODE> (tl.tile + r * tl.sw, NMODE ? (tl.mtile + r * tl.mw) : nullptr, (int) len, (int) j, rb.K, key, left, right, &flipped);
				owner = route_owner<W> (key, rt);
				tag = ((tl.r0 + r) * rb.maxwin + j) | (flipped ? ROUTE_RC : 0);
			}
			stage_chunk<W, SCATTER> (st, s_cnt, s_base, rt.world, valid, owner, key, tag);
		}
		__syncthreads ();	// the tile is overwritten by the next iteration
	}
	stage_flush<SCATTER> (st, s_cnt, rt.world);
}

// the owner's side: n received canonical keys (W words each) -> n hits, in the order received
template <int W>
__global__ void __launch_bounds__ (BLOCK)
route_answer_kernel (const typename SlotOf<W>::type *table, Lookup lk, const u64 *q, u64 n)
{
	for (u64 i = blockIdx.x * (u64) BLOCK + threadIdx.x; i < n; i += (u64) gridDim.x * BLOCK)
	{
		Key<W> key;
#pragma unroll
		for (int w = 0; w < W; w++)
			key.w[w] = q[i * W + w];
		store_hit (lk.out + i, index_probe<W> (table, lk, key, 0u));
	}
}

// the replies to this rank's staged queries (staged order) -> the caller's output, RC put back
__global__ void __launch_bounds__ (BLOCK)
route_unstage_kernel (const Hit *back, const u64 *tag, u64 n, Hit *out)
{
	for (u64 i = blockIdx.x * (u64) BLOCK + threadIdx.x; i < n; i += (u64) gridDim.x * BLOCK)
	{
		const u64 t = tag[i];
		Hit h = back[i];
		if (t & ROUTE_RC)
			h.status |= HIT_RC;
		store_hit (out + (t & ~ROUTE_RC), h);
	}
}

}	// namespace sdt
