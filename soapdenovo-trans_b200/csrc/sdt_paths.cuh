// sdt_paths.cuh — reads mapped onto the edge graph of sdtgpu_edges_build (sdtgpu_edges_map_reads, sdtgpu_arcs_build).
//
// A read (K+1)-mer is a step of the graph when its first k-mer is a node and that node's counter for the read's next
// base, on the read's side, is non-zero: an out-link of DESIGN §4.6.  Every such step is step i of exactly one record
// (edge or cycle), on the record's strand (0) or the reverse one (1); a palindromic record reports strand 0 only.  The
// stamps below make that a constant number of loads per window:
//   stamp[p]    per table slot: a linear node (record << 1 | palindrome, i << 1 | orientation) of its first visit x_i;
//               a vertex (its first walk start, all ones); anything else all ones
//   srec[s]     per walk start: record << 1 | strand, strand 1 for the start that begins the reverse of a kept walk
//   aux[c]      per cycle: for a palindromic one, h, the index of the leader's second visit (x_h = rc (x_0)), so that
//               rc (s_i) = s_((h - 1 - i) mod m); an edge has h = m
// A window at (p, o) with out-base counter x: a linear p stamped (r, i, o0) gives (r, i, 0) if o == o0, else rc of
// s_(i-1) (mod m); a vertex gives the record of its start (p, o, x): s_0 on strand 0, rc (s_(m-1)) on strand 1.
//
// Arcs: a read crosses a vertex v when both link bases of its window at v are present and both counters non-zero (then
// the steps into and out of v are steps of the graph: the two ends of a (K+1)-mer count the same instances).  A
// crossing in v's + orientation with link bases (left, right) adds one to counter 4 * s_in + right, s_in the start
// (v, -, left): the counters of one vertex are then in (left, right) order, and the starts in table-position order.
//
// Kernels:
//   path_starts_kernel    one thread per walk start: each vertex's first start into its stamp
//   path_records_kernel   one thread per record: finds its first k-mer, walks it over the Step records and stamps the
//                         linear nodes, marks the starts of the walk and of its reverse
//   path_map_kernel       one thread per window over the read tile of route_reads_kernel (the windows a push inserts)
//   path_arcs_kernel      one thread per walk start; pass 0 counts the non-zero counters, pass 1 writes them
#pragma once
#include "sdt_edges.cuh"
#include "sdt_skm.cuh"

namespace sdt {

struct __align__(16) ArcRec { u32 from, to, count, unused; };	// sdtgpu_arc

struct PathMap
{
	const u64 *index;
	u64 idx_cap;
	const Step *step;
	const u64 *starts;	// sorted walk starts of the edge build: position << 3 | orientation << 2 | counter index
	const EdgeRec *edges;
	const u64 *seq;
	uint2 *stamp;
	u32 *srec, *aux;
	u32 *ctr;		// arc counters, 4 per start (NULL: the call does not count)
	u32 *cnt;		// arcs per start (path_arcs_kernel)
	const u64 *off;		// their exclusive scan
	ArcRec *arcs;
	uint2 *out;		// sdtgpu_step per window, or NULL
	u64 *small;		// [0] longest record, [1] crossings of the arcs written
	u64 n_starts, n_edges, n_records;
	int K;
};

// bit b set iff the 6-bit counter b of a link word is non-zero
__device__ __forceinline__ u32 link_mask (u64 w)
{
	u32 m = 0;
#pragma unroll
	for (u32 b = 0; b < 4; b++)
		m |= (((u32) w >> (6 * b)) & 63 ? 1u : 0u) << b;
	return m;
}

// the start (v, d, x) of a vertex whose first start is fs: the starts follow (orientation, counter index) order
__device__ __forceinline__ u32 start_of (u32 fs, u32 lm, u32 rm, u32 d, u32 x)
{
	return fs + (d ? __popc (rm) + __popc (lm & ((1u << x) - 1)) : __popc (rm & ((1u << x) - 1)));
}

__global__ void __launch_bounds__ (256)
path_starts_kernel (PathMap g)
{
	for (u64 s = blockIdx.x * (u64) blockDim.x + threadIdx.x; s < g.n_starts; s += (u64) gridDim.x * blockDim.x)
	{
		const u32 v = (u32) (g.starts[s] >> 3);
		if (s == 0 || (u32) (g.starts[s - 1] >> 3) != v)
			g.stamp[v] = make_uint2 ((u32) s, NO_POS);
	}
}

template <int W>
__global__ void __launch_bounds__ (256)
path_records_kernel (const typename SlotOf<W>::type *table, PathMap g)
{
	const int K = g.K;
	u64 longest = 0;
	for (u64 r = blockIdx.x * (u64) blockDim.x + threadIdx.x; r < g.n_records; r += (u64) gridDim.x * blockDim.x)
	{
		const EdgeRec e = g.edges[r];
		const u32 m = e.length, pal = e.flags & EDGE_PALINDROME;
		const bool cyc = e.flags & EDGE_CYCLE;
		longest = max (longest, (u64) m);
		const u64 *sq = g.seq + (e.seq >> 5);
		auto base = [&] (u32 i) { return (u32) (bswap64 (sq[i >> 5]) >> (62 - 2 * (i & 31))) & 3u; };
		Key<W> kk;
#pragma unroll
		for (int q = 0; q < W; q++)
			kk.w[q] = 0;
		for (int i = 0; i < K; i++)
			kk = key_append<W> (kk, base (i), K);
		u32 o;
		u64 s0, s1;
		const u32 v = index_find<W> (table, g.index, g.idx_cap, canonical<W> (kk, K, o), s0, s1);
		if (v == NO_POS)
			continue;	// (a table whose links disagree)
		u32 cu, co, i;
		if (cyc)
		{	// x_0 is the leader read as (p,+)
			cu = v;
			co = 0;
			i = 0;
		}
		else
		{
			const u32 y = base (K);
			g.srec[start_of (g.stamp[v].x, link_mask (s0), link_mask (s1), o, o ? y ^ 2u : y)] = (u32) r << 1;
			cu = index_find<W> (table, g.index, g.idx_cap, canonical<W> (key_append<W> (kk, y, K), K, co), s0, s1);
			i = 1;
		}
		u32 h = m;
		if (cyc && pal)
		{	// the leader's second visit, in the other orientation
			u32 u = cu, uo = co;
			for (u32 k = 1; k < m; k++)
			{
				const Step st = ld_step (g.step + u);
				const u32 nu = st.next[uo];
				uo = (st.meta >> (10 + uo)) & 1u;
				u = nu;
				if (u == v && uo)
				{
					h = k;
					break;
				}
			}
			g.aux[r - g.n_edges] = h;
		}
		for (; i < m && cu != NO_POS; i++)
		{	// a palindrome visits x_i and x_((h - i) mod m) = rc (x_i): stamp the first of the two
			if (!pal || (i < h ? 2 * i <= h : i > h && 2 * i <= h + m))
				g.stamp[cu] = make_uint2 ((u32) r << 1 | pal, i << 1 | co);
			const Step st = ld_step (g.step + cu);
			cu = st.next[co];
			co = (st.meta >> (10 + co)) & 1u;
		}
		if (!cyc && !pal && cu != NO_POS)
		{	// x_m = (cu, co): the reverse walk starts at (cu, !co) and appends comp (first base of x_(m-1))
			const u32 b = base (m - 1);
			Key<W> k;
			load_slot<W> (table + cu, k, s0, s1);
			g.srec[start_of (g.stamp[cu].x, link_mask (s0), link_mask (s1), co ^ 1u, co ? b ^ 2u : b)] = (u32) r << 1 | 1u;
		}
	}
#pragma unroll
	for (int d = 16; d > 0; d >>= 1)
		longest = max (longest, (u64) __shfl_down_sync (0xFFFFFFFFu, longest, d));
	if ((threadIdx.x & 31) == 0 && longest)
		atomicMax ((unsigned long long *) g.small, (unsigned long long) longest);
}

// every window of a batch of reads (the conventions of insert_reads_kernel); window j of read r -> out[r * maxwin + j]
template <int W, bool NMODE>
__global__ void __launch_bounds__ (BLOCK, 4)
path_map_kernel (const typename SlotOf<W>::type *table, ReadBatch rb, PathMap g)
{
	extern __shared__ __align__(16) u32 smem[];
	__shared__ u32 warp_sums[BLOCK / 32];
	ReadTile<NMODE> tl;
	tile_setup<NMODE> (tl, smem, rb);
	const u64 n_tiles = (rb.n_reads + rb.tile_reads - 1) / rb.tile_reads;
	for (u64 t = blockIdx.x; t < n_tiles; t += gridDim.x)
	{
		tile_stage<NMODE, BLOCK> (tl, rb, t, warp_sums);
		for (u32 w = threadIdx.x; w < tl.total; w += BLOCK)
		{
			u32 r, j, len, left, right;
			bool flipped;
			Key<W> key;
			tile_locate<NMODE> (tl, rb.K, w, r, j, len);
			chop_window<W, NMODE> (tl.tile + r * tl.sw, NMODE ? (tl.mtile + r * tl.mw) : nullptr, (int) len, (int) j, rb.K, key, left, right, &flipped);
			const u32 ob = flipped ? left : right;	// the out-link's counter: L[left] read as (p,-), R[right] as (p,+)
			u32 rec = NO_POS, pos = NO_POS;
			if (ob < 4)
			{
				u64 s0 = 0, s1 = 0;
				const u32 p = index_find<W> (table, g.index, g.idx_cap, key, s0, s1);
				const u32 lm = link_mask (s0), rm = link_mask (s1);
				if (p != NO_POS && (((flipped ? lm : rm) >> ob) & 1))
				{
					const uint2 sp = __ldg (g.stamp + p);
					if (__popc (lm) == 1 && __popc (rm) == 1)
					{
						if (sp.x != NO_POS)
						{
							const u32 pal = sp.x & 1u, i0 = sp.y >> 1;
							rec = sp.x >> 1;
							if ((u32) flipped == (sp.y & 1u))
								pos = i0 << 1;
							else if (!pal && i0)
								pos = (i0 - 1) << 1 | 1u;
							else
							{
								const u32 m = __ldg (&g.edges[rec].length);
								if (!pal)	// x_0 of a cycle
									pos = (m - 1) << 1 | 1u;
								else
								{
									const u32 h = rec < g.n_edges ? m : __ldg (g.aux + (rec - g.n_edges));
									pos = ((h + m - i0) % m) << 1;
								}
							}
						}
					}
					else
					{
						const u32 sr = __ldg (g.srec + start_of (sp.x, lm, rm, flipped, ob));
						if (sr != NO_POS)
						{
							rec = sr >> 1;
							pos = sr & 1u ? (__ldg (&g.edges[rec].length) - 1) << 1 | 1u : 0u;
						}
						if (g.ctr && left < 4 && right < 4 && ((lm >> left) & 1) && ((rm >> right) & 1))
							atomicAdd (g.ctr + 4 * (u64) start_of (sp.x, lm, rm, 1u, left) + right, 1u);
					}
				}
			}
			if (g.out)
				g.out[(tl.r0 + r) * rb.maxwin + j] = make_uint2 (rec, pos);
		}
		__syncthreads ();	// the tile is overwritten by the next iteration
	}
}

// PASS 0: cnt[s] = non-zero counters of start s.  PASS 1: they become arcs at off[s], in (right base) order.
template <int W, int PASS>
__global__ void __launch_bounds__ (256)
path_arcs_kernel (const typename SlotOf<W>::type *table, PathMap g)
{
	u64 crossings = 0;
	for (u64 s = blockIdx.x * (u64) blockDim.x + threadIdx.x; s < g.n_starts; s += (u64) gridDim.x * blockDim.x)
	{
		const uint4 c = *reinterpret_cast<const uint4 *> (g.ctr + 4 * s);
		const u32 cs[4] = { c.x, c.y, c.z, c.w };
		if (PASS == 0)
		{
			g.cnt[s] = (c.x != 0) + (c.y != 0) + (c.z != 0) + (c.w != 0);
			continue;
		}
		if (!g.cnt[s])
			continue;
		const u32 v = (u32) (g.starts[s] >> 3);
		const u32 from = g.srec[s], fr = from >> 1;
		Key<W> k;
		u64 s0, s1;
		load_slot<W> (table + v, k, s0, s1);
		const u32 fs = g.stamp[v].x, lm = link_mask (s0), rm = link_mask (s1);
		ArcRec *out = g.arcs + g.off[s];
#pragma unroll
		for (u32 x = 0; x < 4; x++)
		{
			if (!cs[x])
				continue;
			ArcRec a;
			// "from" is the walk that ends entering (v,+): the start's record on the other strand (a palindrome has one)
			a.from = fr == (NO_POS >> 1) ? NO_POS : (g.edges[fr].flags & EDGE_PALINDROME) ? from : from ^ 1u;
			a.to = g.srec[start_of (fs, lm, rm, 0u, x)];
			a.count = cs[x];
			a.unused = 0;
			*out++ = a;
			crossings += cs[x];
		}
	}
	if (PASS == 1)
		add_ctr (g.small + 1, crossings);
}

}	// namespace sdt
