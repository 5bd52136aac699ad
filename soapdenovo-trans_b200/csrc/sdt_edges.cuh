// sdt_edges.cuh — the finalized table compacted into edges between junction k-mers (sdtgpu_edges_build).
//
// A node is read in two orientations: (v,+) reads its canonical key k, (v,-) reads rc(k).  The out-links of (v,+) are
// the right counters R[x] > 0 (successor b1..b(K-1) x), those of (v,-) the left counters L[x] > 0 (successor
// rc(x b0..b(K-2)), base appended comp(x)).  A node with exactly one non-zero counter on each side is linear; a node
// that is neither linear nor deleted is a vertex.  An edge is a walk vertex -> linear ... linear -> vertex, one per
// (oriented vertex, out-link), kept iff its first (K+1)-mer <= the reverse complement of its last one; the linear
// nodes no edge visits form cycles.  DESIGN §4.6 states the definition in full.
//
// Kernels, all over positions of [0, iter_slots) of the table (the index of sdt_lookup.cuh resolves a key to one):
//   edge_links_kernel    one thread per slot: a linear node resolves both neighbours into a Step record (position,
//                        orientation, out-base, count); a vertex writes its number of walk starts
//   edge_starts_kernel   the starts of each vertex at its scanned offset, in (position, orientation, base) order
//   edge_walk_kernel     one thread per start; pass 0 walks to the end and applies the strand rule, pass 1 walks the
//                        kept starts again and writes the record, the bases and the visited marks
//   edge_cycle_kernel    one thread per unvisited linear node; pass 0 elects one leader per cycle (the node with the
//                        smallest hashed position: a node walks until it meets a smaller one or comes back), pass 1
//                        lets the leaders write their cycles
// A walk is a chain of dependent 16-byte loads, so the longest edge bounds the tail of the walk kernels.
#pragma once
#include "sdt_lookup.cuh"

namespace sdt {

static constexpr u32 EDGE_PALINDROME = 1u, EDGE_CYCLE = 2u;	// SDTGPU_EDGE_*
static constexpr u32 NO_POS = 0xFFFFFFFFu;

struct __align__(16) EdgeRec { u64 seq; u32 length, flags; u64 count_sum; u32 link, unused; };	// sdtgpu_edge

// per slot: next[o] = position of the successor of (v,o); meta (linear nodes) = STEP_LINEAR | out-base of (v,+) << 2 |
// out-base of (v,-) << 4 | first base of k << 6 | last base of k << 8 | orientation of next[0] << 10 | of next[1] << 11
// | R counter of the out-link << 12 | L counter << 18; meta = STEP_VERTEX for a vertex, 0 for an empty or deleted slot
struct __align__(16) Step { u32 next[2]; u32 count; u32 meta; };
static constexpr u32 STEP_VERTEX = 1u, STEP_LINEAR = 2u;

struct EdgeGraph
{
	const u64 *index;
	u64 idx_cap;
	Step *step;
	unsigned char *mark;	// linear nodes an edge visits (pass 1)
	u32 *a, *b;		// per slot or per start: vertex starts; kept / leader flag, 32-base words of the sequence
	const u64 *off_a, *off_b;	// exclusive scans of a and b
	u64 *starts;		// position << 3 | orientation << 2 | counter index
	EdgeRec *edges;
	u64 *seq;		// 32 bases per word, stored as the bytes of the tight-string convention
	u64 *ctr;		// sdtgpu_edges_build's out[]: [1] palindromes, [2] cycles, [3] bases, [4] vertices, [5] and [6] linear nodes, [7] dangling links
	u64 slots, n_starts, edge0, unit0, max_m;	// edge0, unit0: id and word offset of the first cycle
	int K, deLowKmer;
};

// the slot of the canonical key `key` (NO_POS if absent) and its payload words; the probe of index_probe
template <int W>
__device__ __forceinline__ u32 index_find (const typename SlotOf<W>::type *table, const u64 *index, u64 idx_cap, const Key<W> &key, u64 &s0, u64 &s1)
{
	const u64 h = key_hash<W> (key);
	const u32 tag = (u32) h;
	u64 j = slot_of (h, idx_cap);
	for (;;)
	{
		const u64 e = ld64_idx (index + j);
		if (e == IDX_EMPTY)
			return NO_POS;
		if ((u32) (e >> 32) == tag)
		{
			Key<W> k;
			load_slot<W> (table + (u32) e, k, s0, s1);
			if (key_eq<W> (k, key))
				return (u32) e;
		}
		if (++j == idx_cap)
			j = 0;
	}
}

// base i of a K-mer (0 = the first, most significant)
template <int W> __device__ __forceinline__ u32 key_base (const Key<W> &k, int K, int i)
{
	const int bit = 2 * (K - 1 - i);
	u32 r = 0;
#pragma unroll
	for (int q = 0; q < W; q++)
		if ((bit >> 6) == W - 1 - q)
			r = (u32) (k.w[q] >> (bit & 63)) & 3u;
	return r;
}

// drop the first base, append b
template <int W> __device__ __forceinline__ Key<W> key_append (const Key<W> &k, u32 b, int K)
{
	Key<W> r;
#pragma unroll
	for (int q = 0; q < W; q++)
	{
		r.w[q] = (k.w[q] << 2) | (q + 1 < W ? k.w[q + 1] >> 62 : (u64) b);
		const int bits = 2 * K - 64 * (W - 1 - q);
		if (bits <= 0)
			r.w[q] = 0;
		else if (bits < 64)
			r.w[q] &= (1ull << bits) - 1;
	}
	return r;
}

// the canonical key of `k`; o = 1 if that is its reverse complement
template <int W> __device__ __forceinline__ Key<W> canonical (const Key<W> &k, int K, u32 &o)
{
	Key<W> rc;
	revcomp<W> (k, K, rc);
	o = key_less<W> (k, rc) ? 0u : 1u;
	return o ? rc : k;
}

__device__ __forceinline__ Step ld_step (const Step *p)
{	// read-only while the walks run; a random 16-byte load fetches 64 bytes into L2, not a whole line
	Step s;
	asm volatile ("ld.global.nc.L2::64B.v4.u32 {%0,%1,%2,%3}, [%4];"
		      : "=r"(s.next[0]), "=r"(s.next[1]), "=r"(s.count), "=r"(s.meta) : "l"(p));
	return s;
}

__device__ __forceinline__ u64 bswap64 (u64 x)
{
	return ((u64) __byte_perm ((u32) x, 0, 0x0123) << 32) | __byte_perm ((u32) (x >> 32), 0, 0x0123);
}

// bases of one edge, 32 to a word; every word of the edge's range is written, the last one zero-padded
struct SeqOut
{
	u64 *p;
	u64 acc;
	u32 n;
	__device__ __forceinline__ void push (u32 b)
	{
		acc = (acc << 2) | b;
		if (++n == 32)
		{
			*p++ = bswap64 (acc);
			acc = 0;
			n = 0;
		}
	}
	template <int W> __device__ __forceinline__ void push_key (const Key<W> &k, int K)
	{
		for (int i = 0; i < K; i++)
			push (key_base<W> (k, K, i));
	}
	__device__ __forceinline__ void flush ()
	{
		if (n)
			*p = bswap64 (acc << (64 - 2 * n));
	}
};

// warp sum into a counter (every lane of the warp must call it)
__device__ __forceinline__ void add_ctr (u64 *ctr, u64 v)
{
#pragma unroll
	for (int d = 16; d > 0; d >>= 1)
		v += __shfl_down_sync (0xFFFFFFFFu, v, d);
	if ((threadIdx.x & 31) == 0 && v)
		atomicAdd ((unsigned long long *) ctr, (unsigned long long) v);
}

template <int W>
__global__ void __launch_bounds__ (256)
edge_links_kernel (const typename SlotOf<W>::type *table, EdgeGraph g)
{
	u64 n_vert = 0, n_dang = 0;
	for (u64 p = blockIdx.x * (u64) blockDim.x + threadIdx.x; p < g.slots; p += (u64) gridDim.x * blockDim.x)
	{
		Step st = { { NO_POS, NO_POS }, 0, 0 };
		u32 n_starts = 0;
		Key<W> k;
		u64 s0, s1;
		if (load_slot<W> (table + p, k, s0, s1))
		{
			const u32 L = (u32) s0 & 0xFFFFFFu, R = (u32) s1 & 0xFFFFFFu;
			u32 nl = 0, nr = 0, xl = 0, xr = 0;
#pragma unroll
			for (u32 b = 0; b < 4; b++)
			{
				if ((L >> (6 * b)) & 63)
				{
					nl++;
					xl = b;
				}
				if ((R >> (6 * b)) & 63)
				{
					nr++;
					xr = b;
				}
			}
			if (nl == 1 && nr == 1)
			{
				const u32 b0 = key_base<W> (k, g.K, 0), bl = (u32) k.w[W - 1] & 3u;
				st.count = (u32) (s1 >> 32);
				st.meta = STEP_LINEAR | xr << 2 | (xl ^ 2u) << 4 | b0 << 6 | bl << 8 | ((R >> (6 * xr)) & 63) << 12 | ((L >> (6 * xl)) & 63) << 18;
				Key<W> rc;
				revcomp<W> (k, g.K, rc);
#pragma unroll
				for (u32 d = 0; d < 2; d++)
				{
					u32 o;
					const Key<W> nk = canonical<W> (key_append<W> (d ? rc : k, d ? xl ^ 2u : xr, g.K), g.K, o);
					u64 t0, t1;
					const u32 u = index_find<W> (table, g.index, g.idx_cap, nk, t0, t1);
					st.next[d] = u;
					st.meta |= o << (10 + d);
					if (u == NO_POS)
					{
						n_dang++;
						continue;
					}
					// the link back: (u, !o) appends comp (f) to reach (v, !d), f the first base of (v, d)
					const u32 f = d ? bl ^ 2u : b0;
					const u32 back = o ? ((u32) t1 >> (6 * (f ^ 2u))) & 63 : ((u32) t0 >> (6 * f)) & 63;
					n_dang += back == 0;
				}
			}
			else if (!(g.deLowKmer > 0 && L == 0 && R == 0))
			{
				st.meta = STEP_VERTEX;
				n_starts = nl + nr;
				n_vert++;
			}
		}
		*reinterpret_cast<uint4 *> (g.step + p) = make_uint4 (st.next[0], st.next[1], st.count, st.meta);
		g.a[p] = n_starts;
	}
	add_ctr (g.ctr + 4, n_vert);
	add_ctr (g.ctr + 7, n_dang);
}

template <int W>
__global__ void __launch_bounds__ (256)
edge_starts_kernel (const typename SlotOf<W>::type *table, EdgeGraph g)
{
	for (u64 p = blockIdx.x * (u64) blockDim.x + threadIdx.x; p < g.slots; p += (u64) gridDim.x * blockDim.x)
	{
		if (!g.a[p])
			continue;
		Key<W> k;
		u64 s0, s1;
		load_slot<W> (table + p, k, s0, s1);
		u64 at = g.off_a[p];
#pragma unroll
		for (u32 d = 0; d < 2; d++)
#pragma unroll
			for (u32 x = 0; x < 4; x++)
				if (((u32) (d ? s0 : s1) >> (6 * x)) & 63)
					g.starts[at++] = p << 3 | d << 2 | x;
	}
}

// PASS 0: a[s] = the walk is kept, b[s] = its words of sequence.  PASS 1: the kept walks write their records.
template <int W, int PASS>
__global__ void __launch_bounds__ (256)
edge_walk_kernel (const typename SlotOf<W>::type *table, EdgeGraph g)
{
	const int K = g.K;
	u64 n_pal = 0, n_bases = 0, n_lin = 0, n_dang = 0;
	for (u64 s = blockIdx.x * (u64) blockDim.x + threadIdx.x; s < g.n_starts; s += (u64) gridDim.x * blockDim.x)
	{
		if (PASS == 1 && !g.a[s])
			continue;
		const u64 e = g.starts[s];
		const u32 v = (u32) (e >> 3), d = (u32) (e >> 2) & 1u, x = (u32) e & 3u;
		Key<W> k, kk;
		u64 s0, s1;
		load_slot<W> (table + v, k, s0, s1);
		if (d)
			revcomp<W> (k, K, kk);
		else
			kk = k;
		const u32 y = d ? x ^ 2u : x;	// the first base appended
		u32 co;
		u64 t0, t1;
		u32 cu = index_find<W> (table, g.index, g.idx_cap, canonical<W> (key_append<W> (kk, y, K), K, co), t0, t1);
		SeqOut out = { g.seq + (PASS == 1 ? g.off_b[s] : 0), 0, 0 };
		if (PASS == 1)
		{
			out.push_key<W> (kk, K);
			out.push (y);
		}
		u32 pf = key_base<W> (kk, K, 0);	// first base of the oriented k-mer before (cu, co)
		u64 m = 1, csum = 0;
		bool ok = cu != NO_POS;
		if (!ok)
			n_dang++;
		while (ok)
		{
			const Step st = ld_step (g.step + cu);
			if ((st.meta & 3u) != STEP_LINEAR)
				break;
			if (m > g.max_m)
			{	// only a table whose links disagree gets here
				ok = false;
				n_dang++;
				break;
			}
			if (PASS == 1)
			{
				g.mark[cu] = 1;
				csum += st.count;
				out.push ((st.meta >> (2 + 2 * co)) & 3u);
			}
			pf = co ? ((st.meta >> 8) & 3u) ^ 2u : (st.meta >> 6) & 3u;
			cu = st.next[co];
			co = (st.meta >> (10 + co)) & 1u;
			ok = cu != NO_POS;	// (counted by edge_links_kernel)
			m++;
		}
		if (!ok)
		{
			if (PASS == 0)
				g.a[s] = g.b[s] = 0;
			continue;
		}
		// the reverse walk starts at (cu, !co) and appends comp (pf): compare its first (K+1)-mer with ours
		Key<W> ke, kr;
		load_slot<W> (table + cu, ke, t0, t1);
		if (co)
			kr = ke;
		else
			revcomp<W> (ke, K, kr);
		const u32 y2 = pf ^ 2u;
		const bool same = key_eq<W> (kk, kr), pal = same && y == y2;
		if (PASS == 0)
		{
			const bool keep = key_less<W> (kk, kr) || (same && y <= y2);
			g.a[s] = keep;
			g.b[s] = keep ? (u32) ((m + K + 31) / 32) : 0u;
		}
		else
		{
			out.flush ();
			EdgeRec r;
			r.seq = g.off_b[s] * 32;
			r.length = (u32) m;
			r.flags = pal ? EDGE_PALINDROME : 0u;
			r.count_sum = csum;
			r.link = ((u32) (d ? s0 : s1) >> (6 * x)) & 63;
			r.unused = 0;
			g.edges[g.off_a[s]] = r;
			n_pal += pal;
			n_bases += m + K;
			n_lin += pal ? (m - 1) / 2 : m - 1;
		}
	}
	if (PASS == 0)
		add_ctr (g.ctr + 7, n_dang);
	else
	{
		add_ctr (g.ctr + 1, n_pal);
		add_ctr (g.ctr + 3, n_bases);
		add_ctr (g.ctr + 5, n_lin);
	}
}

// PASS 0: a[p] = p leads a cycle, b[p] = the cycle's words of sequence.  PASS 1: the leaders write their cycles,
// starting at (p,+).  A cycle that meets (p,-) before it comes back to (p,+) is its own reverse complement (closed by
// two hairpins): it holds each of its nodes twice.
template <int W, int PASS>
__global__ void __launch_bounds__ (256)
edge_cycle_kernel (const typename SlotOf<W>::type *table, EdgeGraph g)
{
	const int K = g.K;
	u64 n_cyc = 0, n_pal = 0, n_bases = 0, n_lin = 0, n_dang = 0;
	for (u64 p = blockIdx.x * (u64) blockDim.x + threadIdx.x; p < g.slots; p += (u64) gridDim.x * blockDim.x)
	{
		if (PASS == 1 && !g.a[p])
			continue;
		Step st = ld_step (g.step + p);
		if (PASS == 0)
		{
			g.a[p] = g.b[p] = 0;
			if ((st.meta & 3u) != STEP_LINEAR || g.mark[p])
				continue;
		}
		const u32 link = (st.meta >> 12) & 63;
		const u64 label = fmix64 (p);
		SeqOut out = { g.seq + (PASS == 1 ? g.unit0 + g.off_b[p] : 0), 0, 0 };
		if (PASS == 1)
		{
			Key<W> k;
			u64 s0, s1;
			load_slot<W> (table + p, k, s0, s1);
			out.push_key<W> (k, K);
		}
		u32 cu = (u32) p, co = 0;
		u64 m = 0, csum = 0;
		bool pal = false, leader = false;
		for (;;)
		{
			csum += st.count;
			const u32 nu = st.next[co], nco = (st.meta >> (10 + co)) & 1u, ob = (st.meta >> (2 + 2 * co)) & 3u;
			m++;
			if (nu == NO_POS)
				break;	// (counted by edge_links_kernel)
			if (nu == (u32) p)
			{
				if (nco == 0)
				{
					leader = true;
					break;
				}
				pal = true;
			}
			else if (PASS == 0 && fmix64 (nu) < label)
				break;
			if (m > g.max_m)
			{
				n_dang++;
				break;
			}
			if (PASS == 1)
				out.push (ob);
			cu = nu;
			co = nco;
			st = ld_step (g.step + cu);
			if ((st.meta & 3u) != STEP_LINEAR)
			{
				n_dang++;
				break;
			}
		}
		if (PASS == 0)
		{
			if (leader)
			{
				g.a[p] = 1;
				g.b[p] = (u32) ((m + K - 1 + 31) / 32);
			}
		}
		else
		{
			out.flush ();
			EdgeRec r;
			r.seq = (g.unit0 + g.off_b[p]) * 32;
			r.length = (u32) m;
			r.flags = EDGE_CYCLE | (pal ? EDGE_PALINDROME : 0u);
			r.count_sum = csum;
			r.link = link;
			r.unused = 0;
			g.edges[g.edge0 + g.off_a[p]] = r;
			n_cyc++;
			n_pal += pal;
			n_bases += m + K - 1;
			n_lin += pal ? m / 2 : m;
		}
	}
	if (PASS == 0)
		add_ctr (g.ctr + 7, n_dang);
	else
	{
		add_ctr (g.ctr + 1, n_pal);
		add_ctr (g.ctr + 2, n_cyc);
		add_ctr (g.ctr + 3, n_bases);
		add_ctr (g.ctr + 6, n_lin);
	}
}

}	// namespace sdt
