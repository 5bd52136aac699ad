// sdt_prune.cuh — the finalized table pruned of minor branches and tips (sdtgpu_prune), in rounds that do not depend
// on slot order.
//
// Terms of sdt_edges.cuh: (v,+) reads the canonical key, (v,-) its reverse complement; the out-links of (v,+) are the R
// counters, those of (v,-) the L counters.  Every non-zero counter has a reciprocal in its neighbour (the same
// (K+1)-mer seen from the other end).  Removing a node zeroes its counters and their reciprocals; a node left without
// a non-zero counter is deleted.  DESIGN §4.8 states the definition in full.
//
// A round is three launches over the positions [0, iter_slots), so that decisions and writes never race: every
// decision reads the table as it was at the start of the round.
//   prune_decide_kernel<PHASE>  one thread per slot.  PHASE 0 (minor branches): a side with two or more non-zero
//                        counters resolves its neighbours and marks those with 100 count < minor_pct x the largest
//                        count.  PHASE 1 and 2 (single and minor tips): a dead end (one non-zero counter) walks at most
//                        2K steps to the first node that is not linear; if the tip is cut it walks again to mark it
//   prune_unlink_kernel  one thread per marked node: the reciprocal of each of its counters goes into the neighbour's
//                        clear mask (8 bits per slot, L counters in bits 0..3, R counters in bits 4..7)
//   prune_apply_kernel   one thread per slot: a marked node loses all its counters, another the masked ones; the mark
//                        and the mask are reset; removals, live and linear nodes are counted
#pragma once
#include "sdt_kernels.cuh"
#include "sdt_edges.cuh"

namespace sdt {

struct Prune
{
	const u64 *index;
	u64 idx_cap;
	unsigned char *mark;	// per slot: removed by this round
	u32 *mask;		// per slot one byte, four to a word: counters to zero
	u64 *ctr;		// sdtgpu_prune's out[]: [0..2] nodes removed by phase, [3] tips cut, [5] live, [6] linear nodes
	u64 slots;
	int K, minor_pct, phase;
};

__device__ __forceinline__ u32 n_links (u32 w)
{
	u32 n = 0;
#pragma unroll
	for (int b = 0; b < 4; b++)
		n += ((w >> (6 * b)) & 63) != 0;
	return n;
}

__device__ __forceinline__ u32 max_link (u32 w)
{
	u32 m = 0;
#pragma unroll
	for (int b = 0; b < 4; b++)
		m = max (m, (w >> (6 * b)) & 63);
	return m;
}

// the base of the only non-zero counter of w
__device__ __forceinline__ u32 only_link (u32 w)
{
	u32 x = 0;
#pragma unroll
	for (u32 b = 0; b < 4; b++)
		if ((w >> (6 * b)) & 63)
			x = b;
	return x;
}

__device__ __forceinline__ bool is_linear (u32 L, u32 R) { return n_links (L) == 1 && n_links (R) == 1; }

// One step along an out-link: kk (an oriented k-mer) becomes its successor with base y appended.  Returns the
// successor's slot (NO_POS if absent) with its payload, the orientation o it is read in, and the bit of the reciprocal
// counter in its clear mask (the link back from (u, !o) appends comp (f), f the first base of kk).
template <int W>
__device__ __forceinline__ u32 prune_hop (const typename SlotOf<W>::type *table, const Prune &g, Key<W> &kk, u32 y, u32 &o, u32 &back_bit, u64 &t0, u64 &t1)
{
	const u32 f = key_base<W> (kk, g.K, 0);
	kk = key_append<W> (kk, y, g.K);
	const u32 u = index_find<W> (table, g.index, g.idx_cap, canonical<W> (kk, g.K, o), t0, t1);
	back_bit = o ? 4 + (f ^ 2u) : f;
	return u;
}

// the out-link of an oriented linear node: the base its successor appends
__device__ __forceinline__ u32 out_base (u32 L, u32 R, u32 o)
{
	return o ? only_link (L) ^ 2u : only_link (R);
}

// (256, 4): with the block size alone ptxas holds the one-word variants to 32 registers and spills there; four resident
// blocks per SM allow 64 registers, and every variant fits that without spilling (38 to 64 registers)
template <int W, int PHASE>
__global__ void __launch_bounds__ (256, 4)
prune_decide_kernel (const typename SlotOf<W>::type *table, Prune g)
{
	u64 n_tips = 0;
	for (u64 p = blockIdx.x * (u64) blockDim.x + threadIdx.x; p < g.slots; p += (u64) gridDim.x * blockDim.x)
	{
		Key<W> k;
		u64 s0, s1;
		if (!load_slot<W> (table + p, k, s0, s1))
			continue;
		const u32 L = (u32) s0 & 0xFFFFFFu, R = (u32) s1 & 0xFFFFFFu;
		if (PHASE == 0)
		{
#pragma unroll
			for (u32 d = 0; d < 2; d++)
			{
				const u32 w = d ? L : R;
				if (n_links (w) < 2)
					continue;
				Key<W> kk;
				if (d)
					revcomp<W> (k, g.K, kk);
				else
					kk = k;
				u32 nb[4], cnt[4], mx = 0;
#pragma unroll
				for (u32 x = 0; x < 4; x++)
				{
					nb[x] = NO_POS;
					cnt[x] = 0;
					if (!((w >> (6 * x)) & 63))
						continue;
					Key<W> t = kk;
					u32 o, bit;
					u64 t0, t1;
					nb[x] = prune_hop<W> (table, g, t, d ? x ^ 2u : x, o, bit, t0, t1);
					cnt[x] = (u32) (t1 >> 32);
					if (nb[x] != NO_POS)
						mx = max (mx, cnt[x]);
				}
#pragma unroll
				for (u32 x = 0; x < 4; x++)
					if (nb[x] != NO_POS && 100ull * cnt[x] < (u64) g.minor_pct * mx)
						g.mark[nb[x]] = 1;
			}
			continue;
		}
		if (n_links (L) + n_links (R) != 1)
			continue;
		// a dead end: orient it so that its counter is an out-link, and walk to the first node that is not linear
		const u32 d0 = n_links (R) ? 0u : 1u;
		Key<W> kk;
		if (d0)
			revcomp<W> (k, g.K, kk);
		else
			kk = k;
		const Key<W> start = kk;
		const u32 y0 = out_base (L, R, d0);
		bool single = (u32) (s1 >> 32) == 1;
		u32 y = y0, u = NO_POS, o = 0, bit = 0, m = 1;
		u64 t0 = 0, t1 = 0;
		bool found = false;
		for (; m <= 2u * (u32) g.K; m++)
		{
			u = prune_hop<W> (table, g, kk, y, o, bit, t0, t1);
			if (u == NO_POS)
				break;	// (a table whose links disagree: nothing is cut)
			const u32 Lu = (u32) t0 & 0xFFFFFFu, Ru = (u32) t1 & 0xFFFFFFu;
			if (!is_linear (Lu, Ru))
			{
				found = true;
				break;
			}
			single &= (u32) (t1 >> 32) == 1;
			y = out_base (Lu, Ru, o);
		}
		if (!found)
			continue;
		// xm = (u, o): its counter toward x(m-1) is the reciprocal, an out-link of (u, !o)
		const u32 Lu = (u32) t0 & 0xFFFFFFu, Ru = (u32) t1 & 0xFFFFFFu;
		const bool isolated = n_links (Lu) + n_links (Ru) == 1;
		const u32 back = ((bit < 4 ? Lu : Ru) >> (6 * (bit & 3u))) & 63;
		const bool cut = isolated || (PHASE == 1 ? single : back < max_link (bit < 4 ? Lu : Ru));
		if (!cut)
			continue;
		n_tips += !isolated || p <= u;	// both ends of an isolated chain find it
		if (isolated)
			g.mark[u] = 1;
		g.mark[p] = 1;
		kk = start;
		y = y0;
		for (u32 i = 1; i < m; i++)
		{
			const u32 v = prune_hop<W> (table, g, kk, y, o, bit, t0, t1);
			g.mark[v] = 1;
			y = out_base ((u32) t0 & 0xFFFFFFu, (u32) t1 & 0xFFFFFFu, o);
		}
	}
	add_ctr (g.ctr + 3, n_tips);
}

template <int W>
__global__ void __launch_bounds__ (256)
prune_unlink_kernel (const typename SlotOf<W>::type *table, Prune g)
{
	for (u64 p = blockIdx.x * (u64) blockDim.x + threadIdx.x; p < g.slots; p += (u64) gridDim.x * blockDim.x)
	{
		if (!g.mark[p])
			continue;
		Key<W> k;
		u64 s0, s1;
		load_slot<W> (table + p, k, s0, s1);
#pragma unroll
		for (u32 d = 0; d < 2; d++)
		{
			const u32 w = (u32) (d ? s0 : s1) & 0xFFFFFFu;
			if (!w)
				continue;
			Key<W> kk;
			if (d)
				revcomp<W> (k, g.K, kk);
			else
				kk = k;
#pragma unroll
			for (u32 x = 0; x < 4; x++)
			{
				if (!((w >> (6 * x)) & 63))
					continue;
				Key<W> t = kk;
				u32 o, bit;
				u64 t0, t1;
				const u32 u = prune_hop<W> (table, g, t, d ? x ^ 2u : x, o, bit, t0, t1);
				if (u != NO_POS)
					atomicOr (g.mask + (u >> 2), 1u << (8 * (u & 3u) + bit));
			}
		}
	}
}

template <int W>
__global__ void __launch_bounds__ (256)
prune_apply_kernel (typename SlotOf<W>::type *table, Prune g)
{
	u64 n_removed = 0, n_live = 0, n_lin = 0;
	unsigned char *mask = reinterpret_cast<unsigned char *> (g.mask);
	for (u64 p = blockIdx.x * (u64) blockDim.x + threadIdx.x; p < g.slots; p += (u64) gridDim.x * blockDim.x)
	{
		u64 s0, s1;	// an empty slot has no counters
		ld128 (&table[p].p, s0, s1);
		const u32 L = (u32) s0 & 0xFFFFFFu, R = (u32) s1 & 0xFFFFFFu;
		const u32 mk = g.mark[p], cm = mask[p];
		u32 nL = L, nR = R;
		if (mk)
			nL = nR = 0;
		else if (cm)
#pragma unroll
			for (int b = 0; b < 4; b++)
			{
				if ((cm >> b) & 1u)
					nL &= ~(63u << (6 * b));
				if ((cm >> (4 + b)) & 1u)
					nR &= ~(63u << (6 * b));
			}
		if (nL != L || nR != R)
			SlotIO<W>::set_links (table + p, nL, nR);
		if (mk)
			g.mark[p] = 0;
		if (cm)
			mask[p] = 0;
		n_removed += (L | R) && !(nL | nR);
		n_live += (nL | nR) != 0;
		n_lin += is_linear (nL, nR);
	}
	add_ctr (g.ctr + g.phase, n_removed);
	add_ctr (g.ctr + 5, n_live);
	add_ctr (g.ctr + 6, n_lin);
}

}	// namespace sdt
