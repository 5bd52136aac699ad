// sdt_lookup.cuh — read-only lookups in a finalized table (sdtgpu_lookup_kmers_device, sdtgpu_lookup_reads_device).
//
// The two insert paths leave their nodes in different places: the single-pass insert in a hashed table with empty
// slots, the sliced build in a compact node store ordered by work item.  One index serves both: an open-addressing
// array of u64 entries over the slots [0, iter_slots), entry = tag32 << 32 | position32, where tag32 is the low half
// of key_hash (slot_of takes the high bits) and the empty entry is all ones.  Linear probing from
// slot_of (key_hash, idx_cap), idx_cap = max (1024, 2 x nodes): load <= 0.5, 16 bytes per node.
//
// A probe loads an entry, compares the tag and only on a tag match loads the slot (ld256, .L2::64B) to compare the key.
// For keys of up to two words the payload is in the slot's 32-byte sector: a hit costs about two random requests, a
// miss about one (a 32-bit tag matches a foreign key once in 2^32 entries).
#pragma once
#include "sdt_device.cuh"

namespace sdt {

static constexpr u32 HIT_WINDOW = 1u, HIT_FOUND = 2u, HIT_RC = 4u;	// SDTGPU_HIT_*
static constexpr u64 IDX_EMPTY = ~0ull;

struct __align__(16) Hit { u32 count, l_links, rword, status; };	// sdtgpu_hit

// what a lookup needs besides the table (insert_reads_kernel MODE 6, lookup_kmers_kernel)
struct Lookup
{
	const u64 *index = nullptr;
	u64 idx_cap = 0;
	Hit *out = nullptr;
	int deLowKmer = 0;
};

// the raw kmer_t word behind l_links as sdtgpu_export_nodes reports it: r_links plus the linear, deleted and
// single flags of the post-pass (finalize has already applied the -d cutoff to the links)
__device__ __forceinline__ u32 node_rword (u32 L, u32 R, u32 count, int deLowKmer)
{
	u32 in_num = 0, out_num = 0;
#pragma unroll
	for (int b = 0; b < 4; b++)
	{
		in_num += ((L >> (6 * b)) & 63) > 0;
		out_num += ((R >> (6 * b)) & 63) > 0;
	}
	u32 rword = R;
	if (in_num == 1 && out_num == 1)
		rword |= 0x01000000u;	// linear  (thread_mark, prlHashReads.c:956-960)
	if (deLowKmer > 0 && L == 0 && R == 0)
		rword |= 0x02000000u;	// deleted (thread_delow, prlHashReads.c:876-880)
	if (count == 1)
		rword |= 0x08000000u;	// single  (newhash.c:39,103,445)
	return rword;
}

__device__ __forceinline__ u64 ld64_idx (const u64 *p)
{	// the index is read-only once built; a random 8-byte load fetches 64 bytes into L2, not a whole line
	u64 v;
	asm volatile ("ld.global.nc.L2::64B.u64 %0, [%1];" : "=l"(v) : "l"(p));
	return v;
}

// key words and payload of a slot of a finalized table; false if the slot is empty
template <int W> __device__ __forceinline__ bool load_slot (const typename SlotOf<W>::type *s, Key<W> &k, u64 &s0, u64 &s1)
{
	u64 a, b, c, d;
	ld256 (s, a, b, c, d);
	if constexpr (W == 1)
	{
		k.w[0] = a;
		s0 = c;
		s1 = d;
		return a != EMPTY64;
	}
	else if constexpr (W == 2)
	{
		k.w[0] = a;
		k.w[1] = b;
		s0 = c;
		s1 = d;
		return !(a == EMPTY64 && b == EMPTY64);
	}
	else
	{
		k.w[0] = a;
		k.w[1] = b;
		k.w[2] = c;
		k.w[3] = d;
		ld128 (&s->p, s0, s1);
		return !(a == EMPTY64 && b == EMPTY64);
	}
}

template <int W> __device__ __forceinline__ bool key_eq (const Key<W> &a, const Key<W> &b)
{
	bool eq = true;
#pragma unroll
	for (int i = 0; i < W; i++)
		eq &= a.w[i] == b.w[i];
	return eq;
}

// one entry per occupied slot of [0, slots); positions fit 32 bits (the host checks slots < 2^32 - 1)
template <int W>
__global__ void __launch_bounds__ (256)
index_build_kernel (const typename SlotOf<W>::type *table, u64 slots, u64 *index, u64 idx_cap)
{
	for (u64 i = blockIdx.x * (u64) blockDim.x + threadIdx.x; i < slots; i += (u64) gridDim.x * blockDim.x)
	{
		Key<W> k;
		u64 s0, s1;
		if (!load_slot<W> (table + i, k, s0, s1))
			continue;
		const u64 h = key_hash<W> (k);
		const u64 e = (h << 32) | i;
		u64 j = slot_of (h, idx_cap);
		while (atomicCAS (index + j, IDX_EMPTY, e) != IDX_EMPTY)
			if (++j == idx_cap)
				j = 0;
	}
}

// the canonical key `key` in the table?  status gets HIT_WINDOW | HIT_FOUND (and rc_flag); count, links, rword
// as the export reports them
template <int W>
__device__ __forceinline__ Hit index_probe (const typename SlotOf<W>::type *table, const Lookup &lk, const Key<W> &key, u32 rc_flag)
{
	Hit r = { 0, 0, 0, HIT_WINDOW | rc_flag };
	const u64 h = key_hash<W> (key);
	const u32 tag = (u32) h;
	u64 j = slot_of (h, lk.idx_cap);
	for (;;)
	{
		const u64 e = ld64_idx (lk.index + j);
		if (e == IDX_EMPTY)
			return r;
		if ((u32) (e >> 32) == tag)
		{
			Key<W> k;
			u64 s0, s1;
			load_slot<W> (table + (u32) e, k, s0, s1);
			if (key_eq<W> (k, key))
			{
				r.l_links = (u32) s0 & 0xFFFFFFu;
				r.count = (u32) (s1 >> 32);
				r.rword = node_rword (r.l_links, (u32) s1 & 0xFFFFFFu, r.count, lk.deLowKmer);
				r.status |= HIT_FOUND;
				return r;
			}
		}
		if (++j == lk.idx_cap)
			j = 0;
	}
}

__device__ __forceinline__ void store_hit (Hit *p, const Hit &h)
{
	*reinterpret_cast<uint4 *> (p) = make_uint4 (h.count, h.l_links, h.rword, h.status);
}

// arbitrary keys in the sdtgpu_node layout (key[0] most significant, the k-mer in the low 2K bits): validated,
// canonicalised (KmerSmaller of the k-mer and its reverse complement, as the chop does), looked up
template <int W>
__global__ void __launch_bounds__ (256)
lookup_kmers_kernel (const typename SlotOf<W>::type *table, Lookup lk, const u64 *keys, u64 n, int K)
{
	for (u64 i = blockIdx.x * (u64) blockDim.x + threadIdx.x; i < n; i += (u64) gridDim.x * blockDim.x)
	{
		const ulonglong2 lo = *reinterpret_cast<const ulonglong2 *> (keys + 4 * i);
		const ulonglong2 hi = *reinterpret_cast<const ulonglong2 *> (keys + 4 * i + 2);
		const u64 q[4] = { lo.x, lo.y, hi.x, hi.y };
		bool ok = true;
#pragma unroll
		for (int w = 0; w < 4; w++)
		{	// word w holds bits 64 (3 - w) .. 64 (3 - w) + 63 of the key; bits at 2K and above must be clear
			const int bits = 2 * K - 64 * (3 - w);
			if (bits <= 0)
				ok &= q[w] == 0;
			else if (bits < 64)
				ok &= (q[w] >> bits) == 0;
		}
		Hit r = { 0, 0, 0, 0 };
		if (ok)
		{
			Key<W> f, rc;
#pragma unroll
			for (int w = 0; w < W; w++)
				f.w[w] = q[4 - W + w];
			revcomp<W> (f, K, rc);
			const bool fwd = key_less<W> (f, rc);
			r = index_probe<W> (table, lk, fwd ? f : rc, fwd ? 0u : HIT_RC);
		}
		store_hit (lk.out + i, r);
	}
}

}	// namespace sdt
