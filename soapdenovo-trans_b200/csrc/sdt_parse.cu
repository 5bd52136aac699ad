// sdt_parse.cu — FASTA/FASTQ files parsed and 2-bit packed on the GPU (include/sdtgpu.h, sdtgpu_reader_*).
//
// The records, their order and every output byte equal what sdtpack_next (host/sdt_readpack.c, one thread,
// one batch) produces.  Per file the text goes to the device in chunks:
//   - the host fills a pinned staging buffer with parallel pread while the kernels of the current chunk run;
//   - a chunk = the unconsumed tail of the previous chunk (a device-to-device copy) + the next chunk_bytes of the
//     file (one cudaMemcpyAsync from the staging buffer).  It always starts at a record boundary: the first
//     unconsumed record (FASTQ) or just after the last consumed sequence line (FASTA), so no parser state crosses
//     chunks except "the first FASTQ header has not been found yet";
//   - a record is consumed when its lines end inside the chunk (FASTA: the sequence line; FASTQ: all four) or the
//     chunk reaches the end of the file.  A chunk that consumes nothing and skips nothing is followed by a larger
//     one (tail = the whole chunk); a junk line that runs past the chunk's end is skipped on the host, so junk never
//     makes a buffer grow.
// Kernels of a chunk, on the reader's stream: newline count per 4 KiB (16-byte loads) -> scan of the counts ->
// newline positions; FASTA: headers are the '>' lines at even offsets of their run of '>' lines, found by a scan of
// a two-state machine (P = "the next '>' line is a sequence line") and compacted into a list of header lines;
// FASTQ: every fourth line from the first header (found once per file by the find_header rule); then one thread
// decides how many records are consumed and where the next chunk starts.  The host reads that back (one small copy)
// and launches the pack kernel, one warp per record, on the caller's stream.
#include "../../include/sdtgpu.h"
#include <cuda_runtime.h>

#include <algorithm>
#include <cerrno>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fcntl.h>
#include <string>
#include <sys/stat.h>
#include <thread>
#include <unistd.h>
#include <vector>

namespace {

typedef unsigned long long u64;
typedef unsigned int u32;

constexpr u32 NONE = 0xFFFFFFFFu;
constexpr int NL_THREADS = 256;				// 16 text bytes each: 4 KiB per block
constexpr u64 NL_BLOCK_BYTES = 16 * NL_THREADS;
constexpr int LINE_THREADS = 256, LINES_PER_THREAD = 4;	// FASTA tiles of 1024 lines
constexpr u32 TILE_LINES = LINE_THREADS * LINES_PER_THREAD;
constexpr int PACK_WARPS = 8;
constexpr u64 DEFAULT_CHUNK = 64ull << 20;
constexpr u64 MAX_CHUNK = 0xFFFF0000ull;		// positions inside a chunk are 32-bit

// what the host reads back per chunk
struct ChunkRes
{
	u32 T;		// newlines in the chunk
	u32 n_lines;	// line starts < len
	u32 H;		// FASTA headers
	u32 h0;		// FASTQ: header line of record 0 (NONE: not found in the first chunk)
	u32 n_rec;	// records consumed
	u32 next;	// start of the next chunk, relative to this one
	u32 junk;	// the line at `next` is junk that runs past the chunk's end
	u32 found;	// FASTQ: the first header has been found
};

// ---- newline index

__device__ __forceinline__ u32 nl_nibble (u32 w)
{
	const u32 e = __vcmpeq4 (w, 0x0A0A0A0Au);
	return ((e >> 7) & 1u) | ((e >> 14) & 2u) | ((e >> 21) & 4u) | ((e >> 28) & 8u);
}

// bit k: text[pos + k] == '\n' and pos + k < len
__device__ __forceinline__ u32 nl_mask16 (const char *text, u64 pos, u32 len)
{
	if (pos >= len)
		return 0;
	const uint4 v = *reinterpret_cast<const uint4 *> (text + pos);
	u32 m = nl_nibble (v.x) | nl_nibble (v.y) << 4 | nl_nibble (v.z) << 8 | nl_nibble (v.w) << 12;
	if (len - pos < 16)
		m &= (1u << (len - pos)) - 1u;
	return m;
}

// exclusive scan of one u32 per thread over a block of `nthreads` (<= 1024); *total = the block's sum
__device__ __forceinline__ u32 block_excl_sum (u32 v, u32 *sh /* [33] */, u32 *total)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
	u32 inc = v;
	for (int d = 1; d < 32; d <<= 1)
	{
		const u32 o = __shfl_up_sync (0xFFFFFFFFu, inc, d);
		if (lane >= d)
			inc += o;
	}
	if (lane == 31)
		sh[warp] = inc;
	__syncthreads ();
	if (warp == 0)
	{
		const u32 w = lane < nw ? sh[lane] : 0;
		u32 wi = w;
		for (int d = 1; d < 32; d <<= 1)
		{
			const u32 o = __shfl_up_sync (0xFFFFFFFFu, wi, d);
			if (lane >= d)
				wi += o;
		}
		if (lane < nw)
			sh[lane] = wi - w;
		if (lane == 31)
			sh[32] = wi;
	}
	__syncthreads ();
	const u32 ex = sh[warp] + inc - v;
	*total = sh[32];
	__syncthreads ();
	return ex;
}

__global__ void __launch_bounds__ (NL_THREADS)
parse_nl_count_kernel (const char *text, u32 len, u32 *blk_cnt)
{
	__shared__ u32 sh[33];
	const u64 pos = ((u64) blockIdx.x * NL_THREADS + threadIdx.x) * 16;
	u32 total;
	block_excl_sum (__popc (nl_mask16 (text, pos, len)), sh, &total);
	if (threadIdx.x == 0)
		blk_cnt[blockIdx.x] = total;
}

// one block of 1024: exclusive scan of the per-block counts; the chunk's line counts and a fresh result record
__global__ void __launch_bounds__ (1024)
parse_nl_scan_kernel (const u32 *blk_cnt, u32 nb, u32 *blk_off, const char *text, u32 len, ChunkRes *res)
{
	__shared__ u32 sh[33];
	u32 carry = 0;
	for (u32 i0 = 0; i0 < nb; i0 += 1024)
	{
		const u32 i = i0 + threadIdx.x;
		const u32 v = i < nb ? blk_cnt[i] : 0;
		u32 total;
		const u32 ex = block_excl_sum (v, sh, &total);
		if (i < nb)
			blk_off[i] = carry + ex;
		carry += total;
	}
	if (threadIdx.x == 0)
	{
		ChunkRes r;
		r.T = carry;
		r.n_lines = carry + (len > 0 && text[len - 1] != '\n' ? 1u : 0u);
		r.H = 0;
		r.h0 = NONE;
		r.n_rec = r.next = r.junk = r.found = 0;
		*res = r;
	}
}

__global__ void __launch_bounds__ (NL_THREADS)
parse_nl_write_kernel (const char *text, u32 len, const u32 *blk_off, u32 *nl)
{
	__shared__ u32 sh[33];
	const u64 pos = ((u64) blockIdx.x * NL_THREADS + threadIdx.x) * 16;
	u32 m = nl_mask16 (text, pos, len), total;
	u32 o = blk_off[blockIdx.x] + block_excl_sum (__popc (m), sh, &total);
	for (; m; m &= m - 1)
		nl[o++] = (u32) pos + (u32) __ffs (m) - 1;
}

__device__ __forceinline__ u32 line_start (const u32 *nl, u32 j) { return j ? nl[j - 1] + 1 : 0; }

// ---- FASTA headers.  State P before a line: 1 if a '>' line there would be the sequence line of the header just
// before it.  A '>' line with P = 0 is a header and sets P = 1; any other line sets P = 0.  Tr is such a step
// (or a run of steps) as a function of the state it starts in: f bit P = state after, c_P = headers passed.

struct Tr
{
	u32 f, c0, c1;
};

__device__ __forceinline__ Tr tr_id () { return Tr{2u, 0u, 0u}; }
__device__ __forceinline__ Tr tr_line (bool gt) { return gt ? Tr{1u, 1u, 0u} : Tr{0u, 0u, 0u}; }
__device__ __forceinline__ u32 tr_state (Tr t, u32 P) { return (t.f >> P) & 1u; }
__device__ __forceinline__ u32 tr_count (Tr t, u32 P) { return P ? t.c1 : t.c0; }

// a, then b
__device__ __forceinline__ Tr tr_then (Tr a, Tr b)
{
	const u32 a0 = a.f & 1u, a1 = (a.f >> 1) & 1u;
	return Tr{tr_state (b, a0) | tr_state (b, a1) << 1, a.c0 + tr_count (b, a0), a.c1 + tr_count (b, a1)};
}

__device__ __forceinline__ Tr tr_shfl_up (Tr t, int d)
{
	return Tr{__shfl_up_sync (0xFFFFFFFFu, t.f, d), __shfl_up_sync (0xFFFFFFFFu, t.c0, d), __shfl_up_sync (0xFFFFFFFFu, t.c1, d)};
}

__device__ __forceinline__ Tr tr_warp_incl (Tr t)
{
	const int lane = threadIdx.x & 31;
	for (int d = 1; d < 32; d <<= 1)
	{
		const Tr o = tr_shfl_up (t, d);
		if (lane >= d)
			t = tr_then (o, t);
	}
	return t;
}

// exclusive scan over a block of LINE_THREADS
__device__ __forceinline__ Tr tr_block_excl (Tr t, Tr *sh /* [17] */, Tr *total)
{
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = LINE_THREADS / 32;
	const Tr inc = tr_warp_incl (t);
	if (lane == 31)
		sh[warp] = inc;
	__syncthreads ();
	if (warp == 0)
	{
		const Tr wi = tr_warp_incl (lane < nw ? sh[lane] : tr_id ());
		Tr we = tr_shfl_up (wi, 1);
		if (lane == 0)
			we = tr_id ();
		if (lane < nw)
			sh[nw + lane] = we;
		if (lane == nw - 1)
			sh[2 * nw] = wi;
	}
	__syncthreads ();
	Tr ex = tr_shfl_up (inc, 1);
	if (lane == 0)
		ex = tr_id ();
	*total = sh[2 * nw];
	return tr_then (sh[nw + warp], ex);
}

__device__ __forceinline__ bool is_gt (const char *text, const u32 *nl, u32 j, u32 n_lines)
{
	return j < n_lines && text[line_start (nl, j)] == '>';
}

__device__ __forceinline__ Tr fa_thread_lines (const char *text, const u32 *nl, u32 n_lines, u32 j0)
{
	Tr t = tr_id ();
#pragma unroll
	for (int k = 0; k < LINES_PER_THREAD; k++)
		t = tr_then (t, tr_line (is_gt (text, nl, j0 + k, n_lines)));
	return t;
}

__global__ void __launch_bounds__ (LINE_THREADS)
parse_fa_tile_kernel (const char *text, const u32 *nl, u32 n_lines, Tr *agg)
{
	__shared__ Tr sh[17];
	const u32 j0 = blockIdx.x * TILE_LINES + threadIdx.x * LINES_PER_THREAD;
	Tr total;
	tr_block_excl (fa_thread_lines (text, nl, n_lines, j0), sh, &total);
	if (threadIdx.x == 0)
		agg[blockIdx.x] = total;
}

// one warp: state and header count at the start of every tile; res->H = all headers
__global__ void parse_fa_tiles_scan_kernel (const Tr *agg, u32 nt, u32 *tile_state, u32 *tile_count, ChunkRes *res)
{
	const int lane = threadIdx.x;
	Tr carry = tr_id ();
	for (u32 i0 = 0; i0 < nt; i0 += 32)
	{
		const u32 i = i0 + lane;
		const Tr inc = tr_warp_incl (i < nt ? agg[i] : tr_id ());
		Tr ex = tr_shfl_up (inc, 1);
		if (lane == 0)
			ex = tr_id ();
		ex = tr_then (carry, ex);
		if (i < nt)
		{
			tile_state[i] = tr_state (ex, 0);
			tile_count[i] = tr_count (ex, 0);
		}
		const Tr all = Tr{__shfl_sync (0xFFFFFFFFu, inc.f, 31), __shfl_sync (0xFFFFFFFFu, inc.c0, 31), __shfl_sync (0xFFFFFFFFu, inc.c1, 31)};
		carry = tr_then (carry, all);
	}
	if (lane == 0)
		res->H = tr_count (carry, 0);
}

__global__ void __launch_bounds__ (LINE_THREADS)
parse_fa_headers_kernel (const char *text, const u32 *nl, u32 n_lines, const u32 *tile_state, const u32 *tile_count, u32 *hdr_line)
{
	__shared__ Tr sh[17];
	const u32 j0 = blockIdx.x * TILE_LINES + threadIdx.x * LINES_PER_THREAD;
	Tr total;
	const Tr ex = tr_block_excl (fa_thread_lines (text, nl, n_lines, j0), sh, &total);
	const u32 Pb = tile_state[blockIdx.x];
	u32 P = tr_state (ex, Pb), c = tile_count[blockIdx.x] + tr_count (ex, Pb);
#pragma unroll
	for (int k = 0; k < LINES_PER_THREAD; k++)
	{
		const bool gt = is_gt (text, nl, j0 + k, n_lines);
		if (gt && P == 0)
			hdr_line[c++] = j0 + k;
		P = gt ? P ^ 1u : 0u;
	}
}

// ---- FASTQ: the first '@' line whose line two further down starts with '+' or is not in the chunk
__global__ void __launch_bounds__ (256)
parse_fq_find_kernel (const char *text, const u32 *nl, u32 n_lines, ChunkRes *res)
{
	const u32 i = blockIdx.x * 256 + threadIdx.x;
	if (i >= n_lines || text[line_start (nl, i)] != '@')
		return;
	if (i + 2 >= n_lines || text[line_start (nl, i + 2)] == '+')
		atomicMin (&res->h0, i);
}

// records consumed and where the next chunk starts
__global__ void parse_finalize_kernel (int fastq, int first, int eof, u32 len, const u32 *nl, const u32 *hdr_line, ChunkRes *res)
{
	ChunkRes r = *res;
	const u32 T = r.T;
	auto start = [&] (u32 j) { return j <= T ? line_start (nl, j) : len; };
	r.n_rec = 0;
	r.junk = 0;
	if (!fastq)
	{
		const u32 H = r.H;
		if (eof)
		{
			r.n_rec = H;
			r.next = len;
		}
		else
		{
			r.n_rec = H && hdr_line[H - 1] + 1 >= T ? H - 1 : H;	// only the last header can lack a complete sequence line
			if (r.n_rec)
				r.next = start (hdr_line[r.n_rec - 1] + 2);
			else if (H)
				r.next = start (hdr_line[0]);
			else
			{
				r.next = start (T);
				r.junk = r.next < len;
			}
		}
		r.h0 = 0;
		*res = r;
		return;
	}
	u32 h0 = 0;
	r.found = 1;
	if (first)
	{
		h0 = r.h0;
		if (h0 == NONE)
		{	// nothing but lines that are not headers
			r.found = 0;
			r.next = eof ? len : start (T);
			r.junk = !eof && r.next < len;
			*res = r;
			return;
		}
		if (!eof && h0 + 2 >= r.n_lines)
		{	// undecided: the line two further down is not in the chunk yet
			r.found = 0;
			r.next = start (h0);
			*res = r;
			return;
		}
	}
	r.h0 = h0;
	if (eof)
	{
		r.n_rec = r.n_lines > h0 ? (r.n_lines - h0 + 3) / 4 : 0;
		r.next = len;
	}
	else
	{
		r.n_rec = T >= h0 ? (T - h0) / 4 : 0;
		r.next = start (h0 + 4 * r.n_rec);
	}
	*res = r;
}

// ---- a shard's summary (sdtgpu_reader_summary): per piece of the rank's byte range, the lines j_lo .. n_lines - 1
// of the piece (line 0 is not a line start of the file when the byte before the piece is not '\n')
struct SumRes
{
	Tr tr;			// FASTA: the lines as one transfer function
	u32 first;		// start of line j_lo (NONE: the piece holds no line start)
	u32 open[2];		// FASTQ: start of the '@' line n_lines - 2 + k if its line two further down is not in the piece
	u64 cand;		// FASTQ: (line << 32 | start) of the first '@' line whose line two further down starts with '+'
};

__global__ void __launch_bounds__ (LINE_THREADS)
shard_fa_tile_kernel (const char *text, const u32 *nl, u32 j_lo, u32 n_lines, Tr *agg)
{
	__shared__ Tr sh[17];
	const u32 j0 = blockIdx.x * TILE_LINES + threadIdx.x * LINES_PER_THREAD;
	Tr t = tr_id ();
#pragma unroll
	for (int k = 0; k < LINES_PER_THREAD; k++)
		if (j0 + k >= j_lo && j0 + k < n_lines)
			t = tr_then (t, tr_line (text[line_start (nl, j0 + k)] == '>'));
	Tr total;
	tr_block_excl (t, sh, &total);
	if (threadIdx.x == 0)
		agg[blockIdx.x] = total;
}

// one warp: the tiles composed into res->tr, and the piece's first line start
__global__ void shard_piece_kernel (const Tr *agg, u32 nt, const u32 *nl, u32 j_lo, u32 n_lines, SumRes *res)
{
	const int lane = threadIdx.x;
	Tr carry = tr_id ();
	for (u32 i0 = 0; i0 < nt; i0 += 32)
	{
		const Tr inc = tr_warp_incl (i0 + lane < nt ? agg[i0 + lane] : tr_id ());
		carry = tr_then (carry, Tr{__shfl_sync (0xFFFFFFFFu, inc.f, 31), __shfl_sync (0xFFFFFFFFu, inc.c0, 31), __shfl_sync (0xFFFFFFFFu, inc.c1, 31)});
	}
	if (lane == 0)
	{
		res->tr = carry;
		res->first = j_lo < n_lines ? line_start (nl, j_lo) : NONE;
	}
}

// the parse_fq_find_kernel rule from line j_lo on; lines whose line two further down lies past the piece are left to
// the host, which reads on in the file
__global__ void __launch_bounds__ (256)
shard_fq_find_kernel (const char *text, const u32 *nl, u32 j_lo, u32 n_lines, SumRes *res)
{
	const u32 i = j_lo + blockIdx.x * 256 + threadIdx.x;
	if (i >= n_lines || text[line_start (nl, i)] != '@')
		return;
	if (i + 2 >= n_lines)
		res->open[i + 2 - n_lines] = line_start (nl, i);
	else if (text[line_start (nl, i + 2)] == '+')
		atomicMin (&res->cand, (u64) i << 32 | line_start (nl, i));
}

// ---- pack: one warp per record, straight to its output row

__device__ __forceinline__ u32 base_code (u32 c, int n_kmer)
{
	if (n_kmer && (c == 'N' || c == 'n'))
		return 4;
	if (c >= 'a' && c <= 'z')
		c -= 'a' - 'A';
	if (c >= 'A' && c <= 'Z')
		return (c & 6u) >> 1;
	return c == '.' ? 0u : 0xFFu;
}

struct PackArgs
{
	const char *text;
	const u32 *nl, *hdr_line;	// hdr_line == NULL: FASTQ, header of record r at line h0 + 4r
	u32 h0, T, len;
	u32 r0, n;			// records r0 .. r0 + n - 1 of the chunk
	u64 out0, out_step;		// go to output rows out0 + i * out_step
	u32 max_read_len, stride;
	int reverse, n_kmer;
	uint8_t *packed, *nmask;
	uint32_t *lens;
};

__global__ void __launch_bounds__ (PACK_WARPS * 32)
parse_pack_kernel (PackArgs a)
{
	extern __shared__ u32 smem[];
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const u32 i = blockIdx.x * PACK_WARPS + warp;
	if (i >= a.n)
		return;
	const u32 pk_words = a.stride / 4, nm_bytes = a.stride / 2, nm_words = a.nmask ? (nm_bytes + 3) / 4 : 0;
	u32 *pk = smem + (size_t) warp * (pk_words + (a.nmask ? (nm_bytes + 3) / 4 : 0)), *nm = pk + pk_words;
	for (u32 w = lane; w < pk_words + nm_words; w += 32)
		pk[w] = 0;
	const u32 r = a.r0 + i;
	const u32 line = (a.hdr_line ? a.hdr_line[r] : a.h0 + 4 * r) + 1;
	const u32 s = line <= a.T ? line_start (a.nl, line) : a.len;
	const u32 e = line < a.T ? a.nl[line] : a.len;
	const u32 raw = min (e - s, a.max_read_len);	// truncation counts raw characters
	const unsigned char *src = reinterpret_cast<const unsigned char *> (a.text) + s;
	u32 n = 0;
	if (a.reverse)
		for (u32 b = 0; b < raw; b += 32)
			n += __popc (__ballot_sync (0xFFFFFFFFu, b + lane < raw && base_code (src[b + lane], a.n_kmer) != 0xFFu));
	__syncwarp ();
	u32 q0 = 0;
	for (u32 b = 0; b < raw; b += 32)
	{
		const u32 c = b + lane < raw ? base_code (src[b + lane], a.n_kmer) : 0xFFu;
		const u32 m = __ballot_sync (0xFFFFFFFFu, c != 0xFFu);
		if (c != 0xFFu)
		{
			const u32 q = q0 + __popc (m & ((1u << lane) - 1u));
			const u32 oq = a.reverse ? n - 1 - q : q;
			const u32 oc = a.reverse && c < 4 ? c ^ 2u : c;
			atomicOr (&pk[oq >> 4], (oc & 3u) << (8 * ((oq >> 2) & 3) + 6 - 2 * (oq & 3)));
			if (oc == 4 && a.nmask)
				atomicOr (&nm[oq >> 5], 1u << (8 * ((oq >> 3) & 3) + 7 - (oq & 7)));
		}
		q0 += __popc (m);
	}
	__syncwarp ();
	const u64 row = a.out0 + (u64) i * a.out_step;
	u32 *dst = reinterpret_cast<u32 *> (a.packed + row * a.stride);
	for (u32 w = lane; w < pk_words; w += 32)
		dst[w] = pk[w];
	if (a.nmask)
		for (u32 b = lane; b < nm_bytes; b += 32)
			a.nmask[row * nm_bytes + b] = (uint8_t) (nm[b >> 2] >> (8 * (b & 3)));
	if (lane == 0)
		a.lens[row] = a.reverse ? n : q0;
}

thread_local std::string g_reader_open_error;	// the last sdtgpu_reader_open failure

struct Slot
{	// one chunk on the device; two per file, used in turn
	char *text = nullptr;
	u64 text_cap = 0;
	u32 *nl = nullptr, *hdr = nullptr;
	u64 nl_cap = 0, hdr_cap = 0;
	cudaEvent_t packed = nullptr;	// the caller's stream has finished the packs that read this slot
};

struct File
{
	int fd = -1;
	u64 size = 0;
	std::string path;
	char *stage[2] = {nullptr, nullptr};	// pinned
	u64 stage_off[2] = {0, 0}, stage_len[2] = {0, 0};
	int stage_next = 0;			// staging buffer of the next upload
	Slot slot[2];
	u32 *scratch = nullptr;			// per 4 KiB block counts and offsets, per tile aggregates
	u64 scratch_cap = 0;
	ChunkRes *d_res = nullptr, *h_res = nullptr;
	int cur = -1;				// slot of the current chunk (-1: none yet)
	u64 chunk_start = 0;
	u32 len = 0, cursor = 0;
	ChunkRes res{};
	bool eof = false, first = true;
	// a shard reader's position: the first chunk starts at `origin`, the next record is record `rec` of the file,
	// and `left` more records may be taken (ALL: no budget, a plain reader)
	u64 origin = 0, rec = 0, left = ~0ull;
	bool placed = false;
	u64 fingerprint = 0;
	bool exhausted () const { return left == 0 || (cur >= 0 && eof && cursor == res.n_rec); }
};

constexpr u64 ALL = ~0ull;
constexpr u64 SUM_MAGIC = 0x31304d5553544453ull;	// "SDTSUM01"

// a run of FASTA lines as a function of the state before it, with 64-bit header counts (host side of Tr)
struct Tr64
{
	u32 f = 2;
	u64 c0 = 0, c1 = 0;
	u32 state (u32 P) const { return (f >> P) & 1u; }
	u64 count (u32 P) const { return P ? c1 : c0; }
	Tr64 then (const Tr64 &b) const
	{
		const u32 a0 = f & 1u, a1 = (f >> 1) & 1u;
		Tr64 t;
		t.f = b.state (a0) | b.state (a1) << 1;
		t.c0 = c0 + b.count (a0);
		t.c1 = c1 + b.count (a1);
		return t;
	}
};

// what a summary holds per file (sdtgpu_reader_summary), for this rank's range of it
struct FileSum
{
	u64 first = ALL;	// offset of the range's first line start (ALL: none)
	u64 n_lines = 0;	// line starts in the range
	Tr64 tr;		// FASTA: those lines
	u64 cand = ALL;		// FASTQ: offset of the first header candidate (ALL: none) ...
	u64 cand_line = 0;	// ... and its line number in the range
};

// where a shard reader enters the ranges of a file: the record numbers before every range (c[q], q = 0 .. world)
// and the start of range q's first record, `skip` lines after its first line start `off`
struct FilePlan
{
	std::vector<u64> c, off;
	std::vector<uint8_t> skip;
};

// records k0 .. k1 - 1 of one file (file 0 or 1), or of both alternately (file -1, a pair segment); ordinals from ord0
struct Seg
{
	int file = 0;
	u64 k0 = 0, k1 = 0, ord0 = 0;
	u64 size () const { return (file < 0 ? 2 : 1) * (k1 - k0); }
};

}	// namespace

struct sdtgpu_reader
{
	int device = 0, n_files = 1, fastq = 0;
	u64 chunk_bytes = DEFAULT_CHUNK, stage_bytes = 0;
	File f[2];
	bool cuda_ready = false;
	cudaStream_t stream = nullptr;
	u64 stats[4] = {0, 0, 0, 0};
	std::string err;
	// shard readers (sdtgpu_reader_open_shard): world = 0 is a plain reader
	int rank = 0, world = 0;
	bool summarized = false, planned = false;
	uint8_t summary[SDTGPU_READER_SUMMARY_BYTES] = {};
	FilePlan plan[2];
	Seg seg[3];			// pairs (or the one file's records), drain, and an empty one past the end
	int seg_i = 0;			// the current segment
	u64 seg_done = 0;		// records of it returned
	bool seg_ready = false;		// the files are placed for it
	SumRes *d_sum = nullptr, *h_sum = nullptr;
};

namespace {

#define RCK(r, call)                                                                                    \
	do                                                                                              \
	{                                                                                               \
		cudaError_t e_ = (call);                                                                \
		if (e_ != cudaSuccess)                                                                  \
		{                                                                                       \
			char b_[512];                                                                   \
			snprintf (b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString (e_), __FILE__, __LINE__); \
			(r)->err = b_;                                                                  \
			return e_ == cudaErrorMemoryAllocation ? SDTGPU_ENOMEM : SDTGPU_ECUDA;          \
		}                                                                                       \
	} while (0)

int reader_fail (sdtgpu_reader *r, int code, const std::string &msg)
{
	r->err = msg;
	return code;
}

// [off, off + len) of the file into dst, by several threads for large ranges
int read_range (sdtgpu_reader *r, File &f, char *dst, u64 off, u64 len)
{
	auto piece = [&f] (char *d, u64 o, u64 n) -> bool {
		while (n)
		{
			const ssize_t got = pread (f.fd, d, (size_t) std::min<u64> (n, 1ull << 30), (off_t) o);
			if (got < 0 && errno == EINTR)
				continue;
			if (got <= 0)
				return false;
			d += got; o += (u64) got; n -= (u64) got;
		}
		return true;
	};
	const unsigned hw = std::max (1u, std::thread::hardware_concurrency ());
	const u64 nt = len < (4ull << 20) ? 1 : std::min<u64> ({8, hw, len >> 20});
	bool ok = true;
	if (nt == 1)
		ok = piece (dst, off, len);
	else
	{
		const u64 per = (len + nt - 1) / nt;
		std::vector<char> oks (nt, 1);
		std::vector<std::thread> th;
		for (u64 t = 1; t < nt; t++)
		{
			const u64 a = t * per, b = std::min (len, a + per);
			th.emplace_back ([&, t, a, b] { oks[t] = a < b ? piece (dst + a, off + a, b - a) : true; });
		}
		oks[0] = piece (dst, off, std::min (len, per));
		for (auto &x : th)
			x.join ();
		for (char o : oks)
			ok = ok && o;
	}
	return ok ? SDTGPU_OK : reader_fail (r, SDTGPU_EINVAL, "cannot read " + f.path + ": " + strerror (errno ? errno : EIO));
}

// staging buffer si holds [off, off + min (stage_bytes, size - off))
int fill_stage (sdtgpu_reader *r, File &f, int si, u64 off)
{
	const u64 n = std::min (r->stage_bytes, f.size - off);
	f.stage_off[si] = off;
	f.stage_len[si] = 0;
	if (n && read_range (r, f, f.stage[si], off, n))
		return SDTGPU_EINVAL;
	f.stage_len[si] = n;
	return SDTGPU_OK;
}

// position after the first '\n' at or after off (or the file size)
int skip_line (sdtgpu_reader *r, File &f, u64 off, u64 *out)
{
	std::vector<char> buf (1 << 16);
	while (off < f.size)
	{
		const u64 n = std::min<u64> (buf.size (), f.size - off);
		if (read_range (r, f, buf.data (), off, n))
			return SDTGPU_EINVAL;
		const char *nl = static_cast<const char *> (memchr (buf.data (), '\n', n));
		if (nl)
		{
			*out = off + (u64) (nl - buf.data ()) + 1;
			return SDTGPU_OK;
		}
		off += n;
	}
	*out = f.size;
	return SDTGPU_OK;
}

int grow (sdtgpu_reader *r, Slot &s, void **p, u64 *cap, u64 need_bytes)
{
	if (*cap >= need_bytes)
		return SDTGPU_OK;
	RCK (r, cudaEventSynchronize (s.packed));
	if (*p)
		RCK (r, cudaFree (*p));
	*p = nullptr;
	*cap = 0;
	const u64 want = need_bytes + need_bytes / 4 + 4096;	// room for chunks a little larger than this one
	RCK (r, cudaMalloc (p, want));
	*cap = want;
	r->stats[3]++;
	return SDTGPU_OK;
}

int grow_scratch (sdtgpu_reader *r, File &f, u64 text_cap)
{
	const u64 need = (2 * (text_cap / NL_BLOCK_BYTES + 2) + 5 * (text_cap / TILE_LINES + 2)) * sizeof (u32);
	if (f.scratch_cap >= need)
		return SDTGPU_OK;
	RCK (r, cudaStreamSynchronize (r->stream));
	if (f.scratch)
		RCK (r, cudaFree (f.scratch));
	f.scratch = nullptr;
	f.scratch_cap = 0;
	RCK (r, cudaMalloc (&f.scratch, need));
	f.scratch_cap = need;
	r->stats[3]++;
	return SDTGPU_OK;
}

#define RET(x)                              \
	do                                  \
	{                                   \
		const int rc_ = (x);        \
		if (rc_)                    \
			return rc_;         \
	} while (0)

// uploads and indexes the next chunk of file f
int load_chunk (sdtgpu_reader *r, File &f)
{
	const bool have = f.cur >= 0;
	u64 start = f.origin, tail = 0;
	if (have)
	{
		start = f.chunk_start + f.res.next;
		tail = f.len - f.res.next;
		if (f.res.junk)
		{	// a junk line runs past the chunk: skip it here instead of growing the chunk over it
			RET (skip_line (r, f, f.chunk_start + f.len, &start));
			tail = 0;
		}
	}
	const u64 fresh_off = start + tail;
	const u64 fresh = std::min (r->chunk_bytes, f.size - fresh_off);
	const u64 len = tail + fresh;
	if (len > MAX_CHUNK)
		return reader_fail (r, SDTGPU_ERANGE, "a record of " + f.path + " is longer than 4 GiB");
	const int si = f.stage_next;
	if (f.stage_off[si] != fresh_off || f.stage_len[si] < fresh)
		RET (fill_stage (r, f, si, fresh_off));
	const int q = have ? f.cur ^ 1 : 0;
	Slot &S = f.slot[q];
	if (!have)
	{	// both slots at once, so that steady state allocates nothing
		const u64 cap0 = std::min (2 * r->chunk_bytes, f.size) + 64;
		for (Slot &s : f.slot)
			RET (grow (r, s, (void **) &s.text, &s.text_cap, cap0));
	}
	RET (grow (r, S, (void **) &S.text, &S.text_cap, len + 64));
	RET (grow_scratch (r, f, S.text_cap));
	RCK (r, cudaStreamWaitEvent (r->stream, S.packed, 0));
	if (tail)
		RCK (r, cudaMemcpyAsync (S.text, f.slot[f.cur].text + f.res.next, tail, cudaMemcpyDeviceToDevice, r->stream));
	if (fresh)
		RCK (r, cudaMemcpyAsync (S.text + tail, f.stage[si], fresh, cudaMemcpyHostToDevice, r->stream));
	r->stats[0] += fresh;
	r->stats[2]++;
	f.stage_next ^= 1;
	const u32 L = (u32) len;
	const u32 nb = (u32) ((len + NL_BLOCK_BYTES - 1) / NL_BLOCK_BYTES);
	u32 *blk_cnt = f.scratch, *blk_off = f.scratch + nb;
	if (nb)
	{
		parse_nl_count_kernel<<<nb, NL_THREADS, 0, r->stream>>> (S.text, L, blk_cnt);
		parse_nl_scan_kernel<<<1, 1024, 0, r->stream>>> (blk_cnt, nb, blk_off, S.text, L, f.d_res);
	}
	else
		RCK (r, cudaMemsetAsync (f.d_res, 0, sizeof (ChunkRes), r->stream));
	RCK (r, cudaGetLastError ());
	RCK (r, cudaMemcpyAsync (f.h_res, f.d_res, sizeof (ChunkRes), cudaMemcpyDeviceToHost, r->stream));
	// while that runs: the bytes after this chunk, which the next chunk most likely starts with
	if (fresh_off + fresh < f.size)
		RET (fill_stage (r, f, f.stage_next, fresh_off + fresh));
	RCK (r, cudaStreamSynchronize (r->stream));
	const u32 T = f.h_res->T, n_lines = f.h_res->n_lines;
	const bool eof = fresh_off + fresh == f.size;
	RET (grow (r, S, (void **) &S.nl, &S.nl_cap, ((u64) T + 1) * sizeof (u32)));
	if (!r->fastq)
		RET (grow (r, S, (void **) &S.hdr, &S.hdr_cap, ((u64) n_lines / 2 + 2) * sizeof (u32)));
	if (nb)
	{
		parse_nl_write_kernel<<<nb, NL_THREADS, 0, r->stream>>> (S.text, L, blk_off, S.nl);
		const u32 nt = (n_lines + TILE_LINES - 1) / TILE_LINES;
		if (!r->fastq && nt)
		{
			u32 *tstate = blk_off + nb, *tcount = tstate + nt;
			Tr *agg = reinterpret_cast<Tr *> (tcount + nt);
			parse_fa_tile_kernel<<<nt, LINE_THREADS, 0, r->stream>>> (S.text, S.nl, n_lines, agg);
			parse_fa_tiles_scan_kernel<<<1, 32, 0, r->stream>>> (agg, nt, tstate, tcount, f.d_res);
			parse_fa_headers_kernel<<<nt, LINE_THREADS, 0, r->stream>>> (S.text, S.nl, n_lines, tstate, tcount, S.hdr);
		}
		if (r->fastq && f.first && n_lines)
			parse_fq_find_kernel<<<(n_lines + 255) / 256, 256, 0, r->stream>>> (S.text, S.nl, n_lines, f.d_res);
		parse_finalize_kernel<<<1, 1, 0, r->stream>>> (r->fastq, f.first, eof, L, S.nl, S.hdr, f.d_res);
		RCK (r, cudaGetLastError ());
		RCK (r, cudaMemcpyAsync (f.h_res, f.d_res, sizeof (ChunkRes), cudaMemcpyDeviceToHost, r->stream));
		RCK (r, cudaStreamSynchronize (r->stream));
		f.res = *f.h_res;
	}
	else
		f.res = ChunkRes{};
	if (r->fastq && f.first && f.res.found)
		f.first = false;
	f.cur = q;
	f.chunk_start = start;
	f.len = L;
	f.eof = eof;
	f.cursor = 0;
	return SDTGPU_OK;
}

// loads chunks until file f has a record to give or has none left
int fill (sdtgpu_reader *r, File &f)
{
	while (!(f.cur >= 0 && f.cursor < f.res.n_rec) && !f.exhausted ())
		RET (load_chunk (r, f));
	if (f.left != ALL && f.left && f.exhausted ())
		return reader_fail (r, SDTGPU_ESTATE, f.path + " holds fewer records than the summaries counted (did it change?)");
	return SDTGPU_OK;
}

struct Out
{
	uint8_t *packed, *nmask;
	uint32_t *lens;
	int max_read_len, n_kmer, reverse;
	u32 stride;
	cudaStream_t stream;
	size_t smem;
};

int pack (sdtgpu_reader *r, File &f, u32 n, u64 out0, u64 step, const Out &o)
{
	Slot &S = f.slot[f.cur];
	PackArgs a;
	a.text = S.text;
	a.nl = S.nl;
	a.hdr_line = r->fastq ? nullptr : S.hdr;
	a.h0 = f.res.h0;
	a.T = f.res.T;
	a.len = f.len;
	a.r0 = f.cursor;
	a.n = n;
	a.out0 = out0;
	a.out_step = step;
	a.max_read_len = (u32) o.max_read_len;
	a.stride = o.stride;
	a.reverse = o.reverse;
	a.n_kmer = o.n_kmer;
	a.packed = o.packed;
	a.nmask = o.n_kmer ? o.nmask : nullptr;
	a.lens = o.lens;
	parse_pack_kernel<<<(n + PACK_WARPS - 1) / PACK_WARPS, PACK_WARPS * 32, o.smem, o.stream>>> (a);
	RCK (r, cudaGetLastError ());
	RCK (r, cudaEventRecord (S.packed, o.stream));
	f.cursor += n;
	f.rec += n;
	if (f.left != ALL)
		f.left -= n;
	r->stats[1] += n;
	r->seg_done += n;
	return SDTGPU_OK;
}

int init_cuda (sdtgpu_reader *r)
{
	RCK (r, cudaStreamCreateWithFlags (&r->stream, cudaStreamNonBlocking));
	u64 biggest = 0;
	for (int i = 0; i < r->n_files; i++)
		biggest = std::max (biggest, r->f[i].size);
	r->stage_bytes = std::max<u64> (1, std::min (r->chunk_bytes, biggest));
	for (int i = 0; i < r->n_files; i++)
	{
		File &f = r->f[i];
		for (int k = 0; k < 2; k++)
		{
			RCK (r, cudaHostAlloc ((void **) &f.stage[k], r->stage_bytes, cudaHostAllocDefault));
			f.stage_off[k] = ~0ull;
			RCK (r, cudaEventCreateWithFlags (&f.slot[k].packed, cudaEventDisableTiming));
		}
		RCK (r, cudaHostAlloc ((void **) &f.h_res, sizeof (ChunkRes), cudaHostAllocDefault));
		RCK (r, cudaMalloc ((void **) &f.d_res, sizeof (ChunkRes)));
	}
	if (r->world)
	{
		RCK (r, cudaHostAlloc ((void **) &r->h_sum, sizeof (SumRes), cudaHostAllocDefault));
		RCK (r, cudaMalloc ((void **) &r->d_sum, sizeof (SumRes)));
	}
	r->cuda_ready = true;
	return SDTGPU_OK;
}

// ---- shard readers: a summary of this rank's byte range of each file, a plan from every rank's summary, and the
// segments of records this rank returns

// rank q's range of a file of `size` bytes starts here
u64 range_lo (u64 size, int q, int world) { return (u64) ((unsigned __int128) size * (u64) q / (u64) world); }

// FNV-1a of the first and last 4 KiB: tells two files of the same size apart in nearly every case
int fingerprint (sdtgpu_reader *r, File &f)
{
	const u64 n = std::min<u64> (4096, f.size);
	std::vector<char> b (2 * n);
	if (n)
	{
		RET (read_range (r, f, b.data (), 0, n));
		RET (read_range (r, f, b.data () + n, f.size - n, n));
	}
	u64 h = 0xcbf29ce484222325ull;
	for (char c : b)
		h = (h ^ (unsigned char) c) * 0x100000001b3ull;
	f.fingerprint = h;
	return SDTGPU_OK;
}

// FASTQ header rule for the '@' line at p, on the host: the line two further down starts with '+' or is past the end
int fq_rule_on_host (sdtgpu_reader *r, File &f, u64 p, bool *yes)
{
	u64 q;
	RET (skip_line (r, f, p, &q));
	RET (skip_line (r, f, q, &q));
	char c = 0;
	if (q < f.size)
		RET (read_range (r, f, &c, q, 1));
	*yes = q >= f.size || c == '+';
	return SDTGPU_OK;
}

// this rank's range of f, streamed through the device in pieces of at most stage_bytes: line starts, the FASTA
// transfer function of those lines and the first FASTQ header candidate
int summarize_file (sdtgpu_reader *r, File &f, FileSum &s)
{
	s = FileSum{};
	const u64 a = range_lo (f.size, r->rank, r->world), b = range_lo (f.size, r->rank + 1, r->world);
	if (a >= b)
		return SDTGPU_OK;
	char prev = '\n';	// the byte before the piece; offset 0 starts a line
	if (a)
		RET (read_range (r, f, &prev, a - 1, 1));
	Slot &S = f.slot[0];
	for (u64 x = a; x < b;)
	{
		const u64 n = std::min (r->stage_bytes, b - x);
		const int si = f.stage_next;
		if (f.stage_off[si] != x || f.stage_len[si] < n)
			RET (fill_stage (r, f, si, x));
		RET (grow (r, S, (void **) &S.text, &S.text_cap, n + 64));
		RET (grow_scratch (r, f, S.text_cap));
		RCK (r, cudaMemcpyAsync (S.text, f.stage[si], n, cudaMemcpyHostToDevice, r->stream));
		r->stats[0] += n;
		r->stats[2]++;
		f.stage_next ^= 1;
		const u32 L = (u32) n, nb = (u32) ((n + NL_BLOCK_BYTES - 1) / NL_BLOCK_BYTES);
		u32 *blk_cnt = f.scratch, *blk_off = f.scratch + nb;
		parse_nl_count_kernel<<<nb, NL_THREADS, 0, r->stream>>> (S.text, L, blk_cnt);
		parse_nl_scan_kernel<<<1, 1024, 0, r->stream>>> (blk_cnt, nb, blk_off, S.text, L, f.d_res);
		RCK (r, cudaGetLastError ());
		RCK (r, cudaMemcpyAsync (f.h_res, f.d_res, sizeof (ChunkRes), cudaMemcpyDeviceToHost, r->stream));
		const char last = f.stage[si][n - 1];
		if (x + n < b)	// while that runs: the next piece
			RET (fill_stage (r, f, f.stage_next, x + n));
		RCK (r, cudaStreamSynchronize (r->stream));
		const u32 T = f.h_res->T, n_lines = f.h_res->n_lines, j_lo = prev == '\n' ? 0 : 1;
		RET (grow (r, S, (void **) &S.nl, &S.nl_cap, ((u64) T + 1) * sizeof (u32)));
		parse_nl_write_kernel<<<nb, NL_THREADS, 0, r->stream>>> (S.text, L, blk_off, S.nl);
		RCK (r, cudaMemsetAsync (r->d_sum, 0xFF, sizeof (SumRes), r->stream));
		const bool find = r->fastq && s.cand == ALL && n_lines > j_lo;
		if (find)
			shard_fq_find_kernel<<<(n_lines - j_lo + 255) / 256, 256, 0, r->stream>>> (S.text, S.nl, j_lo, n_lines, r->d_sum);
		const u32 nt = r->fastq ? 0 : (n_lines + TILE_LINES - 1) / TILE_LINES;
		Tr *agg = reinterpret_cast<Tr *> (blk_off + nb);
		if (nt)
			shard_fa_tile_kernel<<<nt, LINE_THREADS, 0, r->stream>>> (S.text, S.nl, j_lo, n_lines, agg);
		shard_piece_kernel<<<1, 32, 0, r->stream>>> (agg, nt, S.nl, j_lo, n_lines, r->d_sum);
		RCK (r, cudaGetLastError ());
		RCK (r, cudaMemcpyAsync (r->h_sum, r->d_sum, sizeof (SumRes), cudaMemcpyDeviceToHost, r->stream));
		RCK (r, cudaStreamSynchronize (r->stream));
		const SumRes h = *r->h_sum;
		if (s.first == ALL && h.first != NONE)
			s.first = x + h.first;
		if (find && h.cand != ~0ull)
		{
			s.cand = x + (u32) h.cand;
			s.cand_line = s.n_lines + (h.cand >> 32) - j_lo;
		}
		for (int k = 0; find && k < 2 && s.cand == ALL; k++)
			if (h.open[k] != NONE)
			{	// line n_lines - 2 + k: the line two further down is in a later piece, or past the range
				bool yes;
				RET (fq_rule_on_host (r, f, x + h.open[k], &yes));
				if (yes)
				{
					s.cand = x + h.open[k];
					s.cand_line = s.n_lines + (n_lines - 2 + k) - j_lo;
				}
			}
		s.tr = s.tr.then (Tr64{h.tr.f, h.tr.c0, h.tr.c1});
		s.n_lines += n_lines > j_lo ? n_lines - j_lo : 0;
		prev = last;
		x += n;
	}
	return SDTGPU_OK;
}

void encode_summary (sdtgpu_reader *r, const FileSum *fs)
{
	u64 w[SDTGPU_READER_SUMMARY_BYTES / 8] = {};
	w[0] = SUM_MAGIC;
	w[1] = (u64) r->rank;
	w[2] = (u64) r->world;
	w[3] = (u64) r->fastq;
	w[4] = (u64) r->n_files;
	w[5] = r->f[0].size;
	w[6] = r->n_files == 2 ? r->f[1].size : 0;
	for (int i = 0; i < r->n_files; i++)
	{
		u64 *p = w + 8 + 8 * i;
		p[0] = fs[i].first;
		p[1] = fs[i].n_lines;
		p[2] = fs[i].tr.f;
		p[3] = fs[i].tr.c0;
		p[4] = fs[i].tr.c1;
		p[5] = fs[i].cand;
		p[6] = fs[i].cand_line;
		p[7] = r->f[i].fingerprint;
	}
	memcpy (r->summary, w, sizeof w);
}

// host arithmetic only: every rank runs it on the same summaries and gets the same c[] and entries
int make_plan (sdtgpu_reader *r, const uint8_t *all, uint64_t out[4])
{
	r->planned = false;
	const int W = r->world;
	constexpr int WORDS = SDTGPU_READER_SUMMARY_BYTES / 8;
	std::vector<u64> w ((size_t) W * WORDS);
	memcpy (w.data (), all, (size_t) W * SDTGPU_READER_SUMMARY_BYTES);
	for (int q = 0; q < W; q++)
	{
		const u64 *s = &w[(size_t) q * WORDS];
		bool ok = s[0] == SUM_MAGIC && s[1] == (u64) q && s[2] == (u64) W && s[3] == (u64) r->fastq && s[4] == (u64) r->n_files
			  && s[5] == r->f[0].size && s[6] == (r->n_files == 2 ? r->f[1].size : 0);
		for (int i = 0; ok && i < r->n_files; i++)
		{
			const u64 *p = s + 8 + 8 * i;
			ok = p[7] == r->f[i].fingerprint && p[2] < 4 && (p[5] == ALL || p[6] < p[1]);
		}
		if (!ok)
			return reader_fail (r, SDTGPU_EINVAL, "summary " + std::to_string (q) + " is not rank " + std::to_string (q) + " of " +
					    std::to_string (W) + " over the same files (sizes, contents, FASTA/FASTQ) as this reader");
		if (q == r->rank && r->summarized && memcmp (s, r->summary, SDTGPU_READER_SUMMARY_BYTES))
			return reader_fail (r, SDTGPU_EINVAL, "summary " + std::to_string (q) + " is not the one this reader made");
	}
	for (int i = 0; i < r->n_files; i++)
	{
		FilePlan &P = r->plan[i];
		P.c.assign (W + 1, 0);
		P.off.assign (W, ALL);
		P.skip.assign (W, 0);
		auto sum = [&] (int q) { return &w[(size_t) q * WORDS + 8 + 8 * i]; };
		if (!r->fastq)
		{	// the state before range q is the ranks before it composed from state 0
			u32 P_state = 0;
			for (int q = 0; q < W; q++)
			{
				const u64 *p = sum (q);
				const Tr64 t{(u32) p[2], p[3], p[4]};
				P.off[q] = p[0];
				P.skip[q] = (uint8_t) P_state;	// P = 1: the first line is the sequence line of a header before it
				P.c[q + 1] = P.c[q] + t.count (P_state);
				P_state = t.state (P_state);
			}
			continue;
		}
		// FASTQ: headers are lines h0, h0 + 4, ... of the file, h0 the first candidate of any range
		std::vector<u64> L (W + 1, 0);
		int qs = -1;
		for (int q = 0; q < W; q++)
		{
			L[q + 1] = L[q] + sum (q)[1];
			if (qs < 0 && sum (q)[5] != ALL)
				qs = q;
		}
		if (qs < 0)
			continue;
		const u64 h0 = L[qs] + sum (qs)[6];
		for (int q = 0; q <= W; q++)
			P.c[q] = L[q] > h0 ? (L[q] - h0 + 3) / 4 : 0;
		for (int q = qs; q < W; q++)
		{
			P.off[q] = q == qs ? sum (q)[5] : sum (q)[0];
			P.skip[q] = q == qs ? 0 : (uint8_t) ((4 - (L[q] - h0) % 4) % 4);
		}
	}
	const int k = r->rank;
	const std::vector<u64> &c1 = r->plan[0].c;
	const u64 n1 = c1[W], n2 = r->n_files == 2 ? r->plan[1].c[W] : 0;
	if (r->n_files == 1)
	{
		r->seg[0] = Seg{0, c1[k], c1[k + 1], c1[k]};
		r->seg[1] = Seg{};
	}
	else
	{	// pairs of this rank's file-1 records, then this rank's records of the longer file past the pairs
		const u64 m = std::min (n1, n2);
		const u64 p0 = std::min (m, c1[k]), p1 = std::min (m, c1[k + 1]);
		r->seg[0] = Seg{-1, p0, p1, 2 * p0};
		const int lf = n1 >= n2 ? 0 : 1;
		const std::vector<u64> &cl = r->plan[lf].c;
		const u64 d0 = std::max (m, cl[k]), d1 = std::max (m, cl[k + 1]);
		r->seg[1] = Seg{lf, d0, d1, m + d0};
	}
	r->seg[2] = Seg{};
	r->seg_i = 0;
	r->seg_done = 0;
	r->seg_ready = false;
	for (File &f : r->f)
	{
		f.placed = false;
		f.left = 0;
	}
	r->planned = true;
	out[0] = r->seg[0].size () + r->seg[1].size ();
	out[1] = n1 + n2;
	out[2] = n1;
	out[3] = n2;
	return SDTGPU_OK;
}

// file fi at record k (k < its record count): enter the range that holds record k, then consume records without
// packing them up to k.  Entering a range starts a chunk `skip` lines after its first line start (FASTA: past the
// sequence line of a header before the range; FASTQ: on the next line that is 0 mod 4 from the first header)
int seek (sdtgpu_reader *r, int fi, u64 k)
{
	File &f = r->f[fi];
	if (f.placed && f.rec == k)
		return SDTGPU_OK;
	const FilePlan &P = r->plan[fi];
	const int q = (int) (std::upper_bound (P.c.begin (), P.c.end (), k) - P.c.begin ()) - 1;	// c[q] <= k < c[q + 1]
	u64 off = P.off[q];
	for (int i = 0; i < P.skip[q]; i++)
		RET (skip_line (r, f, off, &off));
	f.cur = -1;
	f.origin = off;
	f.eof = false;
	f.first = false;	// FASTQ: the first header is known
	f.res = ChunkRes{};
	f.cursor = 0;
	f.rec = P.c[q];
	f.placed = true;
	for (f.left = k - f.rec; f.left;)
	{
		RET (fill (r, f));
		const u32 n = (u32) std::min<u64> (f.res.n_rec - f.cursor, f.left);
		f.cursor += n;
		f.rec += n;
		f.left -= n;
	}
	return SDTGPU_OK;
}

// places the files for the current segment and gives each its budget
int seg_enter (sdtgpu_reader *r)
{
	if (r->seg_ready)
		return SDTGPU_OK;
	const Seg &s = r->seg[r->seg_i];
	for (int i = 0; i < r->n_files; i++)
		r->f[i].left = 0;
	for (int i = 0; i < r->n_files && s.size (); i++)
		if (s.file < 0 || s.file == i)
		{
			RET (seek (r, i, s.k0));
			r->f[i].left = s.k1 - s.k0;
		}
	r->seg_ready = true;
	return SDTGPU_OK;
}

// the current segment is done: moves to the next one; true if the same call may go on with it (it has records and
// its ordinals follow on, or the call has returned nothing yet)
bool seg_advance (sdtgpu_reader *r, u64 got)
{
	if (r->seg_i >= 2)
		return false;
	const u64 end = r->seg[r->seg_i].ord0 + r->seg[r->seg_i].size ();
	r->seg_i++;
	r->seg_done = 0;
	r->seg_ready = false;
	const Seg &s = r->seg[r->seg_i];
	return s.size () && (got == 0 || s.ord0 == end);
}

}	// namespace

// rank and world of a reader (world 0: a plain reader), for csrc/sdt_nccl.cu
int sdt_reader_shard (const sdtgpu_reader *r, int *rank, int *world)
{
	*rank = r->rank;
	*world = r->world;
	return SDTGPU_OK;
}

extern "C" {

const char *sdtgpu_reader_last_error (const sdtgpu_reader_t *r) { return r ? r->err.c_str () : g_reader_open_error.c_str (); }

void sdtgpu_reader_close (sdtgpu_reader_t *r)
{
	if (!r)
		return;
	if (r->cuda_ready || r->stream)
	{
		cudaSetDevice (r->device);
		if (r->stream)
			cudaStreamSynchronize (r->stream);
		for (File &f : r->f)
		{
			for (Slot &s : f.slot)
			{
				if (s.packed)
				{
					cudaEventSynchronize (s.packed);
					cudaEventDestroy (s.packed);
				}
				cudaFree (s.text);
				cudaFree (s.nl);
				cudaFree (s.hdr);
			}
			cudaFree (f.scratch);
			cudaFree (f.d_res);
			cudaFreeHost (f.h_res);
			cudaFreeHost (f.stage[0]);
			cudaFreeHost (f.stage[1]);
		}
		cudaFree (r->d_sum);
		cudaFreeHost (r->h_sum);
		if (r->stream)
			cudaStreamDestroy (r->stream);
	}
	for (File &f : r->f)
		if (f.fd >= 0)
			close (f.fd);
	delete r;
}

int sdtgpu_reader_open (sdtgpu_reader_t **out, int device, const char *path1, const char *path2, int fastq, uint64_t chunk_bytes)
{
	if (!out || !path1)
	{
		g_reader_open_error = "out and path1 must not be NULL";
		return SDTGPU_EINVAL;
	}
	*out = nullptr;
	sdtgpu_reader *r = new sdtgpu_reader;
	r->device = device;
	r->fastq = fastq != 0;
	r->n_files = path2 ? 2 : 1;
	r->chunk_bytes = chunk_bytes ? std::min<u64> (chunk_bytes, MAX_CHUNK / 2) : DEFAULT_CHUNK;
	const char *paths[2] = {path1, path2};
	for (int i = 0; i < r->n_files; i++)
	{
		File &f = r->f[i];
		struct stat st;
		f.path = paths[i];
		f.fd = open (paths[i], O_RDONLY);
		if (f.fd < 0 || fstat (f.fd, &st) != 0)
		{
			g_reader_open_error = std::string ("cannot open ") + paths[i] + ": " + strerror (errno);
			sdtgpu_reader_close (r);
			return SDTGPU_EINVAL;
		}
		f.size = (u64) st.st_size;
	}
	*out = r;
	return SDTGPU_OK;
}

int sdtgpu_reader_next (sdtgpu_reader_t *r, void *stream, int max_read_len, int n_kmer, int reverse, uint8_t *d_packed,
			uint32_t *d_lens, uint8_t *d_nmask, uint64_t max_reads, uint32_t stride_bytes, uint64_t *n_out)
{
	if (!r)
		return SDTGPU_EINVAL;
	if (!d_packed || !d_lens || !n_out || max_read_len < 1 || (stride_bytes & 3) || (u64) stride_bytes * 4 < (u64) max_read_len ||
	    (n_kmer && !d_nmask) || max_reads < (u64) r->n_files)
		return reader_fail (r, SDTGPU_EINVAL, "bad arguments (the checks of sdtpack_next: stride a multiple of 4 holding max_read_len bases, nmask with n_kmer, max_reads >= number of files)");
	if (((uintptr_t) d_packed | (uintptr_t) d_lens | (n_kmer ? (uintptr_t) d_nmask : 0)) & 15)
		return reader_fail (r, SDTGPU_EINVAL, "device buffers must be 16-byte aligned");
	*n_out = 0;
	const u64 words = stride_bytes / 4 + (n_kmer ? (stride_bytes / 2 + 3) / 4 : 0);
	const size_t smem = (size_t) words * 4 * PACK_WARPS;
	if (smem > 48 * 1024)
		return reader_fail (r, SDTGPU_EINVAL, "stride_bytes too large for the pack kernel (at most 4096 with n_kmer, 6144 without)");
	if (r->world && !r->planned)
		return reader_fail (r, SDTGPU_ESTATE, "a shard reader needs sdtgpu_reader_plan before sdtgpu_reader_next");
	RCK (r, cudaSetDevice (r->device));
	if (!r->cuda_ready)
		RET (init_cuda (r));
	const Out o{d_packed, d_nmask, d_lens, max_read_len, n_kmer, reverse, stride_bytes, (cudaStream_t) stream, smem};
	const u64 M = r->n_files == 2 ? max_reads & ~1ull : max_reads;
	u64 got = 0;
	for (;;)
	{	// a plain reader runs this once; a shard reader once per segment, as long as the ordinals follow on
		if (r->world)
			RET (seg_enter (r));
		while (got < M)
		{
			File &a = r->f[0], &b = r->f[1];
			if (r->n_files == 2 && !a.exhausted () && !b.exhausted ())
			{	// alternate file 1 / file 2 while both have records
				RET (fill (r, a));
				RET (fill (r, b));
				if (a.exhausted () || b.exhausted ())
					continue;
				const u32 n = (u32) std::min<u64> ({a.res.n_rec - a.cursor, b.res.n_rec - b.cursor, a.left, b.left, (M - got) / 2});
				RET (pack (r, a, n, got, 2, o));
				RET (pack (r, b, n, got + 1, 2, o));
				got += 2 * (u64) n;
				continue;
			}
			File &f = r->n_files == 1 || !a.exhausted () ? a : b;	// then the rest of the longer one
			RET (fill (r, f));
			if (f.exhausted ())
				break;
			const u32 n = (u32) std::min<u64> ({f.res.n_rec - f.cursor, f.left, M - got});
			RET (pack (r, f, n, got, 1, o));
			got += n;
		}
		if (!r->world || got == M || !seg_advance (r, got))
			break;
	}
	*n_out = got;
	return SDTGPU_OK;
}

int sdtgpu_reader_open_shard (sdtgpu_reader_t **out, int device, const char *path1, const char *path2, int fastq,
			      uint64_t chunk_bytes, int rank, int world)
{
	if (!out || !path1 || world < 1 || world > 1024 || rank < 0 || rank >= world)
	{
		g_reader_open_error = "sdtgpu_reader_open_shard: need out and path1, and 0 <= rank < world <= 1024";
		return SDTGPU_EINVAL;
	}
	RET (sdtgpu_reader_open (out, device, path1, path2, fastq, chunk_bytes));
	sdtgpu_reader *r = *out;
	r->rank = rank;
	r->world = world;
	for (int i = 0; i < r->n_files; i++)
		if (fingerprint (r, r->f[i]))
		{
			g_reader_open_error = r->err;
			sdtgpu_reader_close (r);
			*out = nullptr;
			return SDTGPU_EINVAL;
		}
	return SDTGPU_OK;
}

int sdtgpu_reader_summary (sdtgpu_reader_t *r, uint8_t out[SDTGPU_READER_SUMMARY_BYTES])
{
	if (!r || !out)
		return SDTGPU_EINVAL;
	if (!r->world)
		return reader_fail (r, SDTGPU_ESTATE, "sdtgpu_reader_summary needs a reader made by sdtgpu_reader_open_shard");
	if (!r->summarized)
	{
		if (r->planned)
			return reader_fail (r, SDTGPU_ESTATE, "sdtgpu_reader_summary comes before sdtgpu_reader_plan");
		RCK (r, cudaSetDevice (r->device));
		if (!r->cuda_ready)
			RET (init_cuda (r));
		FileSum fs[2];
		for (int i = 0; i < r->n_files; i++)
			RET (summarize_file (r, r->f[i], fs[i]));
		encode_summary (r, fs);
		r->summarized = true;
	}
	memcpy (out, r->summary, SDTGPU_READER_SUMMARY_BYTES);
	return SDTGPU_OK;
}

int sdtgpu_reader_plan (sdtgpu_reader_t *r, const uint8_t *summaries, uint64_t out[4])
{
	if (!r || !summaries || !out)
		return SDTGPU_EINVAL;
	if (!r->world)
		return reader_fail (r, SDTGPU_ESTATE, "sdtgpu_reader_plan needs a reader made by sdtgpu_reader_open_shard");
	return make_plan (r, summaries, out);
}

int sdtgpu_reader_tell (const sdtgpu_reader_t *r, uint64_t *ordinal)
{
	if (!r || !ordinal)
		return SDTGPU_EINVAL;
	if (!r->world)
	{
		*ordinal = r->stats[1];
		return SDTGPU_OK;
	}
	if (!r->planned)
		return SDTGPU_ESTATE;
	for (int i = r->seg_i; i < 2; i++)
	{
		const u64 done = i == r->seg_i ? r->seg_done : 0;
		if (done < r->seg[i].size ())
		{
			*ordinal = r->seg[i].ord0 + done;
			return SDTGPU_OK;
		}
	}
	// nothing left: one past the last record this rank returns (where its share starts if it returns none)
	const Seg &s = r->seg[1].size () ? r->seg[1] : r->seg[0];
	*ordinal = s.ord0 + s.size ();
	return SDTGPU_OK;
}

int sdtgpu_reader_stats (const sdtgpu_reader_t *r, uint64_t out[4])
{
	if (!r || !out)
		return SDTGPU_EINVAL;
	for (int i = 0; i < 4; i++)
		out[i] = r->stats[i];
	return SDTGPU_OK;
}

}	// extern "C"
