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
	bool exhausted () const { return cur >= 0 && eof && cursor == res.n_rec; }
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
	u64 start = 0, tail = 0;
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
	r->stats[1] += n;
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
	r->cuda_ready = true;
	return SDTGPU_OK;
}

}	// namespace

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
	RCK (r, cudaSetDevice (r->device));
	if (!r->cuda_ready)
		RET (init_cuda (r));
	const Out o{d_packed, d_nmask, d_lens, max_read_len, n_kmer, reverse, stride_bytes, (cudaStream_t) stream, smem};
	const u64 M = r->n_files == 2 ? max_reads & ~1ull : max_reads;
	u64 got = 0;
	while (got < M)
	{
		File &a = r->f[0], &b = r->f[1];
		if (r->n_files == 2 && !a.exhausted () && !b.exhausted ())
		{	// alternate file 1 / file 2 while both have records
			RET (fill (r, a));
			RET (fill (r, b));
			if (a.exhausted () || b.exhausted ())
				continue;
			const u32 n = (u32) std::min<u64> ({a.res.n_rec - a.cursor, b.res.n_rec - b.cursor, (M - got) / 2});
			RET (pack (r, a, n, got, 2, o));
			RET (pack (r, b, n, got + 1, 2, o));
			got += 2 * (u64) n;
			continue;
		}
		File &f = r->n_files == 1 || !a.exhausted () ? a : b;	// then the rest of the longer one
		RET (fill (r, f));
		if (f.exhausted ())
			break;
		const u32 n = (u32) std::min<u64> (f.res.n_rec - f.cursor, M - got);
		RET (pack (r, f, n, got, 1, o));
		got += n;
	}
	*n_out = got;
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
