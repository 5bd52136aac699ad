// sdt_nccl.cu — the super-k-mer exchange of the sliced build behind the C ABI: one call per epoch does what a
// host would otherwise script around sdtgpu_skm_stage / sdtgpu_skm_import (include/sdtgpu.h): the ordinal
// bound (an all-reduce), the merge and pack by owner, the counts (an all-gather), the records (ONE grouped
// ncclSend / ncclRecv straight into the import buffer) and the build of this rank's slices.  The routed lookups
// (sdtgpu_lookup_kmers_exchange, sdtgpu_lookup_reads_exchange) drive sdtgpu_lookup_stage / _answer / _unstage the
// same way: the queries travel to their owners and the hits come back, one grouped send / recv each way.
//
// Host code only, layered on the public C ABI of the handle.  NCCL is bound at run time (dlopen of
// libnccl.so.2: in a process that already holds an NCCL — torch's — that one is used; a plain C host gets the
// system's), so libsdtgpu.so has no link-time dependency on it and single-GPU users never load it.
// The reference has no counterpart: its workers share one address space (prlHashReads.c:79-88).
#include "../../include/sdtgpu.h"
#include <cuda_runtime.h>
#include <nccl.h>
#include <dlfcn.h>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

namespace {

struct Nccl
{
	void *lib = nullptr;
	ncclResult_t (*GetUniqueId) (ncclUniqueId *) = nullptr;
	ncclResult_t (*CommInitRank) (ncclComm_t *, int, ncclUniqueId, int) = nullptr;
	ncclResult_t (*CommDestroy) (ncclComm_t) = nullptr;
	const char *(*GetErrorString) (ncclResult_t) = nullptr;
	ncclResult_t (*AllReduce) (const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*AllGather) (const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*Send) (const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*Recv) (void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*GroupStart) () = nullptr;
	ncclResult_t (*GroupEnd) () = nullptr;
	std::string err;
};

Nccl g_nccl;
std::string g_comm_err;	// last failure without a communicator

template <class F> bool sym (void *lib, const char *name, F &f)
{
	f = reinterpret_cast<F> (dlsym (lib, name));
	return f != nullptr;
}

bool nccl_load ()
{
	Nccl &n = g_nccl;
	if (n.lib)
		return true;
	const char *names[] = { "libnccl.so.2", "libnccl.so" };
	void *lib = nullptr;
	for (const char *nm : names)
		if ((lib = dlopen (nm, RTLD_NOW | RTLD_LOCAL)))
			break;
	if (!lib)
	{
		const char *why = dlerror ();
		n.err = std::string ("cannot load libnccl.so.2: ") + (why ? why : "?");
		return false;
	}
	const bool ok = sym (lib, "ncclGetUniqueId", n.GetUniqueId) && sym (lib, "ncclCommInitRank", n.CommInitRank) && sym (lib, "ncclCommDestroy", n.CommDestroy)
		&& sym (lib, "ncclGetErrorString", n.GetErrorString) && sym (lib, "ncclAllReduce", n.AllReduce) && sym (lib, "ncclAllGather", n.AllGather)
		&& sym (lib, "ncclSend", n.Send) && sym (lib, "ncclRecv", n.Recv) && sym (lib, "ncclGroupStart", n.GroupStart) && sym (lib, "ncclGroupEnd", n.GroupEnd);
	if (!ok)
	{
		n.err = "libnccl.so.2 lacks a symbol of the point-to-point API (NCCL >= 2.7 is needed)";
		dlclose (lib);
		return false;
	}
	n.lib = lib;
	return true;
}

}	// namespace

struct sdtgpu_comm
{
	ncclComm_t comm = nullptr;
	int device = 0, rank = 0, world = 1;
	unsigned long long *d_buf = nullptr, *h_pin = nullptr;	// [0] mine, [1] reduced, [8 ..) my counts, [8 + world ..) everybody's
	unsigned long long *d_lk = nullptr, *h_lk = nullptr;	// routed lookups: [0, LK_WORDS) mine, then LK_WORDS per rank
	cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr, e3 = nullptr;
	std::string err;
};

namespace {

constexpr size_t LK_WORDS = 80;	// a routed lookup's messages: the 12-word descriptor, or world counts + a status

int comm_fail (sdtgpu_comm *c, int code, const std::string &what)
{
	(c ? c->err : g_comm_err) = what;
	return code;
}

#define NC(c, call) do { ncclResult_t r_ = (call); if (r_ != ncclSuccess) return comm_fail (c, SDTGPU_ECUDA, std::string (#call) + ": " + g_nccl.GetErrorString (r_)); } while (0)
#define CU(c, call) do { cudaError_t r_ = (call); if (r_ != cudaSuccess) return comm_fail (c, SDTGPU_ECUDA, std::string (#call) + ": " + cudaGetErrorString (r_)); } while (0)

}	// namespace

extern "C" {

const char *sdtgpu_comm_last_error (const sdtgpu_comm_t *c)
{
	return c ? c->err.c_str () : g_comm_err.c_str ();
}

int sdtgpu_comm_unique_id (uint8_t id[SDTGPU_COMM_ID_BYTES])
{
	if (!id)
		return SDTGPU_EINVAL;
	if (!nccl_load ())
		return comm_fail (nullptr, SDTGPU_ESTATE, g_nccl.err);
	static_assert (sizeof (ncclUniqueId) == SDTGPU_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
	ncclUniqueId u;
	NC (nullptr, g_nccl.GetUniqueId (&u));
	memcpy (id, &u, sizeof u);
	return SDTGPU_OK;
}

int sdtgpu_comm_create (sdtgpu_comm_t **out, int device, const uint8_t id[SDTGPU_COMM_ID_BYTES], int rank, int world)
{
	if (!out || !id || world < 1 || world > 64 || rank < 0 || rank >= world)
		return comm_fail (nullptr, SDTGPU_EINVAL, "sdtgpu_comm_create: need 0 <= rank < world <= 64");
	*out = nullptr;
	if (!nccl_load ())
		return comm_fail (nullptr, SDTGPU_ESTATE, g_nccl.err);
	sdtgpu_comm *c = new sdtgpu_comm;
	c->device = device;
	c->rank = rank;
	c->world = world;
	auto bail = [&](int rc) { g_comm_err = c->err; sdtgpu_comm_destroy (c); return rc; };
	if (cudaSetDevice (device) != cudaSuccess)
		return bail (comm_fail (c, SDTGPU_ECUDA, "cudaSetDevice failed"));
	ncclUniqueId u;
	memcpy (&u, id, sizeof u);
	ncclResult_t r = g_nccl.CommInitRank (&c->comm, world, u, rank);
	if (r != ncclSuccess)
	{
		c->comm = nullptr;
		return bail (comm_fail (c, SDTGPU_ECUDA, std::string ("ncclCommInitRank: ") + g_nccl.GetErrorString (r)));
	}
	const size_t words = 8 + (size_t) world + (size_t) world * world;
	const size_t lk_words = LK_WORDS * (1 + (size_t) world);
	if (cudaMalloc (&c->d_buf, words * 8) != cudaSuccess || cudaMallocHost (&c->h_pin, words * 8) != cudaSuccess
	    || cudaMalloc (&c->d_lk, lk_words * 8) != cudaSuccess || cudaMallocHost (&c->h_lk, lk_words * 8) != cudaSuccess
	    || cudaEventCreate (&c->e0) != cudaSuccess || cudaEventCreate (&c->e1) != cudaSuccess
	    || cudaEventCreate (&c->e2) != cudaSuccess || cudaEventCreate (&c->e3) != cudaSuccess)
		return bail (comm_fail (c, SDTGPU_ENOMEM, "sdtgpu_comm_create: allocation failed"));
	*out = c;
	return SDTGPU_OK;
}

int sdtgpu_comm_destroy (sdtgpu_comm_t *c)
{
	if (!c)
		return SDTGPU_OK;
	cudaSetDevice (c->device);
	if (c->comm && g_nccl.CommDestroy)
		g_nccl.CommDestroy (c->comm);
	if (c->d_buf)
		cudaFree (c->d_buf);
	if (c->h_pin)
		cudaFreeHost (c->h_pin);
	if (c->d_lk)
		cudaFree (c->d_lk);
	if (c->h_lk)
		cudaFreeHost (c->h_lk);
	for (cudaEvent_t e : { c->e0, c->e1, c->e2, c->e3 })
		if (e)
			cudaEventDestroy (e);
	delete c;
	return SDTGPU_OK;
}

int sdtgpu_skm_exchange (sdtgpu_t *h, sdtgpu_comm_t *c, uint64_t reads_end_this_rank, uint64_t *n_received, double *collective_ms)
{
	if (!h || !c)
		return SDTGPU_EINVAL;
	const int world = c->world, rank = c->rank;
	cudaStream_t s = static_cast<cudaStream_t> (sdtgpu_stream (h));
	CU (c, cudaSetDevice (c->device));
	int rc;
	// 1. reads of all ranks this epoch: 32-bit ordinals in the slice images when they fit
	c->h_pin[0] = reads_end_this_rank;
	CU (c, cudaMemcpyAsync (c->d_buf, c->h_pin, 8, cudaMemcpyHostToDevice, s));
	NC (c, g_nccl.AllReduce (c->d_buf, c->d_buf + 1, 1, ncclUint64, ncclMax, c->comm, s));
	CU (c, cudaMemcpyAsync (c->h_pin + 1, c->d_buf + 1, 8, cudaMemcpyDeviceToHost, s));
	CU (c, cudaStreamSynchronize (s));
	if ((rc = sdtgpu_skm_set_ordinal_bound (h, c->h_pin[1])))
		return comm_fail (c, rc, std::string ("sdtgpu_skm_set_ordinal_bound: ") + sdtgpu_last_error (h));
	// 2. this rank's copies merged, survivors packed by owner
	void *d_rec = nullptr;
	std::vector<uint64_t> starts (world), counts (world), recv (world);
	if ((rc = sdtgpu_skm_stage (h, &d_rec, starts.data (), counts.data ())))
		return comm_fail (c, rc, std::string ("sdtgpu_skm_stage: ") + sdtgpu_last_error (h));
	uint64_t geo[12];
	if ((rc = sdtgpu_slice_geometry (h, geo)))
		return comm_fail (c, rc, "sdtgpu_slice_geometry failed");
	const size_t rec_bytes = (size_t) geo[4], words = rec_bytes / 8;
	// 3. who sends how much to whom
	unsigned long long *h_mine = c->h_pin + 8, *h_all = c->h_pin + 8 + world, *d_mine = c->d_buf + 8, *d_all = c->d_buf + 8 + world;
	for (int r = 0; r < world; r++)
		h_mine[r] = counts[r];
	CU (c, cudaEventRecord (c->e0, s));
	CU (c, cudaMemcpyAsync (d_mine, h_mine, (size_t) world * 8, cudaMemcpyHostToDevice, s));
	NC (c, g_nccl.AllGather (d_mine, d_all, (size_t) world, ncclUint64, c->comm, s));
	CU (c, cudaMemcpyAsync (h_all, d_all, (size_t) world * world * 8, cudaMemcpyDeviceToHost, s));
	CU (c, cudaStreamSynchronize (s));
	uint64_t total = 0;
	for (int src = 0; src < world; src++)
		total += (recv[src] = h_all[(size_t) src * world + rank]);
	// 4. the records, in place: sender's region -> receiver's import buffer (runs arrive in source-rank order)
	void *d_in = nullptr;
	if ((rc = sdtgpu_skm_import_buffer (h, total, &d_in)))
		return comm_fail (c, rc, std::string ("sdtgpu_skm_import_buffer: ") + sdtgpu_last_error (h));
	const char *out_base = static_cast<const char *> (d_rec);
	char *in_base = static_cast<char *> (d_in);
	NC (c, g_nccl.GroupStart ());
	uint64_t off = 0;
	for (int src = 0; src < world; src++)
	{
		const uint64_t n = recv[src];
		char *seg = in_base + off * rec_bytes;
		off += n;
		if (!n)
			continue;
		if (src == rank)	// own records: a device-local copy, never touches the fabric
			CU (c, cudaMemcpyAsync (seg, out_base + starts[rank] * rec_bytes, n * rec_bytes, cudaMemcpyDeviceToDevice, s));
		else
			NC (c, g_nccl.Recv (seg, n * words, ncclUint64, src, c->comm, s));
	}
	for (int dst = 0; dst < world; dst++)
		if (dst != rank && counts[dst])
			NC (c, g_nccl.Send (out_base + starts[dst] * rec_bytes, counts[dst] * words, ncclUint64, dst, c->comm, s));
	NC (c, g_nccl.GroupEnd ());
	CU (c, cudaEventRecord (c->e1, s));
	// 5. this rank's slices
	if ((rc = sdtgpu_skm_import (h, total)))
		return comm_fail (c, rc, std::string ("sdtgpu_skm_import: ") + sdtgpu_last_error (h));
	if (n_received)
		*n_received = total;
	if (collective_ms)
	{
		float ms = 0;
		CU (c, cudaEventSynchronize (c->e1));
		CU (c, cudaEventElapsedTime (&ms, c->e0, c->e1));
		*collective_ms = ms;
	}
	return SDTGPU_OK;
}

}	// extern "C"

namespace {

// one all-gather of n words per rank (n <= LK_WORDS): this rank's in h_lk[0, n), everybody's to h_lk + LK_WORDS
// (rank r's at r * n); synchronises the stream
int lk_allgather (sdtgpu_comm *c, cudaStream_t s, size_t n)
{
	CU (c, cudaMemcpyAsync (c->d_lk, c->h_lk, n * 8, cudaMemcpyHostToDevice, s));
	NC (c, g_nccl.AllGather (c->d_lk, c->d_lk + LK_WORDS, n, ncclUint64, c->comm, s));
	CU (c, cudaMemcpyAsync (c->h_lk + LK_WORDS, c->d_lk + LK_WORDS, (size_t) c->world * n * 8, cudaMemcpyDeviceToHost, s));
	CU (c, cudaStreamSynchronize (s));
	return SDTGPU_OK;
}

// a routed lookup over NCCL, built from the public halves (include/sdtgpu.h): stage (void **, starts, counts) is
// sdtgpu_lookup_stage_kmers or _reads with the caller's queries bound
template <class Stage>
int lookup_exchange (sdtgpu_t *h, sdtgpu_comm *c, Stage stage, sdtgpu_hit *d_out, double *collective_ms)
{
	const int world = c->world, rank = c->rank;
	int rc;
	// 1. this rank's handle must be sharded as the communicator is (no collective yet)
	uint64_t desc[12];
	if ((rc = sdtgpu_lookup_route (h, desc)))
		return comm_fail (c, rc, "sdtgpu_lookup_route failed");
	if (desc[1] != (uint64_t) rank || desc[2] != (uint64_t) world)
	{
		char b[200];
		snprintf (b, sizeof b, "routed lookup: the handle is rank %llu of %llu, the communicator rank %d of %d",
			  (unsigned long long) desc[1], (unsigned long long) desc[2], rank, world);
		return comm_fail (c, SDTGPU_EINVAL, b);
	}
	cudaStream_t s = static_cast<cudaStream_t> (sdtgpu_stream (h));
	CU (c, cudaSetDevice (c->device));
	// 2. every rank's sharding: all equal but the rank, or nobody goes on
	const size_t nd = 12;
	for (size_t i = 0; i < nd; i++)
		c->h_lk[i] = desc[i];
	if ((rc = lk_allgather (c, s, nd)))
		return rc;
	for (int r = 0; r < world; r++)
		for (size_t i = 0; i < nd; i++)
			if (i != 1 && c->h_lk[LK_WORDS + r * nd + i] != desc[i])
			{
				char b[200];
				snprintf (b, sizeof b, "routed lookup: rank %d's sharding differs from rank %d's in word %zu of sdtgpu_lookup_route (%llu vs %llu)",
					  r, rank, i, c->h_lk[LK_WORDS + r * nd + i], (unsigned long long) desc[i]);
				return comm_fail (c, SDTGPU_EINVAL, b);
			}
	if (!desc[11])
		return comm_fail (c, SDTGPU_ESTATE, "routed lookup before sdtgpu_finalize");
	// 3. this rank's queries by owner
	void *d_q = nullptr;
	std::vector<uint64_t> starts (world, 0), counts (world, 0), recv (world), roff (world);
	const int st = stage (&d_q, starts.data (), counts.data ());
	const std::string why = st ? sdtgpu_last_error (h) : "";
	// 4. who sends how much to whom, and whether every stage worked
	CU (c, cudaEventRecord (c->e0, s));
	const size_t nc = (size_t) world + 1;
	for (int r = 0; r < world; r++)
		c->h_lk[r] = st ? 0 : counts[r];
	c->h_lk[world] = (unsigned long long) st;
	if ((rc = lk_allgather (c, s, nc)))
		return rc;
	const unsigned long long *all = c->h_lk + LK_WORDS;	// all[src * nc + dst]: queries src sends to dst; all[src * nc + world]: src's stage status
	if (st)
		return comm_fail (c, st, "sdtgpu_lookup_stage: " + why);
	for (int r = 0; r < world; r++)
		if (all[r * nc + world])
			return comm_fail (c, SDTGPU_ESTATE, "routed lookup: the stage of rank " + std::to_string (r) + " failed");
	uint64_t total = 0;
	for (int src = 0; src < world; src++)
	{
		roff[src] = total;
		total += (recv[src] = all[src * nc + rank]);
	}
	// 5. the queries, in place: sender's region -> owner's answer buffer (runs in source-rank order)
	void *d_aq = nullptr;
	sdtgpu_hit *d_ar = nullptr;
	if ((rc = sdtgpu_lookup_answer_buffer (h, total, &d_aq, &d_ar)))
		return comm_fail (c, rc, std::string ("sdtgpu_lookup_answer_buffer: ") + sdtgpu_last_error (h));
	const size_t qw = (size_t) desc[4], qb = 8 * qw, hw = sizeof (sdtgpu_hit) / 8;
	const char *q_out = static_cast<const char *> (d_q);
	char *q_in = static_cast<char *> (d_aq);
	NC (c, g_nccl.GroupStart ());
	for (int src = 0; src < world; src++)
	{
		if (!recv[src])
			continue;
		if (src == rank)
			CU (c, cudaMemcpyAsync (q_in + roff[src] * qb, q_out + starts[rank] * qb, recv[src] * qb, cudaMemcpyDeviceToDevice, s));
		else
			NC (c, g_nccl.Recv (q_in + roff[src] * qb, recv[src] * qw, ncclUint64, src, c->comm, s));
	}
	for (int dst = 0; dst < world; dst++)
		if (dst != rank && counts[dst])
			NC (c, g_nccl.Send (q_out + starts[dst] * qb, counts[dst] * qw, ncclUint64, dst, c->comm, s));
	NC (c, g_nccl.GroupEnd ());
	CU (c, cudaEventRecord (c->e1, s));
	// 6. this rank answers what it owns
	if ((rc = sdtgpu_lookup_answer (h, total)))
		return comm_fail (c, rc, std::string ("sdtgpu_lookup_answer: ") + sdtgpu_last_error (h));
	// 7. the hits back to the askers, into their unstage buffers in staged order
	sdtgpu_hit *d_back = nullptr;
	if ((rc = sdtgpu_lookup_unstage_buffer (h, &d_back)))
		return comm_fail (c, rc, std::string ("sdtgpu_lookup_unstage_buffer: ") + sdtgpu_last_error (h));
	CU (c, cudaEventRecord (c->e2, s));
	NC (c, g_nccl.GroupStart ());
	for (int dst = 0; dst < world; dst++)
	{
		if (!counts[dst])
			continue;
		if (dst == rank)
			CU (c, cudaMemcpyAsync (d_back + starts[dst], d_ar + roff[rank], counts[dst] * sizeof (sdtgpu_hit), cudaMemcpyDeviceToDevice, s));
		else
			NC (c, g_nccl.Recv (d_back + starts[dst], counts[dst] * hw, ncclUint64, dst, c->comm, s));
	}
	for (int src = 0; src < world; src++)
		if (src != rank && recv[src])
			NC (c, g_nccl.Send (d_ar + roff[src], recv[src] * hw, ncclUint64, src, c->comm, s));
	NC (c, g_nccl.GroupEnd ());
	CU (c, cudaEventRecord (c->e3, s));
	// 8. into the caller's output
	if ((rc = sdtgpu_lookup_unstage (h, d_out)))
		return comm_fail (c, rc, std::string ("sdtgpu_lookup_unstage: ") + sdtgpu_last_error (h));
	CU (c, cudaStreamSynchronize (s));
	if (collective_ms)
	{
		float a = 0, b = 0;
		CU (c, cudaEventElapsedTime (&a, c->e0, c->e1));
		CU (c, cudaEventElapsedTime (&b, c->e2, c->e3));
		*collective_ms = (double) a + b;
	}
	return SDTGPU_OK;
}

}	// namespace

extern "C" {

int sdtgpu_lookup_kmers_exchange (sdtgpu_t *h, sdtgpu_comm_t *c, const uint64_t *d_keys, uint64_t n, sdtgpu_hit *d_out,
				  double *collective_ms)
{
	if (!h || !c || (n && (!d_keys || !d_out)))
		return comm_fail (nullptr, SDTGPU_EINVAL, "sdtgpu_lookup_kmers_exchange: NULL handle, communicator or buffer");
	return lookup_exchange (h, c, [&](void **q, uint64_t *starts, uint64_t *counts) {
		return sdtgpu_lookup_stage_kmers (h, d_keys, n, q, starts, counts);
	}, d_out, collective_ms);
}

int sdtgpu_lookup_reads_exchange (sdtgpu_t *h, sdtgpu_comm_t *c, const uint8_t *d_packed, const uint32_t *d_lens,
				  const uint8_t *d_nmask, uint64_t n_reads, uint32_t uniform_len, uint32_t stride_bytes,
				  sdtgpu_hit *d_out, double *collective_ms)
{
	if (!h || !c || (n_reads && (!d_packed || !d_out)))
		return comm_fail (nullptr, SDTGPU_EINVAL, "sdtgpu_lookup_reads_exchange: NULL handle, communicator or buffer");
	return lookup_exchange (h, c, [&](void **q, uint64_t *starts, uint64_t *counts) {
		return sdtgpu_lookup_stage_reads (h, d_packed, d_lens, d_nmask, n_reads, uniform_len, stride_bytes, q, starts, counts);
	}, d_out, collective_ms);
}

}	// extern "C"

int sdt_reader_shard (const sdtgpu_reader_t *r, int *rank, int *world);	// csrc/sdt_parse.cu

namespace {

// the all-gather of plan_exchange: this rank's 256 bytes in, everybody's out (rank order)
int gather_summaries (sdtgpu_comm *c, const uint8_t *mine, std::vector<uint8_t> &all)
{
	const size_t B = SDTGPU_READER_SUMMARY_BYTES;
	cudaStream_t s = nullptr;
	uint8_t *d = nullptr;
	int rc = SDTGPU_OK;
	auto step = [&] (int code, const std::string &what) { if (!rc && code) rc = comm_fail (c, code, what); };
	auto cu = [&] (cudaError_t e, const char *what) { step (e == cudaSuccess ? SDTGPU_OK : SDTGPU_ECUDA, std::string (what) + ": " + cudaGetErrorString (e)); };
	cu (cudaSetDevice (c->device), "cudaSetDevice");
	if (!rc)
		cu (cudaStreamCreateWithFlags (&s, cudaStreamNonBlocking), "cudaStreamCreateWithFlags");
	if (!rc)
		cu (cudaMalloc (&d, B * (size_t) c->world), "cudaMalloc");
	if (!rc)	// in place: this rank's block is already where the all-gather puts it
		cu (cudaMemcpyAsync (d + B * (size_t) c->rank, mine, B, cudaMemcpyHostToDevice, s), "cudaMemcpyAsync");
	if (!rc)
	{
		const ncclResult_t r = g_nccl.AllGather (d + B * (size_t) c->rank, d, B, ncclUint8, c->comm, s);
		step (r == ncclSuccess ? SDTGPU_OK : SDTGPU_ECUDA, std::string ("ncclAllGather: ") + (r == ncclSuccess ? "" : g_nccl.GetErrorString (r)));
	}
	if (!rc)
		cu (cudaMemcpyAsync (all.data (), d, B * (size_t) c->world, cudaMemcpyDeviceToHost, s), "cudaMemcpyAsync");
	if (s)
		cu (cudaStreamSynchronize (s), "cudaStreamSynchronize");
	if (d)
		cudaFree (d);
	if (s)
		cudaStreamDestroy (s);
	return rc;
}

}	// namespace

extern "C" int sdtgpu_reader_plan_exchange (sdtgpu_reader_t *r, sdtgpu_comm_t *c, uint64_t out[4])
{
	if (!r || !c || !out)
		return comm_fail (nullptr, SDTGPU_EINVAL, "sdtgpu_reader_plan_exchange: NULL reader, communicator or output");
	int rank = 0, world = 0;
	sdt_reader_shard (r, &rank, &world);
	if (!world)
		return comm_fail (c, SDTGPU_ESTATE, "sdtgpu_reader_plan_exchange needs a reader made by sdtgpu_reader_open_shard");
	if (rank != c->rank || world != c->world)
	{
		char b[200];
		snprintf (b, sizeof b, "sdtgpu_reader_plan_exchange: the reader is rank %d of %d, the communicator rank %d of %d", rank, world, c->rank, c->world);
		return comm_fail (c, SDTGPU_EINVAL, b);
	}
	// a rank whose summary fails still takes part: its all-zero block makes every rank's plan refuse
	uint8_t mine[SDTGPU_READER_SUMMARY_BYTES];
	const int src = sdtgpu_reader_summary (r, mine);
	if (src)
		memset (mine, 0, sizeof mine);
	std::vector<uint8_t> all ((size_t) world * SDTGPU_READER_SUMMARY_BYTES);
	int rc = gather_summaries (c, mine, all);
	if (rc)
		return rc;
	if (src)
		return comm_fail (c, src, std::string ("sdtgpu_reader_summary: ") + sdtgpu_reader_last_error (r));
	if ((rc = sdtgpu_reader_plan (r, all.data (), out)))
		return comm_fail (c, rc, std::string ("sdtgpu_reader_plan: ") + sdtgpu_reader_last_error (r));
	return SDTGPU_OK;
}
