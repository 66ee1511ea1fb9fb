// TMA-staged column tiles: the HBM -> shared-memory front end shared by the aggregate, join-probe and filter
// kernels.  A "tile" is TILE consecutive rows of every (flat) input column; one elected thread issues one
// 1-D bulk copy (cp.async.bulk.shared.global, SASS UBLKCP) per column into the next pipeline stage and the
// copies complete on that stage's mbarrier, so the loads of tile i+1..i+S-1 are in flight while the CTA
// computes on tile i.  This is what gives the kernels their memory-level parallelism: bytes in flight per SM
// = (stages-1) x tile bytes, independent of how branchy the per-row code is.
//
// Requirements for the bulk path: flat columns, 16-byte aligned base pointers, TILE a multiple of 128 rows
// (so that every column's tile - including 1-bit validity tiles - is a multiple of 16 bytes).  The ragged
// last tile of a range is copied cooperatively with plain loads.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define TP_MAX_COLS 20

struct TileCol {
	const unsigned char *ptr; // column base (device)
	uint32_t width;           // bytes per row; 0 = bit-packed (validity mask, 1 bit per row)
	uint32_t smem_off;        // byte offset of this column inside a stage (16-byte aligned)
};

struct TileCols {
	TileCol c[TP_MAX_COLS];
	int n;
	uint32_t stage_bytes; // bytes of one stage (sum of column tiles, each rounded up to 16)
	uint32_t tile_rows;
};

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t tp_smem_addr(const void *p) {
	return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void tp_mbar_init(uint64_t *bar, uint32_t count) {
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(tp_smem_addr(bar)), "r"(count) : "memory");
}

__device__ __forceinline__ void tp_fence_mbar_init() {
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void tp_expect_tx(uint64_t *bar, uint32_t bytes) {
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(tp_smem_addr(bar)), "r"(bytes)
	             : "memory");
}

// Input columns are read exactly once: the bulk copies carry an L2 evict-first policy so that they do not push
// the (re-used) hash tables out of L2.
__device__ __forceinline__ uint64_t tp_evict_first_policy() {
	uint64_t pol;
	asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
	return pol;
}

__device__ __forceinline__ void tp_bulk_load(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar) {
	uint64_t pol = tp_evict_first_policy();
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, "
	             "[%3], %4;" ::"r"(tp_smem_addr(smem_dst)),
	             "l"(gmem_src), "r"(bytes), "r"(tp_smem_addr(bar)), "l"(pol)
	             : "memory");
}

__device__ __forceinline__ void tp_wait(uint64_t *bar, uint32_t parity) {
	asm volatile("{\n"
	             ".reg .pred p;\n"
	             "WAIT_LOOP:\n"
	             "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
	             "@p bra DONE;\n"
	             "bra WAIT_LOOP;\n"
	             "DONE:\n"
	             "}\n" ::"r"(tp_smem_addr(bar)),
	             "r"(parity)
	             : "memory");
}

__device__ __forceinline__ void tp_arrive(uint64_t *bar) {
	asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tp_smem_addr(bar)) : "memory");
}

__device__ __forceinline__ uint32_t tp_col_tile_bytes(const TileCol &c, uint32_t rows) {
	return c.width ? rows * c.width : rows / 8;
}

// Issue the bulk copies of a FULL tile starting at row0 into stage buffer `stage` (called by one thread).
__device__ __forceinline__ void tp_issue_full(const TileCols &tc, unsigned char *stage, uint64_t *bar, uint64_t row0) {
	uint32_t total = 0;
	for (int i = 0; i < tc.n; i++) {
		total += tp_col_tile_bytes(tc.c[i], tc.tile_rows);
	}
	tp_expect_tx(bar, total);
	for (int i = 0; i < tc.n; i++) {
		const TileCol &c = tc.c[i];
		const unsigned char *src = c.width ? c.ptr + row0 * c.width : c.ptr + row0 / 8;
		tp_bulk_load(stage + c.smem_off, src, tp_col_tile_bytes(c, tc.tile_rows), bar);
	}
}

// Cooperative copy of a ragged tile (rows < tile_rows) with plain loads; all threads of the CTA call this and
// must __syncthreads() afterwards.  row0 is a multiple of tile_rows (so bit-packed columns start on a byte).
__device__ __forceinline__ void tp_copy_ragged(const TileCols &tc, unsigned char *stage, uint64_t row0, uint32_t rows) {
	for (int i = 0; i < tc.n; i++) {
		const TileCol &c = tc.c[i];
		uint32_t bytes = c.width ? rows * c.width : (rows + 7) / 8;
		const unsigned char *src = c.width ? c.ptr + row0 * c.width : c.ptr + row0 / 8;
		unsigned char *dst = stage + c.smem_off;
		for (uint32_t b = threadIdx.x; b < bytes; b += blockDim.x) {
			dst[b] = src[b];
		}
	}
}

// Simple (non-specialised) tile loop: every thread is a consumer, thread 0 also issues the TMA copies, one
// __syncthreads() per tile.  Measured on B200: for kernels whose body already synchronises the CTA per tile (join
// probe, filter) this is FASTER than the warp-specialised ring below (no 9th warp, no named barriers); the
// aggregate kernels, whose body never synchronises, use the specialised ring.
// bars: S mbarriers.  body(stage_ptr, row0, rows_in_tile) is CTA-uniform and may use __syncthreads().
template <class BODY>
__device__ __forceinline__ void tp_tile_loop_sync(const TileCols &tc, int S, unsigned char *stages, uint64_t *bars,
                                                  uint64_t row_begin, uint64_t row_end, BODY body) {
	const uint32_t TILE = tc.tile_rows;
	const uint64_t total = row_end - row_begin;
	const uint64_t ntiles = (total + TILE - 1) / TILE;
	const uint64_t nfull = total / TILE;
	if (threadIdx.x == 0) {
		for (int s = 0; s < S; s++) {
			tp_mbar_init(&bars[s], 1);
		}
		tp_fence_mbar_init();
	}
	__syncthreads();
	if (threadIdx.x == 0) {
		for (int s = 0; s < S - 1; s++) {
			uint64_t t = blockIdx.x + (uint64_t)s * gridDim.x;
			if (t < nfull) {
				tp_issue_full(tc, stages + (size_t)s * tc.stage_bytes, &bars[s], row_begin + t * TILE);
			}
		}
	}
	int s = 0;          // stage of tile k = k mod S and the parity of its round, kept as counters (S is a run-time
	uint32_t parity = 0; // value: `k % S` and `k / S` were 5 % of the mask kernel's instructions)
	for (uint64_t k = 0;; k++) {
		uint64_t t = blockIdx.x + k * gridDim.x;
		if (t >= ntiles) {
			break;
		}
		unsigned char *stage = stages + (size_t)s * tc.stage_bytes;
		if (threadIdx.x == 0) {
			uint64_t tn = blockIdx.x + (k + S - 1) * gridDim.x;
			if (tn < nfull) {
				int sn = s == 0 ? S - 1 : s - 1; // (k + S - 1) mod S
				tp_issue_full(tc, stages + (size_t)sn * tc.stage_bytes, &bars[sn], row_begin + tn * TILE);
			}
		}
		uint32_t rows_in_tile = TILE;
		uint64_t row0 = row_begin + t * TILE;
		const int s_now = s;
		const uint32_t parity_now = parity;
		if (++s == S) {
			s = 0;
			parity ^= 1u;
		}
		if (t < nfull) {
			tp_wait(&bars[s_now], parity_now);
		} else {
			rows_in_tile = (uint32_t)(total - t * TILE);
			tp_copy_ragged(tc, stage, row0, rows_in_tile);
			__syncthreads();
		}
		body(stage, row0, rows_in_tile);
		__syncthreads(); // everyone is done with this stage before it is refilled
	}
}

// barrier among the NC consumer threads only (named barrier 1; the producer warp never joins it)
__device__ __forceinline__ void tp_consumer_sync(int NC) {
	asm volatile("bar.sync 1, %0;" ::"r"(NC) : "memory");
}

// Generic warp-specialised tile loop.  The CTA is launched with NC consumer threads + ONE producer warp
// (blockDim.x == NC + 32).  The producer's lane 0 walks the CTA's tiles (blockIdx.x, blockIdx.x + gridDim.x, ...)
// of rows [row_begin, row_end), waits for empty[s] and issues the TMA copies that complete on full[s]; the
// consumers call body(stage_ptr, row0, rows_in_tile) once per tile.  Inside body use tp_consumer_sync(NC), never
// __syncthreads().  bars: 2*S mbarriers in shared memory.  row_begin must be a multiple of 128 rows (as tc.tile_rows
// is), so that every column's tile - bit-packed ones included - starts 16-byte aligned.
template <class BODY>
__device__ __forceinline__ void tp_tile_loop(const TileCols &tc, int S, unsigned char *stages, uint64_t *bars,
                                             uint64_t row_begin, uint64_t row_end, int NC, BODY body) {
	const uint32_t TILE = tc.tile_rows;
	const uint64_t total = row_end - row_begin;
	const uint64_t ntiles = (total + TILE - 1) / TILE;
	const uint64_t nfull = total / TILE;
	uint64_t *full = bars, *empty = bars + S;
	if (threadIdx.x == 0) {
		for (int s = 0; s < S; s++) {
			tp_mbar_init(&full[s], 1);
			tp_mbar_init(&empty[s], NC / 32); // one arrival per consumer warp
		}
		tp_fence_mbar_init();
	}
	__syncthreads();
	// the k-th tile of the CTA uses stage k mod S in round k / S; both are kept as counters (S is a run-time value
	// and a 64-bit `k % S` / `k / S` is a call into the division routine)
	int s = 0;
	uint32_t parity = 0; // (k / S) & 1
	if ((int)threadIdx.x >= NC) {
		if ((threadIdx.x & 31) == 0) {
			bool refill = false; // k >= S: wait until the consumers are done with the stage's previous tile
			for (uint64_t t = blockIdx.x; t < nfull; t += gridDim.x) {
				if (refill) {
					tp_wait(&empty[s], parity ^ 1u);
				}
				tp_issue_full(tc, stages + (size_t)s * tc.stage_bytes, &full[s], row_begin + t * TILE);
				if (++s == S) {
					s = 0;
					parity ^= 1u;
					refill = true;
				}
			}
		}
	} else {
		for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
			unsigned char *stage = stages + (size_t)s * tc.stage_bytes;
			uint32_t rows_in_tile = TILE;
			uint64_t row0 = row_begin + t * TILE;
			const int s_now = s;
			const uint32_t parity_now = parity;
			if (++s == S) {
				s = 0;
				parity ^= 1u;
			}
			if (t < nfull) {
				tp_wait(&full[s_now], parity_now);
			} else {
				// ragged last tile: plain cooperative copy by the consumers
				tp_consumer_sync(NC);
				rows_in_tile = (uint32_t)(total - t * TILE);
				for (int i = 0; i < tc.n; i++) {
					const TileCol &c = tc.c[i];
					uint32_t bytes = c.width ? rows_in_tile * c.width : (rows_in_tile + 7) / 8;
					const unsigned char *src = c.width ? c.ptr + row0 * c.width : c.ptr + row0 / 8;
					unsigned char *dst = stage + c.smem_off;
					for (uint32_t q = threadIdx.x; q < bytes; q += NC) {
						dst[q] = src[q];
					}
				}
				tp_consumer_sync(NC);
			}
			body(stage, row0, rows_in_tile);
			__syncwarp();
			if ((threadIdx.x & 31) == 0) {
				tp_arrive(&empty[s_now]);
			}
		}
	}
	__syncthreads();
}
#endif

// host: lay the columns out inside a stage
static inline void tile_cols_finish(TileCols *tc, uint32_t tile_rows) {
	uint32_t off = 0;
	tc->tile_rows = tile_rows;
	for (int i = 0; i < tc->n; i++) {
		tc->c[i].smem_off = off;
		uint32_t b = tc->c[i].width ? tile_rows * tc->c[i].width : tile_rows / 8;
		off += (b + 15) & ~15u;
	}
	tc->stage_bytes = (off + 127) & ~127u;
}

static inline bool tile_ptr_ok(const void *p) {
	return (((uintptr_t)p) & 15) == 0;
}
