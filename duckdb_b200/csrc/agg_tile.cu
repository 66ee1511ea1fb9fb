// K6 shared-memory sink paths of the hash aggregate, fed by TMA-staged column tiles (tile_pipe.cuh).
//
// FAST (<= 16 groups per CTA, packed key <= 7 bytes; TPC-H Q1: 4-6 groups)
//   With a handful of groups every row of a warp updates the same few states, and atomics - global or shared -
//   serialise on those addresses.  Every CTA keeps a tiny directory of group keys in shared memory and EVERY
//   THREAD owns a private copy of the states of each directory slot, laid out [slot][field][thread] so a warp's
//   accesses are bank-conflict free.  A row costs a directory lookup plus LDS/ADD/STS per distinct input: no
//   atomics, no shuffles.  At the end the private copies are reduced in 128-bit and merged into the global
//   table with one atomic per (CTA, group, state).
// MID  (<= ~1-2 K groups per CTA; SSB Q4.1: 35 groups)
//   A per-CTA open-addressing table in shared memory; 128-bit sums are four 32-bit words updated with native
//   32-bit ATOMS and explicit carry propagation (64-bit shared atomics are CAS loops on sm_100).
// Rows that do not fit the per-CTA structure take the global path inline (agg_find_or_create + global atomics)
// and are counted in counters[1] so the host can switch path (b200_agg_sink's adaptation).
//
// Reference semantics are those of agg.cu; the reference's analogue of FAST is the per-chunk ClusteredAggr
// regrouping (src/common/clustered_aggregate.cpp:298-316, sum.cpp:92-137).
#include "agg_tile.cuh"
#include <cstring>
#include <cstdlib>
#include <type_traits>

struct FastLayout {
	int n8, n4;
	int f_sum[MAX_INPUTS], f_min[MAX_INPUTS], f_max[MAX_INPUTS]; // 8-byte field index or -1
	int f_cnt[MAX_INPUTS];                                       // 4-byte field index or -1 (field 0 = rows)
	int slots;
};

struct MidLayout {
	int cap;         // slots (power of two)
	int words;       // 32-bit state words per slot
	int w_rows;      // word offsets inside the slot's state block
	int w_cnt[MAX_INPUTS];
	int w_sum[MAX_INPUTS]; // 4 words (int) or 2 words (double bits)
	int w_min[MAX_INPUTS]; // 2 words
	int w_max[MAX_INPUTS]; // 2 words
};

// ------------------------------------------------------------------ FAST
__global__ void __launch_bounds__(AT_THREADS + 32) agg_fast_kernel(const __grid_constant__ TileArgs A, FastLayout F) {
	extern __shared__ __align__(128) unsigned char smem_raw[];
	__shared__ unsigned long long dir_key[FAST_MAX_SLOTS];
	__shared__ uint64_t bars[2 * AT_MAX_STAGES];
	const int tid = threadIdx.x;
	const int SLOTS = F.slots;
	const AggLayout &L = A.L;
	uint64_t *p8 = (uint64_t *)smem_raw; // [slot][n8][thread]
	size_t p8_bytes = (size_t)SLOTS * F.n8 * AT_THREADS * 8;
	uint32_t *p4 = (uint32_t *)(smem_raw + p8_bytes); // [slot][n4][thread]
	size_t p4_bytes = (size_t)SLOTS * F.n4 * AT_THREADS * 4;
	unsigned char *stages = smem_raw + ((p8_bytes + p4_bytes + 127) & ~(size_t)127);

	if (tid < FAST_MAX_SLOTS) {
		dir_key[tid] = 0;
	}
	for (int s = 0; s < SLOTS && tid < AT_THREADS; s++) {
		for (int i = 0; i < L.ninputs; i++) {
			if (F.f_sum[i] >= 0) {
				p8[(s * F.n8 + F.f_sum[i]) * AT_THREADS + tid] = 0;
			}
			if (F.f_min[i] >= 0) {
				p8[(s * F.n8 + F.f_min[i]) * AT_THREADS + tid] = ~0ULL;
			}
			if (F.f_max[i] >= 0) {
				p8[(s * F.n8 + F.f_max[i]) * AT_THREADS + tid] = 0;
			}
		}
		for (int f = 0; f < F.n4; f++) {
			p4[(s * F.n4 + f) * AT_THREADS + tid] = 0;
		}
	}
	unsigned long long missed = 0;

	tile_loop(A, stages, bars, AT_THREADS, [&](const unsigned char *stage, uint32_t r, uint64_t row) {
		uint64_t kw[KEY_WORDS_MAX];
		stage_pack_key(A, stage, r, kw);
		unsigned long long tagged = kw[0] | (1ULL << 56);
		int slot = -1;
#pragma unroll
		for (int s = 0; s < FAST_MAX_SLOTS; s++) {
			if (s < SLOTS && dir_key[s] == tagged) {
				slot = s;
			}
		}
		if (slot < 0) {
			for (int s = 0; s < SLOTS; s++) {
				unsigned long long old = atomicCAS(&dir_key[s], 0ULL, tagged);
				if (old == 0ULL || old == tagged) {
					slot = s;
					break;
				}
			}
		}
		if (slot < 0) {
			missed++;
			row_to_global(A, stage, r, row, kw);
			return;
		}
		p4[(slot * F.n4 + 0) * AT_THREADS + tid] += 1;
#pragma unroll 1
		for (int i = 0; i < L.ninputs; i++) {
			if (!stage_valid(stage, A.tc, A.sm.in_valid[i], r)) {
				continue;
			}
			if (F.f_cnt[i] >= 0) {
				p4[(slot * F.n4 + F.f_cnt[i]) * AT_THREADS + tid] += 1;
			}
			int t = L.input_type[i];
			uint64_t raw = stage_value(stage, A.tc.c[A.sm.in_data[i]], t, r);
			if (F.f_sum[i] >= 0) {
				uint64_t *acc = &p8[(slot * F.n8 + F.f_sum[i]) * AT_THREADS + tid];
				uint64_t cur = *acc;
				if (b200_type_is_float(t)) {
					*acc = (uint64_t)__double_as_longlong(__longlong_as_double((long long)cur) + raw_as_double(t, raw));
				} else {
					// 64-bit private partial; on (rare) wrap-around push the old partial to the global state first
					uint64_t v = cur + raw;
					bool ovf = b200_type_is_signed_int(t) ? ((int64_t)((cur ^ v) & (raw ^ v)) < 0) : (v < cur);
					if (ovf) {
						uint64_t gs = agg_find_or_create(A.T, L, hash_packed_key(L, kw), kw, ~0ULL);
						uint64_t *st = A.T.slots + gs * (uint64_t)L.stride + L.sum_off[i];
						atomic_add_128(st, st + 1, cur, sign_hi(t, cur));
						v = raw;
					}
					*acc = v;
				}
			}
			if (F.f_min[i] >= 0) {
				uint64_t *acc = &p8[(slot * F.n8 + F.f_min[i]) * AT_THREADS + tid];
				uint64_t e = encode_ordered(t, raw);
				if (e < *acc) {
					*acc = e;
				}
			}
			if (F.f_max[i] >= 0) {
				uint64_t *acc = &p8[(slot * F.n8 + F.f_max[i]) * AT_THREADS + tid];
				uint64_t e = encode_ordered(t, raw);
				if (e > *acc) {
					*acc = e;
				}
			}
		}
	});

	if (missed) {
		atomicAdd(&A.counters[1], missed);
	}
	__syncthreads();
	// flush: warp w reduces slots w, w+8, ...; lane l sums threads l, l+32, ...
	const int lane = tid & 31, warp = tid >> 5;
	for (int s = warp; s < SLOTS && warp < AT_THREADS / 32; s += AT_THREADS / 32) {
		if (dir_key[s] == 0ULL) {
			continue;
		}
		unsigned long long rows = 0;
		for (int k = lane; k < AT_THREADS; k += 32) {
			rows += p4[(s * F.n4 + 0) * AT_THREADS + k];
		}
		for (int off = 16; off; off >>= 1) {
			rows += __shfl_xor_sync(0xffffffffu, rows, off);
		}
		if (rows == 0) {
			continue;
		}
		uint64_t gkw[KEY_WORDS_MAX] = {dir_key[s] & ~(0xffULL << 56), 0, 0, 0};
		uint64_t gs = 0;
		if (lane == 0) {
			gs = agg_find_or_create(A.T, L, hash_packed_key(L, gkw), gkw, ~0ULL);
		}
		gs = __shfl_sync(0xffffffffu, gs, 0);
		uint64_t *grow = A.T.slots + gs * (uint64_t)L.stride;
		if (lane == 0) {
			atomicAdd((unsigned long long *)(grow + L.rows_off), rows);
		}
		for (int i = 0; i < L.ninputs; i++) {
			int t = L.input_type[i];
			if (F.f_cnt[i] >= 0) {
				unsigned long long cnt = 0;
				for (int k = lane; k < AT_THREADS; k += 32) {
					cnt += p4[(s * F.n4 + F.f_cnt[i]) * AT_THREADS + k];
				}
				for (int off = 16; off; off >>= 1) {
					cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
				}
				if (lane == 0 && cnt) {
					atomicAdd((unsigned long long *)(grow + L.cnt_off[i]), cnt);
				}
			}
			if (F.f_sum[i] >= 0) {
				if (b200_type_is_float(t)) {
					double v = 0;
					for (int k = lane; k < AT_THREADS; k += 32) {
						v += __longlong_as_double((long long)p8[(s * F.n8 + F.f_sum[i]) * AT_THREADS + k]);
					}
					for (int off = 16; off; off >>= 1) {
						v += __shfl_xor_sync(0xffffffffu, v, off);
					}
					if (lane == 0) {
						atomicAdd((double *)(grow + L.sum_off[i]), v);
					}
				} else {
					uint64_t lo = 0, hi = 0;
					for (int k = lane; k < AT_THREADS; k += 32) {
						uint64_t x = p8[(s * F.n8 + F.f_sum[i]) * AT_THREADS + k];
						uint64_t v = lo + x;
						hi += sign_hi(t, x) + (v < lo ? 1 : 0);
						lo = v;
					}
					for (int off = 16; off; off >>= 1) {
						uint64_t olo = __shfl_xor_sync(0xffffffffu, lo, off);
						uint64_t ohi = __shfl_xor_sync(0xffffffffu, hi, off);
						uint64_t v = lo + olo;
						hi += ohi + (v < lo ? 1 : 0);
						lo = v;
					}
					if (lane == 0) {
						atomic_add_128(grow + L.sum_off[i], grow + L.sum_off[i] + 1, lo, hi);
					}
				}
			}
			if (F.f_min[i] >= 0) {
				uint64_t v = ~0ULL;
				for (int k = lane; k < AT_THREADS; k += 32) {
					uint64_t x = p8[(s * F.n8 + F.f_min[i]) * AT_THREADS + k];
					v = x < v ? x : v;
				}
				for (int off = 16; off; off >>= 1) {
					uint64_t o = __shfl_xor_sync(0xffffffffu, v, off);
					v = o < v ? o : v;
				}
				if (lane == 0) {
					atomicMin((unsigned long long *)(grow + L.min_off[i]), (unsigned long long)v);
				}
			}
			if (F.f_max[i] >= 0) {
				uint64_t v = 0;
				for (int k = lane; k < AT_THREADS; k += 32) {
					uint64_t x = p8[(s * F.n8 + F.f_max[i]) * AT_THREADS + k];
					v = x > v ? x : v;
				}
				for (int off = 16; off; off >>= 1) {
					uint64_t o = __shfl_xor_sync(0xffffffffu, v, off);
					v = o > v ? o : v;
				}
				if (lane == 0) {
					atomicMax((unsigned long long *)(grow + L.max_off[i]), (unsigned long long)v);
				}
			}
		}
	}
}

// ------------------------------------------------------------------ FASTREG
// FAST specialised for the common TPC-H / SSB shape: <= SLOTS (4 or 8) groups, integer group keys without
// NULLs, every aggregate is sum / avg / count over NON-NULL 8-byte integer inputs (BIGINT / DECIMAL(<=18)).
// The per-thread partial sums live in REGISTERS (pa / pb[slot][sum], below); a row adds each value to every slot
// under that slot's hit predicate - no shared-memory traffic for the states, no atomics, and the adds are
// independent, so the SM issues them back to back.  Values with |x| >= 2^40 take the global path.
//
// A tile is THREADS x FR_ROWS rows, so every consumer thread does the same work.  Thread t owns the row pairs
// (2t, 2t+1) and (2t + 2 THREADS, 2t + 2 THREADS + 1): one pair of an 8-byte column is one 16-byte shared load,
// and a warp's loads cover 512 contiguous bytes (no bank conflicts).  A pair whose rows all hit a known slot with
// small values takes the straight-line path; any other pair, and every row of the ragged last tile, goes through
// fr_row (directory insert, wide values, overflow to the global table).
#define FR_ROWS 4
// dynamic shared memory of one CTA: two CTAs, their static shared memory and the 1 KB per CTA that the
// system reserves fit the 228 KB of an SM
#define FR_SMEM_BUDGET (113 * 1024 - 256)

static constexpr int fr_threads(int slots, int nsum) {
	// registers: SLOTS x NSUM x 2 32-bit accumulators (+ directory + one row pair); two CTAs per SM
	return slots * nsum <= 20 ? 224 : (slots * nsum <= 32 ? 192 : 160); // + 1 producer warp
}

// A value x with |x| < 2^40 is accumulated as its two parts x = a * 2^20 + b, a = x >> 20 (signed) and
// b = x & (2^20 - 1), in 32-bit registers: one predicated 32-bit add per part (2 SASS per slot and sum, no carry
// chain).  2048 rows per thread keep both part sums inside 32 bits (-2^20 <= a < 2^20, 0 <= b < 2^20); the tile
// loop folds them into 128-bit per-warp sums in shared memory every FR_FLUSH_TILES tiles.
#define FR_FLUSH_TILES (2048 / FR_ROWS)

template <int NSUM>
struct FrVals {
	uint32_t a[NSUM], b[NSUM];
	int32_t hmax, hmin; // range of the high words
};

template <int NSUM>
__device__ __forceinline__ void fr_split(FrVals<NSUM> &v, int j, uint64_t x) {
	const uint32_t lo = (uint32_t)x, hi = (uint32_t)(x >> 32);
	v.a[j] = __funnelshift_r(lo, hi, 20);
	v.b[j] = lo & 0xfffffu;
}

// |x| < 2^40 for every value: the high words all lie in [-256, 255]
__device__ __forceinline__ bool fr_small(int32_t hmax, int32_t hmin) {
	return hmax < 256 && hmin >= -256;
}

template <int NSUM>
__device__ __forceinline__ void fr_accumulate(uint32_t (&pa)[NSUM], uint32_t (&pb)[NSUM], uint32_t &rows,
                                              const FrVals<NSUM> &v, bool hit) {
#pragma unroll
	for (int j = 0; j < NSUM; j++) {
		asm("{\n.reg .pred p;\nsetp.ne.u32 p, %4, 0;\n@p add.u32 %0, %0, %2;\n@p add.u32 %1, %1, %3;\n}"
		    : "+r"(pa[j]), "+r"(pb[j])
		    : "r"(v.a[j]), "r"(v.b[j]), "r"((uint32_t)hit));
	}
	asm("{\n.reg .pred p;\nsetp.ne.u32 p, %1, 0;\n@p add.u32 %0, %0, 1;\n}" : "+r"(rows) : "r"((uint32_t)hit));
}

__device__ __forceinline__ uint32_t lds_u16(uint32_t a) {
	unsigned short v;
	asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a));
	return v;
}

__device__ __forceinline__ void lds_v2u32(uint32_t a, uint32_t &x, uint32_t &y) {
	asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(x), "=r"(y) : "r"(a));
}

__device__ __forceinline__ void lds_v2u64(uint32_t a, uint64_t &x, uint64_t &y) {
	asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(x), "=l"(y) : "r"(a));
}

// Group tags.  KW == 1 (every key column one byte wide, key j in byte j) with NK <= 3 key bytes: the packed key
// itself, 32 bits, with ~0 (never a key) marking an empty slot.  Otherwise the packed key | 1 << 56 (the
// directory's format), with 0 marking an empty slot.
template <int KW, int NK>
struct FrTag {
	static constexpr bool narrow = KW == 1 && NK <= 3;
	using T = typename std::conditional<narrow, uint32_t, unsigned long long>::type;
	static constexpr T empty = narrow ? (T)~0u : (T)0;
	__device__ static unsigned long long dir(T t) {
		return narrow ? (unsigned long long)t | (1ULL << 56) : (unsigned long long)t;
	}
	__device__ static T of_packed(uint64_t k) {
		return narrow ? (T)k : (T)(k | (1ULL << 56));
	}
};

// tag of row r of the staged tile
template <int KW, int NK>
__device__ __forceinline__ typename FrTag<KW, NK>::T fr_row_tag(const RegLayout &R, const unsigned char *stage, uint32_t r) {
	uint64_t k = 0;
	if constexpr (KW == 1) {
#pragma unroll
		for (int j = 0; j < NK; j++) {
			k |= (uint64_t)stage[R.key_smem_off[j] + r] << (8 * j);
		}
	} else if constexpr (KW == 4) {
		k = *(const uint32_t *)(stage + R.key_smem_off[0] + (size_t)r * 4);
	} else {
#pragma unroll 1
		for (int j = 0; j < R.nkeys; j++) {
			k |= stage_load_uint(stage + R.key_smem_off[j] + r * R.key_width[j], R.key_width[j]) << R.key_shift[j];
		}
	}
	return FrTag<KW, NK>::of_packed(k);
}

// tags of the row pair (r, r + 1), r even
template <int KW, int NK>
__device__ __forceinline__ void fr_pair_tags(const RegLayout &R, const unsigned char *stage, uint32_t sb, uint32_t r,
                                             typename FrTag<KW, NK>::T &t0, typename FrTag<KW, NK>::T &t1) {
	if constexpr (KW == 1) {
		uint32_t a = 0, b = 0;
#pragma unroll
		for (int j = 0; j < NK; j++) {
			uint32_t k = lds_u16(sb + R.key_smem_off[j] + r);
			a |= (k & 0xffu) << (8 * j);
			b |= (k >> 8) << (8 * j);
		}
		t0 = FrTag<KW, NK>::of_packed(a);
		t1 = FrTag<KW, NK>::of_packed(b);
	} else if constexpr (KW == 4) {
		uint32_t a, b;
		lds_v2u32(sb + R.key_smem_off[0] + r * 4, a, b);
		t0 = FrTag<KW, NK>::of_packed(a);
		t1 = FrTag<KW, NK>::of_packed(b);
	} else {
		t0 = fr_row_tag<KW, NK>(R, stage, r);
		t1 = fr_row_tag<KW, NK>(R, stage, r + 1);
	}
}

// 128-bit sum of the warp's per-thread values (lo, hi) into w[0..1] (lane 0 writes; the warp owns w)
__device__ __forceinline__ void fr_warp_add128(uint64_t *w, uint64_t lo, uint64_t hi) {
	for (int off = 16; off; off >>= 1) {
		uint64_t olo = __shfl_xor_sync(0xffffffffu, lo, off);
		uint64_t ohi = __shfl_xor_sync(0xffffffffu, hi, off);
		uint64_t v = lo + olo;
		hi += ohi + (v < lo ? 1 : 0);
		lo = v;
	}
	if ((threadIdx.x & 31) == 0) {
		uint64_t v = w[0] + lo;
		w[1] += hi + (v < lo ? 1 : 0);
		w[0] = v;
	}
}

// Fold the consumer thread's part sums into its warp's 128-bit sums wsum[warp][slot][NSUM * 2 + 1] and clear them
// (warp-collective).
template <int NSUM, int SLOTS>
__device__ __forceinline__ void fr_flush(uint64_t *wsum, uint32_t (&pa)[SLOTS][NSUM], uint32_t (&pb)[SLOTS][NSUM]) {
	uint64_t *w = wsum + (threadIdx.x >> 5) * SLOTS * (NSUM * 2 + 1);
#pragma unroll
	for (int s = 0; s < SLOTS; s++) {
#pragma unroll
		for (int j = 0; j < NSUM; j++) {
			const int64_t v = (int64_t)(int32_t)pa[s][j] * (1LL << 20) + pb[s][j];
			fr_warp_add128(w + s * (NSUM * 2 + 1) + 2 * j, (uint64_t)v, v < 0 ? ~0ULL : 0ULL);
			pa[s][j] = 0;
			pb[s][j] = 0;
		}
	}
}

// The consumer side of agg_fastreg_kernel for one key shape (NK key columns when KW == 1).
template <int NSUM, int SLOTS, int THREADS, int KW, int NK>
__device__ __forceinline__ void fr_consume(const TileArgs &A, const RegLayout &R, unsigned char *stages, uint64_t *bars,
                                           unsigned long long *dir_key, uint64_t *wsum, uint32_t (&rows)[SLOTS],
                                           unsigned long long &missed) {
	using Tag = typename FrTag<KW, NK>::T;
	const uint32_t tid = threadIdx.x;
	Tag dk[SLOTS];
	uint32_t pa[SLOTS][NSUM], pb[SLOTS][NSUM];
#pragma unroll
	for (int s = 0; s < SLOTS; s++) {
		dk[s] = FrTag<KW, NK>::empty;
#pragma unroll
		for (int j = 0; j < NSUM; j++) {
			pa[s][j] = 0;
			pb[s][j] = 0;
		}
	}
	uint32_t tiles = 0; // since the last flush

	// one row on its own: first sight of a key (directory insert), wide values, more than SLOTS groups
	auto fr_row = [&](const unsigned char *stage, uint32_t r, uint64_t row) {
		const Tag tag = fr_row_tag<KW, NK>(R, stage, r);
		FrVals<NSUM> v;
		v.hmax = INT32_MIN;
		v.hmin = INT32_MAX;
#pragma unroll
		for (int j = 0; j < NSUM; j++) {
			const uint64_t x = *(const uint64_t *)(stage + R.sum_smem_off[j] + (size_t)r * 8);
			fr_split(v, j, x);
			v.hmax = max(v.hmax, (int32_t)(x >> 32));
			v.hmin = min(v.hmin, (int32_t)(x >> 32));
		}
		const bool big = !fr_small(v.hmax, v.hmin);
		int slot = -1;
#pragma unroll
		for (int s = 0; s < SLOTS; s++) {
			if (dk[s] == tag) {
				slot = s;
			}
		}
		if (slot < 0 || big) {
			const unsigned long long tagged = FrTag<KW, NK>::dir(tag);
			slot = -1;
			if (!big) {
				for (int s = 0; s < SLOTS; s++) {
					unsigned long long old = atomicCAS(&dir_key[s], 0ULL, tagged);
					if (old == 0ULL || old == tagged) {
						slot = s;
						break;
					}
				}
			}
			if (slot < 0) {
				if (!big) {
					missed++;
				}
				uint64_t kw[KEY_WORDS_MAX] = {tagged & ~(0xffULL << 56), 0, 0, 0};
				row_to_global(A, stage, r, row, kw);
				return;
			}
#pragma unroll
			for (int s = 0; s < SLOTS; s++) {
				if (s == slot) {
					dk[s] = tag;
				}
			}
		}
#pragma unroll
		for (int s = 0; s < SLOTS; s++) {
			fr_accumulate<NSUM>(pa[s], pb[s], rows[s], v, s == slot);
		}
	};

	tp_tile_loop(A.tc, A.stages, stages, bars, A.row_begin, A.row_end, THREADS,
	             [&](const unsigned char *stage, uint64_t row0, uint32_t rows_in_tile) {
		// bit i: the thread's row i (pair i / 2, row i % 2 of the pair) goes through fr_row
		uint32_t slow = 0;
		if (rows_in_tile == THREADS * FR_ROWS) {
			const uint32_t sb = tp_smem_addr(stage);
#pragma unroll
			for (int p = 0; p < FR_ROWS / 2; p++) {
				const uint32_t r = 2 * tid + p * 2 * THREADS;
				Tag t0, t1;
				fr_pair_tags<KW, NK>(R, stage, sb, r, t0, t1);
				FrVals<NSUM> v0, v1;
				int32_t hmax = INT32_MIN, hmin = INT32_MAX;
#pragma unroll
				for (int j = 0; j < NSUM; j++) {
					uint64_t x0, x1;
					lds_v2u64(sb + R.sum_smem_off[j] + r * 8, x0, x1);
					fr_split(v0, j, x0);
					fr_split(v1, j, x1);
					hmax = __vimax3_s32(hmax, (int32_t)(x0 >> 32), (int32_t)(x1 >> 32));
					hmin = __vimin3_s32(hmin, (int32_t)(x0 >> 32), (int32_t)(x1 >> 32));
				}
				bool h0[SLOTS], h1[SLOTS];
				bool any0 = false, any1 = false;
#pragma unroll
				for (int s = 0; s < SLOTS; s++) {
					h0[s] = dk[s] == t0;
					h1[s] = dk[s] == t1;
					any0 |= h0[s];
					any1 |= h1[s];
				}
				if (any0 && any1 && fr_small(hmax, hmin)) {
#pragma unroll
					for (int s = 0; s < SLOTS; s++) {
						fr_accumulate<NSUM>(pa[s], pb[s], rows[s], v0, h0[s]);
						fr_accumulate<NSUM>(pa[s], pb[s], rows[s], v1, h1[s]);
					}
				} else {
					slow |= 3u << (2 * p);
				}
			}
		} else {
#pragma unroll
			for (int i = 0; i < FR_ROWS; i++) {
				if (2 * tid + (i >> 1) * 2 * THREADS + (i & 1) < rows_in_tile) {
					slow |= 1u << i;
				}
			}
		}
		while (slow) {
			const int i = __ffs(slow) - 1;
			slow &= slow - 1;
			const uint32_t r = 2 * tid + (i >> 1) * 2 * THREADS + (i & 1);
			fr_row(stage, r, row0 + r);
		}
		if (++tiles == FR_FLUSH_TILES) {
			fr_flush<NSUM, SLOTS>(wsum, pa, pb);
			tiles = 0;
		}
	});
	if (tid < THREADS) {
		fr_flush<NSUM, SLOTS>(wsum, pa, pb);
	}
}

// dynamic shared memory of a launch: the stage ring, then the per-warp sums
static constexpr size_t fr_wsum_bytes(int slots, int nsum) {
	return (size_t)(fr_threads(slots, nsum) / 32) * slots * (nsum * 2 + 1) * 8;
}

template <int NSUM, int SLOTS, int THREADS, int KW>
__global__ void __launch_bounds__(THREADS + 32, 2) agg_fastreg_kernel(const __grid_constant__ TileArgs A, RegLayout R) {
	extern __shared__ __align__(128) unsigned char smem_raw[];
	__shared__ unsigned long long dir_key[REG_MAX_SLOTS];
	__shared__ uint64_t gslot[REG_MAX_SLOTS];
	__shared__ uint64_t bars[2 * AT_MAX_STAGES];
	constexpr int per_slot = NSUM * 2 + 1;
	constexpr int nwarps = THREADS / 32;
	const int tid = threadIdx.x;
	const AggLayout &L = A.L;
	unsigned char *stages = smem_raw;
	uint64_t *wsum = (uint64_t *)(smem_raw + (size_t)A.stages * A.tc.stage_bytes); // [warp][slot][per_slot]
	if (tid < REG_MAX_SLOTS) {
		dir_key[tid] = 0;
	}
	for (int i = tid; i < nwarps * SLOTS * per_slot; i += blockDim.x) {
		wsum[i] = 0;
	}
	uint32_t rows[SLOTS];
#pragma unroll
	for (int s = 0; s < SLOTS; s++) {
		rows[s] = 0;
	}
	unsigned long long missed = 0;

	// (tp_tile_loop synchronises the CTA before its first tile and after its last)
	if constexpr (KW == 1) {
		// the number of one-byte key columns is a compile-time value of the row loop
		switch (R.nkeys) {
		case 1:
			fr_consume<NSUM, SLOTS, THREADS, KW, 1>(A, R, stages, bars, dir_key, wsum, rows, missed);
			break;
		case 2:
			fr_consume<NSUM, SLOTS, THREADS, KW, 2>(A, R, stages, bars, dir_key, wsum, rows, missed);
			break;
		case 3:
			fr_consume<NSUM, SLOTS, THREADS, KW, 3>(A, R, stages, bars, dir_key, wsum, rows, missed);
			break;
		default:
			fr_consume<NSUM, SLOTS, THREADS, KW, 4>(A, R, stages, bars, dir_key, wsum, rows, missed);
			break;
		}
	} else {
		fr_consume<NSUM, SLOTS, THREADS, KW, 0>(A, R, stages, bars, dir_key, wsum, rows, missed);
	}

	if (missed) {
		atomicAdd(&A.counters[1], missed);
	}
	const int lane = tid & 31, warp = tid >> 5;
	if (tid < THREADS) {
#pragma unroll
		for (int s = 0; s < SLOTS; s++) {
			unsigned long long rr = rows[s];
			for (int off = 16; off; off >>= 1) {
				rr += __shfl_xor_sync(0xffffffffu, rr, off);
			}
			if (lane == 0) {
				wsum[(warp * SLOTS + s) * per_slot + NSUM * 2] = rr;
			}
		}
	}
	__syncthreads();
	if (tid < SLOTS) {
		unsigned long long rr = 0;
		for (int w = 0; w < nwarps; w++) {
			rr += wsum[(w * SLOTS + tid) * per_slot + NSUM * 2];
		}
		uint64_t gs = SLOT_DEFER;
		if (dir_key[tid] != 0ULL && rr) {
			uint64_t gkw[KEY_WORDS_MAX] = {dir_key[tid] & ~(0xffULL << 56), 0, 0, 0};
			gs = agg_find_or_create(A.T, L, hash_packed_key(L, gkw), gkw, ~0ULL);
			atomicAdd((unsigned long long *)(A.T.slots + gs * (uint64_t)L.stride + L.rows_off), rr);
		}
		gslot[tid] = gs;
	}
	__syncthreads();
	if (tid < SLOTS * NSUM) {
		int s = tid / NSUM, j = tid % NSUM;
		if (gslot[s] != SLOT_DEFER) {
			uint64_t lo = 0, hi = 0;
			for (int w = 0; w < nwarps; w++) {
				uint64_t olo = wsum[(w * SLOTS + s) * per_slot + 2 * j];
				uint64_t ohi = wsum[(w * SLOTS + s) * per_slot + 2 * j + 1];
				uint64_t v = lo + olo;
				hi += ohi + (v < lo ? 1 : 0);
				lo = v;
			}
			uint64_t *st = A.T.slots + gslot[s] * (uint64_t)L.stride + L.sum_off[R.in_of_sum[j]];
			atomic_add_128(st, st + 1, lo, hi);
		}
	}
}

template <int NSUM, int SLOTS, int KW>
static int launch_fastreg(b200_ctx *ctx, const TileArgs &A, const RegLayout &R, uint64_t ntiles) {
	constexpr int THREADS = fr_threads(SLOTS, NSUM);
	static bool attr_set = false;
	if (!attr_set) {
		CUDA_TRY(cudaFuncSetAttribute(agg_fastreg_kernel<NSUM, SLOTS, THREADS, KW>,
		                              cudaFuncAttributeMaxDynamicSharedMemorySize, FR_SMEM_BUDGET));
		attr_set = true;
	}
	size_t smem = (size_t)A.stages * A.tc.stage_bytes + fr_wsum_bytes(SLOTS, NSUM);
	uint64_t max_grid = (uint64_t)ctx->sm_count * 2;
	uint64_t grid = ntiles < max_grid ? ntiles : max_grid;
	agg_fastreg_kernel<NSUM, SLOTS, THREADS, KW><<<(unsigned)grid, THREADS + 32, smem, ctx->stream>>>(A, R);
	return B200_OK;
}

template <int SLOTS, int KW>
static int dispatch_fastreg_kw(b200_ctx *ctx, const TileArgs &A, const RegLayout &R, uint64_t ntiles) {
	switch (R.nsum) {
	case 1:
		return launch_fastreg<1, SLOTS, KW>(ctx, A, R, ntiles);
	case 2:
		return launch_fastreg<2, SLOTS, KW>(ctx, A, R, ntiles);
	case 3:
		return launch_fastreg<3, SLOTS, KW>(ctx, A, R, ntiles);
	case 4:
		return launch_fastreg<4, SLOTS, KW>(ctx, A, R, ntiles);
	case 5:
		return launch_fastreg<5, SLOTS, KW>(ctx, A, R, ntiles);
	default:
		return launch_fastreg<6, SLOTS, KW>(ctx, A, R, ntiles);
	}
}

template <int SLOTS>
static int dispatch_fastreg(b200_ctx *ctx, const TileArgs &A, const RegLayout &R, uint64_t ntiles) {
	bool all1 = R.nkeys <= 4;
	for (int j = 0; j < R.nkeys; j++) {
		all1 = all1 && R.key_width[j] == 1 && R.key_shift[j] == (uint32_t)(8 * j);
	}
	if (all1) {
		return dispatch_fastreg_kw<SLOTS, 1>(ctx, A, R, ntiles);
	}
	if (R.nkeys == 1 && R.key_width[0] == 4 && R.key_shift[0] == 0) {
		return dispatch_fastreg_kw<SLOTS, 4>(ctx, A, R, ntiles);
	}
	return dispatch_fastreg_kw<SLOTS, 0>(ctx, A, R, ntiles);
}

// ------------------------------------------------------------------ MID
// shared-memory table: tag[cap] (u32: 0 empty, bit31 ready, low bits = hash | 1), key[cap][2] (u64),
// state[cap][words] (u32)
__device__ __forceinline__ void smem_add_u128(uint32_t *w, uint64_t lo, uint64_t hi) {
	// add the 128-bit value [lo,hi] into four 32-bit words with native 32-bit shared atomics
	uint32_t x[4] = {(uint32_t)lo, (uint32_t)(lo >> 32), (uint32_t)hi, (uint32_t)(hi >> 32)};
	uint32_t carry = 0;
#pragma unroll
	for (int q = 0; q < 4; q++) {
		uint64_t add = (uint64_t)x[q] + carry;
		carry = (uint32_t)(add >> 32);
		uint32_t a = (uint32_t)add;
		if (a) {
			uint32_t old = atomicAdd(&w[q], a);
			carry += (old + a) < old ? 1u : 0u;
		}
	}
}

__device__ __forceinline__ void smem_min_u64(unsigned long long *p, unsigned long long v) {
	atomicMin(p, v); // CAS loop in shared memory; MIN/MAX are rare on this path
}

__global__ void __launch_bounds__(AT_THREADS + 32) agg_mid_kernel(const __grid_constant__ TileArgs A, MidLayout M) {
	extern __shared__ __align__(128) unsigned char smem_raw[];
	__shared__ uint64_t bars[2 * AT_MAX_STAGES];
	__shared__ unsigned int mcount;
	const int tid = threadIdx.x;
	const AggLayout &L = A.L;
	const uint32_t cap = M.cap, cmask = M.cap - 1;
	uint32_t *mtag = (uint32_t *)smem_raw;
	uint64_t *mkey = (uint64_t *)(smem_raw + (((size_t)cap * 4 + 15) & ~(size_t)15));
	uint32_t *mstate = (uint32_t *)((unsigned char *)mkey + (size_t)cap * 16);
	size_t table_bytes = (((size_t)cap * 4 + 15) & ~(size_t)15) + (size_t)cap * 16 + (size_t)cap * M.words * 4;
	unsigned char *stages = smem_raw + ((table_bytes + 127) & ~(size_t)127);

	for (uint32_t s = tid; s < cap && tid < AT_THREADS; s += AT_THREADS) {
		mtag[s] = 0;
		mkey[2 * s] = mkey[2 * s + 1] = 0;
		for (int w = 0; w < M.words; w++) {
			mstate[(size_t)s * M.words + w] = 0;
		}
		for (int i = 0; i < L.ninputs; i++) {
			if (M.w_min[i] >= 0) {
				mstate[(size_t)s * M.words + M.w_min[i]] = 0xffffffffu;
				mstate[(size_t)s * M.words + M.w_min[i] + 1] = 0xffffffffu;
			}
		}
	}
	if (tid == 0) {
		mcount = 0;
	}
	unsigned long long missed = 0;
	const uint32_t fill_limit = cap - cap / 4;

	tile_loop(A, stages, bars, AT_THREADS, [&](const unsigned char *stage, uint32_t r, uint64_t row) {
		uint64_t kw[KEY_WORDS_MAX];
		stage_pack_key(A, stage, r, kw);
		// cheap in-CTA hash of the packed key (the DuckDB hash is only needed when a group goes global)
		uint64_t hh = murmur64(kw[0] ^ (kw[1] * 0x9e3779b97f4a7c15ULL));
		uint32_t tag_locked = ((uint32_t)(hh >> 32) & 0x7fffffffu) | 1u;
		uint32_t tag_ready = tag_locked | 0x80000000u;
		uint32_t slot = (uint32_t)hh & cmask;
		int found = -1;
		for (int probe = 0; probe < 64; probe++) {
			uint32_t t = *(volatile uint32_t *)&mtag[slot];
			if (t == 0) {
				if (*(volatile unsigned int *)&mcount >= fill_limit) {
					break;
				}
				uint32_t old = atomicCAS(&mtag[slot], 0u, tag_locked);
				if (old == 0) {
					atomicAdd(&mcount, 1u);
					mkey[2 * slot] = kw[0];
					mkey[2 * slot + 1] = kw[1];
					__threadfence_block();
					*(volatile uint32_t *)&mtag[slot] = tag_ready;
					found = (int)slot;
					break;
				}
				t = old;
			}
			if ((t | 0x80000000u) == tag_ready) {
				while (!(t & 0x80000000u)) {
					t = *(volatile uint32_t *)&mtag[slot];
				}
				__threadfence_block();
				if (((volatile uint64_t *)mkey)[2 * slot] == kw[0] && ((volatile uint64_t *)mkey)[2 * slot + 1] == kw[1]) {
					found = (int)slot;
					break;
				}
			}
			slot = (slot + 1) & cmask;
		}
		if (found < 0) {
			missed++;
			row_to_global(A, stage, r, row, kw);
			return;
		}
		uint32_t *st = mstate + (size_t)found * M.words;
		atomicAdd(&st[M.w_rows], 1u);
#pragma unroll 1
		for (int i = 0; i < L.ninputs; i++) {
			if (!stage_valid(stage, A.tc, A.sm.in_valid[i], r)) {
				continue;
			}
			int t = L.input_type[i];
			uint64_t raw = stage_value(stage, A.tc.c[A.sm.in_data[i]], t, r);
			if (M.w_cnt[i] >= 0) {
				atomicAdd(&st[M.w_cnt[i]], 1u);
			}
			if (M.w_sum[i] >= 0) {
				if (b200_type_is_float(t)) {
					atomicAdd((double *)&st[M.w_sum[i]], raw_as_double(t, raw));
				} else {
					smem_add_u128(&st[M.w_sum[i]], raw, sign_hi(t, raw));
				}
			}
			if (M.w_min[i] >= 0) {
				smem_min_u64((unsigned long long *)&st[M.w_min[i]], (unsigned long long)encode_ordered(t, raw));
			}
			if (M.w_max[i] >= 0) {
				atomicMax((unsigned long long *)&st[M.w_max[i]], (unsigned long long)encode_ordered(t, raw));
			}
		}
	});

	if (missed) {
		atomicAdd(&A.counters[1], missed);
	}
	__syncthreads();
	// flush every occupied slot into the global table
	for (uint32_t s = tid; s < cap && tid < AT_THREADS; s += AT_THREADS) {
		if (!mtag[s]) {
			continue;
		}
		const uint32_t *st = mstate + (size_t)s * M.words;
		if (st[M.w_rows] == 0) {
			continue;
		}
		uint64_t kw[KEY_WORDS_MAX] = {mkey[2 * s], mkey[2 * s + 1], 0, 0};
		uint64_t gs = agg_find_or_create(A.T, L, hash_packed_key(L, kw), kw, ~0ULL);
		uint64_t *grow = A.T.slots + gs * (uint64_t)L.stride;
		atomicAdd((unsigned long long *)(grow + L.rows_off), (unsigned long long)st[M.w_rows]);
		for (int i = 0; i < L.ninputs; i++) {
			if (M.w_cnt[i] >= 0 && st[M.w_cnt[i]]) {
				atomicAdd((unsigned long long *)(grow + L.cnt_off[i]), (unsigned long long)st[M.w_cnt[i]]);
			}
			if (M.w_sum[i] >= 0) {
				if (b200_type_is_float(L.input_type[i])) {
					double v = *(const double *)&st[M.w_sum[i]];
					atomicAdd((double *)(grow + L.sum_off[i]), v);
				} else {
					uint64_t lo = (uint64_t)st[M.w_sum[i]] | ((uint64_t)st[M.w_sum[i] + 1] << 32);
					uint64_t hi = (uint64_t)st[M.w_sum[i] + 2] | ((uint64_t)st[M.w_sum[i] + 3] << 32);
					atomic_add_128(grow + L.sum_off[i], grow + L.sum_off[i] + 1, lo, hi);
				}
			}
			if (M.w_min[i] >= 0) {
				atomicMin((unsigned long long *)(grow + L.min_off[i]), *(const unsigned long long *)&st[M.w_min[i]]);
			}
			if (M.w_max[i] >= 0) {
				atomicMax((unsigned long long *)(grow + L.max_off[i]), *(const unsigned long long *)&st[M.w_max[i]]);
			}
		}
	}
}

// ------------------------------------------------------------------ MID2 (experimental, B200_AGG_MID2=1)
// Same per-CTA open-addressing table as MID, but the integer sums are kept CARRY-FREE: a value v with |v| < 2^40 is
// biased to u = v + 2^40 (41 bits) and split into three 14-bit limbs, each added to its own 32-bit word with a
// fire-and-forget shared-memory RED (no return value, no carry chain).  A word absorbs 2^18 additions of a
// 14-bit limb before it could wrap, so the CTA flushes its table into the global table every 2^18 rows
// (flush_tiles tiles) and at the end: sum = w0 + (w1 << 14) + (w2 << 28) - count * 2^40.
// Rows with a value outside +-2^40 take the global path (like the register fast path).  More consumer warps than
// MID (the slot lookup is a chain of dependent shared-memory loads; the REDs are not waited for).
// NOT yet measured on hardware: off by default, see DESIGN.md section 8.
struct Mid2Layout {
	int cap;   // slots (power of two)
	int words; // 32-bit state words per slot
	int w_rows;
	int w_cnt[MAX_INPUTS]; // -1: not tracked
	int w_sum[MAX_INPUTS]; // three limb words, -1: no sum on this input
	int flush_tiles;       // flush the per-CTA table every this many tiles (tile_rows * flush_tiles <= 2^18)
};

#define MID2_LIMB_BITS 14
#define MID2_BIAS_SHIFT 40

// tile_loop with a per-tile hook: AFTER(k) runs on every consumer thread once the CTA's k-th tile has been
// consumed and its stage handed back to the producer (all consumers of a CTA see the same k sequence).
template <class BODY, class AFTER>
__device__ __forceinline__ void tile_loop_hook(const TileArgs &A, unsigned char *stages, uint64_t *bars, int NC,
                                               BODY body, AFTER after_tile) {
	const uint32_t TILE = A.tc.tile_rows;
	const uint64_t total = A.row_end - A.row_begin;
	const uint64_t ntiles = (total + TILE - 1) / TILE;
	const uint64_t nfull = total / TILE;
	const int S = A.stages;
	uint64_t *full = bars, *empty = bars + AT_MAX_STAGES;
	if (threadIdx.x == 0) {
		for (int s = 0; s < S; s++) {
			tp_mbar_init(&full[s], 1);
			tp_mbar_init(&empty[s], NC / 32);
		}
		tp_fence_mbar_init();
	}
	__syncthreads();
	if ((int)threadIdx.x >= NC) {
		if ((threadIdx.x & 31) == 0) {
			for (uint64_t k = 0;; k++) {
				uint64_t t = blockIdx.x + k * gridDim.x;
				if (t >= nfull) {
					break;
				}
				int s = (int)(k % S);
				uint64_t use = k / S;
				if (use >= 1) {
					tp_wait(&empty[s], (uint32_t)((use - 1) & 1));
				}
				tp_issue_full(A.tc, stages + (size_t)s * A.tc.stage_bytes, &full[s], A.row_begin + t * TILE);
			}
		}
	} else {
		for (uint64_t k = 0;; k++) {
			uint64_t t = blockIdx.x + k * gridDim.x;
			if (t >= ntiles) {
				break;
			}
			int s = (int)(k % S);
			unsigned char *stage = stages + (size_t)s * A.tc.stage_bytes;
			uint32_t rows_in_tile = TILE;
			uint64_t row0 = A.row_begin + t * TILE;
			if (t < nfull) {
				tp_wait(&full[s], (uint32_t)((k / S) & 1));
			} else {
				asm volatile("bar.sync 1, %0;" ::"r"(NC) : "memory");
				rows_in_tile = (uint32_t)(total - t * TILE);
				for (int i = 0; i < A.tc.n; i++) {
					const TileCol &c = A.tc.c[i];
					uint32_t bytes = c.width ? rows_in_tile * c.width : (rows_in_tile + 7) / 8;
					const unsigned char *src = c.width ? c.ptr + row0 * c.width : c.ptr + row0 / 8;
					unsigned char *dst = stage + c.smem_off;
					for (uint32_t q = threadIdx.x; q < bytes; q += NC) {
						dst[q] = src[q];
					}
				}
				asm volatile("bar.sync 1, %0;" ::"r"(NC) : "memory");
			}
			for (uint32_t r = threadIdx.x; r < rows_in_tile; r += NC) {
				body(stage, r, row0 + r);
			}
			__syncwarp();
			if ((threadIdx.x & 31) == 0) {
				tp_arrive(&empty[s]);
			}
			after_tile(k);
		}
	}
	__syncthreads();
}

template <int NC>
__global__ void __launch_bounds__(NC + 32, 1) agg_mid2_kernel(const __grid_constant__ TileArgs A, Mid2Layout M) {
	extern __shared__ __align__(128) unsigned char smem_raw[];
	__shared__ uint64_t bars[2 * AT_MAX_STAGES];
	__shared__ unsigned int mcount;
	const int tid = threadIdx.x;
	const AggLayout &L = A.L;
	const uint32_t cap = M.cap, cmask = M.cap - 1;
	uint32_t *mtag = (uint32_t *)smem_raw;
	uint64_t *mkey = (uint64_t *)(smem_raw + (((size_t)cap * 4 + 15) & ~(size_t)15));
	uint32_t *mstate = (uint32_t *)((unsigned char *)mkey + (size_t)cap * 16);
	size_t table_bytes = (((size_t)cap * 4 + 15) & ~(size_t)15) + (size_t)cap * 16 + (size_t)cap * M.words * 4;
	unsigned char *stages = smem_raw + ((table_bytes + 127) & ~(size_t)127);

	for (uint32_t s = tid; s < cap && tid < NC; s += NC) {
		mtag[s] = 0;
		mkey[2 * s] = mkey[2 * s + 1] = 0;
		for (int w = 0; w < M.words; w++) {
			mstate[(size_t)s * M.words + w] = 0;
		}
	}
	if (tid == 0) {
		mcount = 0;
	}
	unsigned long long missed = 0;
	const uint32_t fill_limit = cap - cap / 4;

	// merge every slot with pending rows into the global table and clear its state words (consumers only)
	auto flush = [&]() {
		for (uint32_t s = tid; s < cap; s += NC) {
			if (!mtag[s]) {
				continue;
			}
			uint32_t *st = mstate + (size_t)s * M.words;
			uint32_t rows = st[M.w_rows];
			if (rows == 0) {
				continue;
			}
			st[M.w_rows] = 0;
			uint64_t kw[KEY_WORDS_MAX] = {mkey[2 * s], mkey[2 * s + 1], 0, 0};
			uint64_t gs = agg_find_or_create(A.T, L, hash_packed_key(L, kw), kw, ~0ULL);
			uint64_t *grow = A.T.slots + gs * (uint64_t)L.stride;
			atomicAdd((unsigned long long *)(grow + L.rows_off), (unsigned long long)rows);
			for (int i = 0; i < L.ninputs; i++) {
				uint32_t cnt = rows; // values behind the limbs: every row unless the input's NULLs are tracked
				if (M.w_cnt[i] >= 0) {
					cnt = st[M.w_cnt[i]];
					st[M.w_cnt[i]] = 0;
					if (cnt) {
						atomicAdd((unsigned long long *)(grow + L.cnt_off[i]), (unsigned long long)cnt);
					}
				}
				if (M.w_sum[i] >= 0) {
					uint32_t *w = &st[M.w_sum[i]];
					uint64_t biased = (uint64_t)w[0] + ((uint64_t)w[1] << MID2_LIMB_BITS) +
					                  ((uint64_t)w[2] << (2 * MID2_LIMB_BITS));
					w[0] = w[1] = w[2] = 0;
					int64_t sum = (int64_t)biased - ((int64_t)cnt << MID2_BIAS_SHIFT);
					if (cnt) {
						atomic_add_128(grow + L.sum_off[i], grow + L.sum_off[i] + 1, (uint64_t)sum,
						               sum < 0 ? ~0ULL : 0ULL);
					}
				}
			}
		}
	};

	tile_loop_hook(
	    A, stages, bars, NC,
	    [&](const unsigned char *stage, uint32_t r, uint64_t row) {
		    uint64_t kw[KEY_WORDS_MAX];
		    stage_pack_key(A, stage, r, kw);
		    uint64_t hh = murmur64(kw[0] ^ (kw[1] * 0x9e3779b97f4a7c15ULL));
		    uint32_t tag_locked = ((uint32_t)(hh >> 32) & 0x7fffffffu) | 1u;
		    uint32_t tag_ready = tag_locked | 0x80000000u;
		    uint32_t slot = (uint32_t)hh & cmask;
		    int found = -1;
		    for (int probe = 0; probe < 64; probe++) {
			    uint32_t t = *(volatile uint32_t *)&mtag[slot];
			    if (t == 0) {
				    if (*(volatile unsigned int *)&mcount >= fill_limit) {
					    break;
				    }
				    uint32_t old = atomicCAS(&mtag[slot], 0u, tag_locked);
				    if (old == 0) {
					    atomicAdd(&mcount, 1u);
					    mkey[2 * slot] = kw[0];
					    mkey[2 * slot + 1] = kw[1];
					    __threadfence_block();
					    *(volatile uint32_t *)&mtag[slot] = tag_ready;
					    found = (int)slot;
					    break;
				    }
				    t = old;
			    }
			    if ((t | 0x80000000u) == tag_ready) {
				    while (!(t & 0x80000000u)) {
					    t = *(volatile uint32_t *)&mtag[slot];
				    }
				    __threadfence_block();
				    if (((volatile uint64_t *)mkey)[2 * slot] == kw[0] && ((volatile uint64_t *)mkey)[2 * slot + 1] == kw[1]) {
					    found = (int)slot;
					    break;
				    }
			    }
			    slot = (slot + 1) & cmask;
		    }
		    if (found < 0) {
			    missed++;
			    row_to_global(A, stage, r, row, kw);
			    return;
		    }
		    // a row is applied entirely here or entirely on the global path: check the limb range first
		    bool in_range = true;
#pragma unroll 1
		    for (int i = 0; i < L.ninputs; i++) {
			    if (M.w_sum[i] >= 0 && stage_valid(stage, A.tc, A.sm.in_valid[i], r)) {
				    int64_t v = (int64_t)stage_value(stage, A.tc.c[A.sm.in_data[i]], L.input_type[i], r);
				    in_range = in_range && (uint64_t)(v + (1LL << MID2_BIAS_SHIFT)) < (1ULL << (MID2_BIAS_SHIFT + 1));
			    }
		    }
		    if (!in_range) {
			    row_to_global(A, stage, r, row, kw);
			    return;
		    }
		    uint32_t *st = mstate + (size_t)found * M.words;
		    atomicAdd(&st[M.w_rows], 1u);
#pragma unroll 1
		    for (int i = 0; i < L.ninputs; i++) {
			    if (!stage_valid(stage, A.tc, A.sm.in_valid[i], r)) {
				    continue;
			    }
			    if (M.w_cnt[i] >= 0) {
				    atomicAdd(&st[M.w_cnt[i]], 1u);
			    }
			    if (M.w_sum[i] >= 0) {
				    int64_t v = (int64_t)stage_value(stage, A.tc.c[A.sm.in_data[i]], L.input_type[i], r);
				    uint64_t u = (uint64_t)(v + (1LL << MID2_BIAS_SHIFT));
				    const uint32_t limb_mask = (1u << MID2_LIMB_BITS) - 1;
				    atomicAdd(&st[M.w_sum[i]], (uint32_t)u & limb_mask);
				    atomicAdd(&st[M.w_sum[i] + 1], (uint32_t)(u >> MID2_LIMB_BITS) & limb_mask);
				    atomicAdd(&st[M.w_sum[i] + 2], (uint32_t)(u >> (2 * MID2_LIMB_BITS)));
			    }
		    }
	    },
	    [&](uint64_t k) {
		    if ((k + 1) % (uint64_t)M.flush_tiles == 0) {
			    asm volatile("bar.sync 1, %0;" ::"r"(NC) : "memory");
			    flush();
			    asm volatile("bar.sync 1, %0;" ::"r"(NC) : "memory");
		    }
	    });

	if (missed) {
		atomicAdd(&A.counters[1], missed);
	}
	if (tid < NC) {
		flush();
	}
}

template <int NC>
static int launch_mid2(b200_ctx *ctx, const TileArgs &A, const Mid2Layout &M, unsigned grid, size_t smem) {
	static bool attr_set = false;
	if (!attr_set) {
		CUDA_TRY(cudaFuncSetAttribute(agg_mid2_kernel<NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM_BUDGET));
		attr_set = true;
	}
	agg_mid2_kernel<NC><<<grid, NC + 32, smem, ctx->stream>>>(A, M);
	return B200_OK;
}

// ------------------------------------------------------------------ host
static bool col_stageable(const DCol &c) {
	if (c.vtype != B200_FLAT_VECTOR || !tile_ptr_ok(c.data)) {
		return false;
	}
	if (c.validity && !tile_ptr_ok(c.validity)) {
		return false;
	}
	return true;
}

int b200_agg_tile_eligible(const AggLayout &L, const KeyCols &keys, const AggCols &ac) {
	for (int j = 0; j < L.nkeys; j++) {
		if (!col_stageable(keys.c[j])) {
			return B200_ERR_INVALID;
		}
	}
	for (int i = 0; i < L.ninputs; i++) {
		if (!col_stageable(ac.c[i])) {
			return B200_ERR_INVALID;
		}
	}
	return B200_OK; // (key width limits of the individual paths are checked by b200_agg_sink)
}

static int add_tile_col(TileCols *tc, const void *ptr, uint32_t width) {
	// the same column may be referenced several times (key and input, or two inputs): stage it once
	for (int i = 0; i < tc->n; i++) {
		if (tc->c[i].ptr == (const unsigned char *)ptr && tc->c[i].width == width) {
			return i;
		}
	}
	if (tc->n >= TP_MAX_COLS) {
		return -1;
	}
	tc->c[tc->n].ptr = (const unsigned char *)ptr;
	tc->c[tc->n].width = width;
	return tc->n++;
}

// upper bound on the groups one launch can add to the global table through the end-of-CTA flushes
uint64_t b200_agg_tile_headroom(int mode, int sm_count) {
	return (uint64_t)sm_count * (mode == 0 ? FAST_MAX_SLOTS : (mode == 2 ? 1024 : 4096));
}

// agg_priv.cu
struct PrivDirect;
int b200_agg_priv_launch(b200_ctx *ctx, TileArgs &A, const AggLayout &L, const KeyCols &keys, const AggCols &ac, int groups_hint,
                         const PrivDirect *direct);

int b200_agg_tile_sink(b200_ctx *ctx, int mode, int slots_hint, const AggLayout &L, const AggTable &T,
                       const KeyCols &keys, const AggCols &ac, uint64_t row_begin, uint64_t row_end,
                       uint32_t *deferred, unsigned long long *counters, const PrivDirect *direct) {
	if (row_begin % AT_TILE) {
		b200_set_error("agg tile path: row_begin must be a multiple of %d", AT_TILE);
		return B200_ERR_INVALID;
	}
	TileArgs A;
	memset(&A, 0, sizeof(A));
	A.T = T;
	A.L = L;
	A.keys = keys;
	A.ac = ac;
	A.row_begin = row_begin;
	A.row_end = row_end;
	A.deferred = deferred;
	A.counters = counters;
	A.tc.n = 0;
	bool ok = true;
	for (int j = 0; j < L.nkeys; j++) {
		A.sm.key_data[j] = add_tile_col(&A.tc, keys.c[j].data, b200_type_size(keys.c[j].type));
		A.sm.key_valid[j] = keys.c[j].validity ? add_tile_col(&A.tc, keys.c[j].validity, 0) : -1;
		ok = ok && A.sm.key_data[j] >= 0 && (!keys.c[j].validity || A.sm.key_valid[j] >= 0);
	}
	for (int i = 0; i < L.ninputs; i++) {
		A.sm.in_data[i] = add_tile_col(&A.tc, ac.c[i].data, b200_type_size(ac.c[i].type));
		A.sm.in_valid[i] = ac.c[i].validity ? add_tile_col(&A.tc, ac.c[i].validity, 0) : -1;
		ok = ok && A.sm.in_data[i] >= 0 && (!ac.c[i].validity || A.sm.in_valid[i] >= 0);
	}
	if (!ok) {
		b200_set_error("agg tile path: too many staged columns");
		return B200_ERR_INVALID;
	}
	tile_cols_finish(&A.tc, AT_TILE);
	uint64_t n = row_end - row_begin;
	uint64_t ntiles = (n + AT_TILE - 1) / AT_TILE;
	static bool attr_set = false;
	if (!attr_set) {
		CUDA_TRY(cudaFuncSetAttribute(agg_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM_BUDGET));
		CUDA_TRY(cudaFuncSetAttribute(agg_mid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, AT_SMEM_BUDGET));
		attr_set = true;
	}
	if (mode == 2) {
		// thread-private shared-memory accumulators (agg_priv.cu); shapes it does not take fall back to MID
		int rc = b200_agg_priv_launch(ctx, A, L, keys, ac, slots_hint, direct);
		if (rc == B200_OK) {
			ctx->launches++;
			return B200_OK;
		}
		if (rc != B200_ERR_INVALID) {
			return rc;
		}
		tile_cols_finish(&A.tc, AT_TILE);
		mode = 1;
	}
	if (mode == 0) {
		// register-accumulator specialisation: sums / counts over non-NULL 8-byte integer inputs, integer keys
		RegLayout R;
		memset(&R, 0, sizeof(R));
		bool reg_ok = L.key_bytes <= 7;
		size_t fr_extra = 0;
		R.nkeys = L.nkeys;
		for (int j = 0; j < L.nkeys && reg_ok; j++) {
			reg_ok = b200_type_is_integer(L.key_type[j]) && !keys.c[j].validity;
			R.key_smem_off[j] = A.tc.c[A.sm.key_data[j]].smem_off;
			R.key_width[j] = b200_type_size(L.key_type[j]);
			R.key_shift[j] = L.key_off[j] * 8;
		}
		for (int i = 0; i < L.ninputs && reg_ok; i++) {
			reg_ok = b200_type_is_integer(L.input_type[i]) && !ac.track_cnt[i] && L.min_off[i] < 0 && L.max_off[i] < 0;
			if (reg_ok && L.sum_off[i] >= 0) {
				if (R.nsum >= REG_MAX_SUMS || b200_type_size(L.input_type[i]) != 8) {
					reg_ok = false;
				} else {
					R.sum_smem_off[R.nsum] = A.tc.c[A.sm.in_data[i]].smem_off;
					R.in_of_sum[R.nsum++] = i;
				}
			}
		}
		if (reg_ok && R.nsum >= 1) {
			// tiles of FR_ROWS rows per consumer thread; as many stages (up to 3) as fit two CTAs per SM.  Q1
			// (42 B/row, 896-row tiles): 3 x 37.6 KB, so two tiles per CTA are in flight while it works on a third.
			const int slots = slots_hint <= 4 ? 4 : 8;
			uint32_t rows = (uint32_t)fr_threads(slots, R.nsum) * FR_ROWS;
			tile_cols_finish(&A.tc, rows);
			fr_extra = fr_wsum_bytes(slots, R.nsum);
			A.stages = AT_MAX_STAGES;
			while (A.stages > 2 && (size_t)A.stages * A.tc.stage_bytes + fr_extra > FR_SMEM_BUDGET) {
				A.stages--;
			}
			ntiles = (n + rows - 1) / rows;
			for (int j = 0; j < L.nkeys; j++) {
				R.key_smem_off[j] = A.tc.c[A.sm.key_data[j]].smem_off;
			}
			for (int j = 0; j < R.nsum; j++) {
				R.sum_smem_off[j] = A.tc.c[A.sm.in_data[R.in_of_sum[j]]].smem_off;
			}
		}
		if (reg_ok && R.nsum >= 1 && (size_t)A.stages * A.tc.stage_bytes + fr_extra <= FR_SMEM_BUDGET) {
			// first try 4 slots (TPC-H Q1 has 4 groups); the caller escalates to 8 slots, then MID, then GLOBAL
			int rc = slots_hint <= 4 ? dispatch_fastreg<4>(ctx, A, R, ntiles) : dispatch_fastreg<8>(ctx, A, R, ntiles);
			ctx->launches++;
			B200_TRY(rc);
			CUDA_TRY(cudaGetLastError());
			return B200_OK;
		}
		tile_cols_finish(&A.tc, AT_TILE);
		ntiles = (n + AT_TILE - 1) / AT_TILE;
		FastLayout F;
		memset(&F, 0, sizeof(F));
		F.n8 = 0;
		F.n4 = 1;
		for (int i = 0; i < L.ninputs; i++) {
			F.f_sum[i] = L.sum_off[i] >= 0 ? F.n8++ : -1;
			F.f_min[i] = L.min_off[i] >= 0 ? F.n8++ : -1;
			F.f_max[i] = L.max_off[i] >= 0 ? F.n8++ : -1;
			F.f_cnt[i] = ac.track_cnt[i] ? F.n4++ : -1;
		}
		size_t per_slot = (size_t)AT_THREADS * (F.n8 * 8 + F.n4 * 4);
		int best_slots = 0, best_stages = 0;
		const int cand[][2] = {{16, 3}, {8, 3}, {16, 2}, {8, 2}, {4, 3}, {4, 2}, {2, 2}};
		for (auto &c : cand) {
			size_t need = ((per_slot * c[0] + 127) & ~(size_t)127) + (size_t)c[1] * A.tc.stage_bytes + 256;
			if (need <= AT_SMEM_BUDGET) {
				best_slots = c[0];
				best_stages = c[1];
				break;
			}
		}
		if (!best_slots) {
			b200_set_error("agg fast path: states do not fit shared memory");
			return B200_ERR_INVALID;
		}
		F.slots = best_slots;
		A.stages = best_stages;
		size_t smem = ((per_slot * F.slots + 127) & ~(size_t)127) + (size_t)A.stages * A.tc.stage_bytes;
		uint64_t grid = ntiles < (uint64_t)ctx->sm_count ? ntiles : (uint64_t)ctx->sm_count;
		agg_fast_kernel<<<(unsigned)grid, AT_THREADS + 32, smem, ctx->stream>>>(A, F);
	} else {
		// experimental carry-free variant (B200_AGG_MID2=<consumer threads: 512 | 704 | 960>, any other value > 0 = 704):
		// integer sums / counts only.  Tiles hold 2 rows per consumer thread so that every warp gets the same work.
		const char *mid2_env = getenv("B200_AGG_MID2");
		bool mid2 = mid2_env && atoi(mid2_env) > 0;
		for (int i = 0; i < L.ninputs && mid2; i++) {
			mid2 = b200_type_is_integer(L.input_type[i]) && L.min_off[i] < 0 && L.max_off[i] < 0;
		}
		if (mid2) {
			int nc = atoi(mid2_env);
			nc = (nc == 512 || nc == 960) ? nc : 704;
			Mid2Layout M2;
			memset(&M2, 0, sizeof(M2));
			int w2 = 0;
			M2.w_rows = w2++;
			for (int i = 0; i < L.ninputs; i++) {
				M2.w_cnt[i] = ac.track_cnt[i] ? w2++ : -1;
				M2.w_sum[i] = -1;
				if (L.sum_off[i] >= 0) {
					M2.w_sum[i] = w2;
					w2 += 3;
				}
			}
			M2.words = w2;
			uint32_t rows2 = 2u * (uint32_t)nc; // a multiple of 128 for all three thread counts
			tile_cols_finish(&A.tc, rows2);
			uint64_t ntiles2 = (n + rows2 - 1) / rows2;
			M2.flush_tiles = (int)((1u << 18) / rows2);
			A.stages = 2;
			int cap2 = 4096;
			size_t table2 = 0;
			while (cap2 >= 64) {
				table2 = (((size_t)cap2 * 4 + 15) & ~(size_t)15) + (size_t)cap2 * 16 + (size_t)cap2 * M2.words * 4;
				if (((table2 + 127) & ~(size_t)127) + (size_t)A.stages * A.tc.stage_bytes + 256 <= AT_SMEM_BUDGET) {
					break;
				}
				cap2 >>= 1;
			}
			if (cap2 >= 64 && M2.flush_tiles >= 1) {
				M2.cap = cap2;
				size_t smem2 = ((table2 + 127) & ~(size_t)127) + (size_t)A.stages * A.tc.stage_bytes;
				unsigned grid2 = (unsigned)(ntiles2 < (uint64_t)ctx->sm_count ? ntiles2 : (uint64_t)ctx->sm_count);
				int rc = nc == 512   ? launch_mid2<512>(ctx, A, M2, grid2, smem2)
				         : nc == 960 ? launch_mid2<960>(ctx, A, M2, grid2, smem2)
				                     : launch_mid2<704>(ctx, A, M2, grid2, smem2);
				B200_TRY(rc);
				ctx->launches++;
				CUDA_TRY(cudaGetLastError());
				return B200_OK;
			}
			tile_cols_finish(&A.tc, AT_TILE); // does not fit: back to the MID layout below
		}
		MidLayout M;
		memset(&M, 0, sizeof(M));
		int w = 0;
		M.w_rows = w++;
		for (int i = 0; i < L.ninputs; i++) {
			M.w_cnt[i] = ac.track_cnt[i] ? w++ : -1;
			M.w_sum[i] = M.w_min[i] = M.w_max[i] = -1;
			if (L.sum_off[i] >= 0) {
				w = (w + 1) & ~1; // 8-byte alignment for the double / 64-bit views
				M.w_sum[i] = w;
				w += b200_type_is_float(L.input_type[i]) ? 2 : 4;
			}
			if (L.min_off[i] >= 0) {
				w = (w + 1) & ~1;
				M.w_min[i] = w;
				w += 2;
			}
			if (L.max_off[i] >= 0) {
				w = (w + 1) & ~1;
				M.w_max[i] = w;
				w += 2;
			}
		}
		M.words = (w + 1) & ~1;
		A.stages = 2;
		int cap = 4096;
		while (cap >= 64) {
			size_t table = (((size_t)cap * 4 + 15) & ~(size_t)15) + (size_t)cap * 16 + (size_t)cap * M.words * 4;
			if (((table + 127) & ~(size_t)127) + (size_t)A.stages * A.tc.stage_bytes + 256 <= AT_SMEM_BUDGET) {
				break;
			}
			cap >>= 1;
		}
		if (cap < 64) {
			b200_set_error("agg mid path: states do not fit shared memory");
			return B200_ERR_INVALID;
		}
		M.cap = cap;
		size_t table = (((size_t)cap * 4 + 15) & ~(size_t)15) + (size_t)cap * 16 + (size_t)cap * M.words * 4;
		size_t smem = ((table + 127) & ~(size_t)127) + (size_t)A.stages * A.tc.stage_bytes;
		uint64_t grid = ntiles < (uint64_t)ctx->sm_count ? ntiles : (uint64_t)ctx->sm_count;
		agg_mid_kernel<<<(unsigned)grid, AT_THREADS + 32, smem, ctx->stream>>>(A, M);
	}
	ctx->launches++;
	CUDA_TRY(cudaGetLastError());
	return B200_OK;
}
