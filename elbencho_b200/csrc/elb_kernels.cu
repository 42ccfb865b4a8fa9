/*
 * Hand-written sm_100a kernels for the on-GPU work of the LocalWorker hot path:
 *
 *   K1 fill_pattern   <- LocalWorker::preWriteIntegrityCheckFillBuf   (LocalWorker.cpp:2091-2128)
 *   K2 verify_pattern <- LocalWorker::postReadIntegrityCheckVerifyBuf (LocalWorker.cpp:2137-2179)
 *   K3 fill_random    <- LocalWorker::preWriteBufRandRefillCuda + bufFill (:2185-2203, 2236-2277)
 *
 * All three are HBM-bound byte/integer kernels (K1/K3: 1 byte written per payload byte, K2: 1 byte
 * read per payload byte), so the design follows the streaming rules: 32-byte (256-bit) vector
 * accesses per thread (LDG/STG.E.256 on sm_100), fully coalesced (a warp covers 1 KiB per access),
 * L1 no-allocate hints, several independent accesses in flight per thread, and a grid sized to a
 * multiple of the SM count that walks "tiles" of the whole in-flight window (many blocks per
 * launch) so that one launch covers tens to hundreds of MiB.
 *
 * Staged forms (the worker's default staging engine): the same kernels also move the block between
 * the pinned host ring and the device ring while they work on it, so that a batch's whole GPU
 * stage is ONE launch and no copy engine is involved:
 *   fill + stage-out   : every generated vector is stored to the device slot AND to the host slot
 *                        (zero-copy stores over PCIe)
 *   stage-in + verify  : every vector is loaded from the host slot (zero-copy load over PCIe),
 *                        stored to the device slot and compared
 *   stage copy         : plain slot copy host->device / device->host for runs without --verify /
 *                        fill
 * The host slot of a block is at (device address + hostDelta); both rings have the same layout, so
 * alignment and tile geometry are the same on both sides. Descriptors are read straight from
 * pinned host memory, and the last CTA of a verify launch (device-side ticket) publishes the
 * per-block results to pinned host memory and re-arms the device copies: no descriptor copy, no
 * result copy, no init launch. These launches are PCIe-bound (measured ~47 GiB/s per direction for
 * 1 MiB blocks, profiles/r02_hostpath_exploration.jsonl), the resident forms are HBM-bound.
 *
 * One launch processes an array of block descriptors {devPtr, len, fileOffset, blockCounter}.
 * Tiles are ELB_TILE_BYTES slices of a block's 32-byte-aligned body; unaligned head/tail bytes
 * (device address not 32-byte aligned, or odd lengths) are handled byte-wise by tile 0 of the
 * block. Mismatch counts are reduced per warp (redux.sync) before touching global atomics.
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <atomic>
#include <mutex>
#include <string>

#include "elb_patterns.cuh"
#include "elb_internal.h"

#define ELB_THREADS 256
#define ELB_VEC_BYTES 32
#define ELB_UNROLL 4
#define ELB_TILE_BYTES (ELB_THREADS * ELB_VEC_BYTES * ELB_UNROLL) /* 32 KiB */

struct __align__(32) u64x4
{
	uint64_t a, b, c, d;
};

__device__ __forceinline__ void st_na_256(void* ptr, const u64x4& v)
{
	asm volatile("st.global.L1::no_allocate.v4.u64 [%0], {%1,%2,%3,%4};"
		:: "l"(ptr), "l"(v.a), "l"(v.b), "l"(v.c), "l"(v.d) : "memory");
}

__device__ __forceinline__ u64x4 ld_nc_na_256(const void* ptr)
{
	u64x4 v;
	asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];"
		: "=l"(v.a), "=l"(v.b), "=l"(v.c), "=l"(v.d) : "l"(ptr) );
	return v;
}

/* number of differing bytes between two u64 */
__device__ __forceinline__ unsigned diff_bytes64(uint64_t x, uint64_t y)
{
	const unsigned lo = __vcmpne4( (unsigned)x, (unsigned)y);
	const unsigned hi = __vcmpne4( (unsigned)(x >> 32), (unsigned)(y >> 32) );
	return (__popc(lo) + __popc(hi) ) >> 3;
}

/* index (0..7) of the first differing byte of two unequal u64 */
__device__ __forceinline__ unsigned first_diff_byte64(uint64_t x, uint64_t y)
{
	return (unsigned)(__ffsll( (long long)(x ^ y) ) - 1) >> 3;
}

/* ---- generators ------------------------------------------------------------------------- */

struct PatternGen
{
	uint64_t fileOffset; // file offset of block byte 0
	uint64_t salt;

	/* fast path is valid when the file position of every 32-byte vector is 8-byte aligned */
	__device__ __forceinline__ bool canUseFast(uint64_t headLen) const
		{ return ( (fileOffset + headLen) & 7) == 0; }

	template<bool FAST>
	__device__ __forceinline__ u64x4 vec32(uint64_t pos) const
	{
		u64x4 v;

		if(FAST)
		{ // four consecutive aligned checksum words: offset + salt (LocalWorker.cpp:2110-2112)
			const uint64_t w = fileOffset + pos + salt;
			v.a = w;
			v.b = w + 8;
			v.c = w + 16;
			v.d = w + 24;
		}
		else
		{ // block starts in the middle of a checksum word: funnel-shift neighbours together
			const uint64_t filePos = fileOffset + pos;
			const unsigned shiftBits = (unsigned)(filePos & 7) * 8; // != 0 here
			const uint64_t w0 = (filePos & ~7ULL) + salt;
			const uint64_t w1 = w0 + 8, w2 = w0 + 16, w3 = w0 + 24, w4 = w0 + 32;
			v.a = (w0 >> shiftBits) | (w1 << (64 - shiftBits) );
			v.b = (w1 >> shiftBits) | (w2 << (64 - shiftBits) );
			v.c = (w2 >> shiftBits) | (w3 << (64 - shiftBits) );
			v.d = (w3 >> shiftBits) | (w4 << (64 - shiftBits) );
		}

		return v;
	}

	__device__ __forceinline__ uint8_t byte(uint64_t pos) const
		{ return elb_pattern_byte(fileOffset + pos, salt); }
};

struct RandomGen
{
	uint64_t blockKey;
	uint64_t varFillLen;
	uint64_t remainderVal;

	/* fast path is valid when every 32-byte vector starts on a word boundary of the block */
	__device__ __forceinline__ bool canUseFast(uint64_t headLen) const
		{ return (headLen & 7) == 0; }

	template<bool FAST>
	__device__ __forceinline__ u64x4 vec32(uint64_t pos) const
	{
		u64x4 v;

		if(FAST && ( (pos + ELB_VEC_BYTES) <= varFillLen) )
		{ // four whole random words
			const uint64_t wordIdx = pos >> 3;
			v.a = elb_rand_word(blockKey, wordIdx);
			v.b = elb_rand_word(blockKey, wordIdx + 1);
			v.c = elb_rand_word(blockKey, wordIdx + 2);
			v.d = elb_rand_word(blockKey, wordIdx + 3);
		}
		else if(FAST && (pos >= varFillLen) )
		{ // constant remainder: the same rotation of the repeated u64 four times
			const unsigned rotBits = (unsigned)( (pos - varFillLen) & 7) * 8;
			const uint64_t val = rotBits ?
				( (remainderVal >> rotBits) | (remainderVal << (64 - rotBits) ) ) : remainderVal;
			v.a = v.b = v.c = v.d = val;
		}
		else
		{ // boundary vector or unaligned block start
			v.a = elb_rand_bytes8(pos, blockKey, varFillLen, remainderVal);
			v.b = elb_rand_bytes8(pos + 8, blockKey, varFillLen, remainderVal);
			v.c = elb_rand_bytes8(pos + 16, blockKey, varFillLen, remainderVal);
			v.d = elb_rand_bytes8(pos + 24, blockKey, varFillLen, remainderVal);
		}

		return v;
	}

	__device__ __forceinline__ uint8_t byte(uint64_t pos) const
		{ return elb_rand_byte(pos, blockKey, varFillLen, remainderVal); }
};

/* ---- block geometry --------------------------------------------------------------------- */

struct BlockGeom
{
	uint8_t* ptr;      // device address of block byte 0
	uint64_t len;
	uint64_t headLen;  // bytes before the first 32-byte aligned address (< 32, <= len)
	uint64_t bodyLen;  // multiple of 32
	uint64_t tailLen;  // < 32
	uint64_t numTiles; // >= 1 for len > 0 (tile 0 also does head/tail)
};

__device__ __forceinline__ BlockGeom make_geom(const elb_block_desc& desc)
{
	BlockGeom g;
	g.ptr = (uint8_t*)desc.devPtr;
	g.len = desc.len;

	const uint64_t misalign = (uint64_t)(uintptr_t)g.ptr & (ELB_VEC_BYTES - 1);
	uint64_t headLen = misalign ? (ELB_VEC_BYTES - misalign) : 0;
	if(headLen > g.len)
		headLen = g.len;

	g.headLen = headLen;
	g.bodyLen = (g.len - headLen) & ~(uint64_t)(ELB_VEC_BYTES - 1);
	g.tailLen = g.len - headLen - g.bodyLen;
	g.numTiles = (g.bodyLen + ELB_TILE_BYTES - 1) / ELB_TILE_BYTES;
	if(!g.numTiles && g.len)
		g.numTiles = 1;

	return g;
}

/* ---- fill ------------------------------------------------------------------------------- */

template<bool FAST, bool STAGED, class Gen>
__device__ __forceinline__ void fill_tile(const BlockGeom& g, const Gen& gen, uint64_t tileIdx,
	int64_t hostDelta)
{
	const uint64_t tileStart = tileIdx * ELB_TILE_BYTES; // within body
	uint8_t* bodyPtr = g.ptr + g.headLen;

	if( (tileStart + ELB_TILE_BYTES) <= g.bodyLen)
	{ // full tile: no bounds checks, all stores independent
		#pragma unroll
		for(int u = 0; u < ELB_UNROLL; u++)
		{
			const uint64_t bodyOff = tileStart +
				(uint64_t)(u * ELB_THREADS + threadIdx.x) * ELB_VEC_BYTES;
			const uint64_t pos = g.headLen + bodyOff;
			const u64x4 v = gen.template vec32<FAST>(pos);
			st_na_256(bodyPtr + bodyOff, v);
			if(STAGED)
				st_na_256(bodyPtr + hostDelta + bodyOff, v);
		}
	}
	else
	{
		#pragma unroll
		for(int u = 0; u < ELB_UNROLL; u++)
		{
			const uint64_t bodyOff = tileStart +
				(uint64_t)(u * ELB_THREADS + threadIdx.x) * ELB_VEC_BYTES;
			if(bodyOff < g.bodyLen)
			{
				const uint64_t pos = g.headLen + bodyOff;
				const u64x4 v = gen.template vec32<FAST>(pos);
				st_na_256(bodyPtr + bodyOff, v);
				if(STAGED)
					st_na_256(bodyPtr + hostDelta + bodyOff, v);
			}
		}
	}

	if(!tileIdx && (g.headLen | g.tailLen) )
	{ // unaligned head/tail bytes (at most 31 each)
		if(threadIdx.x < g.headLen)
		{
			const uint8_t b = gen.byte(threadIdx.x);
			g.ptr[threadIdx.x] = b;
			if(STAGED)
				g.ptr[hostDelta + (int64_t)threadIdx.x] = b;
		}

		const uint64_t tailStart = g.headLen + g.bodyLen;
		if(threadIdx.x < g.tailLen)
		{
			const uint8_t b = gen.byte(tailStart + threadIdx.x);
			g.ptr[tailStart + threadIdx.x] = b;
			if(STAGED)
				g.ptr[hostDelta + (int64_t)(tailStart + threadIdx.x)] = b;
		}
	}
}

/* plain slot copy between the rings: IN = host slot -> device slot, else device -> host */
template<bool IN>
__device__ __forceinline__ void copy_tile(const BlockGeom& g, uint64_t tileIdx, int64_t hostDelta)
{
	const uint64_t tileStart = tileIdx * ELB_TILE_BYTES;
	uint8_t* devBody = g.ptr + g.headLen;
	uint8_t* hostBody = devBody + hostDelta;
	const uint8_t* src = IN ? hostBody : devBody;
	uint8_t* dst = IN ? devBody : hostBody;

	if( (tileStart + ELB_TILE_BYTES) <= g.bodyLen)
	{
		u64x4 v[ELB_UNROLL];

		#pragma unroll
		for(int u = 0; u < ELB_UNROLL; u++)
			v[u] = ld_nc_na_256(src + tileStart +
				(uint64_t)(u * ELB_THREADS + threadIdx.x) * ELB_VEC_BYTES);

		#pragma unroll
		for(int u = 0; u < ELB_UNROLL; u++)
			st_na_256(dst + tileStart +
				(uint64_t)(u * ELB_THREADS + threadIdx.x) * ELB_VEC_BYTES, v[u] );
	}
	else
	{
		#pragma unroll
		for(int u = 0; u < ELB_UNROLL; u++)
		{
			const uint64_t bodyOff = tileStart +
				(uint64_t)(u * ELB_THREADS + threadIdx.x) * ELB_VEC_BYTES;
			if(bodyOff < g.bodyLen)
				st_na_256(dst + bodyOff, ld_nc_na_256(src + bodyOff) );
		}
	}

	if(!tileIdx && (g.headLen | g.tailLen) )
	{
		const uint8_t* srcBlock = IN ? (g.ptr + hostDelta) : g.ptr;
		uint8_t* dstBlock = IN ? g.ptr : (g.ptr + hostDelta);

		if(threadIdx.x < g.headLen)
			dstBlock[threadIdx.x] = srcBlock[threadIdx.x];

		const uint64_t tailStart = g.headLen + g.bodyLen;
		if(threadIdx.x < g.tailLen)
			dstBlock[tailStart + threadIdx.x] = srcBlock[tailStart + threadIdx.x];
	}
}

/* ---- verify ----------------------------------------------------------------------------- */

/* compare one 32-byte vector; update thread-local count and first mismatch position (Count: 32
 * bits where the count covers one tile, 64 bits where it covers a whole block of any length) */
template<class Count>
__device__ __forceinline__ void verify_vec(const u64x4& got, const u64x4& exp, uint64_t pos,
	Count& numBad, uint64_t& firstBad)
{
	const uint64_t anyDiff = (got.a ^ exp.a) | (got.b ^ exp.b) | (got.c ^ exp.c) |
		(got.d ^ exp.d);

	if(__builtin_expect(anyDiff != 0, 0) )
	{
		numBad += diff_bytes64(got.a, exp.a) + diff_bytes64(got.b, exp.b) +
			diff_bytes64(got.c, exp.c) + diff_bytes64(got.d, exp.d);

		uint64_t first;
		if(got.a != exp.a)
			first = pos + first_diff_byte64(got.a, exp.a);
		else if(got.b != exp.b)
			first = pos + 8 + first_diff_byte64(got.b, exp.b);
		else if(got.c != exp.c)
			first = pos + 16 + first_diff_byte64(got.c, exp.c);
		else
			first = pos + 24 + first_diff_byte64(got.d, exp.d);

		if(first < firstBad)
			firstBad = first;
	}
}

template<bool FAST, bool STAGED, class Gen>
__device__ __forceinline__ void verify_tile(const BlockGeom& g, const Gen& gen,
	uint64_t tileIdx, elb_verify_result* result, unsigned long long* counters, int64_t hostDelta)
{
	const uint64_t tileStart = tileIdx * ELB_TILE_BYTES;
	uint8_t* devBody = g.ptr + g.headLen;
	const uint8_t* bodyPtr = STAGED ? (devBody + hostDelta) : devBody; // where the data is read

	unsigned numBad = 0;
	uint64_t firstBad = ~0ULL;

	if( (tileStart + ELB_TILE_BYTES) <= g.bodyLen)
	{ // full tile: issue all loads first, then compare
		u64x4 got[ELB_UNROLL];

		#pragma unroll
		for(int u = 0; u < ELB_UNROLL; u++)
		{
			const uint64_t bodyOff = tileStart +
				(uint64_t)(u * ELB_THREADS + threadIdx.x) * ELB_VEC_BYTES;
			got[u] = ld_nc_na_256(bodyPtr + bodyOff);
		}

		#pragma unroll
		for(int u = 0; u < ELB_UNROLL; u++)
		{
			const uint64_t bodyOff = tileStart +
				(uint64_t)(u * ELB_THREADS + threadIdx.x) * ELB_VEC_BYTES;
			const uint64_t pos = g.headLen + bodyOff;
			if(STAGED)
				st_na_256(devBody + bodyOff, got[u] );
			verify_vec(got[u], gen.template vec32<FAST>(pos), pos, numBad, firstBad);
		}
	}
	else
	{
		#pragma unroll
		for(int u = 0; u < ELB_UNROLL; u++)
		{
			const uint64_t bodyOff = tileStart +
				(uint64_t)(u * ELB_THREADS + threadIdx.x) * ELB_VEC_BYTES;
			if(bodyOff < g.bodyLen)
			{
				const uint64_t pos = g.headLen + bodyOff;
				const u64x4 got = ld_nc_na_256(bodyPtr + bodyOff);
				if(STAGED)
					st_na_256(devBody + bodyOff, got);
				verify_vec(got, gen.template vec32<FAST>(pos), pos, numBad, firstBad);
			}
		}
	}

	if(!tileIdx && (g.headLen | g.tailLen) )
	{
		const uint8_t* srcBlock = STAGED ? (g.ptr + hostDelta) : g.ptr;

		if(threadIdx.x < g.headLen)
		{
			const uint8_t got = srcBlock[threadIdx.x];
			if(STAGED)
				g.ptr[threadIdx.x] = got;
			if(got != gen.byte(threadIdx.x) )
			{
				numBad++;
				if(threadIdx.x < firstBad)
					firstBad = threadIdx.x;
			}
		}

		const uint64_t tailStart = g.headLen + g.bodyLen;
		if(threadIdx.x < g.tailLen)
		{
			const uint64_t pos = tailStart + threadIdx.x;
			const uint8_t got = srcBlock[pos];
			if(STAGED)
				g.ptr[pos] = got;
			if(got != gen.byte(pos) )
			{
				numBad++;
				if(pos < firstBad)
					firstBad = pos;
			}
		}
	}

	// warp-reduced mismatch count; global atomics only on the (rare) mismatch path
	const unsigned warpBad = __reduce_add_sync(0xffffffffu, numBad);

	if(__builtin_expect(warpBad != 0, 0) )
	{
		// 64-bit min via two 32-bit redux steps
		const unsigned firstHi = (unsigned)(firstBad >> 32);
		const unsigned minHi = __reduce_min_sync(0xffffffffu, firstHi);
		const unsigned firstLo = (firstHi == minHi) ? (unsigned)firstBad : 0xffffffffu;
		const unsigned minLo = __reduce_min_sync(0xffffffffu, firstLo);

		if( (threadIdx.x & 31) == 0)
		{
			atomicAdd( (unsigned long long*)&result->numMismatchBytes,
				(unsigned long long)warpBad);
			atomicMin( (unsigned long long*)&result->firstMismatchIdx,
				( (unsigned long long)minHi << 32) | minLo);
			if(counters)
				atomicAdd(&counters[ELB_DEVCTR_VERIFY_MISMATCH_BYTES],
					(unsigned long long)warpBad);
		}
	}
}

/* ---- kernels: walk all tiles of all descriptors, round-robin over the grid --------------- */

/* STAGE_NONE: work on the device slot only (kernel level ABI, resident windows). STAGE_PUBLISH:
 * device slot only, but the last CTA of a verify launch publishes the results to pinned host
 * memory (copy-engine staging). STAGE_FULL: the kernel also moves the block between the rings. */
enum { STAGE_NONE = 0, STAGE_PUBLISH = 1, STAGE_FULL = 2 };

enum { MODE_FILL_PATTERN = 0, MODE_VERIFY_PATTERN = 1, MODE_FILL_RANDOM = 2,
	MODE_COPY_IN = 3 /* host slot -> device slot */, MODE_COPY_OUT = 4 /* device -> host */,
	NUM_MODES = 5 };

struct KernelArgs
{
	const elb_block_desc* descs; // device-readable array, or NULL to use inlineDesc
	elb_block_desc inlineDesc;   // single-block launches pass the descriptor by value
	uint32_t numDescs;
	uint64_t salt;         // pattern
	uint64_t seed;         // random
	unsigned pct;          // random
	elb_verify_result* results; // verify
	unsigned long long* counters; // optional device counter block

	// staging (see the header comment); hostDelta == 0: work on the device slot only
	int64_t hostDelta;              // host slot address = device slot address + hostDelta
	elb_verify_result* hostResults; // verify: pinned copy of results, written by the last CTA
	unsigned* doneTicket;           // device counter behind the last-CTA detection (stays 0)
};

/* number of tiles of a block; same rule as make_geom() */
__device__ __forceinline__ uint64_t num_tiles_of(const elb_block_desc& desc)
{
	const uint64_t misalign = (uint64_t)(uintptr_t)desc.devPtr & (ELB_VEC_BYTES - 1);
	uint64_t headLen = misalign ? (ELB_VEC_BYTES - misalign) : 0;
	if(headLen > desc.len)
		headLen = desc.len;

	const uint64_t bodyLen = (desc.len - headLen) & ~(uint64_t)(ELB_VEC_BYTES - 1);
	const uint64_t numTiles = (bodyLen + ELB_TILE_BYTES - 1) / ELB_TILE_BYTES;

	return (!numTiles && desc.len) ? 1 : numTiles;
}

/* process tiles [tileBegin, tileEnd) of one block */
template<int MODE, bool STAGED>
__device__ __forceinline__ void process_block_tiles(const KernelArgs& args,
	const elb_block_desc& desc, uint32_t descIdx, const BlockGeom& g, uint64_t tileBegin,
	uint64_t tileEnd)
{
	const int64_t hostDelta = args.hostDelta;

	if(MODE == MODE_FILL_PATTERN)
	{
		PatternGen gen;
		gen.fileOffset = desc.fileOffset;
		gen.salt = args.salt;

		if(gen.canUseFast(g.headLen) )
			for(uint64_t tileIdx = tileBegin; tileIdx < tileEnd; tileIdx++)
				fill_tile<true, STAGED>(g, gen, tileIdx, hostDelta);
		else
			for(uint64_t tileIdx = tileBegin; tileIdx < tileEnd; tileIdx++)
				fill_tile<false, STAGED>(g, gen, tileIdx, hostDelta);
	}
	else if(MODE == MODE_VERIFY_PATTERN)
	{
		PatternGen gen;
		gen.fileOffset = desc.fileOffset;
		gen.salt = args.salt;

		if(gen.canUseFast(g.headLen) )
			for(uint64_t tileIdx = tileBegin; tileIdx < tileEnd; tileIdx++)
				verify_tile<true, STAGED>(g, gen, tileIdx, &args.results[descIdx], args.counters,
					hostDelta);
		else
			for(uint64_t tileIdx = tileBegin; tileIdx < tileEnd; tileIdx++)
				verify_tile<false, STAGED>(g, gen, tileIdx, &args.results[descIdx], args.counters,
					hostDelta);
	}
	else if(MODE == MODE_FILL_RANDOM)
	{
		RandomGen gen;
		gen.blockKey = elb_rand_block_key(args.seed, desc.blockCounter);
		gen.varFillLen = elb_rand_var_fill_len(desc.len, args.pct);
		gen.remainderVal = elb_rand_remainder_val(gen.blockKey);

		if(gen.canUseFast(g.headLen) )
			for(uint64_t tileIdx = tileBegin; tileIdx < tileEnd; tileIdx++)
				fill_tile<true, STAGED>(g, gen, tileIdx, hostDelta);
		else
			for(uint64_t tileIdx = tileBegin; tileIdx < tileEnd; tileIdx++)
				fill_tile<false, STAGED>(g, gen, tileIdx, hostDelta);
	}
	else
	{
		for(uint64_t tileIdx = tileBegin; tileIdx < tileEnd; tileIdx++)
			copy_tile<MODE == MODE_COPY_IN>(g, tileIdx, hostDelta);
	}
}

/* which device counter a mode accumulates block lengths into (-1: none) */
template<int MODE>
__device__ __forceinline__ int counter_slot_of()
{
	return (MODE == MODE_VERIFY_PATTERN) ? ELB_DEVCTR_VERIFIED_BYTES :
		( (MODE == MODE_FILL_PATTERN) || (MODE == MODE_FILL_RANDOM) ) ? ELB_DEVCTR_FILLED_BYTES : -1;
}

/**
 * End of a verify launch with host-visible results: every CTA (also those that found no work)
 * takes a ticket; the one that draws the last ticket sees all result atomics of the launch, copies
 * the per-block results to pinned host memory, re-arms the device entries that recorded a mismatch
 * and puts the ticket counter back to 0. The host reads hostResults after the launch's event.
 * Must be reached by all threads of the CTA.
 */
__device__ __forceinline__ void publish_results_if_last(const KernelArgs& args)
{
	__shared__ bool sIsLastCTA;

	if(!args.hostResults)
		return;

	__threadfence(); // order this CTA's result atomics before its ticket
	__syncthreads();

	if(!threadIdx.x)
		sIsLastCTA = (atomicAdd(args.doneTicket, 1u) == (gridDim.x - 1) );

	__syncthreads();

	if(!sIsLastCTA)
		return;

	__threadfence();

	for(uint32_t i = threadIdx.x; i < args.numDescs; i += blockDim.x)
	{
		volatile elb_verify_result* devResult = &args.results[i];
		elb_verify_result result;

		result.numMismatchBytes = devResult->numMismatchBytes;
		result.firstMismatchIdx = devResult->firstMismatchIdx;

		args.hostResults[i] = result;

		if(result.numMismatchBytes)
		{
			devResult->numMismatchBytes = 0;
			devResult->firstMismatchIdx = ~0ULL;
		}
	}

	if(!threadIdx.x)
		*args.doneTicket = 0;
}

/* block-wide sum; result valid in all threads. sScratch: one slot per warp. */
__device__ __forceinline__ uint64_t block_sum(uint64_t val, uint64_t* sScratch)
{
	for(int offset = 16; offset > 0; offset >>= 1)
		val += __shfl_xor_sync(0xffffffffu, val, offset);

	__syncthreads(); // protect sScratch from the previous use

	if( !(threadIdx.x & 31) )
		sScratch[threadIdx.x >> 5] = val;

	__syncthreads();

	uint64_t total = 0;

	#pragma unroll
	for(int warp = 0; warp < (ELB_THREADS / 32); warp++)
		total += sScratch[warp];

	return total;
}

/**
 * One launch over the whole window. All tiles of all blocks form one sequence; CTA b takes the
 * contiguous chunk [b*chunk, (b+1)*chunk) of it, so every CTA streams through consecutive
 * addresses and touches only the few descriptors its chunk overlaps. Finding the chunk start
 * needs the prefix sums of the per-block tile counts: the CTA computes them cooperatively
 * (coalesced descriptor loads + a block scan per 256 descriptors), which costs a few
 * microseconds per launch instead of a serial walk over all descriptors per CTA.
 */
template<int MODE, int STAGE>
__global__ void __launch_bounds__(ELB_THREADS, 4)
elb_blocks_kernel(const KernelArgs args)
{
	constexpr bool STAGED = (STAGE == STAGE_FULL);
	constexpr bool PUBLISH = (MODE == MODE_VERIFY_PATTERN) && (STAGE != STAGE_NONE);

	__shared__ uint64_t sScratch[ELB_THREADS / 32];
	__shared__ uint64_t sStartTile;
	__shared__ uint32_t sStartDesc;

	const uint32_t numDescs = args.numDescs;
	const elb_block_desc* descs = args.descs;

	// pass 1: total number of tiles
	uint64_t myTiles = 0;

	if(!descs)
		myTiles = threadIdx.x ? 0 : num_tiles_of(args.inlineDesc);
	else
		for(uint32_t descIdx = threadIdx.x; descIdx < numDescs; descIdx += ELB_THREADS)
			myTiles += num_tiles_of(descs[descIdx] );

	const uint64_t totalTiles = block_sum(myTiles, sScratch);
	const uint64_t chunkTiles = (totalTiles + gridDim.x - 1) / gridDim.x;
	const uint64_t chunkBegin = (uint64_t)blockIdx.x * chunkTiles;

	if(chunkBegin >= totalTiles)
	{ // (uniform for the whole CTA)
		if(PUBLISH)
			publish_results_if_last(args);
		return;
	}

	const uint64_t chunkEnd = (chunkBegin + chunkTiles < totalTiles) ?
		(chunkBegin + chunkTiles) : totalTiles;

	// pass 2: locate the block that contains tile chunkBegin
	uint32_t descIdx = 0;
	uint64_t tileIdx = chunkBegin;

	if(descs)
	{
		uint64_t segmentBase = 0; // tiles of all previous segments (uniform)

		for(uint32_t segment = 0; segment < numDescs; segment += ELB_THREADS)
		{
			const uint32_t myDesc = segment + threadIdx.x;
			const uint64_t tiles = (myDesc < numDescs) ? num_tiles_of(descs[myDesc] ) : 0;

			// inclusive scan inside the warp
			uint64_t inclusive = tiles;
			for(int offset = 1; offset < 32; offset <<= 1)
			{
				const uint64_t other = __shfl_up_sync(0xffffffffu, inclusive, offset);
				if( (threadIdx.x & 31) >= offset)
					inclusive += other;
			}

			__syncthreads();

			if( (threadIdx.x & 31) == 31)
				sScratch[threadIdx.x >> 5] = inclusive;

			__syncthreads();

			uint64_t warpBase = 0;
			uint64_t segmentTotal = 0;

			#pragma unroll
			for(int warp = 0; warp < (ELB_THREADS / 32); warp++)
			{
				if(warp < (int)(threadIdx.x >> 5) )
					warpBase += sScratch[warp];
				segmentTotal += sScratch[warp];
			}

			const uint64_t exclusive = segmentBase + warpBase + inclusive - tiles;

			if(tiles && (chunkBegin >= exclusive) && (chunkBegin < (exclusive + tiles) ) )
			{
				sStartDesc = myDesc;
				sStartTile = chunkBegin - exclusive;
			}

			segmentBase += segmentTotal;

			if(segmentBase > chunkBegin)
				break; // found (uniform)
		}

		__syncthreads();

		descIdx = sStartDesc;
		tileIdx = sStartTile;
	}

	// walk the chunk: consecutive tiles, block after block
	uint64_t tilesLeft = chunkEnd - chunkBegin;

	while(tilesLeft)
	{
		const elb_block_desc desc = descs ? descs[descIdx] : args.inlineDesc;
		const BlockGeom g = make_geom(desc);

		const uint64_t tileEnd = (g.numTiles - tileIdx < tilesLeft) ?
			g.numTiles : (tileIdx + tilesLeft);

		if(tileIdx < tileEnd)
		{
			process_block_tiles<MODE, STAGED>(args, desc, descIdx, g, tileIdx, tileEnd);

			// device-resident stats: one atomic per block, by the CTA that owns its first tile
			if( (counter_slot_of<MODE>() >= 0) && args.counters && !tileIdx && !threadIdx.x)
				atomicAdd(&args.counters[counter_slot_of<MODE>()], (unsigned long long)g.len);

			tilesLeft -= (tileEnd - tileIdx);
		}

		descIdx++;
		tileIdx = 0;
	}

	if(PUBLISH)
		publish_results_if_last(args);
}

/**
 * Hardware-scheduled form for windows whose blocks are (nearly) all the same size: a 1-D grid of
 * numDescs x ctasPerBlock short-lived CTAs, CTA i works on tile (i % ctasPerBlock) of block
 * (i / ctasPerBlock) and exits. No prefix scan, and - the point - the block scheduler hands out
 * tiles dynamically: SMs that get more bandwidth (smaller GPCs, nearer memory partitions) take
 * more tiles, and the set of addresses in flight is a compact window that moves through the
 * buffer. A static partition (the persistent kernel above) ends when the slowest SM is done;
 * measured write-only: 6.2 TB/s static vs 7.5 TB/s dynamic (profiles/, fill_variants2).
 * CTAs past the end of a shorter block exit immediately.
 */
template<int MODE, int STAGE>
__global__ void __launch_bounds__(ELB_THREADS, 4)
elb_blocks_tiled_kernel(const KernelArgs args, const uint32_t ctasPerBlock,
	const uint32_t tilesPerCTA)
{
	constexpr bool STAGED = (STAGE == STAGE_FULL);
	constexpr bool PUBLISH = (MODE == MODE_VERIFY_PATTERN) && (STAGE != STAGE_NONE);

	const uint32_t descIdx = blockIdx.x / ctasPerBlock;
	const uint32_t ctaInBlock = blockIdx.x - descIdx * ctasPerBlock;
	const uint64_t tileIdx = (uint64_t)ctaInBlock * tilesPerCTA;

	const elb_block_desc desc = args.descs ? args.descs[descIdx] : args.inlineDesc;
	const BlockGeom g = make_geom(desc);

	if(tileIdx >= g.numTiles)
	{ // (uniform for the whole CTA)
		if(PUBLISH)
			publish_results_if_last(args);
		return;
	}

	/* the launch shape comes from a size HINT: a block that is longer than the hint said has more
	   tiles than ctasPerBlock CTAs cover, so the last CTA of a block takes all that remain */
	const uint64_t tileEnd = ( (ctaInBlock + 1 == ctasPerBlock) ||
		(tileIdx + tilesPerCTA >= g.numTiles) ) ? g.numTiles : (tileIdx + tilesPerCTA);

	process_block_tiles<MODE, STAGED>(args, desc, descIdx, g, tileIdx, tileEnd);

	// device-resident stats: one atomic per block, by the CTA that owns its first tile
	if( (counter_slot_of<MODE>() >= 0) && args.counters && !tileIdx && !threadIdx.x)
		atomicAdd(&args.counters[counter_slot_of<MODE>()], (unsigned long long)g.len);

	if(PUBLISH)
		publish_results_if_last(args);
}

/* ---- small blocks: one warp per block ---------------------------------------------------------
 *
 * For 4 KiB .. 8 KiB blocks (BASELINE configs[2]: 4 KiB random reads) a CTA per block leaves half
 * of its threads without a vector and pays the descriptor fetch and the block setup once per
 * 4 KiB. Here a CTA takes ELB_WARPS blocks, warp w works on block (cta * ELB_WARPS + w): a lane
 * handles the 32-byte vectors lane, lane+32, ... of the block body (a warp access covers 1 KiB,
 * 4 independent accesses in flight per lane), the verify reduction is the warp's own redux, the
 * device counter gets one atomic per CTA. */

#define ELB_WARPS (ELB_THREADS / 32)
#define ELB_WARP_SPAN (32 * ELB_VEC_BYTES * ELB_UNROLL) /* 4 KiB per unrolled warp iteration */

template<int MODE, bool STAGED, bool FAST, class Gen>
__device__ __forceinline__ void process_block_warp(const KernelArgs& args, const BlockGeom& g,
	const Gen& gen, elb_verify_result* result)
{
	const unsigned lane = threadIdx.x & 31;
	const int64_t hostDelta = args.hostDelta;
	uint8_t* devBody = g.ptr + g.headLen;
	uint8_t* hostBody = devBody + hostDelta;

	/* 64 bits: the warp walks the whole block, and a block may be longer than the size hint that
	   picked this kernel, so the count of one warp is not bounded by 32 bits */
	unsigned long long numBad = 0;
	uint64_t firstBad = ~0ULL;

	for(uint64_t spanStart = 0; spanStart < g.bodyLen; spanStart += ELB_WARP_SPAN)
	{
		if( (MODE == MODE_VERIFY_PATTERN) || (MODE == MODE_COPY_IN) || (MODE == MODE_COPY_OUT) )
		{ // loads first, then the rest
			const uint8_t* src = (MODE == MODE_COPY_OUT) ? devBody :
				( ( (MODE == MODE_COPY_IN) || STAGED) ? hostBody : devBody);
			u64x4 got[ELB_UNROLL];
			bool valid[ELB_UNROLL];

			#pragma unroll
			for(int u = 0; u < ELB_UNROLL; u++)
			{
				const uint64_t bodyOff = spanStart + (uint64_t)(u * 32 + lane) * ELB_VEC_BYTES;
				valid[u] = (bodyOff < g.bodyLen);
				if(valid[u] )
					got[u] = ld_nc_na_256(src + bodyOff);
			}

			#pragma unroll
			for(int u = 0; u < ELB_UNROLL; u++)
			{
				const uint64_t bodyOff = spanStart + (uint64_t)(u * 32 + lane) * ELB_VEC_BYTES;
				if(!valid[u] )
					continue;

				if(MODE == MODE_COPY_OUT)
					st_na_256(hostBody + bodyOff, got[u] );
				else
				if( (MODE == MODE_COPY_IN) || STAGED)
					st_na_256(devBody + bodyOff, got[u] );

				if(MODE == MODE_VERIFY_PATTERN)
				{
					const uint64_t pos = g.headLen + bodyOff;
					verify_vec(got[u], gen.template vec32<FAST>(pos), pos, numBad, firstBad);
				}
			}
		}
		else
		{ // fill
			#pragma unroll
			for(int u = 0; u < ELB_UNROLL; u++)
			{
				const uint64_t bodyOff = spanStart + (uint64_t)(u * 32 + lane) * ELB_VEC_BYTES;
				if(bodyOff < g.bodyLen)
				{
					const u64x4 v = gen.template vec32<FAST>(g.headLen + bodyOff);
					st_na_256(devBody + bodyOff, v);
					if(STAGED)
						st_na_256(hostBody + bodyOff, v);
				}
			}
		}
	}

	if(g.headLen | g.tailLen)
	{ // unaligned head / tail bytes (at most 31 each): one lane per byte
		const uint64_t tailStart = g.headLen + g.bodyLen;

		for(int part = 0; part < 2; part++)
		{
			const uint64_t partLen = part ? g.tailLen : g.headLen;
			const uint64_t pos = (part ? tailStart : 0) + lane;

			if(lane >= partLen)
				continue;

			if( (MODE == MODE_FILL_PATTERN) || (MODE == MODE_FILL_RANDOM) )
			{
				const uint8_t b = gen.byte(pos);
				g.ptr[pos] = b;
				if(STAGED)
					g.ptr[hostDelta + (int64_t)pos] = b;
			}
			else
			if(MODE == MODE_COPY_OUT)
				g.ptr[hostDelta + (int64_t)pos] = g.ptr[pos];
			else
			{
				const bool fromHost = (MODE == MODE_COPY_IN) || STAGED;
				const uint8_t got = fromHost ? g.ptr[hostDelta + (int64_t)pos] : g.ptr[pos];

				if(fromHost)
					g.ptr[pos] = got;

				if( (MODE == MODE_VERIFY_PATTERN) && (got != gen.byte(pos) ) )
				{
					numBad++;
					if(pos < firstBad)
						firstBad = pos;
				}
			}
		}
	}

	if(MODE == MODE_VERIFY_PATTERN)
	{
		const unsigned anyBad = __reduce_or_sync(0xffffffffu, numBad ? 1u : 0u);

		if(__builtin_expect(anyBad != 0, 0) )
		{
			unsigned long long warpBad = numBad; // (redux adds 32 bits only)
			for(int laneMask = 16; laneMask; laneMask >>= 1)
				warpBad += __shfl_xor_sync(0xffffffffu, warpBad, laneMask);

			const unsigned firstHi = (unsigned)(firstBad >> 32);
			const unsigned minHi = __reduce_min_sync(0xffffffffu, firstHi);
			const unsigned firstLo = (firstHi == minHi) ? (unsigned)firstBad : 0xffffffffu;
			const unsigned minLo = __reduce_min_sync(0xffffffffu, firstLo);

			if(!lane)
			{ // (the only writer of this block's result: plain stores would do, atomics keep the
			  //  contract that several launches may accumulate into one result)
				atomicAdd( (unsigned long long*)&result->numMismatchBytes,
					(unsigned long long)warpBad);
				atomicMin( (unsigned long long*)&result->firstMismatchIdx,
					( (unsigned long long)minHi << 32) | minLo);
				if(args.counters)
					atomicAdd(&args.counters[ELB_DEVCTR_VERIFY_MISMATCH_BYTES],
						(unsigned long long)warpBad);
			}
		}
	}
}

template<int MODE, int STAGE>
__global__ void __launch_bounds__(ELB_THREADS, 3)
elb_blocks_warp_kernel(const KernelArgs args)
{
	constexpr bool STAGED = (STAGE == STAGE_FULL);
	constexpr bool PUBLISH = (MODE == MODE_VERIFY_PATTERN) && (STAGE != STAGE_NONE);

	__shared__ unsigned long long sBlockBytes;

	const uint32_t descIdx = blockIdx.x * ELB_WARPS + (threadIdx.x >> 5);

	if(!threadIdx.x)
		sBlockBytes = 0;

	__syncthreads();

	if(descIdx < args.numDescs)
	{ // (uniform per warp)
		const elb_block_desc desc = args.descs ? args.descs[descIdx] : args.inlineDesc;
		const BlockGeom g = make_geom(desc);

		if(g.len)
		{
			if( (MODE == MODE_FILL_PATTERN) || (MODE == MODE_VERIFY_PATTERN) )
			{
				PatternGen gen;
				gen.fileOffset = desc.fileOffset;
				gen.salt = args.salt;

				if(gen.canUseFast(g.headLen) )
					process_block_warp<MODE, STAGED, true>(args, g, gen, &args.results[descIdx] );
				else
					process_block_warp<MODE, STAGED, false>(args, g, gen, &args.results[descIdx] );
			}
			else
			if(MODE == MODE_FILL_RANDOM)
			{
				RandomGen gen;
				gen.blockKey = elb_rand_block_key(args.seed, desc.blockCounter);
				gen.varFillLen = elb_rand_var_fill_len(desc.len, args.pct);
				gen.remainderVal = elb_rand_remainder_val(gen.blockKey);

				if(gen.canUseFast(g.headLen) )
					process_block_warp<MODE, STAGED, true>(args, g, gen, NULL);
				else
					process_block_warp<MODE, STAGED, false>(args, g, gen, NULL);
			}
			else
			{
				PatternGen unused{};
				process_block_warp<MODE, true, true>(args, g, unused, NULL);
			}

			if( (counter_slot_of<MODE>() >= 0) && args.counters && !(threadIdx.x & 31) )
				atomicAdd(&sBlockBytes, (unsigned long long)g.len);
		}
	}

	if( (counter_slot_of<MODE>() >= 0) && args.counters)
	{ // device-resident stats: one global atomic per CTA
		__syncthreads();

		if(!threadIdx.x && sBlockBytes)
			atomicAdd(&args.counters[counter_slot_of<MODE>()], sBlockBytes);
	}

	if(PUBLISH)
		publish_results_if_last(args);
}

__global__ void elb_verify_init_kernel(elb_verify_result* results, uint32_t numDescs)
{
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;

	if(i < numDescs)
	{
		results[i].numMismatchBytes = 0;
		results[i].firstMismatchIdx = ~0ULL;
	}
}

/* ---- host side launchers ------------------------------------------------------------------ */

static std::atomic<uint64_t> gNumKernelLaunches{0};

thread_local std::string elbThreadLastError;

void elb_set_last_error(const std::string& msg)
{
	elbThreadLastError = msg;
}

struct DeviceLaunchInfo
{
	int numSMs{0};
	int ctasPerSM[NUM_MODES]{0, 0, 0, 0, 0};
	/* 32 KiB tiles per CTA of the hardware-scheduled kernel; 0 = always use the persistent
	   kernel for this mode. Tuning knob: ELB_TILES_PER_CTA="fill,verify,random". */
	uint32_t tilesPerCTA[NUM_MODES]{1, 2, 8, 2, 2}; // measured best on B200 (profiles/: sweep_tiles)
};

static DeviceLaunchInfo gDevInfo[ELB_MAX_DEVICES];
static std::once_flag gDevInfoOnce[ELB_MAX_DEVICES];

template<int MODE>
static int queryOccupancy()
{
	int numBlocks = 0;
	cudaOccupancyMaxActiveBlocksPerMultiprocessor(&numBlocks,
		elb_blocks_kernel<MODE, ( (MODE == MODE_COPY_IN) || (MODE == MODE_COPY_OUT) ) ? STAGE_FULL : STAGE_NONE>,
		ELB_THREADS, 0);
	return (numBlocks > 0) ? numBlocks : 1;
}

static const DeviceLaunchInfo* getDeviceLaunchInfo()
{
	int dev = 0;
	cudaError_t devRes = cudaGetDevice(&dev);

	if( (devRes != cudaSuccess) || (dev < 0) || (dev >= ELB_MAX_DEVICES) )
	{
		elb_set_last_error(std::string("cudaGetDevice failed: ") + cudaGetErrorString(devRes) );
		return NULL;
	}

	std::call_once(gDevInfoOnce[dev], [dev]()
	{
		cudaDeviceGetAttribute(&gDevInfo[dev].numSMs, cudaDevAttrMultiProcessorCount, dev);
		gDevInfo[dev].ctasPerSM[MODE_FILL_PATTERN] = queryOccupancy<MODE_FILL_PATTERN>();
		gDevInfo[dev].ctasPerSM[MODE_VERIFY_PATTERN] = queryOccupancy<MODE_VERIFY_PATTERN>();
		gDevInfo[dev].ctasPerSM[MODE_FILL_RANDOM] = queryOccupancy<MODE_FILL_RANDOM>();
		gDevInfo[dev].ctasPerSM[MODE_COPY_IN] = queryOccupancy<MODE_COPY_IN>();
		gDevInfo[dev].ctasPerSM[MODE_COPY_OUT] = queryOccupancy<MODE_COPY_OUT>();

		const char* tilesEnv = getenv("ELB_TILES_PER_CTA");
		if(tilesEnv)
		{
			unsigned vals[3];
			if(sscanf(tilesEnv, "%u,%u,%u", &vals[0], &vals[1], &vals[2]) == 3)
				for(int mode = 0; mode < 3; mode++)
					gDevInfo[dev].tilesPerCTA[mode] = vals[mode];
		}
	});

	if(gDevInfo[dev].numSMs <= 0)
	{
		elb_set_last_error("Unable to query CUDA device attributes (no usable GPU?)");
		return NULL;
	}

	return &gDevInfo[dev];
}

#define ELB_WARP_KERNEL_MAX_BLOCK (8 * 1024)

/* tuning / profiling knob: ELB_NO_WARP_KERNEL=1 sends small blocks through the tile kernels */
static bool smallBlockKernelEnabled()
{
	static const bool enabled = []()
	{
		const char* env = getenv("ELB_NO_WARP_KERNEL");
		return !(env && env[0] && (env[0] != '0') );
	}();

	return enabled;
}

static const char* modeName(int mode)
{
	static const char* names[NUM_MODES] =
		{"fill_pattern", "verify_pattern", "fill_random", "stage_copy_in", "stage_copy_out"};
	return names[mode];
}

static int checkLaunch(const char* what)
{
	cudaError_t res = cudaGetLastError();

	if(res != cudaSuccess)
	{
		elb_set_last_error(std::string(what) + " kernel launch failed: " +
			cudaGetErrorString(res) );
		return -1;
	}

	return 0;
}

/**
 * @totalBytesHint upper bound of bytes covered by the launch (used only to size the grid);
 *    0 = unknown (launch a full persistent grid).
 * @maxBlockLenHint upper bound of the length of any block of the launch; 0 = unknown. With both
 *    hints and blocks of (nearly) uniform size the hardware-scheduled tiled kernel is used,
 *    otherwise (ragged windows: many CTAs would find nothing to do) the persistent one.
 */
template<int MODE, int STAGE>
static int launchBlocksKernelT(const KernelArgs& args, uint64_t totalBytesHint,
	uint64_t maxBlockLenHint, cudaStream_t stream)
{
	if(!args.numDescs)
		return 0;

	const DeviceLaunchInfo* devInfo = getDeviceLaunchInfo();
	if(!devInfo)
		return -1;

	/* staged launches run at PCIe speed: one tile per CTA keeps the most loads in flight */
	const uint32_t tilesPerCTA = (STAGE == STAGE_FULL) ? 1 : devInfo->tilesPerCTA[MODE];

	/* small blocks: one warp per block (a longer block than the hint said is still processed
	   completely, the warp loops over its whole body) */
	if(maxBlockLenHint && (maxBlockLenHint <= ELB_WARP_KERNEL_MAX_BLOCK) && args.descs &&
		smallBlockKernelEnabled() )
	{
		const uint64_t numCTAs = ( (uint64_t)args.numDescs + ELB_WARPS - 1) / ELB_WARPS;

		elb_blocks_warp_kernel<MODE, STAGE><<<(unsigned)numCTAs, ELB_THREADS, 0, stream>>>(args);
		gNumKernelLaunches.fetch_add(1, std::memory_order_relaxed);

		return checkLaunch(modeName(MODE) );
	}

	if(maxBlockLenHint && totalBytesHint && tilesPerCTA)
	{
		const uint64_t ctaBytes = (uint64_t)ELB_TILE_BYTES * tilesPerCTA;
		const uint64_t ctasPerBlock = (maxBlockLenHint + ctaBytes - 1) / ctaBytes;
		const uint64_t numCTAs = ctasPerBlock * args.numDescs;
		const uint64_t neededCTAs = (totalBytesHint + ctaBytes - 1) / ctaBytes + args.numDescs;

		if( (numCTAs <= 0x7fffffffULL) && (numCTAs <= (2 * neededCTAs + 1024) ) )
		{
			elb_blocks_tiled_kernel<MODE, STAGE><<<(unsigned)numCTAs, ELB_THREADS, 0, stream>>>(
				args, (uint32_t)ctasPerBlock, tilesPerCTA);
			gNumKernelLaunches.fetch_add(1, std::memory_order_relaxed);

			return checkLaunch(modeName(MODE) );
		}
	}

	// grid: a multiple of the SM count, never more CTAs than tiles
	uint64_t gridSize = (uint64_t)devInfo->numSMs * devInfo->ctasPerSM[MODE];

	if(totalBytesHint)
	{
		const uint64_t maxTiles =
			(totalBytesHint + ELB_TILE_BYTES - 1) / ELB_TILE_BYTES + args.numDescs;
		if(maxTiles < gridSize)
			gridSize = maxTiles;
	}

	elb_blocks_kernel<MODE, STAGE><<<(unsigned)gridSize, ELB_THREADS, 0, stream>>>(args);
	gNumKernelLaunches.fetch_add(1, std::memory_order_relaxed);

	return checkLaunch(modeName(MODE) );
}

template<int MODE>
static int launchBlocksKernel(const KernelArgs& args, uint64_t totalBytesHint,
	uint64_t maxBlockLenHint, cudaStream_t stream)
{
	if(args.hostDelta || (MODE == MODE_COPY_IN) || (MODE == MODE_COPY_OUT) )
		return launchBlocksKernelT<MODE, STAGE_FULL>(args, totalBytesHint, maxBlockLenHint, stream);

	if constexpr( (MODE == MODE_COPY_IN) || (MODE == MODE_COPY_OUT) )
		return -1; // (not reached: the copy kernels exist in their staged form only)
	else
	{
		if constexpr(MODE == MODE_VERIFY_PATTERN)
			if(args.hostResults)
				return launchBlocksKernelT<MODE, STAGE_PUBLISH>(args, totalBytesHint,
					maxBlockLenHint, stream);

		return launchBlocksKernelT<MODE, STAGE_NONE>(args, totalBytesHint, maxBlockLenHint,
			stream);
	}
}

static void applyStage(KernelArgs& args, const elb_stage_args* stage)
{
	if(!stage)
		return;

	args.hostDelta = stage->hostDelta;
	args.hostResults = stage->hostResults;
	args.doneTicket = stage->doneTicket;
}

int elb_launch_fill_pattern(const elb_block_desc* descs, const elb_block_desc* inlineDesc,
	uint32_t numDescs, uint64_t salt, uint64_t* devCounters, uint64_t totalBytesHint,
	uint64_t maxBlockLenHint, cudaStream_t stream, const elb_stage_args* stage)
{
	KernelArgs args{};
	args.descs = descs;
	if(inlineDesc)
		args.inlineDesc = *inlineDesc;
	args.numDescs = numDescs;
	args.salt = salt;
	args.counters = (unsigned long long*)devCounters;
	applyStage(args, stage);

	return launchBlocksKernel<MODE_FILL_PATTERN>(args, totalBytesHint, maxBlockLenHint, stream);
}

int elb_launch_verify_init(elb_verify_result* devResults, uint32_t numDescs,
	cudaStream_t stream)
{
	if(!numDescs)
		return 0;

	elb_verify_init_kernel<<<(numDescs + 255) / 256, 256, 0, stream>>>(devResults, numDescs);
	gNumKernelLaunches.fetch_add(1, std::memory_order_relaxed);

	return checkLaunch("verify_init");
}

/**
 * @initResults false if the caller knows devResults still holds {0, ~0} entries (true after any
 *    launch that found no mismatch, and always after a launch with stage->hostResults, which
 *    re-arms the entries itself), which saves the init launch.
 */
int elb_launch_verify_pattern(const elb_block_desc* descs, const elb_block_desc* inlineDesc,
	uint32_t numDescs, uint64_t salt, elb_verify_result* devResults, uint64_t* devCounters,
	uint64_t totalBytesHint, uint64_t maxBlockLenHint, bool initResults, cudaStream_t stream,
	const elb_stage_args* stage)
{
	if(!numDescs)
		return 0;

	if(stage && stage->hostResults && !stage->doneTicket)
	{
		elb_set_last_error("verify_pattern: host results need a device ticket counter");
		return -1;
	}

	if(initResults && elb_launch_verify_init(devResults, numDescs, stream) )
		return -1;

	KernelArgs args{};
	args.descs = descs;
	if(inlineDesc)
		args.inlineDesc = *inlineDesc;
	args.numDescs = numDescs;
	args.salt = salt;
	args.results = devResults;
	args.counters = (unsigned long long*)devCounters;
	applyStage(args, stage);

	return launchBlocksKernel<MODE_VERIFY_PATTERN>(args, totalBytesHint, maxBlockLenHint, stream);
}

int elb_launch_fill_random(const elb_block_desc* descs, const elb_block_desc* inlineDesc,
	uint32_t numDescs, unsigned pct, uint64_t seed, uint64_t* devCounters,
	uint64_t totalBytesHint, uint64_t maxBlockLenHint, cudaStream_t stream,
	const elb_stage_args* stage)
{
	KernelArgs args{};
	args.descs = descs;
	if(inlineDesc)
		args.inlineDesc = *inlineDesc;
	args.numDescs = numDescs;
	args.seed = seed;
	args.pct = pct;
	args.counters = (unsigned long long*)devCounters;
	applyStage(args, stage);

	return launchBlocksKernel<MODE_FILL_RANDOM>(args, totalBytesHint, maxBlockLenHint, stream);
}

/* plain copy of the blocks between the rings (runs without --verify / without fill) */
int elb_launch_stage_copy(const elb_block_desc* descs, uint32_t numDescs, bool hostToDevice,
	int64_t hostDelta, uint64_t totalBytesHint, uint64_t maxBlockLenHint, cudaStream_t stream)
{
	KernelArgs args{};
	args.descs = descs;
	args.numDescs = numDescs;
	args.hostDelta = hostDelta;

	if(!descs || !hostDelta)
	{
		elb_set_last_error("stage_copy: descriptor array and host delta are required");
		return -1;
	}

	return hostToDevice ?
		launchBlocksKernel<MODE_COPY_IN>(args, totalBytesHint, maxBlockLenHint, stream) :
		launchBlocksKernel<MODE_COPY_OUT>(args, totalBytesHint, maxBlockLenHint, stream);
}

/* query launch geometry of the current device now (so that no attribute/occupancy query happens
 * later inside a stream capture) */
int elb_kernels_warmup()
{
	return getDeviceLaunchInfo() ? 0 : -1;
}

uint64_t elb_get_num_kernel_launches()
{
	return gNumKernelLaunches.load(std::memory_order_relaxed);
}
