/*
 * C ABI of the kernel level (include/elbencho_b200.h): thin argument checks around the launchers
 * in elb_kernels.cu. These are the entry points a reference-side BLOCK_MODIFIER shim would bind
 * in place of LocalWorker::preWriteIntegrityCheckFillBuf / postReadIntegrityCheckVerifyBuf /
 * preWriteBufRandRefillCuda (source/workers/LocalWorker.cpp:2091-2277).
 */
#include <cuda_runtime.h>

#include <string>

#include "elb_internal.h"

extern thread_local std::string elbThreadLastError;

static int checkRandArgs(unsigned pct, int randAlgo)
{
	if(pct > 100)
	{
		elb_set_last_error("Block variance percent must be in range 0..100. Given: " +
			std::to_string(pct) );
		return -1;
	}

	if(randAlgo != ELB_RANDALGO_SPLITMIX64)
	{
		elb_set_last_error("Unknown random fill algorithm: " + std::to_string(randAlgo) );
		return -1;
	}

	return 0;
}

/* the staged kernels move 32-byte vectors between (devPtr) and (devPtr + hostDelta): both ends of
   a vector are aligned only if hostDelta is */
static int checkHostDelta(const char* what, int64_t hostDelta)
{
	if(hostDelta % ELB_STAGE_ALIGN)
	{
		elb_set_last_error(std::string(what) + ": hostDelta must be a multiple of " +
			std::to_string(ELB_STAGE_ALIGN) + " bytes (alignment of the staged vector copies). "
			"Given: " + std::to_string(hostDelta) );
		return -1;
	}

	return 0;
}

extern "C" {

int elb_abi_version(void)
{
	return ELB_ABI_VERSION;
}

const char* elb_last_error(void)
{
	return elbThreadLastError.c_str();
}

uint64_t elb_num_kernel_launches(void)
{
	return elb_get_num_kernel_launches();
}

int elb_fill_pattern(void* devPtr, uint64_t len, uint64_t fileOffset, uint64_t salt,
	void* stream)
{
	if(!len)
		return 0;

	if(!devPtr)
	{
		elb_set_last_error("elb_fill_pattern: NULL device pointer");
		return -1;
	}

	elb_block_desc desc{devPtr, len, fileOffset, 0};

	return elb_launch_fill_pattern(NULL, &desc, 1, salt, NULL, len, len, (cudaStream_t)stream);
}

int elb_verify_pattern(const void* devPtr, uint64_t len, uint64_t fileOffset, uint64_t salt,
	elb_verify_result* devOut, void* stream)
{
	if(!devOut)
	{
		elb_set_last_error("elb_verify_pattern: NULL result pointer");
		return -1;
	}

	if(!len) // reference returns early on empty buffers (LocalWorker.cpp:2140-2141)
		return elb_launch_verify_init(devOut, 1, (cudaStream_t)stream);

	if(!devPtr)
	{
		elb_set_last_error("elb_verify_pattern: NULL device pointer");
		return -1;
	}

	elb_block_desc desc{const_cast<void*>(devPtr), len, fileOffset, 0};

	return elb_launch_verify_pattern(NULL, &desc, 1, salt, devOut, NULL, len, len,
		true /*initResults*/, (cudaStream_t)stream);
}

int elb_fill_random(void* devPtr, uint64_t len, unsigned pct, uint64_t seed,
	uint64_t blockCounter, int randAlgo, void* stream)
{
	if(checkRandArgs(pct, randAlgo) )
		return -1;

	if(!len)
		return 0;

	if(!devPtr)
	{
		elb_set_last_error("elb_fill_random: NULL device pointer");
		return -1;
	}

	elb_block_desc desc{devPtr, len, 0, blockCounter};

	return elb_launch_fill_random(NULL, &desc, 1, pct, seed, NULL, len, len,
		(cudaStream_t)stream);
}

int elb_fill_pattern_batch_sized(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	uint64_t* devCounters, uint64_t totalBytes, uint64_t maxBlockLen, void* stream)
{
	if(numDescs && !descs)
	{
		elb_set_last_error("elb_fill_pattern_batch: NULL descriptor array");
		return -1;
	}

	return elb_launch_fill_pattern(descs, NULL, numDescs, salt, devCounters, totalBytes,
		maxBlockLen, (cudaStream_t)stream);
}

int elb_verify_pattern_batch_sized(const elb_block_desc* descs, uint32_t numDescs,
	uint64_t salt, elb_verify_result* devResults, uint64_t* devCounters, uint64_t totalBytes,
	uint64_t maxBlockLen, void* stream)
{
	if(numDescs && (!descs || !devResults) )
	{
		elb_set_last_error("elb_verify_pattern_batch: NULL descriptor or result array");
		return -1;
	}

	return elb_launch_verify_pattern(descs, NULL, numDescs, salt, devResults, devCounters,
		totalBytes, maxBlockLen, true /*initResults*/, (cudaStream_t)stream);
}

int elb_fill_random_batch_sized(const elb_block_desc* descs, uint32_t numDescs, unsigned pct,
	uint64_t seed, int randAlgo, uint64_t* devCounters, uint64_t totalBytes, uint64_t maxBlockLen,
	void* stream)
{
	if(checkRandArgs(pct, randAlgo) )
		return -1;

	if(numDescs && !descs)
	{
		elb_set_last_error("elb_fill_random_batch: NULL descriptor array");
		return -1;
	}

	return elb_launch_fill_random(descs, NULL, numDescs, pct, seed, devCounters, totalBytes,
		maxBlockLen, (cudaStream_t)stream);
}

int elb_fill_pattern_staged(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	int64_t hostDelta, uint64_t* devCounters, uint64_t totalBytes, uint64_t maxBlockLen,
	void* stream)
{
	if(checkHostDelta("elb_fill_pattern_staged", hostDelta) )
		return -1;

	if(numDescs && !descs)
	{
		elb_set_last_error("elb_fill_pattern_staged: NULL descriptor array");
		return -1;
	}

	elb_stage_args stage;
	stage.hostDelta = hostDelta;

	return elb_launch_fill_pattern(descs, NULL, numDescs, salt, devCounters, totalBytes,
		maxBlockLen, (cudaStream_t)stream, &stage);
}

int elb_fill_random_staged(const elb_block_desc* descs, uint32_t numDescs, unsigned pct,
	uint64_t seed, int randAlgo, int64_t hostDelta, uint64_t* devCounters, uint64_t totalBytes,
	uint64_t maxBlockLen, void* stream)
{
	if(checkHostDelta("elb_fill_random_staged", hostDelta) )
		return -1;

	if(checkRandArgs(pct, randAlgo) )
		return -1;

	if(numDescs && !descs)
	{
		elb_set_last_error("elb_fill_random_staged: NULL descriptor array");
		return -1;
	}

	elb_stage_args stage;
	stage.hostDelta = hostDelta;

	return elb_launch_fill_random(descs, NULL, numDescs, pct, seed, devCounters, totalBytes,
		maxBlockLen, (cudaStream_t)stream, &stage);
}

int elb_verify_pattern_staged(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	int64_t hostDelta, elb_verify_result* devResults, elb_verify_result* hostResults,
	unsigned* devDoneTicket, uint64_t* devCounters, uint64_t totalBytes, uint64_t maxBlockLen,
	void* stream)
{
	if(checkHostDelta("elb_verify_pattern_staged", hostDelta) )
		return -1;

	if(numDescs && (!descs || !devResults) )
	{
		elb_set_last_error("elb_verify_pattern_staged: NULL descriptor or result array");
		return -1;
	}

	elb_stage_args stage;
	stage.hostDelta = hostDelta;
	stage.hostResults = hostResults;
	stage.doneTicket = devDoneTicket;

	return elb_launch_verify_pattern(descs, NULL, numDescs, salt, devResults, devCounters,
		totalBytes, maxBlockLen, false /*initResults*/, (cudaStream_t)stream, &stage);
}

int elb_stage_copy(const elb_block_desc* descs, uint32_t numDescs, int hostToDevice,
	int64_t hostDelta, uint64_t totalBytes, uint64_t maxBlockLen, void* stream)
{
	if(checkHostDelta("elb_stage_copy", hostDelta) )
		return -1;

	if(!numDescs)
		return 0;

	return elb_launch_stage_copy(descs, numDescs, hostToDevice != 0, hostDelta, totalBytes,
		maxBlockLen, (cudaStream_t)stream);
}

int elb_verify_results_init(elb_verify_result* devResults, uint32_t numDescs, void* stream)
{
	if(numDescs && !devResults)
	{
		elb_set_last_error("elb_verify_results_init: NULL result array");
		return -1;
	}

	return elb_launch_verify_init(devResults, numDescs, (cudaStream_t)stream);
}

int elb_fill_pattern_batch(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	uint64_t* devCounters, void* stream)
{
	return elb_fill_pattern_batch_sized(descs, numDescs, salt, devCounters, 0, 0, stream);
}

int elb_verify_pattern_batch(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	elb_verify_result* devResults, uint64_t* devCounters, void* stream)
{
	return elb_verify_pattern_batch_sized(descs, numDescs, salt, devResults, devCounters, 0, 0,
		stream);
}

int elb_fill_random_batch(const elb_block_desc* descs, uint32_t numDescs, unsigned pct,
	uint64_t seed, int randAlgo, uint64_t* devCounters, void* stream)
{
	return elb_fill_random_batch_sized(descs, numDescs, pct, seed, randAlgo, devCounters, 0, 0,
		stream);
}

} // extern "C"
