/*
 * elbencho_b200 — C ABI of the Blackwell-native GPU I/O benchmark worker.
 *
 * This is the drop-in boundary for elbencho's LocalWorker hot path. The reference has no
 * plugin/FFI mechanism (WorkerManager.cpp:163 hard-codes `new LocalWorker(...)`), so the entry
 * points below mirror, one-to-one, what a thin C++ `Worker` subclass would bind:
 *
 *   kernel level  -> the BLOCK_MODIFIER slots of LocalWorker (source/workers/LocalWorker.h:44-74)
 *   worker level  -> the abstract Worker interface (source/workers/Worker.h:20-226)
 *   manager level -> WorkerManager (source/workers/WorkerManager.cpp:142-324)
 *
 * Every signature uses plain pointers and sizes only. `stream` arguments are `cudaStream_t`
 * passed as `void*` (NULL = the legacy default stream). Device pointers are ordinary CUDA device
 * addresses; no torch types cross this boundary.
 *
 * All entry points return 0 on success and a negative value on error unless stated otherwise;
 * the error text is available through elb_last_error() (thread-local) or
 * elb_worker_last_error()/elb_mgr_last_error() (WorkerException text of the reference, e.g. the
 * byte-identical "Data verification failed. Offset: ..." message of LocalWorker.cpp:2174-2177).
 */
#ifndef ELBENCHO_B200_H_
#define ELBENCHO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ELB_ABI_VERSION 1

/* ---------------------------------------------------------------------------------------------
 * Enums (values follow source/Common.h:142-179 so a shim can cast directly)
 * ------------------------------------------------------------------------------------------- */

enum elb_bench_phase
{
	ELB_PHASE_IDLE = 0,
	ELB_PHASE_TERMINATE = 1,
	ELB_PHASE_CREATEDIRS = 2,
	ELB_PHASE_DELETEDIRS = 3,
	ELB_PHASE_CREATEFILES = 4,
	ELB_PHASE_DELETEFILES = 5,
	ELB_PHASE_READFILES = 6,
	ELB_PHASE_SYNC = 7,
	ELB_PHASE_DROPCACHES = 8,
	ELB_PHASE_STATFILES = 9,
};

enum elb_path_type
{
	ELB_PATH_DIR = 0,
	ELB_PATH_FILE = 1,
	ELB_PATH_BLOCKDEV = 2,
};

/* I/O engines of the per-block loop. SYNC = rwBlockSized semantics (LocalWorker.cpp:1669-1781),
 * AIO = aioBlockSized semantics (:1795-2037) on raw kernel AIO (no libaio dependency). */
enum elb_io_engine
{
	ELB_IOENGINE_AUTO = 0, /* SYNC when iodepth==1, else AIO (LocalWorker.cpp:1243-1244) */
	ELB_IOENGINE_SYNC = 1,
	ELB_IOENGINE_AIO = 2,
};

/* Random-fill generators for --blockvarpct (counter-based, position-keyed; see DESIGN.md) */
enum elb_rand_algo
{
	ELB_RANDALGO_SPLITMIX64 = 0, /* splitmix64 of (seed, block counter, word index); uniform u64 */
};

/* Generators of random offsets for --rand (--randalgo; toolkits/random/RandAlgoSelectorTk.h:10-25).
 * All four streams are bit-identical to the reference's classes for the same injected state. */
enum elb_offset_rand_algo
{
	ELB_OFFSETALGO_XOSHIRO256SS = 0, /* "balanced_single", the default (LocalWorker.cpp:1135-1136) */
	ELB_OFFSETALGO_GOLDENPRIME = 1,  /* "fast" */
	ELB_OFFSETALGO_XOSHIRO256PP = 2, /* "balanced": lane 0 of the reference's 4-way SIMD class */
	ELB_OFFSETALGO_MT19937 = 3,      /* "strong": std::mt19937_64 */
};

/* Histogram kinds for elb_worker_histogram (Worker.h:55-58) */
enum elb_histo_kind
{
	ELB_HISTO_IOPS = 0,
	ELB_HISTO_IOPS_READMIX = 1,
	ELB_HISTO_ENTRIES = 2,
	ELB_HISTO_ENTRIES_READMIX = 3,
};

#define ELB_LATHISTO_NUMBUCKETS 112 /* LatencyHistogram.h:14-18 */

/* ---------------------------------------------------------------------------------------------
 * Kernel level: on-GPU block modifiers / checkers (replace LocalWorker.cpp:2091-2277)
 * ------------------------------------------------------------------------------------------- */

/* Result of an on-GPU integrity check. One per block descriptor.
 * numMismatchBytes: number of bytes differing from the expected pattern (0 = block is good).
 * firstMismatchIdx: index within the block of the first differing byte, ~0ULL if none.
 * (expected/actual byte values follow from the closed form / one 1-byte read; the worker layer
 * produces the reference's exception text from them.) */
typedef struct elb_verify_result
{
	uint64_t numMismatchBytes;
	uint64_t firstMismatchIdx;
} elb_verify_result;

/* One block of the in-flight window: device address, length, file offset, and the block counter
 * that keys the random fill (ignored by pattern fill/verify). */
typedef struct elb_block_desc
{
	void* devPtr;
	uint64_t len;
	uint64_t fileOffset;
	uint64_t blockCounter;
} elb_block_desc;

/* Device-resident counter block of a worker (what the stats reduce sums across GPUs). */
enum elb_dev_counter
{
	ELB_DEVCTR_VERIFY_MISMATCH_BYTES = 0,
	ELB_DEVCTR_VERIFIED_BYTES = 1,
	ELB_DEVCTR_FILLED_BYTES = 2,
	ELB_DEVCTR_NUM = 8,
};

/* K1: buffer byte i <- byte ((fileOffset+i) % 8) of little-endian u64 (((fileOffset+i) & ~7) +
 * salt). Replaces preWriteIntegrityCheckFillBuf (LocalWorker.cpp:2091-2128). Any alignment/len. */
int elb_fill_pattern(void* devPtr, uint64_t len, uint64_t fileOffset, uint64_t salt,
	void* stream);

/* K2: compare device buffer with the pattern; *devOut (device memory, 16 bytes) receives the
 * result. Replaces postReadIntegrityCheckVerifyBuf (LocalWorker.cpp:2137-2179). */
int elb_verify_pattern(const void* devPtr, uint64_t len, uint64_t fileOffset, uint64_t salt,
	elb_verify_result* devOut, void* stream);

/* K3: first varFillLen = (len*pct)/100 bytes (rounded down to a multiple of 4 like the
 * reference's GPU path, LocalWorker.cpp:2253-2256) random, remainder = one repeated u64.
 * Replaces preWriteBufRandRefillCuda (:2236-2277: curandGenerate + host bufFill + H2D copy). */
int elb_fill_random(void* devPtr, uint64_t len, unsigned pct, uint64_t seed,
	uint64_t blockCounter, int randAlgo, void* stream);

/* Batched forms: one launch over the whole in-flight window. `descs` must be readable by the
 * device (device memory or pinned mapped host memory); `numDescs` blocks. `devResults` has one
 * entry per descriptor. `devCounters` (may be NULL) points to ELB_DEVCTR_NUM u64 in device memory
 * that the kernels accumulate into (device-resident stats block). */
int elb_fill_pattern_batch(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	uint64_t* devCounters, void* stream);
int elb_verify_pattern_batch(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	elb_verify_result* devResults, uint64_t* devCounters, void* stream);
int elb_fill_random_batch(const elb_block_desc* descs, uint32_t numDescs, unsigned pct,
	uint64_t seed, int randAlgo, uint64_t* devCounters, void* stream);
/* As above, plus two size hints (0 = unknown) that only pick the launch shape: totalBytes = sum
 * of the descriptor lengths, maxBlockLen = upper bound of any descriptor's length (the block
 * size). With both, windows of (nearly) equally sized blocks run as a grid of short-lived CTAs,
 * one 32 KiB tile each, handed out dynamically by the hardware block scheduler; ragged or
 * unknown windows run on a persistent grid that partitions all tiles statically. The hints are
 * never load-bearing: a descriptor longer than maxBlockLen is still processed completely (the
 * last CTA of its block walks the remaining tiles), only slower. */
int elb_fill_pattern_batch_sized(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	uint64_t* devCounters, uint64_t totalBytes, uint64_t maxBlockLen, void* stream);
int elb_verify_pattern_batch_sized(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	elb_verify_result* devResults, uint64_t* devCounters, uint64_t totalBytes,
	uint64_t maxBlockLen, void* stream);
int elb_fill_random_batch_sized(const elb_block_desc* descs, uint32_t numDescs, unsigned pct,
	uint64_t seed, int randAlgo, uint64_t* devCounters, uint64_t totalBytes, uint64_t maxBlockLen,
	void* stream);

/* Staged forms: the kernels also move each block between a pinned host buffer and its device
 * buffer while they work on it (the worker's default staging engine; replaces
 * cudaMemcpyGPUToHost / cudaMemcpyHostToGPU of LocalWorker.cpp:2285-2321 around the block
 * modifiers). The host copy of a block lives at (devPtr + hostDelta); the host memory must be
 * pinned and device-accessible (cudaHostAlloc / cudaHostRegister), `descs` may live there too.
 *   fill_*_staged   : every generated vector goes to the device buffer AND to the host buffer
 *   verify_*_staged : every vector is loaded from the host buffer, stored to the device buffer and
 *                     compared. devResults must hold {0, ~0} entries (elb_verify_results_init);
 *                     if hostResults and devDoneTicket (one zeroed unsigned in device memory)
 *                     are given, the last CTA of the launch copies the per-block results to
 *                     hostResults (pinned) and re-arms the device entries.
 *   stage_copy      : plain copy host -> device (hostToDevice != 0) or device -> host
 * hostDelta == 0 turns the staging off (verify then still publishes to hostResults).
 * hostDelta must be a multiple of ELB_STAGE_ALIGN (32): the kernels move 32-byte vectors, and both
 * ends of a vector are aligned only then. Page-aligned rings of equal layout satisfy this. Any
 * other hostDelta is rejected with -1 before anything is launched. */
#define ELB_STAGE_ALIGN 32

int elb_fill_pattern_staged(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	int64_t hostDelta, uint64_t* devCounters, uint64_t totalBytes, uint64_t maxBlockLen,
	void* stream);
int elb_fill_random_staged(const elb_block_desc* descs, uint32_t numDescs, unsigned pct,
	uint64_t seed, int randAlgo, int64_t hostDelta, uint64_t* devCounters, uint64_t totalBytes,
	uint64_t maxBlockLen, void* stream);
int elb_verify_pattern_staged(const elb_block_desc* descs, uint32_t numDescs, uint64_t salt,
	int64_t hostDelta, elb_verify_result* devResults, elb_verify_result* hostResults,
	unsigned* devDoneTicket, uint64_t* devCounters, uint64_t totalBytes, uint64_t maxBlockLen,
	void* stream);
int elb_stage_copy(const elb_block_desc* descs, uint32_t numDescs, int hostToDevice,
	int64_t hostDelta, uint64_t totalBytes, uint64_t maxBlockLen, void* stream);
/* devResults[0..numDescs) <- {0, ~0} */
int elb_verify_results_init(elb_verify_result* devResults, uint32_t numDescs, void* stream);

/* Number of kernel launches issued through this library since load (all threads). */
uint64_t elb_num_kernel_launches(void);

/* Thread-local text of the last error returned by any entry point on this thread. */
const char* elb_last_error(void);

/* ABI version of the loaded library (== ELB_ABI_VERSION). */
int elb_abi_version(void);

/* sizeof(elb_cfg) / sizeof(elb_phase_results) as compiled into the library (binding self-check) */
uint32_t elb_cfg_struct_size(void);
uint32_t elb_phase_results_struct_size(void);

/* ---------------------------------------------------------------------------------------------
 * Configuration (the ProgArgs subset that reaches the hot path; SURVEY.md §5 "Config / flags")
 * ------------------------------------------------------------------------------------------- */

typedef struct elb_cfg
{
	uint32_t structSize; /* = sizeof(elb_cfg), for ABI checking */

	/* bench paths (ProgArgs benchPathsVec / benchPathType) */
	const char* const* paths;
	uint32_t numPaths;
	int32_t pathType; /* enum elb_path_type */

	/* -t / --rankoffset / numDataSetThreads */
	uint32_t numThreads;
	uint32_t rankOffset;
	uint32_t numDataSetThreads; /* 0 = numThreads */

	/* -b / -s / --iodepth / --direct */
	uint64_t blockSize;
	uint64_t fileSize;
	uint32_t ioDepth;
	int32_t useDirectIO;
	int32_t ioEngine; /* enum elb_io_engine */

	/* -n / -N / --dirsharing (dir mode) */
	uint64_t numDirs;
	uint64_t numFiles;
	int32_t doDirSharing;

	/* --trunc / --trunctosize / --preallocfile */
	int32_t doTruncate;
	int32_t doTruncToSize;
	int32_t doPreallocFile;

	/* --rand / --randamount / --norandalign / --randalgo / --backward / --strided */
	int32_t useRandomOffsets;
	int32_t useRandomUnaligned;
	int32_t useExplicitRandOffsetAlgo; /* nonzero = user gave --randalgo => no full coverage */
	int32_t doReverseSeqOffsets;
	int32_t useStridedAccess;
	uint64_t randomAmount; /* 0 = default (ProgArgs.cpp:1558-1561) */
	uint64_t randOffsetSeed; /* 0 = self-seed (std::random_device) like the reference */

	/* --verify <salt> / --verifydirect / --readinline */
	uint64_t integrityCheckSalt;
	int32_t doDirectVerify;
	int32_t doReadInline;

	/* --blockvarpct / --blockvaralgo (+ injected seed; 0 = self-seed) */
	uint32_t blockVariancePercent;
	int32_t blockVarianceAlgo; /* enum elb_rand_algo */
	uint64_t blockVarianceSeed;

	/* --rwmixpct */
	uint32_t rwMixReadPercent;

	/* --gpuids / --cufile / --gds / --gdsbufreg / --cuhostbufreg */
	const int32_t* gpuIDs;
	uint32_t numGPUIDs;
	int32_t useCuFile;
	int32_t useGDSBufReg;

	/* pipeline tuning of the staged loop (new; 0 = defaults) */
	uint32_t pipelineBatchBlocks; /* blocks per batched kernel launch / staged copy */
	uint32_t pipelineNumBatches;  /* batches in flight (>= 2 for overlap) */

	int32_t ignoreDelErrors;
	int32_t runAsService; /* disables last-finisher stonewall trigger (Worker.cpp:41-43) */
	int32_t verifyCollectAll; /* nonzero: do not stop at first bad block, count all mismatches */
	/* enum elb_write_gate_mode: buffered (non-O_DIRECT) writes of all workers of this process to the
	 * same file pass a per-file FIFO gate in user space one at a time. Linux serialises buffered
	 * writes to one inode on the inode lock anyway; a ticket queue whose next-in-line spins while
	 * the others sleep hands the file over without the lock's contention (measured on tmpfs,
	 * 16 writers: 3.0 -> 3.7 GiB/s). I/O sizes and order per worker are unchanged; the block's
	 * latency includes the time in the queue (as it includes the inode lock wait without it). */
	int32_t serializeBufferedWrites;

	/* --rwmixthr: the first N local workers read (their share of the data set) during the write
	 * phase; their stats go to the ReadMix counters (LocalWorker.cpp:1028-1041) */
	uint32_t numRWMixReadThreads;
	int32_t randOffsetAlgo; /* enum elb_offset_rand_algo (--randalgo) */

	/* --limitread / --limitwrite: per-thread bytes per second, 0 = unlimited (RateLimiter.h:13-66,
	 * LocalWorker.cpp:1293-1299, 1331-1337); applied per block before its storage call */
	uint64_t limitReadBps;
	uint64_t limitWriteBps;
	/* --infloop: every worker restarts its share of the phase when it reaches the end, until
	 * interrupted or until the time limit (LocalWorker.cpp:196-364) */
	int32_t doInfiniteIOLoop;
	/* --rwmixthrpct: with --rwmixthr, keep the bytes of the reader threads at this percentage
	 * of all bytes of the write phase (RateLimiterRWMixThreads.h:22-197); 0 = no balancing */
	uint32_t rwMixThreadsReadPercent;

	/* Custom tree mode (--treefile, --treeroundup, --sharesize, --treerand): work on the dirs and
	 * files listed in a tree file instead of the generated r<rank>/d<n>/r<rank>-f<n> names
	 * (source/PathStore.cpp, LocalWorker.cpp:2927-3010, 3261-3470). NULL/empty = off. Needs a
	 * directory as the single benchmark path. */
	const char* treeFilePath;
	uint64_t treeRoundUpSize; /* round file sizes up to a multiple of this (0 = off) */
	uint64_t fileShareSize;   /* files of at least this size are shared between workers as block
	                             ranges; 0 = 32 x blockSize (ProgArgs.cpp:52, 1291-1292) */
	int32_t useCustomTreeRandomize; /* shuffle each worker's file list */
	int32_t reserved4;
	uint64_t treeRandomizeSeed;     /* 0 = self-seed (tests inject one) */

	/* --cores / --zones: worker rank r binds itself to cpuCores[r % n] and / or to the CPUs and
	 * memory of NUMA zone numaZones[r % n] first thing in its preparation (Worker.cpp:102-146) */
	const int32_t* cpuCores;
	const int32_t* numaZones;
	uint32_t numCPUCores;
	uint32_t numNumaZones;

	/* --flock range|full: POSIX advisory lock (fcntl F_SETLKW) around every block's storage call,
	 * read lock for reads, write lock for writes (FileTk.h:49-120, LocalWorker.cpp:1701-1750) */
	uint32_t flockType;     /* 0 none, 1 range, 2 full */
	/* --fadv: posix_fadvise on every opened file; bit 1 seq, 2 rand, 4 willneed, 8 dontneed,
	 * 16 noreuse (ProgArgs.h:240-249, FileTk.cpp:138-215) */
	uint32_t fadviseFlags;
	int32_t doStatInline;   /* --statinline: fstat each dir mode file right after open */
	int32_t noDirectIOCheck; /* --nodiocheck: skip the direct IO alignment / size sanity checks */

	/* Who moves a block between the pinned host ring and the device ring (enum
	 * elb_staging_engine): the fill / verify kernels themselves over PCIe (one launch per batch, no
	 * copy engine, no descriptor or result copies), or cudaMemcpyAsync on the batch stream followed
	 * / preceded by the kernel. 0 = auto (kernels). Ignored with --cufile (no host ring). */
	int32_t stagingEngine;
	/* 0: each worker binds itself to the CPUs of its GPU's NUMA node and prefers memory from there
	 * (pinned ring, page cache pages it first touches) unless --zones / --cores are given;
	 * nonzero: no binding (the reference's behaviour without --zones) */
	int32_t noGPUNumaBinding;
	/* --nofdsharing: every worker opens its own file descriptors in file / blockdev mode instead
	 * of using the manager's (ProgArgs.h useNoFDSharing, LocalWorker.cpp:1088-1117) */
	int32_t useNoFDSharing;
	int32_t reserved5;
} elb_cfg;

enum elb_staging_engine
{
	ELB_STAGING_AUTO = 0,
	ELB_STAGING_KERNEL = 1, /* fused: fill + stage-out, stage-in + verify, stage copy */
	ELB_STAGING_COPYENGINE = 2, /* cudaMemcpyAsync + kernel on the device slot */
};

/* elb_cfg::serializeBufferedWrites values */
enum elb_write_gate_mode
{
	ELB_WRITEGATE_AUTO = 0, /* on when several local workers write one file buffered */
	ELB_WRITEGATE_ON = 1,
	ELB_WRITEGATE_OFF = 2,
};

/* ---------------------------------------------------------------------------------------------
 * Stats types (source/LiveOps.h:13-118, source/LiveLatency.h:12-89, LatencyHistogram.h:28-45)
 * ------------------------------------------------------------------------------------------- */

typedef struct elb_liveops
{
	uint64_t numEntriesDone;
	uint64_t numBytesDone;
	uint64_t numIOPSDone;
} elb_liveops;

typedef struct elb_livelat
{
	uint64_t numAvgIOLatValues;
	uint64_t avgIOLatMicroSecsSum;
	uint64_t numAvgIOLatReadMixValues;
	uint64_t avgIOLatReadMixMicroSecsSum;
	uint64_t numAvgEntriesLatValues;
	uint64_t avgEntriesLatMicroSecsSum;
	uint64_t numAvgEntriesLatReadMixValues;
	uint64_t avgEntriesLatReadMixMicrosSecsSum;
} elb_livelat;

/* Sum of the live counters over all workers and GPUs of a manager. With two or more GPUs the
 * per-GPU partial sums (host counters staged to the GPU + the device-resident kernel counters of
 * that GPU's workers) are reduced to the first GPU with one grouped ncclReduce over NVLink; the
 * reference does this sum on the host (source/Statistics.cpp:414-470, :2728-2804). */
typedef struct elb_live_snapshot
{
	elb_liveops ops;
	elb_liveops opsReadMix;
	elb_livelat lat;          /* consumed: add-and-reset like LiveLatency::getAndResetAll */
	uint64_t numWorkersDone;
	uint64_t numWorkersTotal;
	uint64_t devCounters[ELB_DEVCTR_NUM]; /* verify mismatch / verified / filled bytes so far */
	uint32_t numGPUs;
	int32_t reducedWithNccl;  /* 1: summed by ncclReduce; 0: single GPU or NCCL unavailable */
	int32_t gatheredOnDevice; /* 1: device counters read by the gather kernel (no per-worker D2H) */
	int32_t reserved;
} elb_live_snapshot;

typedef struct elb_histogram
{
	uint64_t buckets[ELB_LATHISTO_NUMBUCKETS];
	uint64_t numStoredValues;
	uint64_t numMicroSecTotal;
	uint64_t minMicroSecLat; /* ~0 when empty */
	uint64_t maxMicroSecLat;
} elb_histogram;

/* Aggregated result of one phase (what Statistics::generatePhaseResults computes,
 * Statistics.cpp:1641-1764). */
typedef struct elb_phase_results
{
	uint64_t firstFinishUSec; /* stonewall: fastest worker with work */
	uint64_t lastFinishUSec;
	elb_liveops opsTotal;          /* last done */
	elb_liveops opsStoneWallTotal; /* first done */
	elb_liveops opsPerSec;          /* getPerSecFromUSec(opsTotal, lastFinishUSec) */
	elb_liveops opsStoneWallPerSec; /* getPerSecFromUSec(stonewall, firstFinishUSec) */
	elb_liveops opsReadMixTotal;
	elb_histogram iopsLatHisto;
	elb_histogram entriesLatHisto;
	uint64_t verifyMismatchBytes; /* device counter, summed over workers */
	uint64_t verifiedBytes;
	uint64_t filledBytes;
	uint64_t numKernelLaunches;
	uint64_t h2dBytes;
	uint64_t d2hBytes;
	uint64_t devKernelUSec; /* sum of event-timed kernel durations (fill/verify), microseconds */
	uint32_t numWorkersDone;
	uint32_t numWorkersDoneWithError;
	/* rwmix read side (Statistics.h PhaseResults: ops*ReadMix, *LatHistoReadMix) */
	elb_liveops opsStoneWallReadMixTotal;
	elb_liveops opsReadMixPerSec;
	elb_liveops opsStoneWallReadMixPerSec;
	elb_histogram iopsLatHistoReadMix;
	elb_histogram entriesLatHistoReadMix;
	/* CPU utilisation of this process' host between phase start and first/last finisher
	 * (CPUUtil.cpp; /proc/stat delta), percent */
	uint32_t cpuUtilStoneWallPercent;
	uint32_t cpuUtilPercent;
	/* 1: workers span >= 2 GPUs and the histograms + device counter blocks above were merged by
	 * ncclReduce sum / min / max to the first GPU (SURVEY.md §8e); 0: merged on the host */
	uint32_t statsReducedWithNccl;
	uint32_t reserved2;
} elb_phase_results;

/* ---------------------------------------------------------------------------------------------
 * Worker level (mirrors Worker.h / LocalWorker.h; SURVEY.md §8b)
 * ------------------------------------------------------------------------------------------- */

typedef struct elb_worker elb_worker;
typedef struct elb_mgr elb_mgr;

/* Histogram helpers (LatencyHistogram.h:50-77, :140-159, operator+= :187-202) */
void elb_histogram_reset(elb_histogram* h);
void elb_histogram_add_latency(elb_histogram* h, uint64_t latencyMicroSec);
void elb_histogram_merge(elb_histogram* dst, const elb_histogram* src);
double elb_histogram_percentile(const elb_histogram* h, double percentage);
/* UnitTk::getPerSecFromUSec (toolkits/UnitTk.h:48-56) */
uint64_t elb_per_sec_from_usec(uint64_t totalValue, uint64_t elapsedUSec);

/* Human-readable formats of the result table (toolkits/UnitTk.cpp:90-204, LatencyHistogram.h:
 * 109-178). kind 0: latency in microseconds ("1.23ms"), 1: elapsed milliseconds ("1m1.007s"),
 * 2: elapsed seconds ("1h2m3s"), 3: histogram line of `histo`, 4: percentile of `histo`. Returns the
 * text length (text truncated to outBufLen - 1), -1 on error. */
int64_t elb_format_value(int kind, uint64_t value, double percentage, const elb_histogram* histo,
	char* outBuf, uint64_t outBufLen);
/* UnitTk::numHumanToBytesBinary (toolkits/UnitTk.cpp:18-76): "4k", "1M", "64G"; 0 ok, -1 error */
int elb_num_human_to_bytes(const char* numHuman, uint64_t* outBytes);

/* HashTk::simple128 (toolkits/HashTk.cpp:10-41), the hash of the service password line that
 * travels as "PwHash"; out receives 32 hex digits + NUL */
void elb_simple128_hash(const char* input, char out[33]);

/* The two rate limiters of the per-block loop on their own (toolkits/RateLimiter.h:13-66,
 * toolkits/RateLimiterRWMixThreads.h:22-197). wait calls return 1 if the caller had to sleep, 0 if
 * not, -1 on error (balancer: interrupted, or 600 s without progress). */
typedef struct elb_rate_limiter elb_rate_limiter;
elb_rate_limiter* elb_rate_limiter_create(uint64_t limitPerSec);
int elb_rate_limiter_wait(elb_rate_limiter* limiter, uint64_t nextSize);
void elb_rate_limiter_destroy(elb_rate_limiter* limiter);

typedef struct elb_rwmix_balancer elb_rwmix_balancer;
elb_rwmix_balancer* elb_rwmix_balancer_create(unsigned readRatioPercent, unsigned numReaderThreads,
	unsigned numWriterThreads, uint64_t maxBlockSize);
int elb_rwmix_balancer_wait_read(elb_rwmix_balancer* balancer, uint64_t nextBlockSize);
int elb_rwmix_balancer_wait_write(elb_rwmix_balancer* balancer, uint64_t nextBlockSize);
void elb_rwmix_balancer_interrupt(elb_rwmix_balancer* balancer); /* waiters return -1 */
void elb_rwmix_balancer_destroy(elb_rwmix_balancer* balancer);

/* The FIFO gate in front of buffered writes to one file (elb_cfg::serializeBufferedWrites) as a
 * toolkit object: take a ticket, optionally sleep until near the front (< 2 tickets ahead), wait
 * for the turn, leave. */
typedef struct elb_write_gate elb_write_gate;
elb_write_gate* elb_write_gate_create(void);
uint64_t elb_write_gate_take_ticket(elb_write_gate* gate);
void elb_write_gate_wait_until_near(elb_write_gate* gate, uint64_t ticket);
void elb_write_gate_wait_turn(elb_write_gate* gate, uint64_t ticket);
void elb_write_gate_leave(elb_write_gate* gate);
void elb_write_gate_destroy(elb_write_gate* gate);
/* numThreads threads take turnsPerThread turns of holdUSec each through one gate; returns 0 if
 * every turn was exclusive and the turns were served in ticket order, else the number of
 * violations (self-check of the futex hand-over on this host). */
int64_t elb_write_gate_selftest(uint32_t numThreads, uint32_t turnsPerThread, uint32_t holdUSec);

/* Custom tree mode: the sublist of one worker (PathStore::getWorkerSublistNonShared/-Shared as
 * combined by LocalWorker::prepareCustomTreePathStores, LocalWorker.cpp:1520-1560), as text lines
 * "<path>\t<totalLen>\t<rangeStart>\t<rangeLen>\n". kind 0: directories, 1: files (non-shared
 * files first, then this worker's ranges of the shared files). Returns the length of the full
 * text (which is truncated to outBufLen - 1 bytes in outBuf), or -1 on error. */
int64_t elb_custom_tree_worker_list(const char* treeFilePath, uint64_t blockSize,
	uint64_t fileShareSize, uint64_t treeRoundUpSize, uint64_t workerRank,
	uint64_t numDataSetThreads, int kind, char* outBuf, uint64_t outBufLen);
/* FileTk::scanCustomTree (toolkits/FileTk.cpp:387-470): returns dirs + files found, -1 on error */
int64_t elb_custom_tree_scan(const char* scanPath, const char* outTreeFilePath);

/* ---------------------------------------------------------------------------------------------
 * Offset plans (toolkits/offsetgen/OffsetGenerator.h:27-46 interface; one handle type for all
 * six generators). Exposed so that a reference-side shim can reuse them and so that their
 * sequences can be checked without a GPU. kind: 0 sequential, 1 reverse, 2 random unaligned,
 * 3 random aligned, 4 strided, 5 random aligned full coverage. randState: xoshiro256** state
 * (NULL = self-seed); lcgSeed/haveLCGSeed: start-state source of the full coverage permutation.
 * ------------------------------------------------------------------------------------------- */
typedef struct elb_offset_plan elb_offset_plan;

elb_offset_plan* elb_offset_plan_create(int kind, uint64_t amount, uint64_t rangeLen,
	uint64_t rangeOffset, uint64_t blockSize, uint64_t numDataSetThreads,
	const uint64_t randState[4], uint64_t lcgSeed, int haveLCGSeed);
/* same with an explicit generator (enum elb_offset_rand_algo); randState: 4 words for the
 * xoshiro variants, word 0 = seed for golden prime and mt19937 (NULL = self-seed) */
elb_offset_plan* elb_offset_plan_create_algo(int kind, uint64_t amount, uint64_t rangeLen,
	uint64_t rangeOffset, uint64_t blockSize, uint64_t numDataSetThreads, int randAlgo,
	const uint64_t randState[4], uint64_t lcgSeed, int haveLCGSeed);

/* The offset PRNGs on their own (RandAlgoInterface::next, toolkits/random/RandAlgoInterface.h:27) */
typedef struct elb_rand_algo_handle elb_rand_algo_handle;
elb_rand_algo_handle* elb_rand_algo_create(int randAlgo, const uint64_t state[4]);
uint64_t elb_rand_algo_next(elb_rand_algo_handle* algo);
void elb_rand_algo_destroy(elb_rand_algo_handle* algo);
void elb_offset_plan_destroy(elb_offset_plan* plan);
void elb_offset_plan_restart(elb_offset_plan* plan); /* reset() */
void elb_offset_plan_restart_range(elb_offset_plan* plan, uint64_t rangeLen,
	uint64_t rangeOffset); /* reset(len, offset) */
/* next block; the requested length counts as submitted. returns 0 when nothing is left. */
int elb_offset_plan_next(elb_offset_plan* plan, uint64_t* outOffset, uint64_t* outLen);
uint64_t elb_offset_plan_bytes_total(const elb_offset_plan* plan);
uint64_t elb_offset_plan_bytes_left(const elb_offset_plan* plan);
/* expand an injected 64-bit seed to the xoshiro256** state used for worker `rank` */
void elb_expand_offset_seed(uint64_t seed, uint64_t rank, uint64_t outState[4]);

/* ---------------------------------------------------------------------------------------------
 * Manager level (WorkerManager: owns the workers and their threads, one thread per worker)
 * ------------------------------------------------------------------------------------------- */

/* Create workers (numThreads LocalWorker equivalents, ranks rankOffset..), allocate their rings on
 * GPU gpuIDs[rank % numGPUIDs] (LocalWorker.cpp:1420-1429) and start their threads; returns after
 * all workers finished preparation (WorkerManager.cpp:142-199). NULL on error (elb_last_error). */
elb_mgr* elb_mgr_create(const elb_cfg* cfg);

/* WorkerManager::startNextPhase (:291-324): reset stats, set phase + phaseStartT, wake workers. */
int elb_mgr_start_phase(elb_mgr* m, int benchPhase);

/* Wait up to timeoutMS for all workers to finish the phase (WorkerManager::waitForWorkersDone
 * :245-267). Returns 1 when all are done, 0 on timeout, <0 if a worker ended with an error. */
int elb_mgr_wait_done(elb_mgr* m, int timeoutMS);

/* start + wait in one call. */
int elb_mgr_run_phase(elb_mgr* m, int benchPhase);

/* Statistics::getLiveOps (Statistics.cpp:1333-1345): sum over workers. out[0] = liveOps,
 * out[1] = liveOpsReadMix. */
int elb_mgr_live_ops(elb_mgr* m, elb_liveops out[2]);
int elb_mgr_live_latency(elb_mgr* m, elb_livelat* out); /* add-and-reset */
/* all live counters at once, reduced across the manager's GPUs (NCCL for >= 2 GPUs) */
int elb_mgr_live_snapshot(elb_mgr* m, elb_live_snapshot* out);
/* one line describing how elb_mgr_live_snapshot reduces ("NCCL 22703, 2 GPUs, root GPU 0") */
const char* elb_mgr_live_reduce_info(elb_mgr* m);

/* Phase results (valid after wait_done returned 1). */
int elb_mgr_phase_results(elb_mgr* m, elb_phase_results* out);

/* Expected totals of a phase (WorkerManager::getPhaseNumEntriesAndBytes, :333-487). */
int elb_mgr_expected_totals(elb_mgr* m, int benchPhase, uint64_t* outEntries,
	uint64_t* outBytes);

/* Request friendly interruption of all workers (Worker::interruptExecution). */
int elb_mgr_interrupt(elb_mgr* m);

uint32_t elb_mgr_num_workers(elb_mgr* m);
elb_worker* elb_mgr_worker(elb_mgr* m, uint32_t localIdx);
const char* elb_mgr_last_error(elb_mgr* m);

/* Terminate threads (BenchPhase_TERMINATE), run cleanup, free everything. */
void elb_mgr_destroy(elb_mgr* m);

/* ---------------------------------------------------------------------------------------------
 * Command line front end: the reference's main() (source/Main.cpp:13-68) for the supported option
 * subset, incl. --service / --hosts distributed mode. Returns the process exit code.
 * ------------------------------------------------------------------------------------------- */
int elb_cli_main(int argc, char** argv);

/* Render phase results the way the reference prints/stores them, for the options of the given
 * command line: format 0 = console table rows (Statistics.cpp:1771-2140), 1 = CSV labels line +
 * values line (:2151-2323), 2 = JSON document (:2429-2723). Writes a NUL-terminated string into
 * outBuf (truncated to outBufLen) and returns the full length, or -1 on error (elb_last_error). */
int64_t elb_format_phase_results(int argc, char** argv, int benchPhase,
	const elb_phase_results* results, int format, char* outBuf, uint64_t outBufLen);

/* Per-worker getters (may be called from any thread while the worker runs; Worker.h:83-226) */
uint64_t elb_worker_rank(elb_worker* w);
int elb_worker_gpu_id(elb_worker* w);
int elb_worker_live_ops(elb_worker* w, elb_liveops out[2]);
int elb_worker_stonewall_ops(elb_worker* w, elb_liveops out[2]);
int elb_worker_histogram(elb_worker* w, int kind, elb_histogram* out);
uint64_t elb_worker_elapsed_usec(elb_worker* w); /* 0 if none (no work / error) */
int elb_worker_got_work(elb_worker* w);
int elb_worker_dev_counters(elb_worker* w, uint64_t out[ELB_DEVCTR_NUM]); /* D2H snapshot */
/* device address of the worker's counter block (ELB_DEVCTR_NUM u64) on its GPU — the payload of
 * the NCCL stats reduce; never dereference on the host. */
uint64_t* elb_worker_dev_counters_ptr(elb_worker* w);
const char* elb_worker_last_error(elb_worker* w);

#ifdef __cplusplus
}
#endif

#endif /* ELBENCHO_B200_H_ */
