/*
 * fastsmc_b200 — C ABI of the B200-native FastSMC IBD hot path (libfastsmc_b200.so).
 *
 * This is the drop-in boundary: plain pointers and sizes, int error codes, no exceptions, no C++
 * or torch types.  The C++ host classes (fastsmc_b200/csrc/host: HMM, FastSMC, ASMC) and the
 * Python front end call nothing else.  Each entry point names the reference routine(s) it
 * replaces; paths are relative to the reference's ASMC_SRC/SRC directory.
 *
 * Conventions
 *   - every function returns FSMC_OK (0) or a negative FSMC_E_* code; fsmc_last_error() returns a
 *     thread-local message for the last failure on the calling thread;
 *   - all pointers are HOST pointers unless a name ends in _dev;
 *   - a context owns one GPU's device buffers and one CUDA stream; it is not re-entrant (like the
 *     reference HMM object, HMM.hpp:84-170) — use one context per host thread and GPU;
 *   - there is no CPU fallback: without a CUDA device every call fails with FSMC_E_CUDA.
 */
#ifndef FASTSMC_B200_H
#define FASTSMC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FSMC_OK 0
#define FSMC_E_INVALID (-1)  /* bad argument                                        */
#define FSMC_E_CUDA (-2)     /* CUDA runtime error (message has the CUDA string)    */
#define FSMC_E_STATE (-3)    /* call order: model / haplotypes not set              */
#define FSMC_E_OVERFLOW (-4) /* an output buffer was too small; see the out counts  */
#define FSMC_E_NOMEM (-5)    /* device memory exhausted                             */

#define FSMC_TILE 32 /* pairs per tile == lanes per warp == reference default batchSize */

typedef struct fsmc_ctx fsmc_ctx;

const char* fsmc_last_error(void);
int fsmc_version(void);

/* Number of visible CUDA devices (0 if none / driver missing). */
int fsmc_device_count(void);

/* Create / destroy a context on CUDA device `device`. */
int fsmc_ctx_create(int device, fsmc_ctx** out);
int fsmc_ctx_destroy(fsmc_ctx* ctx);

/* Run all work of this context on an existing CUDA stream (a cudaStream_t passed as void*), e.g.
 * torch's current stream.  NULL restores the context's own stream. */
int fsmc_ctx_set_stream(fsmc_ctx* ctx, void* cuda_stream);

/* ------------------------------------------------------------------------------------------------
 * Model: everything HMM::HMM precomputes (HMM.cpp:65-127) and getNextAlphaBatched /
 * getPreviousBetaBatched look up per site (HMM.cpp:795-797, 951-954).
 *
 * The reference keys transition rows by an exact float distance in an unordered_map
 * (DecodingQuantities.hpp:60-63).  Here the host resolves roundMorgans(gen[pos]-gen[pos-1])
 * (HmmUtils.cpp:65-79) to a row index once per site; the device sees dense tables.
 * ------------------------------------------------------------------------------------------------ */
typedef struct fsmc_model {
  int32_t states;                 /* S                                                       */
  int32_t sites;                  /* L                                                       */
  const float* initialStateProb;  /* [S]    DecodingQuantities::initialStateProb             */
  const float* expectedTimes;     /* [S]    DecodingQuantities::expectedTimes                */
  const float* columnRatios;      /* [S]    DecodingQuantities::columnRatios                 */
  const float* emission1;         /* [L][S] HMM::emission1AtSite        (HMM.cpp:159-256)    */
  const float* emission0minus1;   /* [L][S] HMM::emission0minus1AtSite                       */
  const float* emission2minus0;   /* [L][S] HMM::emission2minus0AtSite                       */
  int32_t numDistances;           /* rows of the four transition tables                      */
  const float* D;                 /* [numDistances][S] Dvectors                              */
  const float* B;                 /* [numDistances][S] Bvectors                              */
  const float* U;                 /* [numDistances][S] Uvectors                              */
  const float* RR;                /* [numDistances][S] rowRatioVectors                       */
  const int32_t* distanceRow;     /* [L] row for the gap (pos-1 -> pos); entry 0 is ignored  */
  int32_t stateThreshold;         /* HMM::getStateThreshold   (HMM.cpp:504-513)              */
  int32_t ageThreshold;           /* HMM.cpp:101-105                                         */
  float probabilityThreshold;     /* HMM.cpp:96-99                                           */
  /* Optional identity of the tables above (0 = none).  A context that already holds a model with the same non-zero tag,
   * state and site counts keeps its device tables and only takes the three thresholds: the jobs of one data set
   * (Data.cpp:62-80) share their emission and transition tables, and a pooled context is handed job after job.          */
  uint64_t modelTag;
} fsmc_model;

int fsmc_set_model(fsmc_ctx* ctx, const fsmc_model* model);

/* ------------------------------------------------------------------------------------------------
 * Haplotypes: the genotype1/genotype2 bit vectors of Data::individuals (Individual.hpp,
 * Data.cpp:472-497), i.e. AFTER minor-allele folding, bit-packed.
 * bits[h * wordsPerHap + s / 64] bit (s % 64) = allele of haplotype h at site s,
 * wordsPerHap = (sites + 63) / 64.  Haplotype h is individual h/2, hap 1 + h%2
 * (HmmUtils.cpp:179-188).
 * ------------------------------------------------------------------------------------------------ */
int fsmc_set_haplotypes(fsmc_ctx* ctx, const uint64_t* bits, int64_t numHaps, int64_t sites);

/* ------------------------------------------------------------------------------------------------
 * Decoding: replaces HMM::decodeBatch (HMM.cpp:639-722: forwardBatch, backwardBatch, combine) and
 * its consumers writePerPairOutputFastSMC (HMM.cpp:1179-1357, segment calling incl.
 * getPosteriorMean / getMAP, HMM.cpp:1087-1107) and writePerPairOutput (HMM.cpp:1360-1410).
 *
 * The unit of work is a TILE: up to 32 haplotype pairs that the reference decodes in one batch,
 * sharing the batch's decode window [from,to) and segment-scan window [scanFrom,scanTo)
 * (HMM.cpp:555-636, 1199-1204).  A reference batch larger than 32 is passed as several tiles with
 * the same windows.  Per-site posteriors never leave the chip; only the outputs asked for do.
 * ------------------------------------------------------------------------------------------------ */

/* fsmc_decode_request.flags */
#define FSMC_CALL_SEGMENTS 0x1u   /* run the IBD segment caller                                   */
#define FSMC_SEG_AGE 0x2u         /* per-segment posterior mean + MAP (doPerPairPosteriorMean/MAP) */
#define FSMC_SITE_MEAN 0x4u       /* per-site posterior mean TMRCA   (HMM.cpp:1378-1392)          */
#define FSMC_SITE_MAP 0x8u        /* per-site MAP state index        (HMM.cpp:1396-1409)          */
#define FSMC_SITE_IBD 0x10u       /* per-site IBD probability  sum_{k<stateThreshold} posterior   */
#define FSMC_EXACT 0x20u          /* unfused mul/add in the reference's NO_SSE operation order:   */
                                  /* results are bit-identical to the reference's NO_SSE build    */
#define FSMC_GENERIC_KERNEL 0x40u /* force the any-S shared-memory kernel (testing)               */
#define FSMC_WIDE_KERNEL 0x80u    /* never use the narrow (no beta round trip) kernel (testing)   */
#define FSMC_ONE_WARP_KERNEL 0x100u /* never use the state-split kernels (one tile per CTA) (testing) */
#define FSMC_SITE_POSTERIOR 0x200u /* full per-site posterior of every pair (HMM.cpp:1372-1389, ASMC::decodePairs
                                      per_pair_posteriors; HMM::decode)                             */
#define FSMC_SUM_POSTERIOR 0x400u  /* per-site posterior summed over the real pairs of the call
                                      (augmentSumOverPairs, HMM.cpp:1044-1085; sum_of_posteriors)   */
#define FSMC_SUM_BY_GENOTYPE 0x800u /* with FSMC_SUM_POSTERIOR: three sums, by the pair's genotype at the site:
                                      both major / heterozygous / both minor (sumOverPairs00/01/11)  */

typedef struct fsmc_segment {
  uint32_t pair;     /* tile * 32 + lane                                                        */
  int32_t posStart;  /* first site of the segment                                               */
  int32_t posEnd;    /* last site of the segment (inclusive)                                    */
  float prob;        /* sum of per-site IBD probabilities (writePairIBD's `prob`)               */
  float postMean;    /* HMM::getPosteriorMean of the per-state sums (if FSMC_SEG_AGE)           */
  float mapTime;     /* HMM::getMAP: expectedTimes[argmax_k sum_k / prior_k] (if FSMC_SEG_AGE)  */
  int32_t mapState;  /* that argmax                                                             */
  int32_t level;     /* 0..3 = threshold 1000x,100x,10x,1x probabilityThreshold                 */
} fsmc_segment;

typedef struct fsmc_decode_request {
  int64_t numTiles;
  const uint32_t* hapA;        /* [numTiles*32] first haplotype of each pair  (unused lanes: any) */
  const uint32_t* hapB;        /* [numTiles*32] second haplotype                                  */
  const int32_t* tilePairs;    /* [numTiles] number of real pairs in the tile (1..32)             */
  const int32_t* tileFrom;     /* [numTiles] decode window start                                  */
  const int32_t* tileTo;       /* [numTiles] decode window end (exclusive)                        */
  const int32_t* tileScanFrom; /* [numTiles] segment scan start   (ignored without CALL_SEGMENTS) */
  const int32_t* tileScanTo;   /* [numTiles] segment scan end (exclusive)                         */
  uint32_t flags;
  /* outputs ------------------------------------------------------------------------------------ */
  fsmc_segment* segments;      /* [segmentCapacity]; sorted by (pair, posStart) on return         */
  int64_t segmentCapacity;
  /* per-site outputs: row-major [numTiles*32][siteStride], row = pair, column = pos - tileFrom.
   * Rows of unused lanes are left untouched.  May be NULL if the flag is not set. */
  float* siteMean;
  int32_t* siteMap;
  float* siteIbd;
  int64_t siteStride;
  /* FSMC_SITE_POSTERIOR: row-major [numTiles*32][states][siteStride], column = pos - tileFrom.      */
  float* sitePosterior;
  /* FSMC_SUM_POSTERIOR: row-major [planes][states][sites], column = absolute site; planes = 3 with
   * FSMC_SUM_BY_GENOTYPE (0: both major, 1: heterozygous, 2: both minor), else 1.  Overwritten with
   * the sums of THIS call (float atomics on the device: the summation order is not fixed, results
   * agree with the reference's sequential sums to rounding).                                        */
  float* sumPosterior;
} fsmc_decode_request;

typedef struct fsmc_decode_stats {
  int64_t numSegments;  /* segments found (may exceed segmentCapacity -> FSMC_E_OVERFLOW)         */
  double pairSites;     /* sum over tiles of real pairs * (to - from)                             */
  float kernelMs;       /* device time of the decode kernels, CUDA events on the context stream   */
  float totalMs;        /* device time of the whole call incl. H2D/D2H copies on that stream      */
  int32_t kernelLaunches;
  int32_t statesKernel; /* S the kernel was specialised for, 0 = generic                          */
  int64_t scratchBytes; /* backward-sweep scratch in HBM                                          */
  int32_t narrowKernel; /* 1 if the kernel without the beta round trip ran (states < threshold only) */
  int32_t tileWarps;    /* warps that shared a tile: 1, or 2 / 4 for the state-split kernels                */
  /* all-state age estimates without the beta round trip (csrc/decode_sparse.cuh): narrow sweeps + checkpoints, then
   * full posteriors only inside the IBD runs                                                                        */
  int32_t sparseKernel;     /* 1 if that path ran                                                  */
  int32_t checkpointSites;  /* sites per checkpoint block                                           */
  int64_t sparseItems;      /* run pieces (one per run and block) refined                           */
  int64_t checkpointBytes;  /* beta checkpoints in HBM                                              */
  /* outputs copied device -> host by the call: segment records, per-site rows and sums (the counter read-back of at most
   * 32 bytes that sizes them is not counted).  0 for fsmc_decode_device.                                              */
  int64_t d2hBytes;
} fsmc_decode_stats;

int fsmc_decode(fsmc_ctx* ctx, const fsmc_decode_request* req, fsmc_decode_stats* stats);

/* ------------------------------------------------------------------------------------------------
 * Device-resident outputs: the per-site outputs of fsmc_decode written by the decode kernels straight into caller-owned
 * device memory of the context's device (e.g. torch tensors), at caller-chosen rows.  Nothing is staged and nothing but
 * the stats crosses to the host.  The request's own output fields are ignored; FSMC_CALL_SEGMENTS is rejected.  The kernel
 * is the one fsmc_decode chooses for the same flags; a request that would run a narrow kernel (FSMC_SITE_IBD without
 * FSMC_SITE_MEAN / FSMC_SITE_MAP) is rejected, since those kernels write pair-numbered rows only: add FSMC_WIDE_KERNEL.
 * All work is enqueued on the context's stream; the call returns when it has completed.
 * ------------------------------------------------------------------------------------------------ */
typedef struct fsmc_device_outputs {
  const int64_t* laneRow;     /* host [numTiles*32]: output row of pair tile*32+lane; ignored for unused lanes          */
  int64_t numRows;            /* rows of every per-pair output below (< 2^31)                                         */
  int64_t siteStride;         /* >= longest window; column = pos - tileFrom                                           */
  float* siteMean_dev;        /* [numRows][siteStride] or NULL (FSMC_SITE_MEAN)                                       */
  int32_t* siteMap_dev;       /* [numRows][siteStride] or NULL (FSMC_SITE_MAP)                                        */
  float* siteIbd_dev;         /* [numRows][siteStride] or NULL (FSMC_SITE_IBD)                                        */
  float* sitePosterior_dev;   /* [numRows][states][siteStride] or NULL (FSMC_SITE_POSTERIOR): posterior * stateWeight[k] */
  /* [planes][states][sites] or NULL (FSMC_SUM_POSTERIOR): ACCUMULATED, out += (sum over the call's pairs) * stateWeight[k]
   * (one rounding per operation, in this order: the host's per-chunk update of ASMC::decodePairs)                          */
  float* sumPosterior_dev;
  const float* stateWeight;   /* host [states] or NULL (= 1): ASMC passes expectedTimes (ref: HMM.cpp:1382-1389)       */
} fsmc_device_outputs;
int fsmc_decode_device(fsmc_ctx* ctx, const fsmc_decode_request* req, const fsmc_device_outputs* out,
                       fsmc_decode_stats* stats);

/* Per column of a row-major device matrix m[rows][ld] (cols <= ld): the minimum over rows and the first row that attains it,
 * as DecodePairsReturnStruct::finaliseCalculations (ref: DecodePairsReturnStruct.hpp:105-118): row 0 is the start value and
 * a later row replaces it only when strictly smaller (so a NaN in row 0 stays, later NaNs are skipped).  Deterministic.
 * Enqueued on the context's stream; returns without waiting.  min_dev / argmin_dev: [cols], device memory.              */
int fsmc_column_min_f32(fsmc_ctx* ctx, const float* m_dev, int64_t rows, int64_t cols, int64_t ld, float* min_dev,
                        int32_t* argmin_dev);
int fsmc_column_min_i32(fsmc_ctx* ctx, const int32_t* m_dev, int64_t rows, int64_t cols, int64_t ld, int32_t* min_dev,
                        int32_t* argmin_dev);

/* Which kernel family a request with these flags would run on the context's model, before any request exists: callers
 * that run several contexts on one device (HMM's pipelined decode workers) must know whether the request sizes its
 * scratch for the whole device.  meanScanSites = expected length of the scan windows (0 for hashing candidates): the
 * sparse age-estimate path is chosen for long windows only.                                                         */
typedef struct fsmc_kernel_info {
  int32_t statesKernel;  /* as fsmc_decode_stats                                                   */
  int32_t narrowKernel;
  int32_t sparseKernel;
  int32_t tileWarps;
  int32_t largeScratch;  /* 1: scratch grows with free device memory (full beta rows or checkpoints): one context per device */
} fsmc_kernel_info;
int fsmc_query_kernel(fsmc_ctx* ctx, uint32_t flags, double meanScanSites, fsmc_kernel_info* out);

/* Split-phase form of the same call, for callers that keep inputs resident in HBM and overlap host
 * work with the kernels (and for timing the kernels without host traffic):
 *   fsmc_plan_create  : validates the request, copies its input arrays to the device, allocates
 *                       device outputs and the backward-sweep scratch;
 *   fsmc_plan_launch  : enqueues the decode kernels on the context stream and returns at once;
 *   fsmc_plan_collect : waits, copies the requested outputs into the host buffers of `out`
 *                       (same layout as fsmc_decode_request; only the output fields are read) and
 *                       sorts the segments.  May be called once per launch. */
typedef struct fsmc_plan fsmc_plan;
int fsmc_plan_create(fsmc_ctx* ctx, const fsmc_decode_request* req, fsmc_plan** out);
int fsmc_plan_launch(fsmc_ctx* ctx, fsmc_plan* plan);
int fsmc_plan_collect(fsmc_ctx* ctx, fsmc_plan* plan, const fsmc_decode_request* out, fsmc_decode_stats* stats);
int fsmc_plan_destroy(fsmc_ctx* ctx, fsmc_plan* plan);


/* ------------------------------------------------------------------------------------------------
 * Seeding: replaces the GERMLINE-style candidate search of FastSMC::run (FastSMC.cpp:144-229):
 * Individuals::getWordHash (HASHING/Individuals.hpp:51-62), SeedHash::insertIndividuals /
 * extendAllPairs incl. the job-window filter (HASHING/SeedHash.hpp:41-135), ExtendHash::extendPair /
 * clearPairsPriorTo / clearAllPairs (HASHING/ExtendHash.hpp:52-116) and the length filter of
 * Match::print (HASHING/Match.hpp:42-52, HASHING/Utils.cpp:22-34).
 *
 * Works on the haplotypes given to fsmc_set_haplotypes.  Word w covers sites [64w, 64w+63]; a
 * trailing partial word is never hashed (FastSMC.cpp:188-196).  Two haplotypes match at w when
 * their 64-SNP words are identical (the reference's hash is the identity on the word, SURVEY F5;
 * minor-allele folding flips both haplotypes alike, so folded words compare like raw ones).  A
 * match interval [startWord, endWord] of a pair a < b starts at a matching word with no match in
 * the preceding gap+1 words, and is extended while the next match is at most gap+1 words ahead
 * (low-complexity words, see fsmc_seed_params.skip, count as neither match nor miss for an open interval
 * and move its end; with fsmc_seed_params.maxSeeds a "match" at w is membership of the same nested bucket and moves the
 * interval's end up to readAhead-1 words past w, see there).
 * Intervals are produced for pairs that pass the job filter on GLOBAL haplotype ids
 * (HASHING/SeedHash.hpp:99-129) and, unless FSMC_SEED_ALL_INTERVALS is set, whose genetic length
 * 100*(gen[min(64*end+63, L-1)] - gen[64*start]) is >= minLengthCm.
 * Output order: ascending (endWord, hapA, hapB) — the canonical candidate order.
 * ------------------------------------------------------------------------------------------------ */
#define FSMC_SEED_ALL_INTERVALS 0x1u /* keep intervals shorter than minLengthCm too (order replay)  */
#define FSMC_SEED_UNSORTED 0x2u      /* skip the canonical sort: intervals in no particular order     */
/* FSMC_SEED_REFERENCE_ORDER: output = the candidates only (length >= minLengthCm), in the order in which the
 * reference's FastSMC::run hands them to HMM::decodeFromHashing, i.e. the iteration order of its SeedHash /
 * ExtendHash maps (boost::unordered_map 1.75; HASHING/SeedHash.hpp:34,80, HASHING/ExtendHash.hpp:29,85-116).  Batch
 * composition, decode windows and therefore segment boundaries depend on this order (HMM.cpp:561-565, 1199-1204).
 * Computed on the device (csrc/seed_order.h).  The seed map is keyed by words of RAW alleles: give flipMask when the
 * haplotypes of fsmc_set_haplotypes are minor-allele folded.                                                        */
#define FSMC_SEED_REFERENCE_ORDER 0x4u

typedef struct fsmc_match {
  uint32_t hapA;      /* smaller local haplotype index                                            */
  uint32_t hapB;      /* larger local haplotype index                                             */
  int32_t startWord;
  int32_t endWord;    /* inclusive                                                                */
} fsmc_match;

typedef struct fsmc_seed_params {
  int32_t gap;                    /* DecodingParams::gap                                          */
  float minLengthCm;              /* DecodingParams::min_m                                        */
  const float* geneticPositions;  /* [sites] Morgans (Data::geneticPositions)                     */
  const uint32_t* globalHapId;    /* [numHaps] id of each loaded haplotype in the whole data set  */
  /* job geometry, in global haplotype ids (Data.cpp:62-80): windows [loI,hiI) x [loJ,hiJ)        */
  uint32_t loI, hiI, loJ, hiJ;
  int32_t lastJob;                /* jobInd == jobs: open-ended windows, strictly below diagonal  */
  int32_t aboveDiag;              /* Data::is_j_above_diag                                        */
  uint32_t flags;
  /* [sites/64] (host) bit s%64 of word s/64 = site s was flipped by folding: raw word = word ^ flipMask[w].
   * NULL = the haplotypes are raw.  Only read with FSMC_SEED_REFERENCE_ORDER.                      */
  const uint64_t* flipMask;
  /* DecodingParams::skip (FastSMC.cpp:208-219, HASHING/ExtendHash.hpp:102-106): a word whose number of distinct
   * haplotype words divided by numHaps is <= skip is "low complexity": no pair is seeded at it, and every interval that is
   * alive there is extended to it.  0 = off (every word has at least one distinct value).                              */
  float skip;
  /* DecodingParams::max_seeds (HASHING/SeedHash.hpp:56-69, 85-93): a bucket of more than maxSeeds identical words is not
   * enumerated; its haplotypes are re-hashed on the next word (recursively, while that word lies inside the reference's
   * read-ahead buffer of readAhead = DecodingParams::constReadAhead words), and the pairs of the final nested bucket are
   * extended to the deepest word.  0 = off.                                                                              */
  int32_t maxSeeds;
  int32_t readAhead;
} fsmc_seed_params;

typedef struct fsmc_seed_stats {
  int64_t numMatches;     /* intervals found (may exceed capacity -> FSMC_E_OVERFLOW)              */
  int64_t pairVisits;     /* sum over words of sum over groups n(n-1)/2                            */
  int64_t numStarts;      /* pair visits that started an interval                                  */
  int32_t numWords;
  int32_t kernelLaunches;
  float kernelMs;         /* device time of the seeding kernels                                    */
  int64_t bytesRead;      /* algorithmic HBM bytes: every word once + grouping traffic             */
  /* FSMC_SEED_REFERENCE_ORDER: numMatches counts the candidates; every interval is a node of the reference's map */
  int64_t numIntervals;   /* intervals of any length                                               */
  int64_t maxLiveNodes;   /* most nodes in the reference's extend map at once                       */
  int32_t orderEpochs;    /* rehashes of that map + 1                                               */
  float orderMs;          /* device time of the ordering passes                                     */
  float rankHostMs;       /* host time of the seed-map iteration ranks (overlaps the seeding kernels) */
} fsmc_seed_stats;

int fsmc_seed(fsmc_ctx* ctx, const fsmc_seed_params* params, fsmc_match* out, int64_t capacity,
              fsmc_seed_stats* stats);

#ifdef __cplusplus
}
#endif
#endif /* FASTSMC_B200_H */
