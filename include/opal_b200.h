/*
 * opal_b200.h -- extended C ABI of libopal_b200.so (beneath the drop-in opal.h).
 *
 * opal.h's opalSearchDatabase packs and uploads the database on every call, as the reference's
 * signature demands (reference src/opal.h:150-154 takes host pointers each time).  Real workloads
 * run many queries against one database, so the same engine is also reachable through a
 * resident-database handle: pack + upload once, search many times.  Plain pointers and sizes
 * only; every function is safe to bind from C, ctypes, cgo, JNI ...
 *
 * Scores / end locations returned here are in CALLER order (index i <-> db[i]), -1 for unset.
 */
#ifndef OPAL_B200_H
#define OPAL_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct OpalB200Db OpalB200Db;
struct OpalSearchResult; /* opal.h */

/* Number of CUDA devices this process can use (0 => every search returns OPAL_ERR_NO_SIMD_SUPPORT). */
int opalb200_device_count(void);

/* Text of the last CUDA / argument error seen by the calling thread ("" if none). */
const char* opalb200_last_error(void);

/*
 * The library recycles device and pinned host allocations between calls instead of returning them to the driver
 * (a drop-in opalSearchDatabase call would otherwise spend more time in cudaMalloc than searching): up to 8 GB of
 * device memory per GPU and 2 GB of pinned memory may sit in that cache.  This returns all of it.
 */
void opalb200_trim_cache(void);

/*
 * Length-sorts the database (longest first), concatenates it in that order and uploads it to
 * `device`'s HBM.  Same db / dbLength / dbSeqLengths meaning as opalSearchDatabase
 * (reference src/opal.h:107-109).  Returns NULL on failure.
 */
OpalB200Db* opalb200_db_create(unsigned char* db[], int dbLength, const int dbSeqLengths[], int device);
/*
 * The same database resident on SEVERAL devices of this host: the sequences, in length order, are dealt round-robin
 * over devices[0 .. numDevices) -- shards of equal residue count (= equal work: cells = queryLength x residues) and
 * equal length mix -- and every search below runs on all of them concurrently, one host thread and one set of
 * streams per device, each device returning its own results, which are scattered into the caller's arrays by an
 * index map (targets are independent: no collective, no peer traffic; SURVEY.md section 8e).  The alignment stage of
 * a target runs on the device that owns it.  opalb200_db_create / _create_sorted with device = -1 take the devices
 * from the environment instead (OPAL_B200_DEVICES = "all" or "0,1,...", else OPAL_B200_DEVICE, else device 0) -- as
 * the drop-in opalSearchDatabase does, which has no device argument.  devices NULL or numDevices <= 0: likewise.
 */
OpalB200Db* opalb200_db_create_multi(unsigned char* db[], int dbLength, const int dbSeqLengths[], const int devices[],
                                     int numDevices);
/* Devices the handle's database is dealt over (1 unless created for several). */
int opalb200_db_devices(const OpalB200Db* handle);
/*
 * Same, from a database that is already packed (the in-memory form of the on-disk format written by
 * opal_makedb_b200, opal_b200/cli/packed_db.h; replaces the per-run parse + sort of readFastaSequences,
 * reference src/opal_aligner.cpp:247-301): `residues` holds all sequences back to back, longest first;
 * sortedLengths[p] is the length of the p-th of them and order[p] the index it has for the caller
 * (order may be NULL: identity).  Results still come back in caller order.  Returns NULL on failure.
 */
OpalB200Db* opalb200_db_create_sorted(const unsigned char* residues, const int sortedLengths[], const int order[],
                                      int dbLength, int device);
void opalb200_db_destroy(OpalB200Db* handle);

/* Sequences / residues held by the handle. */
int opalb200_db_length(const OpalB200Db* handle);
long long opalb200_db_residues(const OpalB200Db* handle);

/*
 * Score (searchType 0) or score + end location (searchType 1) of `query` against every database
 * sequence whose skip[i] is 0 (skip may be NULL).  Arguments as opalSearchDatabase.  Outputs are
 * arrays of dbLength ints in caller order; endQuery/endTarget may be NULL for searchType 0.
 * deviceMs (nullable) receives the CUDA-event time from the first kernel launch to the last kernel
 * end of this search -- the window the reference times around its call (src/opal_aligner.cpp:157-165).
 * Returns 0 or an OPAL_ERR_* code.
 */
int opalb200_db_search(OpalB200Db* handle, const unsigned char query[], int queryLength,
                       int gapOpen, int gapExt, const int* scoreMatrix, int alphabetLength,
                       int searchType, int mode, const unsigned char* skip,
                       int* scores, int* endQuery, int* endTarget, float* deviceMs);

/*
 * Searches with a position-specific scoring matrix (PSSM) instead of a query and a substitution matrix: pssm is
 * queryLength x alphabetLength ints, row-major, and pssm[r * alphabetLength + y] is the score of query position r
 * against database residue code y (as from PSI-BLAST, a family alignment or any per-position scoring).  Everything
 * else is the matrix search: modes, gaps, search types, end-location tie-breaking, skip rule, results of empty
 * queries / targets.  pssm[r * A + y] = scoreMatrix[query[r] * A + y] gives exactly the scores and end locations of
 * the matrix search with (query, scoreMatrix).  Argument rules are the matrix rules, with the extremes taken over all
 * queryLength x alphabetLength entries (OPAL_ERR_OVERFLOW for an entry outside (INT_MIN / 2, INT_MAX / 2));
 * pssm may be NULL only when queryLength is 0 (otherwise OPAL_ERR_INVALID_ARGUMENT).
 * The alignment stage (the _results_pssm / _topk_pssm calls below, OPAL_SEARCH_ALIGNMENT) restates the reference's band
 * (calculateBandBorders) with M = the largest of all PSSM entries instead of the largest matrix entry.  It also takes
 * the residues the PSSM was built for (query, codes < alphabetLength, required at OPAL_SEARCH_ALIGNMENT and ignored
 * otherwise); they are used only to label diagonal steps OPAL_ALIGN_MATCH / OPAL_ALIGN_MISMATCH.
 *
 * Same outputs as opalb200_db_search.
 */
int opalb200_db_search_pssm(OpalB200Db* handle, const int* pssm, int queryLength, int alphabetLength,
                            int gapOpen, int gapExt, int searchType, int mode, const unsigned char* skip,
                            int* scores, int* endQuery, int* endTarget, float* deviceMs);

/*
 * numQueries searches against the resident database (config 3's protocol: many queries, one database), with up
 * to `inFlight` (1..16) queries on the device at a time so that the tail of one query overlaps the bulk of the
 * next and host-side planning / result publishing overlaps kernels.  Same arguments as opalb200_db_search;
 * outputs are numQueries x dbLength ints, row q = query q, in caller order.  batchMs (nullable) receives the
 * CUDA-event time from the start of the batch to the last kernel end.
 */
int opalb200_db_search_batch(OpalB200Db* handle, int numQueries, const unsigned char* const queries[],
                             const int queryLengths[], int gapOpen, int gapExt, const int* scoreMatrix,
                             int alphabetLength, int searchType, int mode,
                             int* scores, int* endQuery, int* endTarget, int inFlight, float* batchMs);

/*
 * The same with a mode per search (modes[s] = OPAL_MODE_*): the reference's performance protocol loops modes x queries
 * over one database (test/perf:15-24); in one batch the tail of the last search of a mode overlaps the first of the next.
 */
int opalb200_db_search_batch_modes(OpalB200Db* handle, int numSearches, const unsigned char* const queries[],
                                   const int queryLengths[], const int modes[], int gapOpen, int gapExt,
                                   const int* scoreMatrix, int alphabetLength, int searchType,
                                   int* scores, int* endQuery, int* endTarget, int inFlight, float* batchMs);

/* opalb200_db_search_batch_modes with one PSSM per search (pssms[s]: queryLengths[s] x alphabetLength, see
 * opalb200_db_search_pssm). */
int opalb200_db_search_batch_pssm(OpalB200Db* handle, int numSearches, const int* const pssms[],
                                  const int queryLengths[], const int modes[], int alphabetLength,
                                  int gapOpen, int gapExt, int searchType,
                                  int* scores, int* endQuery, int* endTarget, int inFlight, float* batchMs);

/*
 * opalSearchDatabase (reference src/opal.h:150-154) against the resident database: same result records, same
 * reuse rule for prefilled entries (:118-122), all three search levels including OPAL_SEARCH_ALIGNMENT --
 * only the db / dbLength / dbSeqLengths arguments are replaced by the handle.  results[] has
 * opalb200_db_length(handle) entries in caller order.
 */
int opalb200_db_search_results(OpalB200Db* handle, const unsigned char query[], int queryLength,
                               int gapOpen, int gapExt, const int* scoreMatrix, int alphabetLength,
                               struct OpalSearchResult* results[], int searchType, int mode);

/* opalb200_db_search_results with a PSSM (see opalb200_db_search_pssm; query labels the alignments' diagonal steps and
 * may be NULL below OPAL_SEARCH_ALIGNMENT). */
int opalb200_db_search_results_pssm(OpalB200Db* handle, const unsigned char query[], const int* pssm,
                                    int queryLength, int alphabetLength, int gapOpen, int gapExt,
                                    struct OpalSearchResult* results[], int searchType, int mode);

/*
 * Score -> top-k -> alignment in one call on the resident database (BASELINE configs[3]: "SCORE pass, take the
 * top 1000, ALIGNMENT on those"): a score + end search over every sequence, selection of the k best (score
 * descending, ties by caller index ascending) and, for searchType OPAL_SEARCH_ALIGNMENT, start location and
 * alignment of just those k -- nothing is re-uploaded and nothing is scored twice, which is what the two
 * opalSearchDatabase calls of the reference protocol cost.  indices[j] receives the caller index of the j-th
 * best sequence and *results[j] its record (same fields as opalSearchDatabase gives it at that search level);
 * both arrays have k entries, *found (nullable) = min(k, dbLength) of them are written.
 */
int opalb200_db_search_topk(OpalB200Db* handle, const unsigned char query[], int queryLength,
                            int gapOpen, int gapExt, const int* scoreMatrix, int alphabetLength,
                            int searchType, int mode, int k, int* indices, struct OpalSearchResult* results[], int* found);

/* opalb200_db_search_topk with a PSSM (see opalb200_db_search_pssm; query labels the alignments' diagonal steps and may
 * be NULL below OPAL_SEARCH_ALIGNMENT). */
int opalb200_db_search_topk_pssm(OpalB200Db* handle, const unsigned char query[], const int* pssm,
                                 int queryLength, int alphabetLength, int gapOpen, int gapExt,
                                 int searchType, int mode, int k, int* indices,
                                 struct OpalSearchResult* results[], int* found);

/*
 * opalb200_db_search_topk for numSearches searches in one call, up to `inFlight` (1..16; <= 0: 3) of them on the device
 * at a time as in opalb200_db_search_batch, with a mode per search (modes[s] = OPAL_MODE_*).  At
 * OPAL_SEARCH_ALIGNMENT the hits of all searches are aligned in the same launches.  indices and results are
 * numSearches x k, row-major: row s starts at s * k and holds exactly what opalb200_db_search_topk returns for search s
 * alone.  *found (nullable) = min(k, dbLength), the count written in every row; later slots are untouched.  Every search
 * is checked before any runs: a fault returns the code of the lowest-index search that has one, writes no record and
 * leaves *found = 0.
 */
int opalb200_db_search_batch_topk(OpalB200Db* handle, int numSearches, const unsigned char* const queries[],
                                  const int queryLengths[], const int modes[], int gapOpen, int gapExt,
                                  const int* scoreMatrix, int alphabetLength, int searchType, int k,
                                  int* indices, struct OpalSearchResult* results[], int* found, int inFlight);

/* opalb200_db_search_batch_topk with one PSSM per search (pssms[s]: queryLengths[s] x alphabetLength, see
 * opalb200_db_search_pssm).  queries[s] labels the alignments' diagonal steps; `queries` and any queries[s] may be NULL
 * below OPAL_SEARCH_ALIGNMENT. */
int opalb200_db_search_batch_topk_pssm(OpalB200Db* handle, int numSearches, const unsigned char* const queries[],
                                       const int* const pssms[], const int queryLengths[], const int modes[],
                                       int alphabetLength, int gapOpen, int gapExt, int searchType, int k,
                                       int* indices, struct OpalSearchResult* results[], int* found, int inFlight);

/* Statistics of the last search on this handle: kernels launched, targets re-run in 32 bits, and the
 * geometry of the last launched class (threads per target pair, query rows per thread, passes over the
 * query, resident warps per SM scheduler partition), and the number of concurrent launch groups. Any pointer may be NULL. */
void opalb200_db_last_stats(const OpalB200Db* handle, int* kernelLaunches, int* rerun32, int* G, int* R, int* passes,
                            int* warpsPerPartition, int* groups);

/* Targets of the last search that were swept "folded": one target per warp, occupying both 16-bit lanes (its
 * second half of the query rows rides 32 columns behind the first), which is how the few longest targets of a
 * database -- each bounds the search time, being swept by a single warp -- are finished sooner. 0 = none. */
int opalb200_db_last_folded(const OpalB200Db* handle);

/* Tasks of the last search whose passes over the query were "chained": a query longer than one strip of rows takes
 * several passes, and for the longest targets every pass runs on a warp of its own at the same time, the boundary row
 * handed from pass to pass through L2 while both sweep -- the target then costs its length in steps once, not once per
 * pass. 0 = none. */
int opalb200_db_last_chained(const OpalB200Db* handle);

/*
 * Measures the packed-DPX issue rate of `device` with a register-only kernel running the SW cell
 * recurrence (6 s16x2 instructions per 2 cells): returns giga cell updates per second that the
 * integer pipe can sustain (the roofline of SURVEY.md section 8d), and through the out-params the
 * thread-instructions/s and the kernel time.
 */
double opalb200_measure_dpx_peak(int device, double* threadInstrPerSec, float* ms);
/* Same with the instruction mix of the recurrence chosen: mix 0 = SW (6 packed instructions per 2 cells, the function
 * above), mix 1 = NW / HW / OV (5: no running maximum per cell). */
double opalb200_measure_dpx_peak_mix(int device, int mix, double* threadInstrPerSec, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* OPAL_B200_H */
