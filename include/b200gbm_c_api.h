/*
 * b200gbm C ABI — the drop-in boundary of the B200-native LightGBM-on-Spark training path.
 *
 * libb200gbm.so exports the subset of the LightGBM 3.2.x C API that MMLSpark calls through the
 * SWIG-generated `lightgbmlib` bindings (SURVEY.md §8b), with the same names, argument order and
 * error convention (every function returns 0 on success, -1 on failure; the message is read with
 * LGBM_GetLastError()).  Handles are opaque pointers; all input arrays are caller-owned and may be
 * freed as soon as the call returns.  Last-error, CUDA-device and network state are thread-local:
 * one host thread drives one (network, dataset, booster) triple, like one Spark task thread.
 *
 * Citations are into /root/reference/lightgbm/src/main/scala/com/microsoft/ml/spark/lightgbm/ (LGB/).
 * Every `data` pointer may be a host pointer OR a CUDA device pointer (detected at run time).
 * There is no CPU fallback: calls that need the GPU fail with -1 when no CUDA device is present.
 */
#ifndef B200GBM_C_API_H_
#define B200GBM_C_API_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* DatasetHandle;
typedef void* BoosterHandle;

#define C_API_DTYPE_FLOAT32 (0) /* LGB/dataset/LightGBMDataset.scala:35-41 */
#define C_API_DTYPE_FLOAT64 (1)
#define C_API_DTYPE_INT32 (2)
#define C_API_DTYPE_INT64 (3)

#define C_API_PREDICT_NORMAL (0) /* LGB/booster/LightGBMBooster.scala:144-150 */
#define C_API_PREDICT_RAW_SCORE (1)
#define C_API_PREDICT_LEAF_INDEX (2)
#define C_API_PREDICT_CONTRIB (3)

/* ---- error ------------------------------------------------------------------------------ */
/* LGB/LightGBMUtils.scala:22-34 (validate: rc == -1 -> LGBM_GetLastError) */
const char* LGBM_GetLastError(void);

/* ---- network (replaces LightGBM's TCP collectives with NCCL over NVLink) ------------------ */
/* LGB/TrainUtils.scala:279-295: LGBM_NetworkInit(nodes, localListenPort, 120, numNodes).
 * `machines` = "ip:port,ip:port,..."; the rank is the position of the entry whose port equals
 * local_listen_port.  Rank 0 hands its ncclUniqueId to every other rank over one TCP connection
 * to that rank's listen port; afterwards all traffic is NCCL. */
int LGBM_NetworkInit(const char* machines, int local_listen_port, int listen_time_out, int num_machines);
/* LGB/LightGBMBase.scala:379 */
int LGBM_NetworkFree(void);

/* ---- dataset ---------------------------------------------------------------------------- */
/* LGB/dataset/DatasetAggregator.scala:335-343 (dense) */
int LGBM_DatasetCreateFromMat(const void* data, int data_type, int32_t nrow, int32_t ncol, int is_row_major,
                              const char* parameters, const DatasetHandle reference, DatasetHandle* out);
/* LGB/dataset/DatasetAggregator.scala:442-453 (sparse) */
int LGBM_DatasetCreateFromCSR(const void* indptr, int indptr_type, const int32_t* indices, const void* data,
                              int data_type, int64_t nindptr, int64_t nelem, int64_t num_col,
                              const char* parameters, const DatasetHandle reference, DatasetHandle* out);
/* LightGBM streaming ingestion (not used by the reference revision; offered as the bulk path of
 * SURVEY.md §8f-1): create from a column-wise sample, then push row blocks (host or device). */
int LGBM_DatasetCreateFromSampledColumn(double** sample_data, int** sample_indices, int32_t ncol,
                                        const int* num_per_col, int32_t num_sample_row, int32_t num_total_row,
                                        const char* parameters, DatasetHandle* out);
int LGBM_DatasetPushRows(DatasetHandle dataset, const void* data, int data_type, int32_t nrow, int32_t ncol,
                         int32_t start_row);
/* LGB/dataset/LightGBMDataset.scala:85-169 ("label"/"weight" f32, "init_score" f64, "group" i32) */
int LGBM_DatasetSetField(DatasetHandle handle, const char* field_name, const void* field_data, int num_element, int type);
/* LGB/dataset/LightGBMDataset.scala:22-47 (borrowed pointer into the dataset) */
int LGBM_DatasetGetField(DatasetHandle handle, const char* field_name, int* out_len, const void** out_ptr, int* out_type);
/* LGB/dataset/LightGBMDataset.scala:52-69 */
int LGBM_DatasetGetNumData(DatasetHandle handle, int* out);
int LGBM_DatasetGetNumFeature(DatasetHandle handle, int* out);
/* LGB/dataset/LightGBMDataset.scala:178-186 */
int LGBM_DatasetSetFeatureNames(DatasetHandle handle, const char** feature_names, int num_feature_names);
/* LGB/dataset/LightGBMDataset.scala:188-191 */
int LGBM_DatasetFree(DatasetHandle handle);

/* ---- booster life cycle ------------------------------------------------------------------ */
/* LGB/booster/LightGBMBooster.scala:230-243 */
int LGBM_BoosterCreate(const DatasetHandle train_data, const char* parameters, BoosterHandle* out);
/* LGB/booster/LightGBMBooster.scala:41-48 */
int LGBM_BoosterLoadModelFromString(const char* model_str, int* out_num_iterations, BoosterHandle* out);
/* LGB/booster/LightGBMBooster.scala:252-256 */
int LGBM_BoosterMerge(BoosterHandle handle, BoosterHandle other_handle);
/* LGB/booster/LightGBMBooster.scala:258-264 */
int LGBM_BoosterAddValidData(BoosterHandle handle, const DatasetHandle valid_data);
/* LGB/booster/LightGBMBooster.scala:152-157 */
int LGBM_BoosterFree(BoosterHandle handle);

/* ---- training (the hot path) ------------------------------------------------------------- */
/* LGB/booster/LightGBMBooster.scala:351-361 — one boosting iteration: gradients -> per-partition
 * histograms (K4) -> NCCL histogram allreduce (C2) -> best-split scan (K5) -> row partition (K7) */
int LGBM_BoosterUpdateOneIter(BoosterHandle handle, int* is_finished);
/* LGB/booster/LightGBMBooster.scala:368-388 (custom objective: grad/hess of length num_data*num_class) */
int LGBM_BoosterUpdateOneIterCustom(BoosterHandle handle, const float* grad, const float* hess, int* is_finished);
/* LGB/booster/LightGBMBooster.scala:315-318 ("learning_rate=<x>") */
int LGBM_BoosterResetParameter(BoosterHandle handle, const char* parameters);

/* ---- evaluation / introspection ---------------------------------------------------------- */
int LGBM_BoosterGetEvalCounts(BoosterHandle handle, int* out_len);
/* LGB/booster/LightGBMBooster.scala:279-294 (through the SWIG string-array helper) */
int LGBM_BoosterGetEvalNames(BoosterHandle handle, const int len, int* out_len, const size_t buffer_len,
                             size_t* out_buffer_len, char** out_strs);
/* LGB/booster/LightGBMBooster.scala:296-310 */
int LGBM_BoosterGetEval(BoosterHandle handle, int data_idx, int* out_len, double* out_results);
int LGBM_BoosterGetNumPredict(BoosterHandle handle, int data_idx, int64_t* out_len);
/* LGB/booster/LightGBMBooster.scala:327-346 */
int LGBM_BoosterGetPredict(BoosterHandle handle, int data_idx, int64_t* out_len, double* out_result);
/* LGB/booster/LightGBMBooster.scala:159-197 */
int LGBM_BoosterGetNumClasses(BoosterHandle handle, int* out_len);
int LGBM_BoosterNumModelPerIteration(BoosterHandle handle, int* out_tree_per_iteration);
int LGBM_BoosterNumberOfTotalModel(BoosterHandle handle, int* out_models);
int LGBM_BoosterGetNumFeature(BoosterHandle handle, int* out_len);
int LGBM_BoosterGetCurrentIteration(BoosterHandle handle, int* out_iteration);
/* LGB/booster/LightGBMBooster.scala:491-498 */
int LGBM_BoosterFeatureImportance(BoosterHandle handle, int num_iteration, int importance_type, double* out_results);

/* ---- model (de)serialisation ------------------------------------------------------------- */
/* LGB/booster/LightGBMBooster.scala:269-274 (SWIG helper retries with out_len when the buffer is short) */
int LGBM_BoosterSaveModelToString(BoosterHandle handle, int start_iteration, int num_iteration,
                                  int feature_importance_type, int64_t buffer_len, int64_t* out_len, char* out_str);
/* LGB/booster/LightGBMBooster.scala:465-472 */
int LGBM_BoosterDumpModel(BoosterHandle handle, int start_iteration, int num_iteration, int feature_importance_type,
                          int64_t buffer_len, int64_t* out_len, char* out_str);

/* ---- prediction (per-row UDF semantics of the reference; host side) ------------------------ */
/* LGB/booster/LightGBMBooster.scala:528-545 */
int LGBM_BoosterPredictForMatSingle(BoosterHandle handle, const void* data, int data_type, int ncol, int is_row_major,
                                    int predict_type, int start_iteration, int num_iteration, const char* parameter,
                                    int64_t* out_len, double* out_result);
/* LGB/booster/LightGBMBooster.scala:510-526 */
int LGBM_BoosterPredictForCSRSingle(BoosterHandle handle, const void* indptr, int indptr_type, const int32_t* indices,
                                    const void* data, int data_type, int64_t nindptr, int64_t nelem, int64_t num_col,
                                    int predict_type, int start_iteration, int num_iteration, const char* parameter,
                                    int64_t* out_len, double* out_result);
int LGBM_BoosterPredictForMat(BoosterHandle handle, const void* data, int data_type, int32_t nrow, int32_t ncol,
                              int is_row_major, int predict_type, int start_iteration, int num_iteration,
                              const char* parameter, int64_t* out_len, double* out_result);
int LGBM_BoosterCalcNumPredict(BoosterHandle handle, int num_row, int predict_type, int start_iteration,
                               int num_iteration, int64_t* out_len);

/* ---- ChunkedArray<T> (LGB/swig/SwigUtils.scala:22-90): growable chunk list for row streams ---- */
typedef void* ChunkedArrayHandle;
int B200GBM_ChunkedArrayCreate(int data_type, int64_t chunk_size, ChunkedArrayHandle* out);
int B200GBM_ChunkedArrayAdd(ChunkedArrayHandle h, double value);
int B200GBM_ChunkedArrayAddMany(ChunkedArrayHandle h, const void* values, int64_t n);
int64_t B200GBM_ChunkedArrayGetAddCount(ChunkedArrayHandle h);
int64_t B200GBM_ChunkedArrayGetChunksCount(ChunkedArrayHandle h);
int64_t B200GBM_ChunkedArrayGetLastChunkAddCount(ChunkedArrayHandle h);
double B200GBM_ChunkedArrayGetItem(ChunkedArrayHandle h, int64_t chunk, int64_t index, double on_fail);
int B200GBM_ChunkedArrayCoalesceTo(ChunkedArrayHandle h, void* out);
int B200GBM_ChunkedArrayRelease(ChunkedArrayHandle h);
int B200GBM_ChunkedArrayFree(ChunkedArrayHandle h);

/* ---- engine extensions (instrumentation, parity and benchmark support) ----------------------- */
int B200GBM_SetDevice(int ordinal);                 /* thread-local CUDA device of the calling rank-thread */
int B200GBM_GetDevice(int* ordinal);
int B200GBM_DeviceAlloc(size_t bytes, void** out);  /* cudaMalloc / cudaFree on the thread's device */
int B200GBM_DeviceFree(void* ptr);
int B200GBM_HostAllocPinned(size_t bytes, void** out);
int B200GBM_HostFreePinned(void* ptr);
int B200GBM_Memcpy(void* dst, const void* src, size_t bytes);   /* cudaMemcpyDefault + sync */
/* LightGBM's LCG row sampler (the rows that define the bins) */
int B200GBM_SampleIndices(int num_total_row, int sample_cnt, int seed, int* out, int* out_len);
/* counter-based synthetic generators (SURVEY.md §8d): kind 0 = regression, 1 = binary, 2 = graded relevance 0..4 (ranking),
 * 3 = 10 classes with the last ncol/16 columns categorical (log-uniform ids, cardinality 10^3..10^5) and a 70 %-zero first quarter.
 * x(row, col) and label(row) are pure functions of (seed, row, col). */
int B200GBM_SyntheticFill(void* dev_x_f32, void* dev_label_f32, int64_t row_start, int32_t nrow, int32_t ncol,
                          uint64_t seed, int kind);
int B200GBM_SyntheticRows(const int* rows, int32_t nrows, int32_t ncol, uint64_t seed, int kind, double* host_out,
                          float* host_label_out);
/* dataset introspection for the bit-exact bin parity tests */
int B200GBM_DatasetGetBins(DatasetHandle handle, uint8_t* out_row_major);          /* [num_data][num_feature] */
int B200GBM_DatasetGetBins16(DatasetHandle handle, uint16_t* out_row_major);       /* same, uint16: datasets with features of more than 256 bins */
int B200GBM_DatasetGetBinToCat(DatasetHandle handle, int feature, int* out, int* out_len);   /* categorical feature: bin -> category value (out: >= num_bin ints) */
/* bins of the selected rows only, gathered on the device: out [nrows][num_feature] uint16 (trivial features 0).  Lets a test or
 * bench.py check rows of a dataset far too large to download (the 100M x 512 benchmark matrix) against host-side binning. */
int B200GBM_DatasetGetBinsRows(DatasetHandle handle, const int32_t* rows, int32_t nrows, uint16_t* out);
/* {min, max} of the sampled values of a feature (the feature_infos entry of the model text) */
int B200GBM_DatasetGetFeatureRange(DatasetHandle handle, int feature, double* out2);
int B200GBM_DatasetGetFeatureInfo(DatasetHandle handle, int feature, int* out5);   /* num_bin, missing, default_bin, most_freq_bin, trivial */
int B200GBM_DatasetGetUpperBounds(DatasetHandle handle, int feature, double* out, int* out_len);
int B200GBM_DatasetGetIngestMs(DatasetHandle handle, double* out_ms);
/* kernel-level entry: fixed-point histogram (K4) of the given rows on the dataset's bins, returned as
 * fp64 [num_feature][256][2]; grad/hess/idx are host arrays; idx == NULL means rows 0..cnt-1 */
int B200GBM_DatasetHistogram(DatasetHandle handle, const float* grad, const float* hess, const int32_t* idx,
                             int32_t cnt, double* out);
/* timing of the engine stream, CUDA events: out = {hist_ms, total_ms, hist_rows, hist_launches, launches, iterations} */
int B200GBM_BoosterSetProfile(BoosterHandle handle, int profile_hist);
int B200GBM_BoosterGetTiming(BoosterHandle handle, double* out6, int reset);
int B200GBM_BoosterGetScores(BoosterHandle handle, int data_idx, double* out);    /* raw scores, class-major */
/* for tests: the objective's gradients and hessians at the current training scores (the init_score before the first iteration),
 * class-major [num_class][num_data] fp32; classes the objective does not train read 0.  Changes neither the model nor the scores. */
int B200GBM_BoosterGetGradients(BoosterHandle handle, float* out_grad, float* out_hess);
/* batched GPU prediction (SURVEY §8f-2): row-major matrix on the host or the device, predict_type NORMAL / RAW_SCORE / LEAF_INDEX /
 * CONTRIB (TreeSHAP, [nrow][num_class][num_feature+1]); values equal LGBM_BoosterPredictForMatSingle row by row (raw scores and leaf
 * indices bit for bit, contributions to 1e-12); out_result is a host buffer sized by LGBM_BoosterCalcNumPredict; elapsed_ms (may be
 * NULL) = CUDA-event time.  Replaces the per-row UDF calls of LightGBMBooster.scala:390-423,528-545 for whole partitions. */
int B200GBM_BoosterPredictForMatDevice(BoosterHandle handle, const void* data, int data_type, int64_t nrow, int32_t ncol, int predict_type,
                                       int start_iteration, int num_iteration, int64_t* out_len, double* out_result, double* elapsed_ms);
/* out = {num_machines, rank, histogram reduce mode (0 = ncclAllReduce, 1 = reduce-scatter + scan of the owned feature slice over NVLink
 * peer memory, 2 = two-shot all-reduce kernel over peer memory + replicated scan), constant_hessian} */
int B200GBM_BoosterGetInfo(BoosterHandle handle, int* out4);
/* out = {bytes of the optional column-major copy of the training bins kept for the partition kernel (0 = not kept: it is built before the
 * first tree only if it leaves a reserve of device memory, B200GBM_COLUMN_COPY=0 disables it), free device memory in bytes} */
int B200GBM_BoosterGetMemoryInfo(BoosterHandle handle, int64_t* out2);

#ifdef __cplusplus
}
#endif
#endif /* B200GBM_C_API_H_ */
