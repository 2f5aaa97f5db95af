// C ABI of libb200gbm (see include/b200gbm_c_api.h for the reference call sites each entry replaces).
#include "../../include/b200gbm_c_api.h"

#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "engine.cu"   // unity build: one translation unit, so the kernels in kernels.cuh have a single definition

using namespace b200gbm;

static thread_local std::string t_last_error = "Everything is fine";

static int Fail(const char* what) {
  t_last_error = what;
  return -1;
}
#define API_BEGIN() try {
#define API_END()                                                        \
  }                                                                      \
  catch (const std::exception& ex) { return Fail(ex.what()); }           \
  catch (const std::string& ex) { return Fail(ex.c_str()); }             \
  catch (...) { return Fail("unknown exception"); }                      \
  return 0;

struct DatasetBox { std::unique_ptr<Dataset> ds; };
static Dataset* DS(DatasetHandle h) {
  if (!h) Fatal("dataset handle is null");
  return static_cast<Dataset*>(h);
}
static Booster* BS(BoosterHandle h) {
  if (!h) Fatal("booster handle is null");
  return static_cast<Booster*>(h);
}

extern "C" {

const char* LGBM_GetLastError(void) { return t_last_error.c_str(); }

int LGBM_NetworkInit(const char* machines, int local_listen_port, int listen_time_out, int num_machines) {
  API_BEGIN();
  NetworkInit(machines, local_listen_port, listen_time_out, num_machines);
  API_END();
}
int LGBM_NetworkFree(void) {
  API_BEGIN();
  NetworkFree();
  API_END();
}

// ------------------------------------------------------------------------------------ dataset
int LGBM_DatasetCreateFromMat(const void* data, int data_type, int32_t nrow, int32_t ncol, int is_row_major, const char* parameters,
                              const DatasetHandle reference, DatasetHandle* out) {
  API_BEGIN();
  *out = Dataset::CreateFromMat(data, data_type, nrow, ncol, is_row_major, parameters, static_cast<const Dataset*>(reference));
  API_END();
}
int LGBM_DatasetCreateFromCSR(const void* indptr, int indptr_type, const int32_t* indices, const void* data, int data_type, int64_t nindptr,
                              int64_t nelem, int64_t num_col, const char* parameters, const DatasetHandle reference, DatasetHandle* out) {
  API_BEGIN();
  *out = Dataset::CreateFromCSR(indptr, indptr_type, indices, data, data_type, nindptr, nelem, num_col, parameters,
                                static_cast<const Dataset*>(reference));
  API_END();
}
int LGBM_DatasetCreateFromSampledColumn(double** sample_data, int** sample_indices, int32_t ncol, const int* num_per_col, int32_t num_sample_row,
                                        int32_t num_total_row, const char* parameters, DatasetHandle* out) {
  API_BEGIN();
  *out = Dataset::CreateFromSampledColumn(sample_data, sample_indices, ncol, num_per_col, num_sample_row, num_total_row, parameters);
  API_END();
}
int LGBM_DatasetPushRows(DatasetHandle dataset, const void* data, int data_type, int32_t nrow, int32_t ncol, int32_t start_row) {
  API_BEGIN();
  DS(dataset)->PushRows(data, data_type, nrow, ncol, start_row);
  API_END();
}
int LGBM_DatasetSetField(DatasetHandle handle, const char* field_name, const void* field_data, int num_element, int type) {
  API_BEGIN();
  DS(handle)->SetField(field_name, field_data, num_element, type);
  API_END();
}
int LGBM_DatasetGetField(DatasetHandle handle, const char* field_name, int* out_len, const void** out_ptr, int* out_type) {
  API_BEGIN();
  DS(handle)->GetField(field_name, out_len, out_ptr, out_type);
  if (*out_ptr == nullptr) Fatal(std::string("Field ") + field_name + " is empty");
  API_END();
}
int LGBM_DatasetGetNumData(DatasetHandle handle, int* out) {
  API_BEGIN();
  *out = DS(handle)->num_data;
  API_END();
}
int LGBM_DatasetGetNumFeature(DatasetHandle handle, int* out) {
  API_BEGIN();
  *out = DS(handle)->num_total_features;
  API_END();
}
int LGBM_DatasetSetFeatureNames(DatasetHandle handle, const char** feature_names, int num_feature_names) {
  API_BEGIN();
  DS(handle)->SetFeatureNames(feature_names, num_feature_names);
  API_END();
}
int LGBM_DatasetFree(DatasetHandle handle) {
  API_BEGIN();
  delete static_cast<Dataset*>(handle);
  API_END();
}

// ------------------------------------------------------------------------------------ booster
int LGBM_BoosterCreate(const DatasetHandle train_data, const char* parameters, BoosterHandle* out) {
  API_BEGIN();
  *out = new Booster(DS(train_data), parameters);
  API_END();
}
int LGBM_BoosterLoadModelFromString(const char* model_str, int* out_num_iterations, BoosterHandle* out) {
  API_BEGIN();
  if (!model_str) Fatal("model string is null");
  Booster* b = new Booster(std::string(model_str));
  *out_num_iterations = b->model.NumIterations();
  *out = b;
  API_END();
}
int LGBM_BoosterMerge(BoosterHandle handle, BoosterHandle other_handle) {
  API_BEGIN();
  BS(handle)->MergeFrom(BS(other_handle));
  API_END();
}
int LGBM_BoosterAddValidData(BoosterHandle handle, const DatasetHandle valid_data) {
  API_BEGIN();
  BS(handle)->AddValidData(DS(valid_data));
  API_END();
}
int LGBM_BoosterFree(BoosterHandle handle) {
  API_BEGIN();
  delete static_cast<Booster*>(handle);
  API_END();
}
int LGBM_BoosterUpdateOneIter(BoosterHandle handle, int* is_finished) {
  API_BEGIN();
  *is_finished = BS(handle)->UpdateOneIter() ? 1 : 0;
  API_END();
}
int LGBM_BoosterUpdateOneIterCustom(BoosterHandle handle, const float* grad, const float* hess, int* is_finished) {
  API_BEGIN();
  if (!grad || !hess) Fatal("grad / hess should not be null");
  *is_finished = BS(handle)->UpdateOneIterCustom(grad, hess) ? 1 : 0;
  API_END();
}
int LGBM_BoosterResetParameter(BoosterHandle handle, const char* parameters) {
  API_BEGIN();
  BS(handle)->ResetParameter(parameters);
  API_END();
}
int LGBM_BoosterGetEvalCounts(BoosterHandle handle, int* out_len) {
  API_BEGIN();
  *out_len = static_cast<int>(BS(handle)->EvalNames().size());
  API_END();
}
int LGBM_BoosterGetEvalNames(BoosterHandle handle, const int len, int* out_len, const size_t buffer_len, size_t* out_buffer_len, char** out_strs) {
  API_BEGIN();
  std::vector<std::string> names = BS(handle)->EvalNames();
  *out_len = static_cast<int>(names.size());
  *out_buffer_len = 0;
  for (size_t i = 0; i < names.size(); ++i) {
    *out_buffer_len = std::max(*out_buffer_len, names[i].size() + 1);
    if (static_cast<int>(i) < len && out_strs && out_strs[i] && buffer_len > 0) {
      std::strncpy(out_strs[i], names[i].c_str(), buffer_len - 1);
      out_strs[i][buffer_len - 1] = '\0';
    }
  }
  API_END();
}
int LGBM_BoosterGetEval(BoosterHandle handle, int data_idx, int* out_len, double* out_results) {
  API_BEGIN();
  std::vector<double> v = BS(handle)->GetEval(data_idx);
  *out_len = static_cast<int>(v.size());
  for (size_t i = 0; i < v.size(); ++i) out_results[i] = v[i];
  API_END();
}
int LGBM_BoosterGetNumPredict(BoosterHandle handle, int data_idx, int64_t* out_len) {
  API_BEGIN();
  *out_len = BS(handle)->NumPredict(data_idx);
  API_END();
}
int LGBM_BoosterGetPredict(BoosterHandle handle, int data_idx, int64_t* out_len, double* out_result) {
  API_BEGIN();
  BS(handle)->GetPredict(data_idx, out_len, out_result);
  API_END();
}
int LGBM_BoosterGetNumClasses(BoosterHandle handle, int* out_len) {
  API_BEGIN();
  *out_len = BS(handle)->model.num_class;
  API_END();
}
int LGBM_BoosterNumModelPerIteration(BoosterHandle handle, int* out) {
  API_BEGIN();
  *out = BS(handle)->model.num_tree_per_iteration;
  API_END();
}
int LGBM_BoosterNumberOfTotalModel(BoosterHandle handle, int* out) {
  API_BEGIN();
  *out = static_cast<int>(BS(handle)->model.trees.size());
  API_END();
}
int LGBM_BoosterGetNumFeature(BoosterHandle handle, int* out_len) {
  API_BEGIN();
  *out_len = BS(handle)->model.max_feature_idx + 1;
  API_END();
}
int LGBM_BoosterGetCurrentIteration(BoosterHandle handle, int* out_iteration) {
  API_BEGIN();
  *out_iteration = BS(handle)->model.NumIterations();
  API_END();
}
int LGBM_BoosterFeatureImportance(BoosterHandle handle, int num_iteration, int importance_type, double* out_results) {
  API_BEGIN();
  std::vector<double> v = BS(handle)->model.FeatureImportance(num_iteration, importance_type);
  for (size_t i = 0; i < v.size(); ++i) out_results[i] = v[i];
  API_END();
}
static void CopyOut(const std::string& s, int64_t buffer_len, int64_t* out_len, char* out_str) {
  *out_len = static_cast<int64_t>(s.size()) + 1;
  if (*out_len <= buffer_len && out_str) std::memcpy(out_str, s.c_str(), s.size() + 1);
}
int LGBM_BoosterSaveModelToString(BoosterHandle handle, int start_iteration, int num_iteration, int feature_importance_type, int64_t buffer_len,
                                  int64_t* out_len, char* out_str) {
  API_BEGIN();
  CopyOut(BS(handle)->SaveModelToString(start_iteration, num_iteration, feature_importance_type), buffer_len, out_len, out_str);
  API_END();
}
int LGBM_BoosterDumpModel(BoosterHandle handle, int start_iteration, int num_iteration, int feature_importance_type, int64_t buffer_len,
                          int64_t* out_len, char* out_str) {
  API_BEGIN();
  (void)feature_importance_type;
  CopyOut(BS(handle)->DumpModelJson(start_iteration, num_iteration), buffer_len, out_len, out_str);
  API_END();
}

// ------------------------------------------------------------------------------------ predict
static void RowToDouble(const void* data, int data_type, int ncol, std::vector<double>* row) {
  row->resize(ncol);
  if (data_type == C_API_DTYPE_FLOAT64) std::memcpy(row->data(), data, sizeof(double) * ncol);
  else if (data_type == C_API_DTYPE_FLOAT32) for (int i = 0; i < ncol; ++i) (*row)[i] = static_cast<const float*>(data)[i];
  else Fatal("Unknown data type in predict");
}
int LGBM_BoosterPredictForMatSingle(BoosterHandle handle, const void* data, int data_type, int ncol, int is_row_major, int predict_type,
                                    int start_iteration, int num_iteration, const char* parameter, int64_t* out_len, double* out_result) {
  API_BEGIN();
  (void)is_row_major; (void)parameter;
  std::vector<double> row;
  RowToDouble(data, data_type, ncol, &row);
  *out_len = BS(handle)->model.PredictRow(row.data(), ncol, predict_type, start_iteration, num_iteration, out_result);
  API_END();
}
int LGBM_BoosterPredictForCSRSingle(BoosterHandle handle, const void* indptr, int indptr_type, const int32_t* indices, const void* data, int data_type,
                                    int64_t nindptr, int64_t nelem, int64_t num_col, int predict_type, int start_iteration, int num_iteration,
                                    const char* parameter, int64_t* out_len, double* out_result) {
  API_BEGIN();
  (void)parameter; (void)nindptr;
  Booster* b = BS(handle);
  int64_t ncol = std::max<int64_t>(num_col, b->model.max_feature_idx + 1);
  std::vector<double> row(ncol, 0.0);
  int64_t a = indptr_type == C_API_DTYPE_INT32 ? static_cast<const int32_t*>(indptr)[0] : static_cast<const int64_t*>(indptr)[0];
  int64_t e = indptr_type == C_API_DTYPE_INT32 ? static_cast<const int32_t*>(indptr)[1] : static_cast<const int64_t*>(indptr)[1];
  if (e > nelem) e = nelem;
  for (int64_t k = a; k < e; ++k) {
    double v = data_type == C_API_DTYPE_FLOAT32 ? static_cast<const float*>(data)[k] : static_cast<const double*>(data)[k];
    if (indices[k] >= 0 && indices[k] < ncol) row[indices[k]] = v;
  }
  *out_len = b->model.PredictRow(row.data(), static_cast<int>(ncol), predict_type, start_iteration, num_iteration, out_result);
  API_END();
}
static int64_t PerRow(const HostModel& m, int predict_type, int start_iteration, int num_iteration) {
  int t0, t1;
  m.IterRange(start_iteration, num_iteration, &t0, &t1);
  if (predict_type == C_API_PREDICT_LEAF_INDEX) return t1 - t0;
  if (predict_type == C_API_PREDICT_CONTRIB) return static_cast<int64_t>(m.num_tree_per_iteration) * (m.max_feature_idx + 2);
  return m.num_tree_per_iteration;
}
int LGBM_BoosterCalcNumPredict(BoosterHandle handle, int num_row, int predict_type, int start_iteration, int num_iteration, int64_t* out_len) {
  API_BEGIN();
  *out_len = PerRow(BS(handle)->model, predict_type, start_iteration, num_iteration) * num_row;
  API_END();
}
int LGBM_BoosterPredictForMat(BoosterHandle handle, const void* data, int data_type, int32_t nrow, int32_t ncol, int is_row_major, int predict_type,
                              int start_iteration, int num_iteration, const char* parameter, int64_t* out_len, double* out_result) {
  API_BEGIN();
  (void)parameter;
  const HostModel& m = BS(handle)->model;
  const int64_t per = PerRow(m, predict_type, start_iteration, num_iteration);
#pragma omp parallel
  {
    std::vector<double> row(ncol);
#pragma omp for schedule(static)
    for (int i = 0; i < nrow; ++i) {
      for (int f = 0; f < ncol; ++f) {
        size_t at = is_row_major ? static_cast<size_t>(i) * ncol + f : static_cast<size_t>(f) * nrow + i;
        row[f] = data_type == C_API_DTYPE_FLOAT32 ? static_cast<const float*>(data)[at] : static_cast<const double*>(data)[at];
      }
      m.PredictRow(row.data(), ncol, predict_type, start_iteration, num_iteration, out_result + per * i);
    }
  }
  *out_len = per * nrow;
  API_END();
}

// ------------------------------------------------------------------------------------ ChunkedArray
struct ChunkedArray {
  int data_type;
  size_t elem, chunk_size, last_count = 0;
  std::vector<std::vector<unsigned char>> chunks;
  ChunkedArray(int t, int64_t cs) : data_type(t), elem(t == C_API_DTYPE_FLOAT64 ? 8 : 4), chunk_size(static_cast<size_t>(cs)) { NewChunk(); }
  void NewChunk() { chunks.emplace_back(chunk_size * elem); last_count = 0; }
  void Add(double v) {
    if (last_count == chunk_size) NewChunk();
    unsigned char* p = chunks.back().data() + last_count * elem;
    if (data_type == C_API_DTYPE_FLOAT64) *reinterpret_cast<double*>(p) = v;
    else if (data_type == C_API_DTYPE_FLOAT32) *reinterpret_cast<float*>(p) = static_cast<float>(v);
    else *reinterpret_cast<int32_t*>(p) = static_cast<int32_t>(v);
    ++last_count;
  }
  size_t Count() const { return chunks.empty() ? 0 : (chunks.size() - 1) * chunk_size + last_count; }
};
int B200GBM_ChunkedArrayCreate(int data_type, int64_t chunk_size, ChunkedArrayHandle* out) {
  API_BEGIN();
  if (chunk_size <= 0) Fatal("ChunkedArray: chunk size must be positive");
  if (data_type != C_API_DTYPE_FLOAT32 && data_type != C_API_DTYPE_FLOAT64 && data_type != C_API_DTYPE_INT32) Fatal("ChunkedArray: unsupported type");
  *out = new ChunkedArray(data_type, chunk_size);
  API_END();
}
int B200GBM_ChunkedArrayAdd(ChunkedArrayHandle h, double value) {
  API_BEGIN();
  static_cast<ChunkedArray*>(h)->Add(value);
  API_END();
}
int B200GBM_ChunkedArrayAddMany(ChunkedArrayHandle h, const void* values, int64_t n) {
  API_BEGIN();
  ChunkedArray* c = static_cast<ChunkedArray*>(h);
  const unsigned char* src = static_cast<const unsigned char*>(values);
  while (n > 0) {
    if (c->last_count == c->chunk_size) c->NewChunk();
    size_t room = c->chunk_size - c->last_count, take = std::min<size_t>(room, static_cast<size_t>(n));
    std::memcpy(c->chunks.back().data() + c->last_count * c->elem, src, take * c->elem);
    c->last_count += take; src += take * c->elem; n -= static_cast<int64_t>(take);
  }
  API_END();
}
int64_t B200GBM_ChunkedArrayGetAddCount(ChunkedArrayHandle h) { return static_cast<int64_t>(static_cast<ChunkedArray*>(h)->Count()); }
int64_t B200GBM_ChunkedArrayGetChunksCount(ChunkedArrayHandle h) { return static_cast<int64_t>(static_cast<ChunkedArray*>(h)->chunks.size()); }
int64_t B200GBM_ChunkedArrayGetLastChunkAddCount(ChunkedArrayHandle h) { return static_cast<int64_t>(static_cast<ChunkedArray*>(h)->last_count); }
double B200GBM_ChunkedArrayGetItem(ChunkedArrayHandle h, int64_t chunk, int64_t index, double on_fail) {
  ChunkedArray* c = static_cast<ChunkedArray*>(h);
  if (chunk < 0 || chunk >= static_cast<int64_t>(c->chunks.size()) || index < 0) return on_fail;
  size_t lim = static_cast<size_t>(chunk) + 1 == c->chunks.size() ? c->last_count : c->chunk_size;
  if (static_cast<size_t>(index) >= lim) return on_fail;
  const unsigned char* p = c->chunks[chunk].data() + static_cast<size_t>(index) * c->elem;
  if (c->data_type == C_API_DTYPE_FLOAT64) return *reinterpret_cast<const double*>(p);
  if (c->data_type == C_API_DTYPE_FLOAT32) return *reinterpret_cast<const float*>(p);
  return *reinterpret_cast<const int32_t*>(p);
}
int B200GBM_ChunkedArrayCoalesceTo(ChunkedArrayHandle h, void* out) {
  API_BEGIN();
  ChunkedArray* c = static_cast<ChunkedArray*>(h);
  unsigned char* dst = static_cast<unsigned char*>(out);
  for (size_t i = 0; i < c->chunks.size(); ++i) {
    size_t cnt = i + 1 == c->chunks.size() ? c->last_count : c->chunk_size;
    std::memcpy(dst, c->chunks[i].data(), cnt * c->elem);
    dst += cnt * c->elem;
  }
  API_END();
}
int B200GBM_ChunkedArrayRelease(ChunkedArrayHandle h) {
  API_BEGIN();
  ChunkedArray* c = static_cast<ChunkedArray*>(h);
  c->chunks.clear(); c->chunks.shrink_to_fit(); c->last_count = 0;
  API_END();
}
int B200GBM_ChunkedArrayFree(ChunkedArrayHandle h) {
  API_BEGIN();
  delete static_cast<ChunkedArray*>(h);
  API_END();
}

// ------------------------------------------------------------------------------------ extensions
int B200GBM_SetDevice(int ordinal) {
  API_BEGIN();
  SetThreadDevice(ordinal);
  EnsureDevice();
  API_END();
}
int B200GBM_GetDevice(int* ordinal) {
  API_BEGIN();
  *ordinal = CurrentDevice();
  API_END();
}
int B200GBM_DeviceAlloc(size_t bytes, void** out) {
  API_BEGIN();
  EnsureDevice();
  B200_CUDA(cudaMalloc(out, bytes));
  API_END();
}
int B200GBM_DeviceFree(void* ptr) {
  API_BEGIN();
  EnsureDevice();
  B200_CUDA(cudaFree(ptr));
  API_END();
}
int B200GBM_HostAllocPinned(size_t bytes, void** out) {
  API_BEGIN();
  EnsureDevice();
  B200_CUDA(cudaMallocHost(out, bytes));
  API_END();
}
int B200GBM_HostFreePinned(void* ptr) {
  API_BEGIN();
  B200_CUDA(cudaFreeHost(ptr));
  API_END();
}
int B200GBM_Memcpy(void* dst, const void* src, size_t bytes) {
  API_BEGIN();
  EnsureDevice();
  B200_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDefault));
  API_END();
}
int B200GBM_SampleIndices(int num_total_row, int sample_cnt, int seed, int* out, int* out_len) {
  API_BEGIN();
  LcgRandom r(seed);
  std::vector<int> v = r.Sample(num_total_row, std::min(sample_cnt, num_total_row));
  for (size_t i = 0; i < v.size(); ++i) out[i] = v[i];
  *out_len = static_cast<int>(v.size());
  API_END();
}
}  // extern "C"

// counter-based generator: every value is a pure function of (seed, row, col)
__device__ __forceinline__ unsigned long long syn_mix(unsigned long long x) {
  x += 0x9E3779B97F4A7C15ULL;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
  return x ^ (x >> 31);
}
__device__ __forceinline__ float syn_u(unsigned long long seed, long long row, int col) {
  unsigned long long h = syn_mix(seed ^ syn_mix(static_cast<unsigned long long>(row) * 0x100000001B3ULL + static_cast<unsigned long long>(col)));
  return static_cast<float>(h >> 40) * (1.0f / 16777216.0f);
}
// kind 3 (BASELINE.json configs[4]): the last ncol/16 columns are categorical with a log-uniform (Zipf-like) id distribution and
// cardinalities from 10^3 to 10^5; the first quarter of the columns is 70 % zeros; the rest is dense numeric like the other kinds
__device__ __forceinline__ int syn_ncat(int ncol, int kind) { return kind == 3 ? max(ncol / 16, 1) : 0; }
__device__ __forceinline__ float syn_x(unsigned long long seed, long long row, int col, int ncol, int kind) {
  const float u = syn_u(seed, row, col);
  if (kind == 3) {
    const int ncat = syn_ncat(ncol, kind);
    if (col >= ncol - ncat) {
      const int j = col - (ncol - ncat);
      const float log10c = 3.0f + (ncat > 1 ? 2.0f * j / (ncat - 1) : 0.0f);
      return floorf(__powf(10.0f, u * log10c)) - 1.0f;                       // ids 0 .. 10^log10c - 1, P(id) ~ 1/(id+1)
    }
    if (col < ncol / 4 && syn_u(seed ^ 0x5151515151ULL, row, col) < 0.7f) return 0.0f;
  }
  return u * (1.0f + static_cast<float>(col % 7)) - static_cast<float>(col % 5);
}
__device__ float syn_label(unsigned long long seed, long long row, int ncol, int kind) {
  const int m = ncol < 16 ? ncol : 16;
  float s = 0.f;
  for (int j = 0; j < m; ++j) s += __sinf(6.2831853f * syn_u(seed, row, j)) * (1.0f + 0.1f * j);
  if (ncol >= 2) s += 2.0f * (syn_u(seed, row, 0) - 0.5f) * (syn_u(seed, row, 1) - 0.5f) * 4.0f;
  const float noise = syn_u(seed ^ 0xABCDEF12345ULL, row, 1 << 20) + syn_u(seed ^ 0xABCDEF12345ULL, row, (1 << 20) + 1) - 1.0f;
  if (kind == 0) return s + 0.1f * noise * 2.449f;
  if (kind == 2) return fminf(fmaxf(floorf(2.0f + 0.6f * s + 1.5f * noise), 0.0f), 4.0f);      // graded relevance 0..4 (lambdarank, BASELINE cfg4)
  if (kind == 3) {                                                                              // 10 ordinal classes, shifted by the first categorical column
    const int ncat = syn_ncat(ncol, kind);
    const float c0 = syn_x(seed, row, ncol - ncat, ncol, kind);
    const float shift = (static_cast<int>(c0) % 3) - 1.0f;
    return fminf(fmaxf(floorf(5.0f + 0.7f * s + 1.2f * shift + 1.5f * noise), 0.0f), 9.0f);
  }
  const float p = 1.0f / (1.0f + __expf(-s));
  return syn_u(seed ^ 0x55AA55AA55ULL, row, 1 << 21) < p ? 1.0f : 0.0f;
}
__global__ void k_syn_fill(float* x, float* label, long long row_start, int nrow, int ncol, unsigned long long seed, int kind) {
  const long long total = static_cast<long long>(nrow) * ncol;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total; e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = e / ncol;
    const int c = static_cast<int>(e % ncol);
    x[e] = syn_x(seed, row_start + r, c, ncol, kind);
    if (c == 0 && label) label[r] = syn_label(seed, row_start + r, ncol, kind);
  }
}
__global__ void k_syn_rows(const int* rows, int nrows, int ncol, unsigned long long seed, int kind, double* out, float* label) {
  const long long total = static_cast<long long>(nrows) * ncol;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total; e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(e / ncol), c = static_cast<int>(e % ncol);
    out[e] = static_cast<double>(syn_x(seed, rows[i], c, ncol, kind));
    if (c == 0 && label) label[i] = syn_label(seed, rows[i], ncol, kind);
  }
}

extern "C" {
int B200GBM_SyntheticFill(void* dev_x_f32, void* dev_label_f32, int64_t row_start, int32_t nrow, int32_t ncol, uint64_t seed, int kind) {
  API_BEGIN();
  EnsureDevice();
  k_syn_fill<<<148 * 16, 256>>>(static_cast<float*>(dev_x_f32), static_cast<float*>(dev_label_f32), row_start, nrow, ncol, seed, kind);
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaDeviceSynchronize());
  API_END();
}
int B200GBM_SyntheticRows(const int* rows, int32_t nrows, int32_t ncol, uint64_t seed, int kind, double* host_out, float* host_label_out) {
  API_BEGIN();
  EnsureDevice();
  DevBuf<int> dr; dr.Alloc(nrows);
  DevBuf<double> dx; dx.Alloc(static_cast<size_t>(nrows) * ncol);
  DevBuf<float> dl; dl.Alloc(nrows);
  B200_CUDA(cudaMemcpy(dr.p, rows, sizeof(int) * nrows, cudaMemcpyHostToDevice));
  k_syn_rows<<<148 * 8, 256>>>(dr.p, nrows, ncol, seed, kind, dx.p, dl.p);
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaMemcpy(host_out, dx.p, sizeof(double) * static_cast<size_t>(nrows) * ncol, cudaMemcpyDeviceToHost));
  if (host_label_out) B200_CUDA(cudaMemcpy(host_label_out, dl.p, sizeof(float) * nrows, cudaMemcpyDeviceToHost));
  API_END();
}
int B200GBM_DatasetGetBins(DatasetHandle handle, uint8_t* out_row_major) {
  API_BEGIN();
  EnsureDevice();
  DS(handle)->GetBinsRowMajor(out_row_major);
  API_END();
}
int B200GBM_DatasetGetBins16(DatasetHandle handle, uint16_t* out_row_major) {
  API_BEGIN();
  EnsureDevice();
  DS(handle)->GetBinsRowMajor16(out_row_major);
  API_END();
}
int B200GBM_DatasetGetBinToCat(DatasetHandle handle, int feature, int* out, int* out_len) {
  API_BEGIN();
  const FeatureBins& fb = DS(handle)->mappers.at(feature);
  for (size_t i = 0; i < fb.bin_to_cat.size(); ++i) out[i] = fb.bin_to_cat[i];
  *out_len = static_cast<int>(fb.bin_to_cat.size());
  API_END();
}
int B200GBM_DatasetGetBinsRows(DatasetHandle handle, const int32_t* rows, int32_t nrows, uint16_t* out) {
  API_BEGIN();
  EnsureDevice();
  DS(handle)->GetBinsOfRows(rows, nrows, out);
  API_END();
}
int B200GBM_DatasetGetFeatureRange(DatasetHandle handle, int feature, double* out2) {
  API_BEGIN();
  const FeatureBins& fb = DS(handle)->mappers.at(feature);
  out2[0] = fb.min_val; out2[1] = fb.max_val;
  API_END();
}
int B200GBM_DatasetGetFeatureInfo(DatasetHandle handle, int feature, int* out5) {
  API_BEGIN();
  const FeatureBins& fb = DS(handle)->mappers.at(feature);
  out5[0] = fb.num_bin; out5[1] = fb.missing_type; out5[2] = static_cast<int>(fb.default_bin); out5[3] = static_cast<int>(fb.most_freq_bin);
  out5[4] = fb.trivial ? 1 : 0;
  API_END();
}
int B200GBM_DatasetGetUpperBounds(DatasetHandle handle, int feature, double* out, int* out_len) {
  API_BEGIN();
  const FeatureBins& fb = DS(handle)->mappers.at(feature);
  for (size_t i = 0; i < fb.upper.size(); ++i) out[i] = fb.upper[i];
  *out_len = static_cast<int>(fb.upper.size());
  API_END();
}
int B200GBM_DatasetGetIngestMs(DatasetHandle handle, double* out_ms) {
  API_BEGIN();
  *out_ms = DS(handle)->ingest_ms;
  API_END();
}
int B200GBM_DatasetHistogram(DatasetHandle handle, const float* grad, const float* hess, const int32_t* idx, int32_t cnt, double* out) {
  API_BEGIN();
  DS(handle)->Histogram(grad, hess, idx, cnt, out);
  API_END();
}
int B200GBM_BoosterSetProfile(BoosterHandle handle, int profile_hist) {
  API_BEGIN();
  BS(handle)->profile_hist = profile_hist != 0;
  API_END();
}
int B200GBM_BoosterGetTiming(BoosterHandle handle, double* out6, int reset) {
  API_BEGIN();
  Booster* b = BS(handle);
  out6[0] = b->timing.hist_ms; out6[1] = b->timing.total_ms; out6[2] = static_cast<double>(b->timing.hist_rows);
  out6[3] = static_cast<double>(b->timing.hist_launches); out6[4] = static_cast<double>(b->timing.launches); out6[5] = b->iter;
  if (reset) b->timing = Booster::Timing();
  API_END();
}
int B200GBM_BoosterPredictForMatDevice(BoosterHandle handle, const void* data, int data_type, int64_t nrow, int32_t ncol, int predict_type,
                                       int start_iteration, int num_iteration, int64_t* out_len, double* out_result, double* elapsed_ms) {
  API_BEGIN();
  Booster* b = BS(handle);
  *out_len = b->PredictBatch(data, data_type, nrow, ncol, predict_type, start_iteration, num_iteration, out_result);
  if (elapsed_ms) *elapsed_ms = b->last_predict_ms;
  API_END();
}
int B200GBM_BoosterGetInfo(BoosterHandle handle, int* out4) {
  API_BEGIN();
  BS(handle)->GetInfo(out4);
  API_END();
}
int B200GBM_BoosterGetMemoryInfo(BoosterHandle handle, int64_t* out2) {
  API_BEGIN();
  BS(handle)->GetMemoryInfo(out2);
  API_END();
}
int B200GBM_BoosterGetScores(BoosterHandle handle, int data_idx, double* out) {
  API_BEGIN();
  BS(handle)->GetRawScores(data_idx, out);
  API_END();
}
int B200GBM_BoosterGetGradients(BoosterHandle handle, float* out_grad, float* out_hess) {
  API_BEGIN();
  BS(handle)->GetGradients(out_grad, out_hess);
  API_END();
}
}  // extern "C"
