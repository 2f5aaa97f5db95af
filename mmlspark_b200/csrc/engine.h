// b200gbm engine: device dataset, data-parallel network state, booster (GBDT driver + tree learner).
// Everything below the C ABI (include/b200gbm_c_api.h).  One host thread drives one
// (network, dataset, booster) triple, exactly like one Spark task thread in the reference
// (SURVEY.md fact 8): network / device / last-error state are thread_local.
#pragma once
#include <cuda_runtime.h>
#include <nccl.h>

#include <cstdint>
#include <memory>
#include <stdexcept>
#include <map>
#include <string>
#include <vector>

#include "bin_mapper.h"
#include "config.h"
#include "kernels.cuh"
#include "model.h"

namespace b200gbm {

#define B200_CUDA(x)                                                                                      \
  do {                                                                                                    \
    cudaError_t e__ = (x);                                                                                \
    if (e__ != cudaSuccess)                                                                               \
      throw std::runtime_error(std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " + __FILE__ + ":" + std::to_string(__LINE__)); \
  } while (0)
#define B200_NCCL(x)                                                                                      \
  do {                                                                                                    \
    ncclResult_t r__ = (x);                                                                               \
    if (r__ != ncclSuccess)                                                                               \
      throw std::runtime_error(std::string("NCCL error: ") + ncclGetErrorString(r__) + " at " + __FILE__ + ":" + std::to_string(__LINE__)); \
  } while (0)

[[noreturn]] inline void Fatal(const std::string& m) { throw std::runtime_error(m); }

// ---- per-thread device + network state -------------------------------------------------------
struct Network {
  bool active = false;
  int rank = 0, world = 1;
  ncclComm_t comm = nullptr;
};
Network& Net();                 // thread-local
int CurrentDevice();            // thread-local CUDA ordinal (selects on first use)
void SetThreadDevice(int ordinal);
void EnsureDevice();            // cudaSetDevice(CurrentDevice()) + fail loudly when no GPU
void NetworkInit(const char* machines, int local_listen_port, int listen_time_out_sec, int num_machines);
void NetworkFree();
void AllReduceHost(double* v, int n, ncclRedOp_t op, cudaStream_t s);      // small host-value collective; no-op without a network

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() {}
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { Free(); }
  void Alloc(size_t count) {
    Free();
    n = count;
    if (count) B200_CUDA(cudaMalloc(reinterpret_cast<void**>(&p), count * sizeof(T)));
  }
  void Free() { if (p) { cudaFree(p); p = nullptr; } n = 0; }
  void Zero(cudaStream_t s) { if (p) B200_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), s)); }
  void Upload(const T* h, size_t count, cudaStream_t s) { B200_CUDA(cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, s)); }
  void Download(T* h, size_t count, cudaStream_t s) const { B200_CUDA(cudaMemcpyAsync(h, p, count * sizeof(T), cudaMemcpyDeviceToHost, s)); }
};

// ---- dataset -----------------------------------------------------------------------------------
class Dataset {
 public:
  ~Dataset();
  // data: host or device pointer (detected); data_type 0=f32 1=f64; reference != null => reuse its bins
  static Dataset* CreateFromMat(const void* data, int data_type, int nrow, int ncol, int is_row_major, const char* params,
                                const Dataset* reference);
  static Dataset* CreateFromCSR(const void* indptr, int indptr_type, const int32_t* indices, const void* data, int data_type,
                                int64_t nindptr, int64_t nelem, int64_t num_col, const char* params, const Dataset* reference);
  // LightGBM streaming ingestion: bins from a column-wise sample, then row blocks pushed in place
  static Dataset* CreateFromSampledColumn(double** sample_data, int** sample_indices, int ncol, const int* num_per_col,
                                          int num_sample_row, int num_total_row, const char* params);
  void PushRows(const void* data, int data_type, int nrow, int ncol, int start_row);
  void GetBinsRowMajor(uint8_t* out) const;                 // fails when a feature has more than 256 bins
  void GetBinsRowMajor16(uint16_t* out) const;
  void GetBinsOfRows(const int32_t* rows, int nrows, uint16_t* out) const;      // [nrows][num_total_features], gathered on the device
  // K4 on this dataset's bins for the given rows (kernel-level parity entry), fp64 [F][256][2]
  void Histogram(const float* grad, const float* hess, const int32_t* idx, int cnt, double* out) const;
  void SetField(const char* name, const void* data, int n, int type);
  void GetField(const char* name, int* out_len, const void** out_ptr, int* out_type) const;
  void SetFeatureNames(const char** names, int n);

  int device = 0;
  int num_data = 0, num_total_features = 0;
  Config cfg;
  std::vector<FeatureBins> mappers;          // [num_total_features]
  std::vector<int> used;                     // inner -> real
  std::vector<int> inner_of;                 // real -> inner or -1
  std::vector<FeatMeta> meta_host;
  int nf = 0, nf_pad = 0, num_tiles = 0;
  int nfn = 0, nw = 0;                       // inner features [0, nfn) live in uint8 tiles, [nfn, nf) are wide (> 256 bins, uint16 columns)
  size_t hist_pairs = 0;                     // (g,h) pairs of one histogram slot: num_tiles*32*256 for the tiles + the wide features' bins
  std::vector<int> sample_order;             // used features in real-index order -> inner index (ColSampler draws in that order)
  size_t rows_stride = 0;
  DevBuf<uint8_t> bins;                      // [num_tiles][rows_stride][32]
  DevBuf<uint16_t> bins16;                   // [nw][rows_stride]
  std::vector<WideMeta> wide_host;
  DevBuf<WideMeta> wide_meta;
  DevBuf<int> wide_cats;                     // sorted category values of all wide features (slices per WideMeta)
  DevBuf<unsigned short> wide_catbin;        // ... and their bins
  DevBuf<double> wide_ub;                    // bin upper bounds of the wide numerical features (max_bin > 255)
  BinView View() const { return BinView{bins.p, rows_stride, bins16.p, nfn}; }
  DevBuf<FeatMeta> meta;
  DevBuf<double> ub;                         // [nf][256] bin upper bounds (categorical: sorted category values)
  DevBuf<uint8_t> catbin;                    // [nf][256] categorical: bin of the i-th sorted category
  bool has_categorical = false;
  std::vector<float> label, weight;
  std::vector<double> init_score;
  std::vector<int32_t> query_boundaries, group_sizes;
  DevBuf<float> d_label, d_weight;
  DevBuf<int> d_qb;
  std::vector<std::string> feature_names;
  cudaStream_t stream = nullptr;
  double ingest_ms = 0.0;                    // H2D + binning time of the last create (CUDA events)

 private:
  void FindBins(const void* data, bool on_device, int data_type, int is_row_major);
  void FindBinsFromColumns(std::vector<std::vector<double>>* nz, int sample_cnt);
  void BinBlock(const void* data, bool on_device, int data_type, int is_row_major, long long nrow, long long start_row);
  // persistent H2D staging of the host ingestion path (two device chunks, a copy stream, events); released once every row is in
  DevBuf<unsigned char> ingest_buf_[2];
  cudaStream_t ingest_copy_stream_ = nullptr;
  cudaEvent_t ingest_copied_[2] = {nullptr, nullptr}, ingest_binned_[2] = {nullptr, nullptr};
  long long ingest_rows_done_ = 0;
  void ReleaseIngestStaging();
  void UploadMeta();
};

// ---- booster -----------------------------------------------------------------------------------
class Objective;       // objective.cuh

struct ValidSet {
  const Dataset* ds = nullptr;
  DevBuf<double> score;   // [K][n]
};

class Booster {
 public:
  Booster(const Dataset* train, const char* params);      // training booster
  explicit Booster(const std::string& model_text);        // prediction-only booster
  ~Booster();

  bool UpdateOneIter();                                   // returns is_finished
  bool UpdateOneIterCustom(const float* grad, const float* hess);
  void ResetParameter(const char* params);
  void AddValidData(const Dataset* valid);
  void MergeFrom(const Booster* other);
  std::vector<std::string> EvalNames() const;
  std::vector<double> GetEval(int data_idx);
  void ValidateMetrics() const;
  void CheckMetricLabels(const Dataset* ds, const Config& c) const;      // ndcg: labels index label_gain
  void GetPredict(int data_idx, int64_t* out_len, double* out);
  int64_t NumPredict(int data_idx) const;
  void GetRawScores(int data_idx, double* out);
  void GetGradients(float* out_g, float* out_h);         // [K][n] at the current training scores (a test hook)
  // batched GPU prediction over a row-major matrix (host or device pointer); predict_type 0 normal, 1 raw, 2 leaf index.
  // Returns the number of doubles written to `out` (host).  last_predict_ms = kernel time (CUDA events), incl. H2D for host input.
  int64_t PredictBatch(const void* data, int data_type, int64_t nrow, int ncol, int predict_type, int start_iteration, int num_iteration, double* out);
  double last_predict_ms = 0.0;
  void GetInfo(int* out4) const;
  std::string SaveModelToString(int start_iteration, int num_iteration, int importance_type) const;
  std::string DumpModelJson(int start_iteration, int num_iteration) const;

  // instrumentation for bench.py / parity tests (B200GBM_* extensions of the C ABI)
  struct Timing { double hist_ms = 0, total_ms = 0; long long hist_rows = 0; long long hist_launches = 0, launches = 0; };
  Timing timing;
  std::map<std::string, double> split_op_ms_; int split_op_trees_ = 0;      // B200GBM_SPLIT_TIMING debug accounting
  bool profile_hist = false;                              // time K4 with events on the engine stream
  std::vector<double> trace;                              // per split records (see B200GBM_BoosterGetTrace)

  Config cfg;
  HostModel model;
  const Dataset* train = nullptr;
  int K = 1;
  int iter = 0;
  int num_init_iteration = 0;

 private:
  void InitTraining();
  void ComputeGradients();
  bool TrainTrees(const float* custom_g, const float* custom_h);
  void TrainOneTree(int class_id, HostTree* out, bool const_hessian);
  void LaunchPartition(int grid, int last);
  int part_max_blocks_ = 148;
  double BoostFromAverage(int class_id);

  int device_ = 0;
  cudaStream_t stream_ = nullptr;
  bool parallel_ = false;
  std::unique_ptr<Objective> obj_;      // null in a prediction-only booster
  bool has_init_score_ = false;
  double shrinkage_ = 0.1;
  LcgRandom col_rand_{2};               // ColSampler (feature_fraction)
  std::vector<uint8_t> feature_used_host_;
  DevBuf<uint8_t> feature_used_;
  void ResetFeaturesByTree();
  // row subsampling: bagging / GOSS / random forest (SURVEY §8f-3)
  bool is_rf_ = false, is_goss_ = false, bagging_ = false, balanced_bagging_ = false, use_bag_ = false, need_re_bagging_ = false;
  int bag_count_ = 0, bag_blocks_ = 0;
  DevBuf<unsigned> bag_lcg_;            // one LCG state per 1024-row block
  DevBuf<LcgJump> bag_jump_;
  DevBuf<uint8_t> in_bag_;
  DevBuf<int> bag_block_cnt_, bag_idx_, bag_total_;
  std::vector<double> rf_init_scores_;
  void Bagging(int it);
  void ComputeGradientsAt(const double* score);
  // percentile objectives: regression_l1 / quantile / mape renew the leaf outputs after the tree is grown (renew_kernel.cuh)
  DevBuf<unsigned long long> rn_keys_a_, rn_keys_b_;
  DevBuf<unsigned> rn_pos_a_, rn_pos_b_, rn_leaf_of_pos_, rn_leaf_a_, rn_leaf_b_;
  DevBuf<double> rn_res_, rn_cdf_, rn_out_;      // rn_out_: [2][num_leaves] outputs, has-rows flags
  DevBuf<int> rn_row_, rn_seg_;
  DevBuf<unsigned char> rn_tmp_;
  size_t rn_tmp_bytes_ = 0;
  void RenewTreeOutput(int class_id, double rf_pred);
  // DART (SURVEY §8f-3): every trained tree keeps its device blob so dropped trees can be re-applied to the binned data
  bool is_dart_ = false, dart_dropped_this_iter_ = false;
  LcgRandom drop_rand_{4};
  std::vector<int> drop_index_;
  std::vector<double> tree_weight_;
  double sum_weight_ = 0.0;
  std::vector<std::unique_ptr<DevBuf<unsigned char>>> tree_store_;     // [iteration * K + class]
  void DroppingTrees();
  void DartNormalize();
  void AddStoredTree(int iter_index, int class_id, bool to_train, bool to_valid);
  TreeDev RebasedTree(unsigned char* base) const;
  SplitParams sp_{};
  // device state
  DevBuf<double> score_;        // [K][n]
  DevBuf<float> grad_, hess_;   // [K][n]
  DevBuf<int4> qgh_, qord_;     // per-row fixed-point (g,h) words; the same in leaf order for the leaf being built
  DevBuf<int> idx0_, idx1_;
  DevBuf<long long> H_;         // scratch histogram of the current smaller leaf
  DevBuf<long long> pool_;      // [num_leaves] leaf histograms
  size_t slot_elems_ = 0;
  DevBuf<uint8_t> flags_;       // [num_leaves][nf_pad]
  DevBuf<SplitCand> cands_;     // [2][nf_pad]
  DevBuf<LeafState> leaves_;
  DevBuf<TreeCtrl> ctrl_;
  DevBuf<unsigned char> tree_blob_;
  TreeDev tree_dev_{};
  size_t tree_blob_bytes_ = 0;
  unsigned char* tree_host_ = nullptr;   // pinned mirror of tree_blob_
  TreeCtrl* ctrl_host_ = nullptr;        // pinned
  LeafState* leaves_host_ = nullptr;     // pinned
  DevBuf<uint8_t> bins_cols_;      // optional [feature][row] copy of the uint8 tiles for the partition kernel
  size_t cols_stride_ = 0;
  bool cols_tried_ = false;
  void EnsureColumnCopy();
 public:
  void GetMemoryInfo(int64_t* out2);
 private:
  DevBuf<unsigned> part_bits_;
  DevBuf<int> part_chunks_;
  // fused data-parallel reduce (peer memory over NVLink); falls back to NCCL when peers cannot map each other
  bool fused_ = false;
  bool p2p_allreduce_ = false;          // B200GBM_FUSED_REDUCE=2: the per-split histogram all-reduce is k_allreduce_p2p instead of ncclAllReduce
  PeerTables peers_{};
  DevBuf<SplitCand> mailbox_;
  DevBuf<unsigned> peer_flags_;
  DevBuf<int> peer_error_;
  std::vector<void*> ipc_opened_;
  unsigned epoch_ = 0;
  void SetupPeerReduce();
  // flattened forest for PredictBatch
  struct ForestBufs { DevBuf<int> tree_offset, leaf_offset, num_leaves, split_feature, decision_type, left_child, right_child, cat_begin, cat_len; DevBuf<double> threshold, leaf_value, node_count, leaf_count, expected; DevBuf<unsigned> cat_words; size_t trees = 0; int max_depth = 0; };
  std::unique_ptr<ForestBufs> forest_;
  void UploadForest();
  std::vector<ValidSet*> valids_;
  // device-side evaluation scratch (metric_kernels.cuh)
  DevBuf<double> met_partial_, met_out_, auc_wpos_, auc_wneg_, auc_ppos_, auc_pneg_;
  DevBuf<unsigned long long> auc_keys_a_, auc_keys_b_;
  DevBuf<int> auc_rows_a_, auc_rows_b_, auc_head_, auc_start_;
  DevBuf<unsigned char> auc_tmp_;
  int num_sms_ = 148;
  cudaEvent_t ev_a_ = nullptr, ev_b_ = nullptr;
};

}  // namespace b200gbm
