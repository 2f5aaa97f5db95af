// Training objectives: the K1/K2 gradient kernels and class Objective, which owns everything the booster needs to know about the
// loss being minimised (label checks, class counts and weights, init scores, gradient launches, leaf-output renewal).  The booster
// (engine.cu) asks it questions and never compares objective names itself.
//
// Two kinds of objective parameters, kept as they are:
//   * read from the live Config at every gradient launch, so LGBM_BoosterResetParameter changes them between iterations: alpha (huber
//     and the quantile gradient), fair_c, poisson_max_delta_step, tweedie_variance_power, sigmoid, lambdarank_truncation_level and
//     lambdarank_norm.  Objective keeps a reference to the booster's Config for these;
//   * captured when the booster is created and kept for its life: the objective itself (a reset `objective` is ignored), the number
//     of classes (score, gradient and class-weight buffers are sized by it), the quantile renewal alpha (RenewAlpha), the class
//     weights of is_unbalance / scale_pos_weight, label_gain and the range of the lambdarank sigmoid table.
#pragma once
#include <algorithm>
#include <cmath>
#include <functional>
#include <limits>
#include <numeric>
#include <string>
#include <vector>

#include "engine.h"

namespace b200gbm {

// ---------------------------------------------------------------- K1 gradients
// [UPSTREAM RegressionL2loss::GetGradients]
__global__ void k_grad_l2(const double* __restrict__ score, const float* __restrict__ label, const float* __restrict__ weight,
                          float* __restrict__ g, float* __restrict__ h, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (weight) { g[i] = static_cast<float>((score[i] - label[i]) * weight[i]); h[i] = weight[i]; }
    else { g[i] = static_cast<float>(score[i] - label[i]); h[i] = 1.0f; }
  }
}
// [UPSTREAM RegressionHuberLoss / FairLoss / PoissonLoss / GammaLoss / TweedieLoss ::GetGradients]; kind 1..5
__global__ void k_grad_regvar(const double* __restrict__ score, const float* __restrict__ label, const float* __restrict__ weight,
                              float* __restrict__ g, float* __restrict__ h, int n, int kind, double alpha, double c, double mds, double rho) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double s = score[i], lab = label[i];
    double gg, hh;
    if (kind == 1) { const double diff = s - lab; gg = fabs(diff) <= alpha ? diff : d_sign(diff) * alpha; hh = 1.0; }
    else if (kind == 2) { const double x = s - lab; gg = c * x / (fabs(x) + c); hh = c * c / ((fabs(x) + c) * (fabs(x) + c)); }
    else if (kind == 3) { gg = exp(s) - lab; hh = exp(s + mds); }
    else if (kind == 4) { gg = 1.0 - lab * exp(-s); hh = lab * exp(-s); }
    else { gg = -lab * exp((1 - rho) * s) + exp((2 - rho) * s); hh = -lab * (1 - rho) * exp((1 - rho) * s) + (2 - rho) * exp((2 - rho) * s); }
    if (weight) { gg *= weight[i]; hh *= weight[i]; }
    g[i] = static_cast<float>(gg); h[i] = static_cast<float>(hh);
  }
}
// [LightGBM RegressionL1loss / RegressionQuantileloss / RegressionMAPELOSS ::GetGradients]; kind 1 l1, 2 quantile, 3 mape
__global__ void k_grad_percentile(const double* __restrict__ score, const float* __restrict__ label, const float* __restrict__ weight,
                                  const float* __restrict__ label_weight, float* __restrict__ g, float* __restrict__ h, int n, int kind, float alpha) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    if (kind == 2) {
      const float delta = static_cast<float>(score[i] - label[i]);
      const float gg = delta >= 0 ? (1.0f - alpha) : -alpha;
      g[i] = weight ? __fmul_rn(gg, weight[i]) : gg;
    } else {
      const double diff = score[i] - label[i];
      const int sgn = (diff > 0.0) - (diff < 0.0);
      if (kind == 1) g[i] = weight ? static_cast<float>(sgn * static_cast<double>(weight[i])) : static_cast<float>(sgn);
      else g[i] = static_cast<float>(sgn * static_cast<double>(label_weight[i]));
    }
    h[i] = weight ? weight[i] : 1.0f;
  }
}
// [UPSTREAM BinaryLogloss::GetGradients]
__global__ void k_grad_binary(const double* __restrict__ score, const float* __restrict__ label, const float* __restrict__ weight,
                              float* __restrict__ g, float* __restrict__ h, int n, double sigmoid, double w_neg, double w_pos) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int is_pos = label[i] > 0;
    const double lab = is_pos ? 1.0 : -1.0;
    const double lw = is_pos ? w_pos : w_neg;
    const double response = -lab * sigmoid / (1.0 + exp(lab * sigmoid * score[i]));
    const double abs_response = fabs(response);
    double gg = response * lw, hh = abs_response * (sigmoid - abs_response) * lw;
    if (weight) { gg *= weight[i]; hh *= weight[i]; }
    g[i] = static_cast<float>(gg); h[i] = static_cast<float>(hh);
  }
}
// [UPSTREAM MulticlassOVA::GetGradients]: class k is a BinaryLogloss on (label == k); cw = per-class {w_neg, w_pos}, need = per-class need_train
__global__ void k_grad_ova(const double* __restrict__ score, const float* __restrict__ label, const float* __restrict__ weight, float* __restrict__ g,
                           float* __restrict__ h, int n, int K, double sigmoid, const double* __restrict__ cw, const uint8_t* __restrict__ need) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int li = static_cast<int>(label[i]);
    for (int k = 0; k < K; ++k) {
      if (!need[k]) continue;
      const size_t id = static_cast<size_t>(n) * k + i;
      const int is_pos = li == k;
      const double lab = is_pos ? 1.0 : -1.0;
      const double lw = cw[2 * k + is_pos];
      const double response = -lab * sigmoid / (1.0 + exp(lab * sigmoid * score[id]));
      const double abs_response = fabs(response);
      double gg = response * lw, hh = abs_response * (sigmoid - abs_response) * lw;
      if (weight) { gg *= weight[i]; hh *= weight[i]; }
      g[id] = static_cast<float>(gg); h[id] = static_cast<float>(hh);
    }
  }
}
// [UPSTREAM CrossEntropy::GetGradients]: labels are probabilities
__global__ void k_grad_xent(const double* __restrict__ score, const float* __restrict__ label, const float* __restrict__ weight, float* __restrict__ g,
                            float* __restrict__ h, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double z = 1.0 / (1.0 + exp(-score[i]));
    double gg = z - label[i], hh = z * (1.0 - z);
    if (weight) { gg *= weight[i]; hh *= weight[i]; }
    g[i] = static_cast<float>(gg); h[i] = static_cast<float>(hh);
  }
}
// [UPSTREAM MulticlassSoftmax::GetGradients]; score/g/h are class-major [K][n]
__global__ void k_grad_softmax(const double* __restrict__ score, const float* __restrict__ label, const float* __restrict__ weight,
                               float* __restrict__ g, float* __restrict__ h, int n, int K, double factor) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    double wmax = score[i];
    for (int k = 1; k < K; ++k) wmax = fmax(wmax, score[static_cast<size_t>(n) * k + i]);
    double wsum = 0;
    for (int k = 0; k < K; ++k) wsum += exp(score[static_cast<size_t>(n) * k + i] - wmax);
    const int lab = static_cast<int>(label[i]);
    const double w = weight ? weight[i] : 1.0;
    for (int k = 0; k < K; ++k) {
      double p = exp(score[static_cast<size_t>(n) * k + i] - wmax) / wsum;
      double gg = (lab == k) ? p - 1.0 : p, hh = factor * p * (1.0 - p);
      if (weight) { gg *= w; hh *= w; }
      g[static_cast<size_t>(n) * k + i] = static_cast<float>(gg);
      h[static_cast<size_t>(n) * k + i] = static_cast<float>(hh);
    }
  }
}

// [UPSTREAM LambdarankNDCG::GetGradientsForOneQuery] — one block per query (K2).
// Sorting: stable rank by score descending (rank counting out of shared memory; queries are ~100 docs).
// Pairs (i, j), i < min(truncation, cnt-1), j > i, are evaluated ONCE, tile by tile over j, by all threads (balanced) into a
// shared-memory matrix M[i][j] = (+-p_lambda, p_hessian) as fp32; then one thread per DOCUMENT adds its entries in the reference's own
// pair order — for document p: (0,p), (1,p) .. (p-1,p), then (p,p+1) .. (p,cnt-1) — with fp32 adds on a score_t accumulator.  No atomics
// (shared-memory float atomicAdd is a CAS loop on sm_100a), no double evaluation (the pair math is fp64 with a software division and a
// table look-up: the first version of this kernel, which evaluated every pair once per side, was FP64-bound at 2.4 ms per 50k queries),
// and every document's lambda / hessian is the same sequence of fp32 additions as the sequential reference: gradients are reproducible
// and equal to the oracle's up to the fp64 rounding of the normalisation factor.  discount[] = 1 / log2(2 + pos) is the host-computed
// table the reference uses (DCGCalculator), not a device log2.
constexpr int kLrThreads = 128;
__host__ __device__ inline int lr_tile(int truncation) {          // j-tile width: M = truncation x (tile + 1) float2 within 48 KB
  int t = (48 * 1024 / 8) / max(truncation, 1) - 1;
  t = min(t, 128);                 // queries are ~100 documents: one tile, and 20 KB per block keeps 8+ blocks per SM
  return max(t & ~31, 32);
}
__global__ void __launch_bounds__(kLrThreads)
k_grad_lambdarank(const double* __restrict__ score, const float* __restrict__ label, const float* __restrict__ weight,
                  const int* __restrict__ qb, int nq, const double* __restrict__ inv_max_dcg, const double* __restrict__ label_gain,
                  const double* __restrict__ discount, const float* __restrict__ sig_table, int sig_bins, double min_in, double max_in,
                  double idx_factor, double sigmoid, int truncation, int norm, float* __restrict__ g, float* __restrict__ h, int max_q) {
  extern __shared__ unsigned char lr_smem[];
  double* r_score = reinterpret_cast<double*>(lr_smem);                  // [max_q] scores in document order
  double* s_score = r_score + max_q;                                     // [max_q] scores by sorted position
  int* s_lab = reinterpret_cast<int*>(s_score + max_q);                  // label by sorted position
  int* s_orig = s_lab + max_q;                                           // document index by sorted position
  float* s_lam = reinterpret_cast<float*>(s_orig + max_q);               // accumulators by sorted position
  float* s_hes = s_lam + max_q;
  float2* M = reinterpret_cast<float2*>(s_hes + max_q);                  // [truncation][T + 1]; 32 * max_q bytes precede it: 8-byte aligned
  __shared__ double s_part[kLrThreads];
  const int T = lr_tile(truncation), TS = T + 1;
  for (int q = blockIdx.x; q < nq; q += gridDim.x) {
    const int start = qb[q], cnt = qb[q + 1] - start;
    __syncthreads();
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) r_score[i] = score[start + i];
    __syncthreads();
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
      const double si = r_score[i];
      int rank = 0;
      for (int j = 0; j < cnt; ++j) {
        const double sj = r_score[j];
        rank += (sj > si) || (sj == si && j < i);
      }
      s_score[rank] = si; s_lab[rank] = static_cast<int>(label[start + i]); s_orig[rank] = i;
      s_lam[rank] = 0.f; s_hes[rank] = 0.f;
    }
    __syncthreads();
    const double imd = inv_max_dcg[q];
    const double best_score = s_score[0];
    int worst_idx = cnt - 1;
    if (worst_idx > 0 && s_score[worst_idx] == kNegInf) worst_idx -= 1;
    const double worst_score = s_score[worst_idx];
    const bool do_div = norm && best_score != worst_score;
    const int teff = min(truncation, cnt - 1);          // pairs exist for i < teff
    double local_sum = 0.0;
    for (int j0 = 0; j0 < cnt; j0 += T) {
      const int tcnt = min(T, cnt - j0);
      // ---- phase A: every pair of the tile once
      for (int e = threadIdx.x; e < teff * tcnt; e += blockDim.x) {
        const int i = e / tcnt, jj = e - i * tcnt, j = j0 + jj;
        float2 m = make_float2(0.f, 0.f);
        if (j > i) {
          const double sci = s_score[i], scj = s_score[j];
          const int li = s_lab[i], lj = s_lab[j];
          if (sci != kNegInf && scj != kNegInf && li != lj) {
            const bool ih = li > lj;                     // position i holds the higher label
            const int hr = ih ? i : j, lr = ih ? j : i;
            const double delta_score = ih ? sci - scj : scj - sci;
            const double dcg_gap = label_gain[ih ? li : lj] - label_gain[ih ? lj : li];
            const double paired_discount = fabs(discount[hr] - discount[lr]);
            double delta = dcg_gap * paired_discount * imd;
            if (do_div) delta /= (0.01f + fabs(delta_score));
            double pl;
            if (delta_score <= min_in) pl = sig_table[0];
            else if (delta_score >= max_in) pl = sig_table[sig_bins - 1];
            else pl = sig_table[static_cast<size_t>((delta_score - min_in) * idx_factor)];
            double ph = pl * (1.0f - pl);
            pl *= -sigmoid * delta;
            ph *= sigmoid * sigmoid * delta;
            local_sum -= 2 * pl;
            const float fl = static_cast<float>(pl);
            m = make_float2(ih ? fl : -fl, static_cast<float>(ph));      // lambdas[i] += m.x, lambdas[j] -= m.x (x - y == x + (-y) exactly)
          }
        }
        M[i * TS + jj] = m;
      }
      __syncthreads();
      // ---- phase B: one thread per document, the reference's order of additions
      for (int p = threadIdx.x; p < cnt; p += blockDim.x) {
        const bool as_j = p >= j0 && p < j0 + tcnt, as_i = p < teff && p + 1 < j0 + tcnt;
        if (!as_j && !as_i) continue;
        float lam = s_lam[p], hes = s_hes[p];
        if (as_j) {
          const int ilim = min(p, teff);
          for (int i = 0; i < ilim; ++i) { const float2 m = M[i * TS + (p - j0)]; lam = __fsub_rn(lam, m.x); hes = __fadd_rn(hes, m.y); }
        }
        if (as_i) {
          for (int j = max(j0, p + 1); j < j0 + tcnt; ++j) { const float2 m = M[p * TS + (j - j0)]; lam = __fadd_rn(lam, m.x); hes = __fadd_rn(hes, m.y); }
        }
        s_lam[p] = lam; s_hes[p] = hes;
      }
      __syncthreads();
    }
    s_part[threadIdx.x] = local_sum;
    __syncthreads();
    double sum_lambdas = 0.0;
    if (norm) for (int t = 0; t < static_cast<int>(blockDim.x); ++t) sum_lambdas += s_part[t];      // fixed order: reproducible
    double nf = 1.0;
    const bool do_norm = norm && sum_lambdas > 0;
    if (do_norm) nf = log2(1 + sum_lambdas) / sum_lambdas;
    for (int r = threadIdx.x; r < cnt; r += blockDim.x) {
      float lam = s_lam[r], hes = s_hes[r];
      if (do_norm) { lam = static_cast<float>(lam * nf); hes = static_cast<float>(hes * nf); }
      const int o = start + s_orig[r];
      if (weight) { lam = static_cast<float>(lam * weight[o]); hes = static_cast<float>(hes * weight[o]); }
      g[o] = lam; h[o] = hes;
    }
  }
}

// ---- host percentiles for the init score of regression_l1 / quantile / mape
// [LightGBM regression_objective.hpp PercentileFun / WeightedPercentileFun, T = label_t]: the alpha percentile counted from the
// top of the descending order d[]: fp = (cnt-1)(1-alpha), interpolation between d[int(fp)] and d[int(fp)+1]; weighted: upper_bound on
// the running weight sum.
static float LabelPercentile(const float* y, int cnt, double alpha) {
  if (cnt <= 1) return y[0];
  const double float_pos = static_cast<double>(cnt - 1) * (1.0 - alpha);
  const int pos = static_cast<int>(float_pos) + 1;
  if (pos < 1) return *std::max_element(y, y + cnt);
  if (pos >= cnt) return *std::min_element(y, y + cnt);
  std::vector<float> v(y, y + cnt);
  std::nth_element(v.begin(), v.begin() + pos, v.end(), std::greater<float>());      // v[pos] = (pos+1)-th largest, larger ones before it
  const float v2 = v[pos], v1 = *std::min_element(v.begin(), v.begin() + pos);
  return static_cast<float>(v1 - (v1 - v2) * (float_pos - (pos - 1)));
}
static float LabelWeightedPercentile(const float* y, const float* w, int cnt, double alpha) {
  if (cnt <= 1) return y[0];
  std::vector<int> order(cnt);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return y[a] < y[b]; });
  std::vector<double> cdf(cnt);
  cdf[0] = w[order[0]];
  for (int i = 1; i < cnt; ++i) cdf[i] = cdf[i - 1] + w[order[i]];
  const double threshold = cdf[cnt - 1] * alpha;
  size_t pos = std::upper_bound(cdf.begin(), cdf.end(), threshold) - cdf.begin();
  pos = std::min(pos, static_cast<size_t>(cnt - 1));
  if (pos == 0 || pos == static_cast<size_t>(cnt - 1)) return y[order[pos]];
  const float v1 = y[order[pos - 1]], v2 = y[order[pos]];
  if (cdf[pos + 1] - cdf[pos] >= 1.0f) return static_cast<float>((threshold - cdf[pos]) / (cdf[pos + 1] - cdf[pos]) * (v2 - v1) + v1);
  return v2;
}

// ---- ranking labels (lambdarank objective, ndcg metric)
// label_gain, or LightGBM's default 2^i - 1 for the labels 0..30
static std::vector<double> RankLabelGain(const Config& cfg) {
  std::vector<double> lg = cfg.label_gain;
  if (lg.empty()) { lg.push_back(0.0); for (int i = 1; i < 31; ++i) lg.push_back(static_cast<double>((1 << i) - 1)); }
  return lg;
}
// [LightGBM DCGCalculator::CheckLabel] a ranking label indexes label_gain: an integer in [0, num_gain)
static void CheckRankLabels(const std::vector<float>& label, size_t num_gain) {
  for (const float l : label) {
    if (std::fabs(l - static_cast<float>(static_cast<int>(l))) > 1e-15f)
      Fatal("label should be int type (met " + std::to_string(l) + ") for ranking task,\nfor the gain of label, please set the label_gain parameter");
    if (!(l >= 0)) Fatal("Label should be non-negative (met " + std::to_string(l) + ") for ranking task");
    if (static_cast<size_t>(l) >= num_gain)
      Fatal("Label " + std::to_string(static_cast<size_t>(l)) + " is not less than the number of label mappings (" + std::to_string(num_gain) + ")");
  }
}

// dynamic shared memory of k_grad_lambdarank: per-document arrays + the pair matrix of one j-tile
static size_t LambdarankSmem(int max_q, int truncation) {
  return static_cast<size_t>(max_q) * (8 + 8 + 4 + 4 + 4 + 4) + 8 + static_cast<size_t>(truncation) * (lr_tile(truncation) + 1) * 8;
}

class Objective {
 public:
  // Parses the objective name; fails on an unknown one and on a quantile alpha outside (0, 1)
  Objective(const Config& cfg, const Dataset* train) : cfg_(cfg), train_(train) {
    static const std::pair<const char*, Kind> kNames[] = {
        {"regression", kRegression}, {"huber", kHuber}, {"fair", kFair}, {"poisson", kPoisson}, {"gamma", kGamma}, {"tweedie", kTweedie},
        {"regression_l1", kL1}, {"quantile", kQuantile}, {"mape", kMape}, {"binary", kBinary}, {"multiclass", kMulticlass},
        {"multiclassova", kMulticlassOva}, {"cross_entropy", kCrossEntropy}, {"lambdarank", kLambdarank}};
    bool known = false;
    for (const auto& kn : kNames) if (cfg.objective == kn.first) { kind_ = kn.second; known = true; }
    if (kind_ == kQuantile && !(cfg.alpha > 0.0 && cfg.alpha < 1.0)) Fatal("Check failed: alpha_ > 0 && alpha_ < 1");
    renew_alpha_ = kind_ == kQuantile ? static_cast<double>(static_cast<float>(cfg.alpha)) : 0.5;     // quantile keeps alpha as score_t
    if (!known) Fatal("Unknown/unsupported objective type name: " + cfg.objective);
    num_model_ = (kind_ == kMulticlass || kind_ == kMulticlassOva) ? cfg.num_class : 1;
  }

  // The configuration / dataset checks LightGBM runs before training starts
  void CheckData() const {
    if (train_->label.empty()) Fatal("label should not be empty for training");
    if ((kind_ == kMulticlass || kind_ == kMulticlassOva) && num_model_ < 2) Fatal("Number of classes should be specified and greater than 1 for multiclass training");
    if (kind_ == kLambdarank && train_->query_boundaries.empty()) Fatal("Ranking tasks require query information");
  }

  int NumModelPerIteration() const { return num_model_; }
  bool IsBinary() const { return kind_ == kBinary; }
  bool IsOva() const { return kind_ == kMulticlassOva; }
  std::string ToString() const {      // the objective line of the model text
    if (kind_ == kBinary) return "binary sigmoid:" + Config::Num(cfg_.sigmoid);
    if (kind_ == kMulticlass) return "multiclass num_class:" + std::to_string(num_model_);
    if (kind_ == kMulticlassOva) return "multiclassova num_class:" + std::to_string(num_model_) + " sigmoid:" + Config::Num(cfg_.sigmoid);
    return cfg_.objective;
  }

  // Label statistics, class weights and device tables; the class counts are global (AllReduceHost) in distributed training
  void Init(cudaStream_t stream, int num_sms) {
    stream_ = stream;
    num_sms_ = num_sms;
    parallel_ = Net().active && Net().world > 1;
    const Dataset* train = train_;
    const int n = train->num_data;
    const int K = NumModelPerIteration();
    class_need_train_.assign(K, true);
    switch (kind_) {
      case kRegression:
        const_hessian_ = train->weight.empty();
        break;
      case kHuber: case kFair:
        break;
      case kPoisson: case kGamma: case kTweedie:
        for (int i = 0; i < n; ++i) if (train->label[i] < 0) Fatal("[" + cfg_.objective + "]: at least one target label is negative");
        break;
      case kL1: case kQuantile: case kMape:
        const_hessian_ = train->weight.empty();
        if (kind_ == kMape) {       // [LightGBM RegressionMAPELOSS::Init] label_weight = 1 / max(1, |label|) (* weight)
          label_weight_host_.resize(n);
          for (int i = 0; i < n; ++i) {
            label_weight_host_[i] = 1.0f / std::max(1.0f, std::fabs(train->label[i]));
            if (!train->weight.empty()) label_weight_host_[i] *= train->weight[i];
          }
          label_weight_.Alloc(n); label_weight_.Upload(label_weight_host_.data(), n, stream_);
        }
        break;
      case kBinary: {
        double cnt[2] = {0, 0};
        for (int i = 0; i < n; ++i) cnt[train->label[i] > 0 ? 1 : 0] += 1;
        AllReduceHost(cnt, 2, ncclSum, stream_);          // global class counts (R14)
        binary_need_train_ = !(cnt[0] == 0 || cnt[1] == 0);
        binary_w_[0] = binary_w_[1] = 1.0;
        if (cfg_.is_unbalance && cnt[0] > 0 && cnt[1] > 0) {
          if (cnt[1] > cnt[0]) { binary_w_[1] = 1.0; binary_w_[0] = cnt[1] / cnt[0]; }
          else { binary_w_[1] = cnt[0] / cnt[1]; binary_w_[0] = 1.0; }
        }
        binary_w_[1] *= cfg_.scale_pos_weight;
        class_need_train_[0] = binary_need_train_;
        break;
      }
      case kMulticlass: {
        class_init_probs_.assign(K + 1, 0.0);
        for (int i = 0; i < n; ++i) {
          int l = static_cast<int>(train->label[i]);
          if (l < 0 || l >= K) Fatal("Label must be in [0, " + std::to_string(K) + "), but found " + std::to_string(l) + " in label");
          double w = train->weight.empty() ? 1.0 : train->weight[i];
          class_init_probs_[l] += w; class_init_probs_[K] += w;
        }
        AllReduceHost(class_init_probs_.data(), K + 1, ncclSum, stream_);
        for (int k = 0; k < K; ++k) {
          class_init_probs_[k] /= class_init_probs_[K];
          class_need_train_[k] = !(std::fabs(class_init_probs_[k]) <= kEps || std::fabs(class_init_probs_[k]) >= 1.0 - kEps);
        }
        break;
      }
      case kMulticlassOva: {       // [UPSTREAM MulticlassOVA::Init]: one BinaryLogloss::Init per class on (label == k)
        std::vector<double> cnt(K, 0.0);
        for (int i = 0; i < n; ++i) {
          const int l = static_cast<int>(train->label[i]);
          if (l < 0 || l >= K) Fatal("Label must be in [0, " + std::to_string(K) + "), but found " + std::to_string(l) + " in label");
          cnt[l] += 1;
        }
        double total = n;
        AllReduceHost(cnt.data(), K, ncclSum, stream_);
        AllReduceHost(&total, 1, ncclSum, stream_);
        std::vector<double> cw(2 * static_cast<size_t>(K), 1.0);
        std::vector<uint8_t> need(K, 1);
        for (int k = 0; k < K; ++k) {
          const double pos = cnt[k], neg = total - cnt[k];
          class_need_train_[k] = !(pos == 0 || neg == 0);
          need[k] = class_need_train_[k] ? 1 : 0;
          if (cfg_.is_unbalance && pos > 0 && neg > 0) {
            if (pos > neg) { cw[2 * k + 1] = 1.0; cw[2 * k] = pos / neg; }
            else { cw[2 * k + 1] = neg / pos; cw[2 * k] = 1.0; }
          }
          cw[2 * k + 1] *= cfg_.scale_pos_weight;
        }
        ova_w_.Alloc(cw.size()); ova_w_.Upload(cw.data(), cw.size(), stream_);
        ova_need_.Alloc(K); ova_need_.Upload(need.data(), K, stream_);
        B200_CUDA(cudaStreamSynchronize(stream_));
        break;
      }
      case kCrossEntropy:      // [UPSTREAM CrossEntropy::Init]
        for (int i = 0; i < n; ++i)
          if (!(train->label[i] >= 0.0f && train->label[i] <= 1.0f)) Fatal("[cross_entropy]: does not tolerate label " + std::to_string(train->label[i]) + " outside [0, 1]");
        if (!train->weight.empty()) {
          double sw = 0;
          for (int i = 0; i < n; ++i) { if (train->weight[i] < 0) Fatal("[cross_entropy]: at least one weight is negative"); sw += train->weight[i]; }
          if (!(sw > 0)) Fatal("[cross_entropy]: sum of weights is zero");
        }
        break;
      case kLambdarank: {
        const std::vector<double> lg = RankLabelGain(cfg_);
        CheckRankLabels(train->label, lg.size());
        const int nq = static_cast<int>(train->query_boundaries.size()) - 1;
        std::vector<double> imd(nq);
        lr_max_q_ = 0;
        for (int q = 0; q < nq; ++q) {
          const int s = train->query_boundaries[q], cnt = train->query_boundaries[q + 1] - s;
          lr_max_q_ = std::max(lr_max_q_, cnt);
          std::vector<int> label_cnt(lg.size(), 0);
          for (int i = 0; i < cnt; ++i) ++label_cnt[static_cast<int>(train->label[s + i])];
          int top = static_cast<int>(lg.size()) - 1, k = std::min(cfg_.lambdarank_truncation_level, cnt);
          double m = 0;
          for (int j = 0; j < k; ++j) {
            while (top > 0 && label_cnt[top] <= 0) --top;
            m += (1.0 / std::log2(2.0 + j)) * lg[top];      // discount_[j] * label_gain_[top] as [UPSTREAM DCGCalculator::CalMaxDCGAtK]
            --label_cnt[top];
          }
          imd[q] = m > 0.0 ? 1.0 / m : m;
        }
        lr_inv_max_dcg_.Alloc(nq); lr_inv_max_dcg_.Upload(imd.data(), nq, stream_);
        lr_label_gain_.Alloc(lg.size()); lr_label_gain_.Upload(lg.data(), lg.size(), stream_);
        const size_t bins_n = kLrSigBins;
        lr_min_in_ = -50.0 / cfg_.sigmoid / 2; lr_max_in_ = 50.0 / cfg_.sigmoid / 2;
        lr_idx_factor_ = bins_n / (lr_max_in_ - lr_min_in_);
        std::vector<float> tab(bins_n);
        for (size_t i = 0; i < bins_n; ++i) tab[i] = static_cast<float>(1.0 / (1.0 + std::exp((i / lr_idx_factor_ + lr_min_in_) * cfg_.sigmoid)));
        lr_sig_table_.Alloc(bins_n); lr_sig_table_.Upload(tab.data(), bins_n, stream_);
        std::vector<double> disc(static_cast<size_t>(std::max(lr_max_q_, 1)) + 1);       // [UPSTREAM DCGCalculator::Init] discount table, host log2
        for (size_t i = 0; i < disc.size(); ++i) disc[i] = 1.0 / std::log2(2.0 + i);
        lr_discount_.Alloc(disc.size()); lr_discount_.Upload(disc.data(), disc.size(), stream_);
        B200_CUDA(cudaStreamSynchronize(stream_));
        if (cfg_.lambdarank_truncation_level < 1 || cfg_.lambdarank_truncation_level > 180) Fatal("lambdarank_truncation_level should be in [1, 180]");
        size_t smem = LambdarankSmem(lr_max_q_, cfg_.lambdarank_truncation_level);
        if (smem > 200 * 1024) Fatal("a query group is too large for the lambdarank kernel");
        B200_CUDA(cudaFuncSetAttribute(k_grad_lambdarank, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(std::max<size_t>(smem, 1024))));
        break;
      }
    }
  }

  // Before the booster's overrides: GOSS and custom gradients never have a constant hessian
  bool IsConstantHessian() const { return const_hessian_; }
  bool ClassNeedTrain(int k) const { return class_need_train_[k]; }

  // [LightGBM ObjectiveFunction::BoostFromScore] init score of class k; averaged over the ranks in distributed training
  double BoostFromScore(int k) {
    const Dataset* train = train_;
    const int n = train->num_data;
    switch (kind_) {
      case kRegression: case kHuber: case kFair: case kPoisson: case kGamma: case kTweedie: {
        double suml = 0, sumw = 0;
        if (!train->weight.empty()) for (int i = 0; i < n; ++i) { suml += static_cast<double>(train->label[i]) * train->weight[i]; sumw += train->weight[i]; }
        else { sumw = n; for (int i = 0; i < n; ++i) suml += train->label[i]; }
        double v = suml / sumw;
        if (kind_ == kPoisson || kind_ == kGamma || kind_ == kTweedie) v = v > 0 ? std::log(v) : -std::numeric_limits<double>::infinity();
        if (parallel_) { AllReduceHost(&v, 1, ncclSum, stream_); v /= Net().world; }   // GlobalSyncUpByMean (R11)
        return v;
      }
      case kL1: case kQuantile: case kMape: {
        const float* y = train->label.data();
        double v;
        if (kind_ == kMape) v = LabelWeightedPercentile(y, label_weight_host_.data(), n, 0.5);
        else if (train->weight.empty()) v = LabelPercentile(y, n, renew_alpha_);
        else v = LabelWeightedPercentile(y, train->weight.data(), n, renew_alpha_);
        if (parallel_) { AllReduceHost(&v, 1, ncclSum, stream_); v /= Net().world; }   // GlobalSyncUpByMean
        return v;
      }
      case kMulticlass:
        return std::log(std::max(kEps, class_init_probs_[k]));
      case kBinary: case kMulticlassOva: case kCrossEntropy: {
        // BinaryLogloss::BoostFromScore on (label > 0) / on (label == k) for class k of OVA / CrossEntropy::BoostFromScore on the label
        double s[2] = {0, 0};
        for (int i = 0; i < n; ++i) {
          const double w = train->weight.empty() ? 1.0 : static_cast<double>(train->weight[i]);
          const double y = kind_ == kBinary ? (train->label[i] > 0 ? 1.0 : 0.0)
                         : kind_ == kMulticlassOva ? (static_cast<int>(train->label[i]) == k ? 1.0 : 0.0) : static_cast<double>(train->label[i]);
          s[0] += y * w; s[1] += w;
        }
        AllReduceHost(s, 2, ncclSum, stream_);
        double pavg = s[0] / s[1];
        pavg = std::min(pavg, 1.0 - kEps);
        pavg = std::max(pavg, kEps);
        return std::log(pavg / (1.0 - pavg)) / (kind_ == kCrossEntropy ? 1.0 : cfg_.sigmoid);
      }
      case kLambdarank:
        break;
    }
    return 0.0;
  }

  // K1/K2: gradients and hessians of every class at `score` ([K][n]) into g, h ([K][n]); one launch at most
  void GetGradients(const double* score, float* g, float* h) const {
    const Dataset* train = train_;
    const int n = train->num_data;
    const int grid = num_sms_ * 8;
    const float* w = train->weight.empty() ? nullptr : train->d_weight.p;
    const float* y = train->d_label.p;
    switch (kind_) {
      case kRegression:
        k_grad_l2<<<grid, 256, 0, stream_>>>(score, y, w, g, h, n);
        break;
      case kL1: case kQuantile: case kMape:
        k_grad_percentile<<<grid, 256, 0, stream_>>>(score, y, w, kind_ == kMape ? label_weight_.p : nullptr, g, h, n, kind_ - kL1 + 1,
                                                     static_cast<float>(cfg_.alpha));
        break;
      case kHuber: case kFair: case kPoisson: case kGamma: case kTweedie:
        k_grad_regvar<<<grid, 256, 0, stream_>>>(score, y, w, g, h, n, kind_ - kHuber + 1, cfg_.alpha, cfg_.fair_c, cfg_.poisson_max_delta_step,
                                                 cfg_.tweedie_variance_power);
        break;
      case kBinary:
        if (binary_need_train_) k_grad_binary<<<grid, 256, 0, stream_>>>(score, y, w, g, h, n, cfg_.sigmoid, binary_w_[0], binary_w_[1]);
        break;
      case kMulticlass: {
        const int K = NumModelPerIteration();
        k_grad_softmax<<<grid, 256, 0, stream_>>>(score, y, w, g, h, n, K, static_cast<double>(K) / (K - 1.0));
        break;
      }
      case kMulticlassOva:
        k_grad_ova<<<grid, 256, 0, stream_>>>(score, y, w, g, h, n, NumModelPerIteration(), cfg_.sigmoid, ova_w_.p, ova_need_.p);
        break;
      case kCrossEntropy:
        k_grad_xent<<<grid, 256, 0, stream_>>>(score, y, w, g, h, n);
        break;
      case kLambdarank: {
        const int nq = static_cast<int>(train->query_boundaries.size()) - 1;
        size_t smem = std::max<size_t>(LambdarankSmem(lr_max_q_, cfg_.lambdarank_truncation_level), 1024);
        k_grad_lambdarank<<<std::min(nq, num_sms_ * 16), kLrThreads, smem, stream_>>>(
            score, y, w, train->d_qb.p, nq, lr_inv_max_dcg_.p, lr_label_gain_.p, lr_discount_.p, lr_sig_table_.p, kLrSigBins, lr_min_in_,
            lr_max_in_, lr_idx_factor_, cfg_.sigmoid, cfg_.lambdarank_truncation_level, cfg_.lambdarank_norm ? 1 : 0, g, h, lr_max_q_);
        break;
      }
    }
  }

  // regression_l1 / quantile / mape: the tree's leaf outputs are replaced by the alpha percentile of the leaf's residuals
  // (renew_kernel.cuh), weighted by RenewWeights() when that is not null
  bool IsRenewTreeOutput() const { return kind_ == kL1 || kind_ == kQuantile || kind_ == kMape; }
  double RenewAlpha() const { return renew_alpha_; }
  const float* RenewWeights() const { return kind_ == kMape ? label_weight_.p : (train_->weight.empty() ? nullptr : train_->d_weight.p); }

 private:
  // huber..tweedie and regression_l1..mape are consecutive, in the order of the `kind` argument of k_grad_regvar / k_grad_percentile
  enum Kind { kRegression, kHuber, kFair, kPoisson, kGamma, kTweedie, kL1, kQuantile, kMape, kBinary, kMulticlass, kMulticlassOva, kCrossEntropy,
              kLambdarank };
  static constexpr int kLrSigBins = 1024 * 1024;      // entries of the lambdarank sigmoid table
  const Config& cfg_;          // the booster's: LGBM_BoosterResetParameter changes what the gradient launches read
  const Dataset* train_;
  Kind kind_ = kRegression;
  int num_model_ = 1;           // trees per iteration: num_class for multiclass / multiclassova
  cudaStream_t stream_ = nullptr;
  int num_sms_ = 148;
  bool parallel_ = false;
  bool const_hessian_ = false;
  std::vector<bool> class_need_train_;
  // binary: class weights {w_neg, w_pos} and whether both classes occur
  double binary_w_[2] = {1.0, 1.0};
  bool binary_need_train_ = true;
  std::vector<double> class_init_probs_;      // multiclass: weighted class frequencies, [K] = total weight
  DevBuf<double> ova_w_;                      // multiclassova: [K][2] {w_neg, w_pos}
  DevBuf<uint8_t> ova_need_;                  // multiclassova: [K] class has both positives and negatives
  double renew_alpha_ = 0.5;                  // percentile of the leaf renewal and of the init score
  std::vector<float> label_weight_host_;      // mape: 1 / max(1, |label|) (* weight)
  DevBuf<float> label_weight_;
  // lambdarank
  DevBuf<double> lr_inv_max_dcg_, lr_label_gain_, lr_discount_;
  DevBuf<float> lr_sig_table_;
  double lr_min_in_ = -50, lr_max_in_ = 50, lr_idx_factor_ = 0;
  int lr_max_q_ = 0;
};

}  // namespace b200gbm
