// Evaluation metrics on the device (LGBM_BoosterGetEval, reference call sites TrainUtils.scala:125-151 and
// LightGBMBooster.scala:296-310).  Round 1 downloaded all K*n fp64 scores and looped on one host thread (0.8 GB per call at 100M rows);
// here every metric is a reduction over the device-resident scores and only a handful of doubles cross PCIe.
//   point-wise losses  [UPSTREAM regression_metric.hpp / binary_metric.hpp / multiclass_metric.hpp / xentropy_metric.hpp]:
//                      k_metric_pointwise -> per-block partial sums -> k_metric_finish (fixed summation order: reproducible)
//   auc                [UPSTREAM binary_metric.hpp AUCMetric]: radix sort by score (cub, library code off the training path), prefix sums of
//                      the positive / negative weights, one term per group of tied scores
//   ndcg@k / map@k     [UPSTREAM rank_metric.hpp, dcg_calculator.cpp, map_metric.hpp]: one block per query, stable rank by counting
#pragma once
#include <cub/cub.cuh>
#include <cuda_runtime.h>

#include <cstdint>

namespace b200gbm {

enum MetricKind {
  kMetL2 = 0, kMetL1, kMetHuber, kMetFair, kMetPoisson, kMetGamma, kMetTweedie, kMetQuantile, kMetMape, kMetBinLogloss, kMetBinError,
  kMetMultiLogloss, kMetMultiError, kMetXent, kMetGammaDeviance
};
struct MetricParams {
  int kind, K, ova, pad;
  double alpha, fair_c, rho, sigmoid;
};

// loss of one row; r[] = raw scores of the row's K classes
__device__ __forceinline__ double d_point_loss(const MetricParams& mp, const double* __restrict__ score, size_t n, size_t i, double lab) {
  const double eps = 1e-15;
  double s0 = score[i];
  switch (mp.kind) {
    case kMetL2: { const double d = s0 - lab; return d * d; }
    case kMetL1: return fabs(s0 - lab);
    case kMetHuber: { const double d = s0 - lab; return fabs(d) <= mp.alpha ? 0.5 * d * d : mp.alpha * (fabs(d) - 0.5 * mp.alpha); }
    case kMetFair: { const double x = fabs(s0 - lab), c = mp.fair_c; return c * x - c * c * log(1.0 + x / c); }
    case kMetPoisson: { double sc = exp(s0); sc = fmax(sc, 1e-10); return sc - lab * log(sc); }
    case kMetGamma: {
      const double sc = exp(s0), theta = -1.0 / sc, b = -(-theta > 0 ? log(-theta) : -INFINITY);
      const double ll = lab > 0 ? log(lab) : -INFINITY, cc = ll - ll;      // psi = 1: (1/psi) log(label/psi) - log(label) - lgamma(1/psi)
      return -((lab * theta - b) + cc);
    }
    case kMetGammaDeviance: { const double sc = exp(s0), tmp = lab / (sc + 1e-9); return tmp - (tmp > 0 ? log(tmp) : -INFINITY) - 1; }
    case kMetTweedie: {
      double sc = fmax(exp(s0), 1e-10);
      const double rho = mp.rho;
      return -lab * exp((1 - rho) * log(sc)) / (1 - rho) + exp((2 - rho) * log(sc)) / (2 - rho);
    }
    case kMetQuantile: { const double delta = lab - s0; return delta < 0 ? (mp.alpha - 1.0) * delta : mp.alpha * delta; }
    case kMetMape: return fabs(lab - s0) / fmax(1.0, fabs(lab));
    case kMetBinLogloss: case kMetBinError: {
      const double p = 1.0 / (1.0 + exp(-mp.sigmoid * s0));
      if (mp.kind == kMetBinError) return ((p <= 0.5) == (lab > 0)) ? 1.0 : 0.0;
      const double pl = lab > 0 ? p : 1.0 - p;
      return pl > eps ? -log(pl) : -log(eps);
    }
    case kMetXent: {
      const double p = 1.0 / (1.0 + exp(-s0));
      const double a = lab * (p > 1e-12 ? log(p) : log(1e-12)), b = (1.0 - lab) * (1.0 - p > 1e-12 ? log(1.0 - p) : log(1e-12));
      return -(a + b);
    }
    case kMetMultiLogloss: case kMetMultiError: {
      // probabilities by the objective's ConvertOutput: softmax, or a sigmoid per class for multiclassova
      const int K = mp.K, l = static_cast<int>(lab);
      double pl = 0.0;
      int larger = 0;
      if (mp.ova) {
        pl = 1.0 / (1.0 + exp(-mp.sigmoid * score[static_cast<size_t>(l) * n + i]));
        if (mp.kind == kMetMultiError)
          for (int k = 0; k < K; ++k) larger += (1.0 / (1.0 + exp(-mp.sigmoid * score[static_cast<size_t>(k) * n + i]))) >= pl;
      } else {
        double mx = s0;
        for (int k = 1; k < K; ++k) mx = fmax(mx, score[static_cast<size_t>(k) * n + i]);
        double sum = 0;
        for (int k = 0; k < K; ++k) sum += exp(score[static_cast<size_t>(k) * n + i] - mx);
        pl = exp(score[static_cast<size_t>(l) * n + i] - mx) / sum;
        if (mp.kind == kMetMultiError)
          for (int k = 0; k < K; ++k) larger += (exp(score[static_cast<size_t>(k) * n + i] - mx) / sum) >= pl;
      }
      if (mp.kind == kMetMultiError) return larger > 1 ? 1.0 : 0.0;
      return pl > eps ? -log(pl) : -log(eps);
    }
  }
  return 0.0;
}

constexpr int kMetricBlock = 256;
__device__ __forceinline__ void d_block_sum2(double& a, double& b, double* sm /*[2*8]*/) {
  for (int o = 16; o; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sm[warp] = a; sm[8 + warp] = b; }
  __syncthreads();
  if (threadIdx.x == 0) { a = 0; b = 0; for (int w = 0; w < kMetricBlock / 32; ++w) { a += sm[w]; b += sm[8 + w]; } }
}
__global__ void __launch_bounds__(kMetricBlock)
k_metric_pointwise(const double* __restrict__ score, const float* __restrict__ label, const float* __restrict__ weight, int n, MetricParams mp,
                   double* __restrict__ partial) {
  __shared__ double sm[16];
  double loss = 0, sw = 0;
  // contiguous row ranges per block and a fixed thread stride: the summation order does not depend on the grid schedule
  const long long per = (static_cast<long long>(n) + gridDim.x - 1) / gridDim.x;
  const long long r0 = per * blockIdx.x, r1 = min(r0 + per, static_cast<long long>(n));
  for (long long i = r0 + threadIdx.x; i < r1; i += kMetricBlock) {
    const double w = weight ? static_cast<double>(weight[i]) : 1.0;
    loss += d_point_loss(mp, score, static_cast<size_t>(n), static_cast<size_t>(i), static_cast<double>(label[i])) * w;
    sw += w;
  }
  d_block_sum2(loss, sw, sm);
  if (threadIdx.x == 0) { partial[2 * blockIdx.x] = loss; partial[2 * blockIdx.x + 1] = sw; }
}
// out[c] = sum over blocks of partial[b * stride + c], c < stride <= 32: one warp, lane = column, sequential over blocks
__global__ void k_metric_finish(const double* __restrict__ partial, int blocks, int stride, double* __restrict__ out) {
  const int c = threadIdx.x;
  if (c >= stride) return;
  double s = 0;
  for (int b = 0; b < blocks; ++b) s += partial[static_cast<size_t>(b) * stride + c];
  out[c] = s;
}

// ---------------------------------------------------------------- AUC
__device__ __forceinline__ unsigned long long d_sortable(double v) {
  unsigned long long b = static_cast<unsigned long long>(__double_as_longlong(v));
  return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}
__global__ void k_auc_keys(const double* __restrict__ score, int n, unsigned long long* __restrict__ keys, int* __restrict__ rows) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { keys[i] = d_sortable(score[i]); rows[i] = i; }
}
// sorted position i (descending score): weights of the row split by class, and the head marker of its tie group
__global__ void k_auc_weights(const unsigned long long* __restrict__ keys, const int* __restrict__ rows, const float* __restrict__ label,
                              const float* __restrict__ weight, int n, double* __restrict__ wpos, double* __restrict__ wneg, int* __restrict__ head) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int r = rows[i];
    const double w = weight ? static_cast<double>(weight[r]) : 1.0;
    const bool pos = label[r] > 0;
    wpos[i] = pos ? w : 0.0; wneg[i] = pos ? 0.0 : w;
    head[i] = (i == 0 || keys[i] != keys[i - 1]) ? i : 0;
  }
}
// one term per tie group, taken at the group's last position t: neg_g * (pos_g / 2 + positives ranked strictly above)
__global__ void __launch_bounds__(kMetricBlock)
k_auc_terms(const unsigned long long* __restrict__ keys, const int* __restrict__ start, const double* __restrict__ ppos, const double* __restrict__ pneg,
            int n, double* __restrict__ partial) {
  __shared__ double sm[16];
  double acc = 0, unused = 0;
  const long long per = (static_cast<long long>(n) + gridDim.x - 1) / gridDim.x;
  const long long r0 = per * blockIdx.x, r1 = min(r0 + per, static_cast<long long>(n));
  for (long long t = r0 + threadIdx.x; t < r1; t += kMetricBlock) {
    if (t != n - 1 && keys[t] == keys[t + 1]) continue;
    const int s = start[t];
    const double before_p = s > 0 ? ppos[s - 1] : 0.0, before_n = s > 0 ? pneg[s - 1] : 0.0;
    const double pos_g = ppos[t] - before_p, neg_g = pneg[t] - before_n;
    acc += neg_g * (pos_g * 0.5 + before_p);
  }
  d_block_sum2(acc, unused, sm);
  if (threadIdx.x == 0) { partial[2 * blockIdx.x] = acc; partial[2 * blockIdx.x + 1] = 0.0; }
}

// ---------------------------------------------------------------- ndcg@k / map@k : one block per query
// out partial[q_block][2 * nk]: ndcg sums then map sums for the nk cut-offs (ks ascending as the reference sorts eval_at)
constexpr int kMaxEvalAt = 16;
struct RankEvalParams { int nk; int ks[kMaxEvalAt]; int want_ndcg, want_map; };
// dynamic shared memory of k_metric_rank: score, sorted label, label and relevance flag per document, plus the label histogram
inline size_t RankMetricSmem(int max_q, int num_gain) {
  return static_cast<size_t>(max_q) * (8 + 4 + 4 + 1) + static_cast<size_t>(num_gain) * 4;
}
__global__ void __launch_bounds__(128)
k_metric_rank(const double* __restrict__ score, const float* __restrict__ label, const int* __restrict__ qb, int nq, const double* __restrict__ label_gain,
              int num_gain, const double* __restrict__ discount, RankEvalParams rp, int max_q, double* __restrict__ partial) {
  extern __shared__ unsigned char rk_smem[];                     // RankMetricSmem(max_q, num_gain) bytes
  double* r_score = reinterpret_cast<double*>(rk_smem);          // [max_q] document order
  int* s_lab = reinterpret_cast<int*>(r_score + max_q);          // [max_q] label by sorted position (ndcg: an index of label_gain)
  float* r_lab = reinterpret_cast<float*>(s_lab + max_q);        // [max_q] label in document order
  int* s_cnt = reinterpret_cast<int*>(r_lab + max_q);            // [num_gain] label value histogram
  unsigned char* s_rel = reinterpret_cast<unsigned char*>(s_cnt + num_gain);     // [max_q] relevant for MAP (label > 0.5) by sorted position
  double acc[2 * kMaxEvalAt];
  for (int k = 0; k < 2 * kMaxEvalAt; ++k) acc[k] = 0.0;
  const long long per = (static_cast<long long>(nq) + gridDim.x - 1) / gridDim.x;
  const long long q0 = per * blockIdx.x, q1 = min(q0 + per, static_cast<long long>(nq));
  for (long long q = q0; q < q1; ++q) {
    const int start = qb[q], cnt = qb[q + 1] - start;
    __syncthreads();
    for (int v = threadIdx.x; v < num_gain; v += blockDim.x) s_cnt[v] = 0;
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) { r_score[i] = score[start + i]; r_lab[i] = label[start + i]; }
    __syncthreads();
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
      const double si = r_score[i];
      int rank = 0;
      for (int j = 0; j < cnt; ++j) { const double sj = r_score[j]; rank += (sj > si) || (sj == si && j < i); }
      const int li = static_cast<int>(r_lab[i]);
      s_lab[rank] = li;
      s_rel[rank] = r_lab[i] > 0.5f;
      if (li >= 0 && li < num_gain) atomicAdd(&s_cnt[li], 1);      // ndcg labels are checked on the host; map-only labels may be anything
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      if (rp.want_ndcg) {
        // [UPSTREAM DCGCalculator::CalMaxDCG] then CalDCG, both sequential in position order; the walk consumes s_cnt (reset per query)
        double maxdcg[kMaxEvalAt];
        {
          int top = num_gain - 1, left = 0;
          double cur = 0;
          for (int e = 0; e < rp.nk; ++e) {
            const int ck = min(rp.ks[e], cnt);
            for (int j = left; j < ck; ++j) {
              while (top > 0 && s_cnt[top] <= 0) --top;
              if (top < 0) break;
              cur += discount[j] * label_gain[top];
              --s_cnt[top];
            }
            maxdcg[e] = cur;
            left = ck;
          }
        }
        if (!(maxdcg[0] > 0.0)) {
          for (int e = 0; e < rp.nk; ++e) acc[e] += 1.0;
        } else {
          double cur = 0;
          int left = 0;
          for (int e = 0; e < rp.nk; ++e) {
            const int ck = min(rp.ks[e], cnt);
            for (int j = left; j < ck; ++j) cur += label_gain[s_lab[j]] * discount[j];
            acc[e] += cur * (1.0 / maxdcg[e]);
            left = ck;
          }
        }
      }
      if (rp.want_map) {
        // [UPSTREAM MapMetric::CalMapAtK]
        int npos = 0;
        for (int j = 0; j < cnt; ++j) npos += s_rel[j];
        int num_hit = 0, left = 0;
        double sum_ap = 0;
        for (int e = 0; e < rp.nk; ++e) {
          const int ck = min(rp.ks[e], cnt);
          for (int j = left; j < ck; ++j)
            if (s_rel[j]) { ++num_hit; sum_ap += num_hit / (j + 1.0f); }
          acc[kMaxEvalAt + e] += npos > 0 ? sum_ap / min(npos, ck) : 1.0;
          left = ck;
        }
      }
    }
  }
  if (threadIdx.x == 0)
    for (int k = 0; k < 2 * kMaxEvalAt; ++k) partial[static_cast<size_t>(blockIdx.x) * 2 * kMaxEvalAt + k] = acc[k];
}

}  // namespace b200gbm
