// sm_100a kernels of the b200gbm training engine other than K4 (hist_kernel.cuh) and the K1/K2 gradients (objective.cuh).
// Kernel numbering follows SURVEY.md §2.5.  Everything a tree needs lives in device memory
// (leaf table, control block, tree arrays) so the host enqueues a whole tree without a sync.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "hist_kernel.cuh"

namespace b200gbm {

constexpr double kEpsD = 1e-15;
#define kNegInf (-__longlong_as_double(0x7ff0000000000000LL))   /* -inf, usable in device code */

struct FeatMeta {          // per inner (used) feature
  int num_bin;
  int missing_type;        // 0 none, 2 NaN
  int default_bin;
  int offset;              // 1 iff most_freq_bin == 0  ([UPSTREAM] storage convention, affects NaN forward scan)
  int real_index;
  int is_categorical;      // bins are category ranks; splits are bin bitsets
  int num_sorted_cats;     // categorical: entries of the sorted category table (ub row = categories, catbin row = their bins)
  int hist_off;            // first (g,h) pair of the feature in a histogram slot: u * 256 for a tile feature, beyond the tiles for a wide one
};

// "Wide" features: more than 256 bins.  LightGBM does not cap a categorical feature at max_bin — it keeps categories until 99 % of the
// sampled mass is covered (BinMapper::FindBin) — so a 10^3..10^5-cardinality column (BASELINE.json configs[4]) needs thousands of bins.
// They live outside the uint8 feature tiles: one uint16 column per feature, their own histogram kernel (k4_hist_wide) and scan
// (k_scan_wide); inner index = nfn + w.  A categorical split on one sends at most max_cat_threshold bins left, carried as a bin list.
constexpr int kWideHistSeg = 8192;       // bins one k4_hist_wide CTA accumulates: 4 planes x 8192 x 4 B = 128 KB of shared memory
constexpr int kWideMaxBins = 16384;      // per feature (k_scan_wide sorts (ctr, bin) keys in 160 KB of shared memory); more fails loudly
constexpr int kCatListMax = 64;          // >= max_cat_threshold (default 32) when wide features exist
struct WideMeta {
  int num_bin, hist_off, cat_off, num_cats;      // hist_off in (g,h) pairs; categorical: slice of the sorted category table (cat_off, num_cats);
                                                 // numerical (max_bin > 255): cat_off = first entry of the feature's upper bounds in the wide ub table
  int default_bin, missing_type, real_index, is_cat;
  int offset, pad0, pad1, pad2;                  // offset: 1 iff most_freq_bin == 0 (as FeatMeta::offset)
};
struct BinView {                         // where a row's bin of inner feature u is stored
  const uint8_t* bins; size_t rows_stride; const uint16_t* bins16; int nfn;
  __device__ __forceinline__ unsigned at(int u, size_t row) const {
    return u < nfn ? bins[(static_cast<size_t>(u >> 5) * rows_stride + row) * 32 + (u & 31)] : bins16[static_cast<size_t>(u - nfn) * rows_stride + row];
  }
};

struct SplitParams {
  double l1, l2, max_delta_step, min_gain_to_split, min_sum_hessian;
  int min_data_in_leaf, max_depth, num_leaves, parallel;
  int nf, nf_pad, num_tiles, nfn;                              // nfn: features stored in uint8 tiles; [nfn, nf) are wide
  double cat_l2, cat_smooth;                                   // categorical split search ([UPSTREAM] defaults 10, 10)
  int max_cat_threshold, max_cat_to_onehot, min_data_per_group, pad3;   // 32, 4, 100
};

struct SplitCand {         // best threshold of one (leaf, feature)
  double gain;             // best_gain - min_gain_shift, or -inf
  double left_g, left_h;   // best_sum_left_gradient / _hessian (hessian still carries +kEpsilon)
  int threshold, left_count, default_left, feature;   // feature = inner index
  double l2_extra;         // cat_l2 for a many-vs-many categorical split (leaf outputs use lambda_l2 + l2_extra)
  unsigned cat_bits[8];    // categorical: bins that go LEFT
  int is_cat, cat_list_len;
  unsigned short cat_list[kCatListMax];      // wide categorical feature: the bins that go LEFT (cat_bits unused)
};

struct LeafBest {
  double gain;
  double left_g, left_h, right_g, right_h;   // sums as stored in SplitInfo (epsilon removed)
  double left_out, right_out;
  int feature, threshold, default_left, left_count, right_count, is_cat;
  unsigned cat_bits[8];
  int cat_list_len, pad;
  unsigned short cat_list[kCatListMax];
};

struct LeafState {
  int begin, count, buf, depth;
  int global_count, identity, hist_slot, parent_node;
  double sum_g, sum_h;
  LeafBest best;
};

struct TreeCtrl {
  int num_leaves, left_leaf, right_leaf, smaller, larger, go, finished, split_leaf;
  int split_feature, split_threshold, split_default_left, split_missing_type, split_num_bin, new_leaf, pending, pad;
  int part_begin, part_count, part_buf, part_identity, part_left_total, smaller_rows, round, split_is_cat;
  unsigned split_cat_bits[8];
  HistWork hist_work;
  unsigned absmax_bits[2];     // max|g|, max|h| as float bits (non-negative floats order like uints)
  int exp_g, exp_h;            // fixed-point exponents: q = rint(x * 2^exp)
  double inv_g, inv_h;         // hist value -> real value
  long long root_q[4];         // sum q_g, sum q_h, local rows, unused  (allreduced)
  long long trace_rows;        // sum of rows scanned by K4 this tree (for the roofline byte model)
  unsigned scan_ticket;        // blocks of k_scan that finished this round (the last one runs the pick step)
  int q_side;                  // (unused since the fused partition kernel decides the side itself)
  unsigned part_barrier;       // k_partition: grid-barrier arrive counter (reset by its last block)
  unsigned part_ticket;        // k_partition: finished-block ticket (the last block runs the next round's controller)
  unsigned part_next[2];       // k_partition: next chunk of phase 1 / phase 3 (dynamic hand-out; reset by its last block)
  int split_wide;              // wide index (inner feature - nfn) of the split feature, or -1
  int split_cat_list_len;
  unsigned short split_cat_list[kCatListMax];
};

struct TreeDev {               // SoA tree under construction (sizes: num_leaves / num_leaves-1)
  int* left_child; int* right_child; int* split_feature_inner; int* threshold_bin; int* decision_type;
  float* split_gain; double* leaf_value; double* leaf_weight; int* leaf_count; double* internal_value;
  double* internal_weight; int* internal_count; int* leaf_parent; int* leaf_depth; int* num_leaves;
  unsigned* cat_bits;          // [num_leaves-1][8] inner (bin) bitset of categorical nodes
  unsigned short* cat_list;    // [num_leaves-1][kCatListMax] bins going left at a categorical node on a wide feature
  int* cat_list_len;           // [num_leaves-1] 0 for every other node
};

// ---------------------------------------------------------------- helpers
__device__ __forceinline__ double d_sign(double x) { return (x > 0.0) - (x < 0.0); }
__device__ __forceinline__ double d_threshold_l1(double s, double l1) {
  double r = fmax(0.0, fabs(s) - l1);
  return d_sign(s) * r;
}
__device__ __forceinline__ double d_calc_output(double g, double h, const SplitParams& p) {
  double ret = (p.l1 > 0) ? -d_threshold_l1(g, p.l1) / (h + p.l2) : -g / (h + p.l2);
  if (p.max_delta_step > 0 && fabs(ret) > p.max_delta_step) ret = d_sign(ret) * p.max_delta_step;
  return ret;
}
// NOT inlined on purpose: the split scan evaluates it ~40 times per lane; inlined and unrolled (each call holds a software fp64 division)
// k_scan grew to 15.8K SASS instructions that every warp ran through once, and ncu showed 55 % of its stall samples in stall_no_inst
// (instruction-cache misses), 39 us per launch.  As a function its body is fetched once.
__device__ __noinline__ double d_leaf_gain(double g, double h, const SplitParams& p) {
  if (!(p.max_delta_step > 0)) {
    if (p.l1 > 0) { double sg = d_threshold_l1(g, p.l1); return (sg * sg) / (h + p.l2); }
    return (g * g) / (h + p.l2);
  }
  double out = d_calc_output(g, h, p);
  double sg = (p.l1 > 0) ? d_threshold_l1(g, p.l1) : g;
  return -(2.0 * sg * out + (h + p.l2) * out * out);
}

// ---------------------------------------------------------------- binning (dataset creation)
// One warp per row-of-a-tile: lane = feature of the tile.  Upper bounds of the tile's 32 features sit
// in shared memory ([32][256] doubles = 64 KB).  ValueToBin: lower-bound search `value <= ub[m]`.
template <typename T>
__global__ void __launch_bounds__(256)
k_bin_rows(const T* __restrict__ X, long long nrow, int ncol, int row_major, long long ld, const FeatMeta* __restrict__ meta,
           const double* __restrict__ ub, const uint8_t* __restrict__ catbin, int nf, uint8_t* __restrict__ bins, long long rows_stride,
           long long row_offset) {
  extern __shared__ double s_ub[];   // [256 bins][32 lanes]: lane l always hits bank pair 2l -> no conflicts beyond the 64-bit 2-phase
  const int tile = blockIdx.y;
  for (int e = threadIdx.x; e < 32 * 256; e += blockDim.x) {
    int f = tile * 32 + (e >> 8);
    s_ub[(e & 255) * 32 + (e >> 8)] = f < nf ? ub[static_cast<size_t>(f) * 256 + (e & 255)] : 0.0;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int u = tile * 32 + lane;
  FeatMeta m;
  m.num_bin = 1; m.missing_type = 0; m.real_index = 0; m.is_categorical = 0; m.num_sorted_cats = 0;
  if (u < nf) m = meta[u];
  const double* myub = s_ub + lane;
  for (long long r = blockIdx.x * 8LL + warp; r < nrow; r += gridDim.x * 8LL) {
    unsigned bin = 0;
    if (u < nf) {
      double v = row_major ? static_cast<double>(X[r * ld + m.real_index]) : static_cast<double>(X[static_cast<long long>(m.real_index) * ld + r]);
      if (m.is_categorical) {     // category -> bin: binary search in the sorted category table; NaN / negative / unseen -> bin 0
        if (!isnan(v)) {
          const int iv = static_cast<int>(v);
          if (iv >= 0) {
            int lo = 0, hi = m.num_sorted_cats;
            while (lo < hi) { int mid = (lo + hi) >> 1; if (static_cast<int>(myub[mid * 32]) < iv) lo = mid + 1; else hi = mid; }
            if (lo < m.num_sorted_cats && static_cast<int>(myub[lo * 32]) == iv) bin = catbin[static_cast<size_t>(u) * 256 + lo];
          }
        }
      } else {
        if (isnan(v)) {
          if (m.missing_type == 2) bin = m.num_bin - 1; else v = 0.0;
        }
        if (!isnan(v)) {
          int lo = 0, hi = m.num_bin - 1 - (m.missing_type == 2 ? 1 : 0);
          while (lo < hi) {
            int mid = (hi + lo - 1) / 2;
            if (v <= myub[mid * 32]) hi = mid; else lo = mid + 1;
          }
          bin = lo;
        }
      }
    }
    bins[(static_cast<size_t>(tile) * rows_stride + row_offset + r) * 32 + lane] = static_cast<uint8_t>(bin);
  }
}

// ---------------------------------------------------------------- quantisation + root sums (K3)
__global__ void k_absmax(const float* __restrict__ g, const float* __restrict__ h, int n, TreeCtrl* ctrl) {
  float mg = 0.f, mh = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    mg = fmaxf(mg, fabsf(g[i])); mh = fmaxf(mh, fabsf(h[i]));
  }
  for (int o = 16; o; o >>= 1) { mg = fmaxf(mg, __shfl_xor_sync(0xffffffffu, mg, o)); mh = fmaxf(mh, __shfl_xor_sync(0xffffffffu, mh, o)); }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&ctrl->absmax_bits[0], __float_as_uint(mg));
    atomicMax(&ctrl->absmax_bits[1], __float_as_uint(mh));
  }
}
// exponents so that |q| < 2^35:  e = 34 - ilogb(max)
__global__ void k_set_scale(TreeCtrl* ctrl, int const_hessian, double hess_const) {
  float mg = __uint_as_float(ctrl->absmax_bits[0]), mh = __uint_as_float(ctrl->absmax_bits[1]);
  int eg = (mg > 0.f && isfinite(mg)) ? 34 - ilogbf(mg) : 0;
  int eh = (mh > 0.f && isfinite(mh)) ? 34 - ilogbf(mh) : 0;
  eg = max(min(eg, 1000), -1000); eh = max(min(eh, 1000), -1000);
  ctrl->exp_g = eg; ctrl->exp_h = eh;
  ctrl->inv_g = ldexp(1.0, -eg);
  ctrl->inv_h = const_hessian ? hess_const : ldexp(1.0, -eh);
  ctrl->root_q[0] = 0; ctrl->root_q[1] = 0; ctrl->root_q[2] = 0; ctrl->root_q[3] = 0;
}
__global__ void __launch_bounds__(256)
k_quantize(const float* __restrict__ g, const float* __restrict__ h, int n, int4* __restrict__ qgh, TreeCtrl* ctrl, int const_hessian,
           const uint8_t* __restrict__ in_bag, int bag_count) {
  const int eg = ctrl->exp_g, eh = ctrl->exp_h;
  long long sg = 0, sh = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    long long qg = __double2ll_rn(ldexp(static_cast<double>(g[i]), eg));
    int4 q;
    q.x = static_cast<int>(qg >> kLoBits); q.y = static_cast<int>(qg & ((1LL << kLoBits) - 1));
    long long qh;
    if (const_hessian) { qh = 1; q.z = 1; q.w = 0; }
    else { qh = __double2ll_rn(ldexp(static_cast<double>(h[i]), eh)); q.z = static_cast<int>(qh >> kLoBits); q.w = static_cast<int>(qh & ((1LL << kLoBits) - 1)); }
    qgh[i] = q;
    if (!in_bag || in_bag[i]) { sg += qg; sh += qh; }       // root sums run over the in-bag rows only
  }
  for (int o = 16; o; o >>= 1) { sg += __shfl_xor_sync(0xffffffffu, sg, o); sh += __shfl_xor_sync(0xffffffffu, sh, o); }
  __shared__ long long s_g[8], s_h[8];
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { s_g[warp] = sg; s_h[warp] = sh; }
  __syncthreads();
  if (threadIdx.x == 0) {
    long long a = 0, b = 0;
    for (int w = 0; w < 8; ++w) { a += s_g[w]; b += s_h[w]; }
    atomicAdd(reinterpret_cast<unsigned long long*>(&ctrl->root_q[0]), static_cast<unsigned long long>(a));
    atomicAdd(reinterpret_cast<unsigned long long*>(&ctrl->root_q[1]), static_cast<unsigned long long>(b));
    if (blockIdx.x == 0) atomicAdd(reinterpret_cast<unsigned long long*>(&ctrl->root_q[2]), static_cast<unsigned long long>(in_bag ? bag_count : n));
  }
}

// ---------------------------------------------------------------- tree init / round controller
__global__ void __launch_bounds__(256)
k_tree_init(TreeCtrl* ctrl, LeafState* leaves, TreeDev tree, uint8_t* flags, SplitParams p, int n_local, const uint8_t* feature_used,
            int root_is_bag) {
  for (int u = threadIdx.x; u < p.nf_pad; u += blockDim.x) flags[u] = (u < p.nf && (!feature_used || feature_used[u])) ? 1 : 0;
  for (int l = threadIdx.x; l < p.num_leaves; l += blockDim.x) {
    leaves[l].best.gain = kNegInf; leaves[l].best.feature = -1;
    tree.leaf_parent[l] = -1; tree.leaf_depth[l] = 0; tree.leaf_value[l] = 0; tree.leaf_weight[l] = 0; tree.leaf_count[l] = 0;
  }
  if (threadIdx.x == 0) {
    LeafState& r = leaves[0];
    r.begin = 0; r.count = n_local; r.buf = 0; r.depth = 0; r.identity = root_is_bag ? 0 : 1; r.hist_slot = 0; r.parent_node = -1;
    r.global_count = static_cast<int>(ctrl->root_q[2]);
    r.sum_g = static_cast<double>(ctrl->root_q[0]) * ctrl->inv_g;
    r.sum_h = static_cast<double>(ctrl->root_q[1]) * ctrl->inv_h;
    ctrl->num_leaves = 1; ctrl->left_leaf = 0; ctrl->right_leaf = -1; ctrl->smaller = 0; ctrl->larger = -1;
    ctrl->go = 0; ctrl->finished = 0; ctrl->split_leaf = -1; ctrl->pending = 0; ctrl->round = 0; ctrl->trace_rows = 0;
    *tree.num_leaves = 1;
  }
}

// Applies the split chosen in the previous round (Tree::Split + leaf bookkeeping, using the TRUE row
// counts in the serial learner and the hessian-reconstructed global counts in the data-parallel one),
// then runs SerialTreeLearner::BeforeFindBestSplit for the coming round.  One block; thread 0 does the bookkeeping, all threads copy
// the inherited is_splittable flags.  Runs as its own kernel before a tree's first round and, for every later round, in the last
// block of the partition kernel of the previous round (k_partition) — one launch and one kernel boundary less per split.
__device__ __forceinline__ void
d_round_ctl(TreeCtrl* ctrl, LeafState* leaves, const TreeDev& tree, uint8_t* flags, const FeatMeta* __restrict__ meta, const SplitParams& p, int last,
            int* s_copy) {       // s_copy: 2 shared ints
  if (threadIdx.x == 0) {
    s_copy[0] = -1; s_copy[1] = -1;
    if (ctrl->pending) {
      ctrl->pending = 0;
      const int leaf = ctrl->split_leaf, nl = ctrl->new_leaf;
      LeafState& L = leaves[leaf];
      LeafState& R = leaves[nl];
      LeafBest b = L.best;
      // written by another block of the same kernel when this runs as the tail of k_partition: read through L2
      const int true_left = __ldcg(&ctrl->part_left_total), true_right = ctrl->part_count - true_left;
      if (!p.parallel) { b.left_count = true_left; b.right_count = true_right; }
      // Tree::Split
      const int node = ctrl->num_leaves - 1;
      const int parent = tree.leaf_parent[leaf];
      if (parent >= 0) {
        if (tree.left_child[parent] == ~leaf) tree.left_child[parent] = node; else tree.right_child[parent] = node;
      }
      tree.split_feature_inner[node] = b.feature;
      tree.split_gain[node] = static_cast<float>(b.gain + p.min_gain_to_split);
      tree.left_child[node] = ~leaf; tree.right_child[node] = ~nl;
      tree.leaf_parent[leaf] = node; tree.leaf_parent[nl] = node;
      tree.internal_weight[node] = tree.leaf_weight[leaf];
      tree.internal_value[node] = tree.leaf_value[leaf];
      tree.internal_count[node] = b.left_count + b.right_count;
      tree.leaf_value[leaf] = isnan(b.left_out) ? 0.0 : b.left_out;
      tree.leaf_weight[leaf] = b.left_h; tree.leaf_count[leaf] = b.left_count;
      tree.leaf_value[nl] = isnan(b.right_out) ? 0.0 : b.right_out;
      tree.leaf_weight[nl] = b.right_h; tree.leaf_count[nl] = b.right_count;
      tree.leaf_depth[nl] = tree.leaf_depth[leaf] + 1; tree.leaf_depth[leaf] += 1;
      const FeatMeta fm = meta[b.feature];
      if (b.is_cat) {
        tree.decision_type[node] = 1 | (fm.missing_type << 2);
        tree.threshold_bin[node] = 0;
      } else {
        tree.decision_type[node] = (b.default_left ? 2 : 0) | (fm.missing_type << 2);
        tree.threshold_bin[node] = b.threshold;
      }
      for (int wd = 0; wd < 8; ++wd) tree.cat_bits[node * 8 + wd] = b.is_cat ? b.cat_bits[wd] : 0u;
      tree.cat_list_len[node] = b.is_cat ? b.cat_list_len : 0;
      if (b.is_cat) for (int k = 0; k < b.cat_list_len && k < kCatListMax; ++k) tree.cat_list[node * kCatListMax + k] = b.cat_list[k];
      ctrl->num_leaves += 1; *tree.num_leaves = ctrl->num_leaves;
      // data partition bookkeeping: children live in the other index buffer
      const int dst_buf = L.identity ? 0 : (L.buf ^ 1);
      R.begin = L.begin + true_left; R.count = true_right; R.buf = dst_buf; R.identity = 0; R.depth = L.depth + 1;
      L.count = true_left; L.buf = dst_buf; L.identity = 0; L.depth += 1;
      L.global_count = b.left_count; R.global_count = b.right_count;
      L.sum_g = b.left_g; L.sum_h = b.left_h; R.sum_g = b.right_g; R.sum_h = b.right_h;
      R.hist_slot = nl;
      L.best.gain = kNegInf; L.best.feature = -1; R.best.gain = kNegInf; R.best.feature = -1;
      ctrl->left_leaf = leaf; ctrl->right_leaf = nl;
    }
    ctrl->go = 0; ctrl->smaller = -1; ctrl->larger = -1; ctrl->split_leaf = -1;
    ctrl->hist_work.count = 0; ctrl->part_count = 0;
    if (!ctrl->finished && !last && ctrl->num_leaves < p.num_leaves) {
      const int ll = ctrl->left_leaf, rl = ctrl->right_leaf;
      bool go = true;
      if (p.max_depth > 0 && tree.leaf_depth[ll] >= p.max_depth) go = false;
      const int nl_cnt = leaves[ll].global_count, nr_cnt = rl >= 0 ? leaves[rl].global_count : 0;
      if (go && nr_cnt < p.min_data_in_leaf * 2 && nl_cnt < p.min_data_in_leaf * 2) go = false;
      if (!go) {
        leaves[ll].best.gain = kNegInf;
        if (rl >= 0) leaves[rl].best.gain = kNegInf;
      } else {
        int smaller = ll, larger = -1;
        if (rl >= 0) {
          if (nl_cnt < nr_cnt) { smaller = ll; larger = rl; } else { smaller = rl; larger = ll; }
          // parent's histogram sits in the slot of `ll`; the larger child inherits it
          if (larger == rl) { int t = leaves[ll].hist_slot; leaves[ll].hist_slot = leaves[rl].hist_slot; leaves[rl].hist_slot = t; }
          s_copy[0] = ll; s_copy[1] = rl;
        }
        ctrl->smaller = smaller; ctrl->larger = larger; ctrl->go = 1;
        const LeafState& S = leaves[smaller];
        ctrl->hist_work.begin = S.begin; ctrl->hist_work.count = S.count; ctrl->hist_work.use_idx = S.identity ? 0 : 1;
        ctrl->hist_work.buf = S.buf;       // K4 reads the row list from index buffer `buf`
        ctrl->smaller_rows = S.count;
        ctrl->trace_rows += S.count;
      }
    }
    ctrl->round += 1;
  }
  __syncthreads();
  if (s_copy[0] >= 0)   // children inherit the parent's per-feature is_splittable flags
    for (int u = threadIdx.x; u < p.nf_pad; u += blockDim.x) flags[static_cast<size_t>(s_copy[1]) * p.nf_pad + u] = flags[static_cast<size_t>(s_copy[0]) * p.nf_pad + u];
}
__global__ void __launch_bounds__(256)
k_round_ctl(TreeCtrl* ctrl, LeafState* leaves, TreeDev tree, uint8_t* flags, const FeatMeta* __restrict__ meta, SplitParams p,
            int last) {
  __shared__ int s_copy[2];
  d_round_ctl(ctrl, leaves, tree, flags, meta, p, last, s_copy);
}

// ---------------------------------------------------------------- K5/K6 split scan
// One warp per (which in {smaller, larger}, feature).  Lane l owns bins 8l..8l+7.  All prefix sums are
// exact int64; gains are fp64.  Replaces FeatureHistogram::FindBestThresholdSequentially (+Subtract).
__device__ __forceinline__ long long warp_suffix_excl(long long v, int lane) {   // sum over lanes > lane
  long long inc = v;
  for (int o = 1; o < 32; o <<= 1) { long long t = __shfl_down_sync(0xffffffffu, inc, o); if (lane + o < 32) inc += t; }
  return inc - v;
}
__device__ __forceinline__ long long warp_prefix_excl(long long v, int lane) {   // sum over lanes < lane
  long long inc = v;
  for (int o = 1; o < 32; o <<= 1) { long long t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
  return inc - v;
}

// the per-feature scan shared by k_scan and k_scan_dp: qg/qh = this lane's 8 bins of the (global) histogram
// The bin loops are deliberately NOT unrolled (qg/qh/cnt are then indexed dynamically and live in L1-cached local memory): unrolled, the two
// scan directions alone were ~5K instructions of straight-line fp64 code per warp and the kernel was bound by instruction fetch.
__device__ __forceinline__ void d_scan_feature(const long long (&qg)[8], const long long (&qh)[8], int lane, const FeatMeta m, const LeafState& L,
                                               double inv_g, double inv_h, const SplitParams& p, uint8_t* flag, SplitCand* outp) {
  SplitCand& out = *outp;
  const double sum_g = L.sum_g, sum_h = L.sum_h + 2 * kEpsD;
  const int num_data = L.global_count;
  const double cnt_factor = num_data / sum_h;
  const double min_gain_shift = d_leaf_gain(sum_g, sum_h, p) + p.min_gain_to_split;
  const bool two_way = (m.num_bin > 2 && m.missing_type == 2);
  const int na = two_way ? 1 : 0;

  int cnt[8];
#pragma unroll 1
  for (int j = 0; j < 8; ++j) cnt[j] = static_cast<int>(static_cast<double>(qh[j]) * inv_h * cnt_factor + 0.5);

  // ---- reverse pass: bins num_bin-1-na .. 1, candidate threshold = b-1
  double best_gain = kNegInf, best_lg = 0, best_lh = 0;
  int best_thr = -1, best_lc = 0, best_dl = 1;
  bool any_valid = false;
  {
    const int hi = m.num_bin - 1 - na;
    long long lg = 0, lh = 0, lc = 0;
#pragma unroll 1
    for (int j = 0; j < 8; ++j) { const int b = lane * 8 + j; if (b >= 1 && b <= hi) { lg += qg[j]; lh += qh[j]; lc += cnt[j]; } }
    long long rg = warp_suffix_excl(lg, lane), rh = warp_suffix_excl(lh, lane), rc = warp_suffix_excl(lc, lane);
#pragma unroll 1
    for (int j = 7; j >= 0; --j) {
      const int b = lane * 8 + j;
      if (b < 1 || b > hi) continue;
      rg += qg[j]; rh += qh[j]; rc += cnt[j];
      const double srg = static_cast<double>(rg) * inv_g;
      const double srh = kEpsD + static_cast<double>(rh) * inv_h;
      const int right_count = static_cast<int>(rc);
      if (right_count < p.min_data_in_leaf || srh < p.min_sum_hessian) continue;
      const int left_count = num_data - right_count;
      if (left_count < p.min_data_in_leaf) continue;
      const double slh = sum_h - srh;
      if (slh < p.min_sum_hessian) continue;
      const double slg = sum_g - srg;
      const double gain = d_leaf_gain(slg, slh, p) + d_leaf_gain(srg, srh, p);
      if (gain <= min_gain_shift) continue;
      any_valid = true;
      if (gain > best_gain) { best_gain = gain; best_lg = slg; best_lh = slh; best_thr = b - 1; best_lc = left_count; }
    }
    // warp argmax: higher gain, ties -> higher threshold (first seen in the right-to-left scan)
    for (int o = 16; o; o >>= 1) {
      double og = __shfl_xor_sync(0xffffffffu, best_gain, o);
      int ot = __shfl_xor_sync(0xffffffffu, best_thr, o);
      double olg = __shfl_xor_sync(0xffffffffu, best_lg, o), olh = __shfl_xor_sync(0xffffffffu, best_lh, o);
      int olc = __shfl_xor_sync(0xffffffffu, best_lc, o);
      if (og > best_gain || (og == best_gain && ot > best_thr)) { best_gain = og; best_thr = ot; best_lg = olg; best_lh = olh; best_lc = olc; }
    }
  }
  // ---- forward pass (NaN-as-missing features only): bins 0 .. num_bin-2, threshold = b, NaN goes right
  if (two_way) {
    const int hi = m.num_bin - 2;
    long long ag = 0, ah = 0, ac = 0;     // everything stored except bin 0 (incl. the NaN bin)
    long long lg = 0, lh = 0, lc = 0;
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
      const int b = lane * 8 + j;
      if (b >= 1 && b < m.num_bin) { ag += qg[j]; ah += qh[j]; ac += cnt[j]; }
      if (b >= m.offset && b <= hi) { lg += qg[j]; lh += qh[j]; lc += cnt[j]; }
    }
    for (int o = 16; o; o >>= 1) { ag += __shfl_xor_sync(0xffffffffu, ag, o); ah += __shfl_xor_sync(0xffffffffu, ah, o); ac += __shfl_xor_sync(0xffffffffu, ac, o); }
    long long pg = warp_prefix_excl(lg, lane), ph = warp_prefix_excl(lh, lane), pc = warp_prefix_excl(lc, lane);
    double base_g = 0.0, base_h = kEpsD; int base_c = 0;
    if (m.offset == 1) {   // implicit bin 0 = leaf total - everything stored  [UPSTREAM NA_AS_MISSING && offset==1]
      base_g = sum_g - static_cast<double>(ag) * inv_g;
      base_h = (sum_h - kEpsD) - static_cast<double>(ah) * inv_h;
      base_c = num_data - static_cast<int>(ac);
    }
    double f_gain = kNegInf, f_lg = 0, f_lh = 0; int f_thr = 1 << 30, f_lc = 0;
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
      const int b = lane * 8 + j;
      if (b > hi) continue;
      if (b >= m.offset) { pg += qg[j]; ph += qh[j]; pc += cnt[j]; }
      const double slg = base_g + static_cast<double>(pg) * inv_g;
      const double slh = base_h + static_cast<double>(ph) * inv_h;
      const int left_count = base_c + static_cast<int>(pc);
      if (left_count < p.min_data_in_leaf || slh < p.min_sum_hessian) continue;
      const int right_count = num_data - left_count;
      if (right_count < p.min_data_in_leaf) continue;
      const double srh = sum_h - slh;
      if (srh < p.min_sum_hessian) continue;
      const double srg = sum_g - slg;
      const double gain = d_leaf_gain(slg, slh, p) + d_leaf_gain(srg, srh, p);
      if (gain <= min_gain_shift) continue;
      any_valid = true;
      if (gain > f_gain) { f_gain = gain; f_lg = slg; f_lh = slh; f_thr = b; f_lc = left_count; }
    }
    for (int o = 16; o; o >>= 1) {
      double og = __shfl_xor_sync(0xffffffffu, f_gain, o);
      int ot = __shfl_xor_sync(0xffffffffu, f_thr, o);
      double olg = __shfl_xor_sync(0xffffffffu, f_lg, o), olh = __shfl_xor_sync(0xffffffffu, f_lh, o);
      int olc = __shfl_xor_sync(0xffffffffu, f_lc, o);
      if (og > f_gain || (og == f_gain && ot < f_thr)) { f_gain = og; f_thr = ot; f_lg = olg; f_lh = olh; f_lc = olc; }
    }
    if (f_gain > best_gain) { best_gain = f_gain; best_thr = f_thr; best_lg = f_lg; best_lh = f_lh; best_lc = f_lc; best_dl = 0; }
  } else if (m.missing_type == 2) {
    best_dl = 0;
  }
  any_valid = __any_sync(0xffffffffu, any_valid);
  if (lane == 0) {
    *flag = any_valid ? 1 : 0;
    if (any_valid && best_gain > min_gain_shift) {
      out.gain = best_gain - min_gain_shift; out.left_g = best_lg; out.left_h = best_lh; out.threshold = best_thr;
      out.left_count = best_lc; out.default_left = best_dl;
    }
  }
}

// Categorical split search for one feature by one warp (FeatureHistogram::FindBestThresholdCategoricalInner [UPSTREAM]):
// one-hot when num_bin <= max_cat_to_onehot; otherwise the bins holding >= cat_smooth rows are ranked by g/(h+cat_smooth)
// (stable, ties by bin) and accumulated from both ends, at most max_cat_threshold bins, lambda_l2 += cat_l2.
// ws = this warp's shared scratch: g[256], h[256], ctr[256] doubles + order[256] + used[256] bytes.
__device__ __noinline__ void d_scan_feature_cat(const long long (&qg)[8], const long long (&qh)[8], int lane, const FeatMeta m, const LeafState& L,
                                                   double inv_g, double inv_h, const SplitParams& p, uint8_t* flag, SplitCand* outp, double* ws) {
  SplitCand& out = *outp;
  double* sg = ws; double* sh = ws + 256; double* sc = ws + 512;
  unsigned char* order = reinterpret_cast<unsigned char*>(ws + 768);
  const double sum_g = L.sum_g, sum_h = L.sum_h + 2 * kEpsD;
  const int num_data = L.global_count;
  const double cnt_factor = num_data / sum_h;
  SplitParams pshift = p;
  if (!(p.max_delta_step > 0)) pshift.max_delta_step = 0;
  const double min_gain_shift = d_leaf_gain(sum_g, sum_h, pshift) + p.min_gain_to_split;
  const bool onehot = m.num_bin <= p.max_cat_to_onehot;
  bool any_valid = false;
  double best_gain = kNegInf, best_lg = 0, best_lh = 0;
  int best_t = 0x7fffffff, best_lc = 0;
  unsigned used_mask = 0;      // bit j: my bin j is "used" (enough rows)
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int b = lane * 8 + j;
    const double g = static_cast<double>(qg[j]) * inv_g, h = static_cast<double>(qh[j]) * inv_h;
    sg[b] = g; sh[b] = h;
    const int cnt = static_cast<int>(h * cnt_factor + 0.5);
    const bool in_range = b >= 1 && b < m.num_bin;
    if (onehot) {
      if (in_range && !(cnt < p.min_data_in_leaf || h < p.min_sum_hessian)) {
        const int other = num_data - cnt;
        const double oh = sum_h - h - kEpsD;
        if (other >= p.min_data_in_leaf && oh >= p.min_sum_hessian) {
          const double gain = d_leaf_gain(sum_g - g, oh, p) + d_leaf_gain(g, h + kEpsD, p);
          if (gain > min_gain_shift) {
            any_valid = true;
            if (gain > best_gain) { best_gain = gain; best_t = b; best_lg = g; best_lh = h + kEpsD; best_lc = cnt; }
          }
        }
      }
    } else {
      const bool used = in_range && cnt >= p.cat_smooth;
      if (used) used_mask |= 1u << j;
      sc[b] = g / (h + p.cat_smooth);
    }
  }
  __syncwarp();
  if (onehot) {
    for (int o = 16; o; o >>= 1) {        // first seen = smallest bin wins ties
      const double og = __shfl_xor_sync(0xffffffffu, best_gain, o);
      const int ot = __shfl_xor_sync(0xffffffffu, best_t, o), oc = __shfl_xor_sync(0xffffffffu, best_lc, o);
      const double olg = __shfl_xor_sync(0xffffffffu, best_lg, o), olh = __shfl_xor_sync(0xffffffffu, best_lh, o);
      if (og > best_gain || (og == best_gain && ot < best_t)) { best_gain = og; best_t = ot; best_lg = olg; best_lh = olh; best_lc = oc; }
    }
    any_valid = __any_sync(0xffffffffu, any_valid);
    if (lane == 0) {
      *flag = any_valid ? 1 : 0;
      if (any_valid) {
        out.gain = best_gain - min_gain_shift; out.left_g = best_lg; out.left_h = best_lh; out.threshold = 0; out.left_count = best_lc;
        out.default_left = 0; out.is_cat = 1; out.l2_extra = 0;
        out.cat_bits[best_t >> 5] |= 1u << (best_t & 31);
      }
    }
    return;
  }
  // ---- rank the used bins by ctr (stable): rank = #{used j : ctr_j < ctr_i  or (== and j < i)}.
  // Uniform loop over the bins: sc[bj] / usedb[bj] are broadcast loads, the 8 comparisons of a lane are independent.
  unsigned char* usedb = order + 256;
  int used_bin = 0;
  double ci[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int b = lane * 8 + j;
    const bool u = (used_mask >> j) & 1u;
    usedb[b] = u ? 1 : 0;
    ci[j] = sc[b];
    used_bin += __popc(__ballot_sync(0xffffffffu, u));
  }
  __syncwarp();
  int rank[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) rank[j] = 0;
  for (int bj = 1; bj < m.num_bin; ++bj) {
    if (!usedb[bj]) continue;             // same bj in every lane: no divergence
    const double cj = sc[bj];
#pragma unroll
    for (int j = 0; j < 8; ++j) rank[j] += (cj < ci[j]) || (cj == ci[j] && bj < lane * 8 + j);
  }
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if ((used_mask >> j) & 1u) order[rank[j]] = static_cast<unsigned char>(lane * 8 + j);
  __syncwarp();
  if (lane == 0) {
    SplitParams pc = p;
    pc.l2 += p.cat_l2;
    const int max_num_cat = min(p.max_cat_threshold, (used_bin + 1) / 2);
    int best_i = -1, best_dir = 1;
    for (int d = 0; d < 2; ++d) {
      const int dir = d == 0 ? 1 : -1;
      int pos = d == 0 ? 0 : used_bin - 1;
      int cnt_cur_group = 0, left_count = 0;
      double slg = 0.0, slh = kEpsD;
      for (int i = 0; i < used_bin && i < max_num_cat; ++i) {
        const int t = order[pos];
        pos += dir;
        const double g = sg[t], h = sh[t];
        const int cnt = static_cast<int>(h * cnt_factor + 0.5);
        slg += g; slh += h; left_count += cnt; cnt_cur_group += cnt;
        if (left_count < p.min_data_in_leaf || slh < p.min_sum_hessian) continue;
        const int right_count = num_data - left_count;
        if (right_count < p.min_data_in_leaf || right_count < p.min_data_per_group) break;
        const double srh = sum_h - slh;
        if (srh < p.min_sum_hessian) break;
        if (cnt_cur_group < p.min_data_per_group) continue;
        cnt_cur_group = 0;
        const double gain = d_leaf_gain(slg, slh, pc) + d_leaf_gain(sum_g - slg, srh, pc);
        if (gain <= min_gain_shift) continue;
        any_valid = true;
        if (gain > best_gain) { best_gain = gain; best_lg = slg; best_lh = slh; best_lc = left_count; best_i = i; best_dir = dir; }
      }
    }
    *flag = any_valid ? 1 : 0;
    if (any_valid) {
      out.gain = best_gain - min_gain_shift; out.left_g = best_lg; out.left_h = best_lh; out.threshold = 0; out.left_count = best_lc;
      out.default_left = 0; out.is_cat = 1; out.l2_extra = p.cat_l2;
      for (int i = 0; i <= best_i; ++i) {
        const int t = best_dir == 1 ? order[i] : order[used_bin - 1 - i];
        out.cat_bits[t >> 5] |= 1u << (t & 31);
      }
    }
  }
}

__device__ __forceinline__ void d_choose_leaf(TreeCtrl* ctrl, LeafState* leaves, const FeatMeta* __restrict__ meta, const SplitParams& p, int lane) {
  double bg = kNegInf; int bf = 0x7fffffff, bl = 0x7fffffff;
  const int nl = ctrl->num_leaves;
  for (int l = lane; l < nl; l += 32) {
    const double g = leaves[l].best.gain;
    const int fi = leaves[l].best.feature;
    const int f = fi < 0 ? 0x7fffffff : meta[fi].real_index;
    if (g > bg || (g == bg && (f < bf || (f == bf && l < bl)))) { bg = g; bf = f; bl = l; }
  }
  for (int o = 16; o; o >>= 1) {
    const double og = __shfl_xor_sync(0xffffffffu, bg, o);
    const int of = __shfl_xor_sync(0xffffffffu, bf, o), ol = __shfl_xor_sync(0xffffffffu, bl, o);
    if (og > bg || (og == bg && (of < bf || (of == bf && ol < bl)))) { bg = og; bf = of; bl = ol; }
  }
  if (lane != 0) return;
  const int best_leaf = bl == 0x7fffffff ? 0 : bl;
  const LeafBest& b = leaves[best_leaf].best;
  if (!(b.gain > 0.0) || ctrl->num_leaves >= p.num_leaves) {
    ctrl->finished = 1; ctrl->split_leaf = -1; ctrl->part_count = 0;
  } else {
    const LeafState& L = leaves[best_leaf];
    const FeatMeta fm = meta[b.feature];
    ctrl->split_leaf = best_leaf; ctrl->new_leaf = ctrl->num_leaves; ctrl->pending = 1;
    ctrl->split_feature = b.feature; ctrl->split_threshold = b.threshold; ctrl->split_default_left = b.default_left;
    ctrl->split_missing_type = fm.missing_type; ctrl->split_num_bin = fm.num_bin;
    ctrl->split_is_cat = b.is_cat;
    for (int wd = 0; wd < 8; ++wd) ctrl->split_cat_bits[wd] = b.cat_bits[wd];
    ctrl->split_wide = b.feature >= p.nfn ? b.feature - p.nfn : -1;
    ctrl->split_cat_list_len = b.cat_list_len;
    for (int k = 0; k < b.cat_list_len && k < kCatListMax; ++k) ctrl->split_cat_list[k] = b.cat_list[k];
    ctrl->part_begin = L.begin; ctrl->part_count = L.count; ctrl->part_buf = L.buf; ctrl->part_identity = L.identity;
    ctrl->part_left_total = 0;
  }
}

// candidates are written by other blocks of the same kernel: read them through L2 (ld.global.cg), never from this SM's L1
__device__ __forceinline__ SplitCand d_load_cand(const SplitCand* c) {
  static_assert(sizeof(SplitCand) % 8 == 0, "SplitCand is copied in 8-byte words");
  SplitCand out;
  const unsigned long long* src = reinterpret_cast<const unsigned long long*>(c);
  unsigned long long* dst = reinterpret_cast<unsigned long long*>(&out);
#pragma unroll
  for (int i = 0; i < static_cast<int>(sizeof(SplitCand) / 8); ++i) dst[i] = __ldcg(src + i);
  return out;
}
// best candidate per leaf (argmax over features, ties -> smaller real feature index), then the leaf to split; one 256-thread block.
// The two leaves of the round are handled side by side (threads 0..127: smaller, 128..255: larger) with warp-shuffle argmaxes — the
// first version looped over the two leaves with an 8-step shared-memory tree each (18 block barriers) and ncu showed this serial tail
// taking longer than the scan itself.  The order (gain desc, real feature index asc) is total, so any reduction shape picks the same winner.
__device__ __noinline__ void
d_pick_block(TreeCtrl* ctrl, LeafState* leaves, const FeatMeta* __restrict__ meta, const SplitCand* cands, const SplitParams& p) {
  __shared__ double s_gain[8];
  __shared__ int s_feat[8], s_idx[8];
  const int which = threadIdx.x >> 7, t = threadIdx.x & 127, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int leaf = ctrl->go ? (which ? ctrl->larger : ctrl->smaller) : -1;
  double bg = kNegInf; int bf = 0x7fffffff, bi = -1;
  if (leaf >= 0) {
    for (int u = t; u < p.nf; u += 128) {
      const double cg = __ldcg(&cands[which * p.nf_pad + u].gain);
      const int rf = meta[u].real_index;
      if (cg > bg || (cg == bg && rf < bf)) { bg = cg; bf = rf; bi = u; }
    }
  }
  for (int o = 16; o; o >>= 1) {
    const double og = __shfl_xor_sync(0xffffffffu, bg, o);
    const int of = __shfl_xor_sync(0xffffffffu, bf, o), oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (og > bg || (og == bg && of < bf)) { bg = og; bf = of; bi = oi; }
  }
  if (lane == 0) { s_gain[warp] = bg; s_feat[warp] = bf; s_idx[warp] = bi; }
  __syncthreads();
  if (t == 0 && leaf >= 0) {
    for (int w = which * 4; w < which * 4 + 4; ++w)
      if (s_gain[w] > bg || (s_gain[w] == bg && s_feat[w] < bf)) { bg = s_gain[w]; bf = s_feat[w]; bi = s_idx[w]; }
    LeafState& L = leaves[leaf];
    LeafBest b;
    b.gain = kNegInf; b.feature = -1; b.threshold = 0; b.default_left = 1; b.left_count = 0; b.right_count = 0;
    b.left_g = b.left_h = b.right_g = b.right_h = b.left_out = b.right_out = 0; b.is_cat = 0; b.cat_list_len = 0; b.pad = 0;
    for (int wd = 0; wd < 8; ++wd) b.cat_bits[wd] = 0u;
    if (bi >= 0 && bg > kNegInf) {
      const SplitCand c = d_load_cand(&cands[which * p.nf_pad + bi]);
      b.cat_list_len = c.cat_list_len;
      for (int k = 0; k < c.cat_list_len && k < kCatListMax; ++k) b.cat_list[k] = c.cat_list[k];
      const double sum_h = L.sum_h + 2 * kEpsD;
      b.gain = c.gain; b.feature = c.feature; b.threshold = c.threshold; b.default_left = c.default_left;
      b.left_count = c.left_count; b.right_count = L.global_count - c.left_count;
      b.left_g = c.left_g; b.left_h = c.left_h - kEpsD;
      b.right_g = L.sum_g - c.left_g; b.right_h = sum_h - c.left_h - kEpsD;
      SplitParams pc = p;
      pc.l2 += c.l2_extra;
      b.left_out = d_calc_output(c.left_g, c.left_h, pc);
      b.right_out = d_calc_output(L.sum_g - c.left_g, sum_h - c.left_h, pc);
      b.is_cat = c.is_cat;
      for (int wd = 0; wd < 8; ++wd) b.cat_bits[wd] = c.cat_bits[wd];
    }
    L.best = b;
  }
  __syncthreads();
  if (threadIdx.x < 32 && !ctrl->finished) d_choose_leaf(ctrl, leaves, meta, p, threadIdx.x);
}
__global__ void __launch_bounds__(256)
k_pick(TreeCtrl* ctrl, LeafState* leaves, const FeatMeta* __restrict__ meta, const SplitCand* cands, SplitParams p) {
  d_pick_block(ctrl, leaves, meta, cands, p);
}

// ---------------------------------------------------------------- fused data-parallel reduce + scan (C2 + K5 + C3)
// Replaces  K4 -> ncclAllReduce(histogram) -> K5  by LightGBM's reduce-scatter scheme executed over NVLink peer
// memory inside the scan kernel: rank r owns a contiguous slice of feature tiles; after a flag barrier ("all local
// histograms are complete") its scan warps read the slice from EVERY rank's scratch histogram with P2P loads, sum it
// (exact int64), scan only the owned features, and post the rank's two best candidates into every peer's mailbox.
constexpr int kMaxPeers = 16;
struct PeerTables {
  const long long* H[kMaxPeers];       // every rank's scratch histogram (own entry = local pointer)
  SplitCand* mail[kMaxPeers];          // every rank's mailbox [world][2]
  unsigned* flags[kMaxPeers];          // every rank's flag block: [0..15] = "hist ready" epochs, [16..31] = "candidates posted"
  int rank, world, feat0, feat1;       // owned inner-feature range [feat0, feat1)
  int* error;                          // set when a spin-wait times out
};

__device__ __forceinline__ void peer_wait(const volatile unsigned* f, int world, unsigned epoch, int* error) {
  const long long t0 = clock64();
  for (int r = 0; r < world; ++r) {
    while (static_cast<int>(f[r] - epoch) < 0) {
      if (clock64() - t0 > 4000000000LL) { *error = 1; return; }   // ~2 s: a peer died; fail instead of hanging the GPU
      __nanosleep(100);
    }
  }
  __threadfence_system();
}
// one small kernel after K4: tell every peer that this rank's scratch histogram is complete
__global__ void k_peer_signal_hist(PeerTables pt, unsigned epoch) {
  __threadfence_system();
  const int r = threadIdx.x;
  if (r < pt.world) *reinterpret_cast<volatile unsigned*>(&pt.flags[r][pt.rank]) = epoch;
}

__global__ void __launch_bounds__(256)
k_scan_dp(const TreeCtrl* __restrict__ ctrl, const LeafState* __restrict__ leaves, const FeatMeta* __restrict__ meta, PeerTables pt,
          long long* __restrict__ pool, size_t slot_elems, uint8_t* __restrict__ flags, SplitCand* __restrict__ cands, SplitParams p,
          unsigned epoch) {
  if (!ctrl->go) return;
  const int which = blockIdx.y;
  const int leaf = which ? ctrl->larger : ctrl->smaller;
  if (leaf < 0) return;
  // "my scratch histogram is complete" (K4 finished: stream order) -> every peer; then wait for all peers
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x < pt.world) {
    __threadfence_system();
    *reinterpret_cast<volatile unsigned*>(&pt.flags[threadIdx.x][pt.rank]) = epoch;
  }
  if (threadIdx.x == 0) peer_wait(pt.flags[pt.rank], pt.world, epoch, pt.error);
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int u = pt.feat0 + blockIdx.x * 8 + warp;
  if (u >= pt.feat1 || u >= p.nf) return;
  SplitCand out;
  out.gain = kNegInf; out.left_g = 0; out.left_h = 0; out.threshold = 0; out.left_count = 0; out.default_left = 1; out.feature = u;
  out.l2_extra = 0; out.is_cat = 0; out.cat_list_len = 0;
  for (int wd = 0; wd < 8; ++wd) out.cat_bits[wd] = 0u;
  uint8_t* flag = &flags[static_cast<size_t>(leaf) * p.nf_pad + u];
  if (!*flag) { if (lane == 0) cands[which * p.nf_pad + u] = out; return; }

  const LeafState& L = leaves[leaf];
  long long* dst = pool + static_cast<size_t>(L.hist_slot) * slot_elems + static_cast<size_t>(u) * 512;
  long long qg[8], qh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { qg[j] = 0; qh[j] = 0; }
  // reduce-scatter: sum the owned slice over all ranks.  P2P loads bypass L1 (volatile); 4 peers are in flight at a time so
  // the ~2 us NVLink round trips overlap instead of serialising.
  for (int r0 = 0; r0 < pt.world; r0 += 4) {
    longlong2 v[4][8];
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const int r = min(r0 + rr, pt.world - 1);
      const long long* src = pt.H[r] + static_cast<size_t>(u) * 512;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        asm volatile("ld.volatile.global.v2.s64 {%0, %1}, [%2];\n" : "=l"(v[rr][j].x), "=l"(v[rr][j].y) : "l"(src + (lane * 8 + j) * 2));
    }
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      if (r0 + rr < pt.world) {
#pragma unroll
        for (int j = 0; j < 8; ++j) { qg[j] += v[rr][j].x; qh[j] += v[rr][j].y; }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int b = lane * 8 + j;
    if (which) {
      longlong2 pr = *reinterpret_cast<const longlong2*>(dst + b * 2);
      qg[j] = pr.x - qg[j]; qh[j] = pr.y - qh[j];
    }
    longlong2 sv; sv.x = qg[j]; sv.y = qh[j];
    *reinterpret_cast<longlong2*>(dst + b * 2) = sv;
  }
  d_scan_feature(qg, qh, lane, meta[u], L, ctrl->inv_g, ctrl->inv_h, p, flag, &out);
  if (lane == 0) cands[which * p.nf_pad + u] = out;
}

// ---------------------------------------------------------------- C2 as ONE kernel: two-shot all-reduce over NVLink peer memory
// B200GBM_FUSED_REDUCE=2.  The histogram all-reduce of a split is 2-4 MB of int64 — far below the size where NCCL's ring / tree protocols
// pay off; ncclAllReduce costs ~50 us of launch + protocol latency per split at 8 ranks.  Here every rank runs this kernel on its own stream:
//   barrier A  "my scratch histogram is complete" -> flag in every peer's flag block; wait for all peers
//   shot 1     rank r sums slice r (1/world of the histogram) over all peers' scratch histograms with 16-byte P2P loads ...
//   shot 2     ... and stores the sums into slice r of EVERY peer's scratch histogram (nobody else touches slice r)
//   barrier B  raised by the block that finishes last; the kernel does not return before all peers raised theirs, so the scan that follows
//              in stream order sees the complete reduced histogram.  Exact int64 sums: identical bits on every rank.
__global__ void __launch_bounds__(256)
k_allreduce_p2p(const TreeCtrl* __restrict__ ctrl, PeerTables pt, size_t elems, unsigned epoch, unsigned* __restrict__ ticket) {
  __shared__ int s_last;
  if (!ctrl->go) return;                 // same decision on every rank (global counts); nothing was built
  if (blockIdx.x == 0 && threadIdx.x < pt.world) {
    __threadfence_system();
    *reinterpret_cast<volatile unsigned*>(&pt.flags[threadIdx.x][pt.rank]) = epoch;
  }
  if (threadIdx.x == 0) peer_wait(pt.flags[pt.rank], pt.world, epoch, pt.error);
  __syncthreads();
  const size_t n2 = elems / 2;                                   // longlong2 units
  const size_t per = (n2 + pt.world - 1) / pt.world;
  const size_t lo = per * pt.rank, hi = min(lo + per, n2);
  for (size_t i = lo + blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < hi; i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    long long sx = 0, sy = 0;
    for (int r0 = 0; r0 < pt.world; r0 += 4) {                   // 4 peers in flight: the NVLink round trips overlap
      long long vx[4], vy[4];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const int r = min(r0 + rr, pt.world - 1);
        asm volatile("ld.volatile.global.v2.s64 {%0, %1}, [%2];\n" : "=l"(vx[rr]), "=l"(vy[rr]) : "l"(pt.H[r] + i * 2));
      }
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) if (r0 + rr < pt.world) { sx += vx[rr]; sy += vy[rr]; }
    }
    for (int r = 0; r < pt.world; ++r)
      asm volatile("st.volatile.global.v2.s64 [%0], {%1, %2};\n" ::"l"(const_cast<long long*>(pt.H[r]) + i * 2), "l"(sx), "l"(sy) : "memory");
  }
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
  __syncthreads();
  if (!s_last) return;
  if (threadIdx.x == 0) *ticket = 0u;
  __threadfence_system();
  if (threadIdx.x < pt.world) *reinterpret_cast<volatile unsigned*>(&pt.flags[threadIdx.x][16 + pt.rank]) = epoch;
  if (threadIdx.x == 0) peer_wait(pt.flags[pt.rank] + 16, pt.world, epoch, pt.error);
  __syncthreads();
}

// leaf choice by warp 0: ArgMax over leaves with SplitInfo::operator> (gain desc, real feature asc, first index), stop on gain <= 0

// argmax over features per leaf (gain desc, real feature index asc), then over leaves
// (SplitInfo::operator> : gain desc, feature asc; ArrayArgs::ArgMax keeps the first on full ties).


// data-parallel pick: local argmax over the OWNED features, exchange of the per-rank winners through the peers'
// mailboxes (C3, SyncUpGlobalBestSplit), global argmax with the same tie-breaks on every rank, then the usual leaf choice.
__global__ void __launch_bounds__(256)
k_pick_dp(TreeCtrl* ctrl, LeafState* leaves, const FeatMeta* __restrict__ meta, const SplitCand* __restrict__ cands, SplitParams p,
          PeerTables pt, unsigned epoch) {
  __shared__ double s_gain[256];
  __shared__ int s_feat[256], s_idx[256];
  const bool go = ctrl->go != 0;
  if (go) {
    for (int which = 0; which < 2; ++which) {
      const int leaf = which ? ctrl->larger : ctrl->smaller;
      double bg = kNegInf; int bf = 0x7fffffff, bi = -1;
      if (leaf >= 0) {
        for (int u = pt.feat0 + threadIdx.x; u < pt.feat1 && u < p.nf; u += blockDim.x) {
          const SplitCand& c = cands[which * p.nf_pad + u];
          const int rf = meta[u].real_index;
          if (c.gain > bg || (c.gain == bg && rf < bf)) { bg = c.gain; bf = rf; bi = u; }
        }
      }
      s_gain[threadIdx.x] = bg; s_feat[threadIdx.x] = bf; s_idx[threadIdx.x] = bi;
      __syncthreads();
      for (int s = 128; s; s >>= 1) {
        if (threadIdx.x < s) {
          double og = s_gain[threadIdx.x + s]; int of = s_feat[threadIdx.x + s];
          if (og > s_gain[threadIdx.x] || (og == s_gain[threadIdx.x] && of < s_feat[threadIdx.x])) {
            s_gain[threadIdx.x] = og; s_feat[threadIdx.x] = of; s_idx[threadIdx.x] = s_idx[threadIdx.x + s];
          }
        }
        __syncthreads();
      }
      if (threadIdx.x < pt.world) {      // post this rank's winner into every peer's mailbox
        SplitCand c;
        c.gain = kNegInf; c.left_g = 0; c.left_h = 0; c.threshold = 0; c.left_count = 0; c.default_left = 1; c.feature = -1;
        if (s_idx[0] >= 0 && s_gain[0] > kNegInf) c = cands[which * p.nf_pad + s_idx[0]];
        SplitCand* dst = pt.mail[threadIdx.x] + pt.rank * 2 + which;
        volatile double* dd = reinterpret_cast<volatile double*>(dst);
        dd[0] = c.gain; dd[1] = c.left_g; dd[2] = c.left_h;
        volatile int* di = reinterpret_cast<volatile int*>(dd + 3);
        di[0] = c.threshold; di[1] = c.left_count; di[2] = c.default_left; di[3] = c.feature;
      }
      __syncthreads();
    }
  }
  // barrier B: "candidates posted" (also means: every peer is done reading this rank's scratch histogram)
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x < pt.world) *reinterpret_cast<volatile unsigned*>(&pt.flags[threadIdx.x][16 + pt.rank]) = epoch;
  if (threadIdx.x == 0) peer_wait(pt.flags[pt.rank] + 16, pt.world, epoch, pt.error);
  __syncthreads();
  if (threadIdx.x == 0 && go) {
    for (int which = 0; which < 2; ++which) {
      const int leaf = which ? ctrl->larger : ctrl->smaller;
      if (leaf < 0) continue;
      SplitCand best;
      best.gain = kNegInf; best.feature = -1; best.left_g = best.left_h = 0; best.threshold = 0; best.left_count = 0; best.default_left = 1;
      int best_rf = 0x7fffffff;
      const SplitCand* mb = pt.mail[pt.rank];
      for (int r = 0; r < pt.world; ++r) {
        SplitCand c;
        const volatile double* dd = reinterpret_cast<const volatile double*>(mb + r * 2 + which);
        c.gain = dd[0]; c.left_g = dd[1]; c.left_h = dd[2];
        const volatile int* di = reinterpret_cast<const volatile int*>(dd + 3);
        c.threshold = di[0]; c.left_count = di[1]; c.default_left = di[2]; c.feature = di[3];
        const int rf = c.feature < 0 ? 0x7fffffff : meta[c.feature].real_index;
        if (c.gain > best.gain || (c.gain == best.gain && rf < best_rf)) { best = c; best_rf = rf; }
      }
      LeafState& L = leaves[leaf];
      LeafBest b;
      b.gain = kNegInf; b.feature = -1; b.threshold = 0; b.default_left = 1; b.left_count = 0; b.right_count = 0;
      b.left_g = b.left_h = b.right_g = b.right_h = b.left_out = b.right_out = 0; b.is_cat = 0; b.cat_list_len = 0; b.pad = 0;
      for (int wd = 0; wd < 8; ++wd) b.cat_bits[wd] = 0u;
      if (best.feature >= 0 && best.gain > kNegInf) {
        const double sum_h = L.sum_h + 2 * kEpsD;
        b.gain = best.gain; b.feature = best.feature; b.threshold = best.threshold; b.default_left = best.default_left;
        b.left_count = best.left_count; b.right_count = L.global_count - best.left_count;
        b.left_g = best.left_g; b.left_h = best.left_h - kEpsD;
        b.right_g = L.sum_g - best.left_g; b.right_h = sum_h - best.left_h - kEpsD;
        b.left_out = d_calc_output(best.left_g, best.left_h, p);
        b.right_out = d_calc_output(L.sum_g - best.left_g, sum_h - best.left_h, p);
      }
      L.best = b;
    }
  }
  __syncthreads();
  if (threadIdx.x < 32 && !ctrl->finished) d_choose_leaf(ctrl, leaves, meta, p, threadIdx.x);
}

// ---------------------------------------------------------------- column-major copy of the uint8 tiles (for the partition kernel)
// The tile layout [tile][row][32 features] is what K4 streams, but the partition kernel needs ONE feature of every row of a leaf and pays
// a 32-byte sector for each byte (62 % of its DRAM bytes at 100M rows).  When device memory allows, the booster keeps a second copy
// [feature][row] (cols_stride = rows rounded up to 256), built once by this kernel.
__global__ void __launch_bounds__(256)
k_tiles_to_columns(const uint8_t* __restrict__ bins, size_t rows_stride, int num_tiles, long long nrow, uint8_t* __restrict__ cols, size_t cols_stride) {
  __shared__ uint4 s_t[256 * 2 + 16];                      // 256 rows x 32 bytes
  const long long per_tile = (nrow + 255) / 256;
  for (long long w = blockIdx.x; w < per_tile * num_tiles; w += gridDim.x) {
    const int tile = static_cast<int>(w / per_tile);
    const long long r0 = (w % per_tile) * 256;
    const int rows = static_cast<int>(min(256LL, nrow - r0));
    const uint4* src = reinterpret_cast<const uint4*>(bins + (static_cast<size_t>(tile) * rows_stride + static_cast<size_t>(r0)) * 32);
    __syncthreads();
    for (int i = threadIdx.x; i < rows * 2; i += 256) s_t[i] = src[i];
    __syncthreads();
    const uint8_t* sb = reinterpret_cast<const uint8_t*>(s_t);
    const int f = threadIdx.x >> 3, g = threadIdx.x & 7;   // feature of the tile, group of 32 rows
    unsigned wv[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      unsigned v = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) { const int r = g * 32 + k * 4 + j; v |= (r < rows ? static_cast<unsigned>(sb[r * 32 + f]) : 0u) << (8 * j); }
      wv[k] = v;
    }
    uint4* dst = reinterpret_cast<uint4*>(cols + (static_cast<size_t>(tile) * 32 + f) * cols_stride + static_cast<size_t>(r0) + g * 32);
    dst[0] = make_uint4(wv[0], wv[1], wv[2], wv[3]);       // cols_stride is a multiple of 256: padding rows exist and are never read
    dst[1] = make_uint4(wv[4], wv[5], wv[6], wv[7]);
  }
}

// ---------------------------------------------------------------- K7 row partition (stable), one cooperative kernel per split
// Replaces [UPSTREAM] DataPartition::Split.  Round 1 ran three kernels (decision bits + per-chunk left counts, single-block scan of the
// chunk counts, scatter) plus a memset of the scratch histogram and the next round's controller: five launches on the per-split
// critical path.  They are now the phases of ONE cooperatively launched kernel separated by software grid barriers (all blocks are
// resident; the arrive counter lives in TreeCtrl):
//   phase 0  zero the scratch histogram H for the next K4 (the scan kernel consumed it; stream order)
//   phase 1  decision bit per row (ballot words) and the left count of every 2048-row chunk
//   ---- grid barrier
//   phase 2  chunk prefix: leaves of <= 2048 chunks (4M rows) are scanned redundantly by every block in shared memory (no second
//            barrier); larger ones in two levels (one block per 2048 counts, second barrier, every block scans the totals)
//   phase 3  stable scatter into the other index buffer (lefts first, then rights, original order kept); the (g,h) words of the
//            child K4 scans next go into partition order (qord)
//   tail     the block that finishes last applies the split to the tree and prepares the next round (d_round_ctl)
constexpr int kPartChunk = 2048;     // rows per chunk = 256 threads x 8
constexpr int kPartLocalScan = 2048; // chunk counts a block scans by itself
__device__ __forceinline__ bool d_goes_left(unsigned bin, const TreeCtrl* c) {
  if (c->split_is_cat) return (c->split_cat_bits[bin >> 5] >> (bin & 31u)) & 1u;
  if (c->split_missing_type == 2 && bin == static_cast<unsigned>(c->split_num_bin - 1)) return c->split_default_left != 0;
  return bin <= static_cast<unsigned>(c->split_threshold);
}
// all blocks of a cooperative launch: arrive on a monotone counter, spin until `target` arrivals
__device__ __forceinline__ void d_grid_barrier(unsigned* counter, unsigned target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    while (*reinterpret_cast<volatile unsigned*>(counter) < target) __nanosleep(32);
    __threadfence();
  }
  __syncthreads();
}
__global__ void __launch_bounds__(256, 3)
k_partition(TreeCtrl* ctrl, LeafState* leaves, TreeDev tree, uint8_t* flags, const FeatMeta* __restrict__ meta, SplitParams p, int last,
            const uint8_t* __restrict__ bins, size_t rows_stride, int* __restrict__ idx0, int* __restrict__ idx1, unsigned* __restrict__ bits,
            int* __restrict__ chunk_left, const int4* __restrict__ qgh, int4* __restrict__ qord, long long* __restrict__ H, size_t h_elems,
            const uint16_t* __restrict__ bins16, int tickets_per_block, const uint8_t* __restrict__ cols, size_t cols_stride, int* __restrict__ super_tot) {
  __shared__ int s_pref[kPartLocalScan + 1];
  __shared__ unsigned short s_list[kCatListMax];
  __shared__ int s_wl[64];
  __shared__ int s_cnt[8];
  __shared__ int s_copy[2];
  __shared__ int s_last;
  __shared__ int s_chunk;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // ---- phase 0: H := 0 (16-byte stores; H is L2-resident)
  {
    longlong2* h2 = reinterpret_cast<longlong2*>(H);
    const size_t n2 = h_elems / 2;
    const longlong2 z = make_longlong2(0, 0);
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n2; i += static_cast<size_t>(gridDim.x) * blockDim.x) h2[i] = z;
  }
  const int n = ctrl->part_count;
  if (n > 0) {
    const int* src = ctrl->part_buf ? idx1 : idx0;
    int* dst = ctrl->part_identity ? idx0 : (ctrl->part_buf ? idx0 : idx1);
    const int begin = ctrl->part_begin, identity = ctrl->part_identity;
    const int f = ctrl->split_feature;
    const int wide = ctrl->split_wide;
    const uint8_t* col = bins + (static_cast<size_t>((wide >= 0 ? 0 : f) >> 5) * rows_stride) * 32 + ((wide >= 0 ? 0 : f) & 31);
    const uint16_t* wcol = wide >= 0 ? bins16 + static_cast<size_t>(wide) * rows_stride : nullptr;
    const uint8_t* ccol = (cols != nullptr && wide < 0) ? cols + static_cast<size_t>(f) * cols_stride : nullptr;      // column-major copy, if kept
    const bool wide_cat = wide >= 0 && ctrl->split_is_cat;
    const int list_len = wide_cat ? ctrl->split_cat_list_len : 0;
    if (threadIdx.x < list_len) s_list[threadIdx.x] = ctrl->split_cat_list[threadIdx.x];
    __syncthreads();
    const int chunks = (n + kPartChunk - 1) / kPartChunk;
    // ---- phase 1 (no block-wide barrier: every warp adds the left count of its 256 rows to the chunk's counter, which the tail of
    // the previous partition kernel left at zero)
    // chunks are handed out dynamically (one atomic per chunk): the rows' DRAM latency varies, and the grid barrier waits for the slowest block
    // a ticket grants `grp` consecutive chunks: a 100M-row leaf has 48K chunks, and one same-address atomic per chunk and phase is a
    // serial ~100 us; with ~tickets_per_block tickets per block the hand-out stays dynamic and the atomics are negligible
    const int grp = tickets_per_block > 0 ? max(1, chunks / (static_cast<int>(gridDim.x) * tickets_per_block)) : 1;
    for (;;) {
      __syncthreads();
      if (threadIdx.x == 0) s_chunk = static_cast<int>(atomicAdd(&ctrl->part_next[0], 1u));
      __syncthreads();
      const int cbase = s_chunk * grp;
      if (cbase >= chunks) break;
      for (int c = cbase; c < min(cbase + grp, chunks); ++c) {
      // the 8 rows of a thread: all index loads first, then all bin loads, then the ballots — two dependent memory latencies per chunk
      // instead of sixteen (ncu, 100M-row table: the kernel ran at 2 TB/s with long_scoreboard as the only stall reason)
      int local = 0;
      int rr[8]; unsigned bb[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int i = c * kPartChunk + k * 256 + threadIdx.x;
        rr[k] = i < n ? (identity ? (begin + i) : src[begin + i]) : -1;
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        bb[k] = 0u;
        if (rr[k] >= 0)
          bb[k] = wide >= 0 ? static_cast<unsigned>(wcol[rr[k]]) : (ccol ? static_cast<unsigned>(ccol[rr[k]]) : static_cast<unsigned>(col[static_cast<size_t>(rr[k]) * 32]));
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        bool left = false;
        if (rr[k] >= 0) {
          const unsigned bin = bb[k];
          if (wide_cat) { for (int kk = 0; kk < list_len; ++kk) left |= (bin == s_list[kk]); }
          else left = d_goes_left(bin, ctrl);
        }
        const unsigned bal = __ballot_sync(0xffffffffu, left);
        if (lane == 0) { bits[(c * kPartChunk + k * 256 + threadIdx.x) >> 5] = bal; local += __popc(bal); }
      }
      if (lane == 0 && local) atomicAdd(&chunk_left[c], local);
      }
    }
    d_grid_barrier(&ctrl->part_barrier, gridDim.x);
    // ---- phase 2: exclusive prefix of the chunk counts + total
    int total_left;
    const bool local_scan = chunks <= kPartLocalScan;
    if (local_scan) {
      // 256 threads x 8 consecutive counts, warp scan of the per-thread sums, then the block total
      int v[8], sum = 0;
#pragma unroll
      for (int k = 0; k < 8; ++k) { const int i = threadIdx.x * 8 + k; v[k] = i < chunks ? __ldcg(chunk_left + i) : 0; sum += v[k]; }
      int inc = sum;
      for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
      if (lane == 31) s_cnt[warp] = inc;
      __syncthreads();
      int woff = 0;
      for (int w = 0; w < warp; ++w) woff += s_cnt[w];
      int run = woff + inc - sum;
#pragma unroll
      for (int k = 0; k < 8; ++k) { s_pref[threadIdx.x * 8 + k] = run; run += v[k]; }
      if (threadIdx.x == 255) s_pref[kPartLocalScan] = run;
      __syncthreads();
      total_left = s_pref[kPartLocalScan];
    } else {
      // two levels: block s scans the 2048 counts of "super-chunk" s in place (prefix relative to the super-chunk) and publishes its total;
      // after the second barrier every block scans the totals.  (The first version had block 0 scan all counts alone: ~190 us for the 48K
      // chunks of a 100M-row root while every other block waited at the barrier.)
      const int supers = (chunks + kPartLocalScan - 1) / kPartLocalScan;
      for (int sp = blockIdx.x; sp < supers; sp += gridDim.x) {
        int v[8], sum = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = sp * kPartLocalScan + threadIdx.x * 8 + k; v[k] = i < chunks ? __ldcg(chunk_left + i) : 0; sum += v[k]; }
        int inc = sum;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        __syncthreads();
        if (lane == 31) s_cnt[warp] = inc;
        __syncthreads();
        int woff = 0;
        for (int w = 0; w < warp; ++w) woff += s_cnt[w];
        int run = woff + inc - sum;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = sp * kPartLocalScan + threadIdx.x * 8 + k; if (i < chunks) chunk_left[i] = run; run += v[k]; }
        if (threadIdx.x == 255) super_tot[sp] = run;
      }
      d_grid_barrier(&ctrl->part_barrier, 2 * gridDim.x);
      {   // exclusive scan of the super-chunk totals (at most 2048 of them: 8.6G rows) into s_pref
        int v[8], sum = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) { const int i = threadIdx.x * 8 + k; v[k] = i < supers ? __ldcg(super_tot + i) : 0; sum += v[k]; }
        int inc = sum;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        __syncthreads();
        if (lane == 31) s_cnt[warp] = inc;
        __syncthreads();
        int woff = 0;
        for (int w = 0; w < warp; ++w) woff += s_cnt[w];
        int run = woff + inc - sum;
#pragma unroll
        for (int k = 0; k < 8; ++k) { s_pref[threadIdx.x * 8 + k] = run; run += v[k]; }
        if (threadIdx.x == 255) s_pref[kPartLocalScan] = run;
        __syncthreads();
        total_left = s_pref[kPartLocalScan];
      }
    }
    // the child K4 scans next is the one with fewer rows by the rule of d_round_ctl (global counts of the split in data-parallel
    // mode, true counts otherwise; ties -> right): its (g,h) words are written in partition order (qord)
    const LeafBest& bsp = leaves[ctrl->split_leaf].best;
    const int lc = p.parallel ? bsp.left_count : total_left, rc = p.parallel ? bsp.right_count : n - total_left;
    const bool q_left = lc < rc;
    // ---- phase 3
    for (;;) {
      __syncthreads();
      if (threadIdx.x == 0) s_chunk = static_cast<int>(atomicAdd(&ctrl->part_next[1], 1u));
      __syncthreads();
      const int cbase = s_chunk * grp;
      if (cbase >= chunks) break;
      for (int c = cbase; c < min(cbase + grp, chunks); ++c) {
      const int wbase = c * (kPartChunk / 32);     // 64 ballot words per chunk; word w covers rows c*2048 + w*32 ..
      if (threadIdx.x < 64) {
        const int i0 = c * kPartChunk + threadIdx.x * 32;
        s_wl[threadIdx.x] = i0 < n ? __popc(__ldcg(bits + wbase + threadIdx.x)) : 0;
      }
      __syncthreads();
      if (warp == 0) {   // exclusive scan of the 64 word counts (two per lane)
        const int a = s_wl[lane * 2], b = s_wl[lane * 2 + 1];
        const int sum = a + b;
        int inc = sum;
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        const int ex = inc - sum;
        s_wl[lane * 2] = ex; s_wl[lane * 2 + 1] = ex + a;
      }
      __syncthreads();
      const int left_base = local_scan ? s_pref[c] : s_pref[c / kPartLocalScan] + __ldcg(chunk_left + c);
      const int right_base = c * kPartChunk - left_base;
      // same batching as phase 1: the 8 index loads, then the (g,h) words of the rows that go to the child K4 scans next, then the stores
      int rr[8], pp[8]; bool qq[8]; int4 qv[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int w = k * 8 + warp;                 // word index inside the chunk
        const int i = c * kPartChunk + w * 32 + lane;
        rr[k] = -1; pp[k] = 0; qq[k] = false;
        if (i < n) {
          const unsigned word = __ldcg(bits + wbase + w);
          const bool left = (word >> lane) & 1u;
          const int lefts_before = s_wl[w] + __popc(word & ((1u << lane) - 1u));
          rr[k] = identity ? (begin + i) : src[begin + i];
          pp[k] = left ? begin + left_base + lefts_before : begin + total_left + right_base + (w * 32 + lane - lefts_before);
          qq[k] = (left == q_left);
        }
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) if (qq[k]) qv[k] = qgh[rr[k]];      // replaces a separate gather pass before K4 (k_gather_q)
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        if (rr[k] < 0) continue;
        dst[pp[k]] = rr[k];
        if (qq[k]) qord[pp[k]] = qv[k];
      }
      __syncthreads();      // s_wl is rewritten for the next chunk
      }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) ctrl->part_left_total = total_left;
  }
  // ---- tail: the last block to finish runs the controller of the next round
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned t = atomicAdd(&ctrl->part_ticket, 1u);
    s_last = (t == gridDim.x - 1) ? 1 : 0;
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    if (threadIdx.x == 0) { ctrl->part_ticket = 0u; ctrl->part_barrier = 0u; ctrl->part_next[0] = 0u; ctrl->part_next[1] = 0u; }
    if (n > 0) for (int c = threadIdx.x; c < (n + kPartChunk - 1) / kPartChunk; c += blockDim.x) chunk_left[c] = 0;      // phase 1 of the next launch accumulates into zeros
    d_round_ctl(ctrl, leaves, tree, flags, meta, p, last, s_copy);
  }
}

// ---------------------------------------------------------------- wide features (> 256 bins): binning, histogram, categorical scan
// value -> bin of the wide columns of a row block (categorical lookup: binary search in the feature's sorted category table)
// value -> bin of one wide feature (shared by the dense and CSR ingestion kernels)
__device__ __forceinline__ unsigned d_wide_bin(double v, const WideMeta& m, const int* __restrict__ cats, const unsigned short* __restrict__ catbin,
                                               const double* __restrict__ wub) {
  unsigned bin = 0;
  if (m.is_cat) {
    if (!isnan(v)) {
      const int iv = static_cast<int>(v);
      if (iv >= 0) {
        const int* c = cats + m.cat_off;
        int lo = 0, hi = m.num_cats;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (c[mid] < iv) lo = mid + 1; else hi = mid; }
        if (lo < m.num_cats && c[lo] == iv) bin = catbin[m.cat_off + lo];
      }
    }
    return bin;
  }
  if (isnan(v)) { if (m.missing_type == 2) return static_cast<unsigned>(m.num_bin - 1); v = 0.0; }
  const double* ub = wub + m.cat_off;
  int lo = 0, hi = m.num_bin - 1 - (m.missing_type == 2 ? 1 : 0);
  while (lo < hi) { const int mid = (hi + lo - 1) / 2; if (v <= ub[mid]) hi = mid; else lo = mid + 1; }
  return static_cast<unsigned>(lo);
}
template <typename T>
__global__ void k_bin_wide(const T* __restrict__ X, long long nrow, int row_major, long long ld, const WideMeta* __restrict__ wm, int nw,
                           const int* __restrict__ cats, const unsigned short* __restrict__ catbin, const double* __restrict__ wub,
                           uint16_t* __restrict__ bins16, size_t rows_stride, long long row_offset) {
  const long long total = nrow * nw;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total; e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int w = static_cast<int>(e / nrow);
    const long long r = e - static_cast<long long>(w) * nrow;
    const WideMeta m = wm[w];
    const double v = row_major ? static_cast<double>(X[r * ld + m.real_index]) : static_cast<double>(X[static_cast<long long>(m.real_index) * ld + r]);
    bins16[static_cast<size_t>(w) * rows_stride + row_offset + r] = static_cast<uint16_t>(d_wide_bin(v, m, cats, catbin, wub));
  }
}

// K4 for wide features.  One CTA = (wide feature, row range of the leaf): the sub-histogram is [NATOM planes][num_bin] in shared memory
// with the same fixed-point fields as the tile kernel; lanes read consecutive rows of the uint16 column (or gather through the leaf's
// index list), so the atomics of a warp fall on data-dependent banks — these features are a few percent of a wide table's columns and
// run at a fraction of the tile kernel's rate, which is acceptable.  Flush every 2^14 rows (field headroom) into the int64 histogram.
constexpr int kWideThreads = 1024;     // one CTA per SM (128 KB of planes): the loop is latency-bound, so as many rows in flight as the SM allows
template <int NATOM>
__global__ void __launch_bounds__(kWideThreads, 1)
k4_hist_wide(const uint16_t* __restrict__ bins16, size_t rows_stride, const WideMeta* __restrict__ wm, const int4* __restrict__ qgh,
             const int4* __restrict__ qord, const int* __restrict__ idx0, const int* __restrict__ idx1, const HistWork* __restrict__ work,
             unsigned long long* __restrict__ hist) {
  extern __shared__ __align__(16) unsigned wplane[];        // [NATOM][nb_pad]
  const HistWork w = *work;
  const int n = w.count;
  if (n <= 0) return;
  const int active = min(static_cast<int>(gridDim.x), (n + 4095) / 4096);
  if (static_cast<int>(blockIdx.x) >= active) return;
  const WideMeta m = wm[blockIdx.y];
  const unsigned lo = blockIdx.z * kWideHistSeg;              // this CTA accumulates bins [lo, lo + nb) of the feature
  if (static_cast<int>(lo) >= m.num_bin) return;
  const int nb = min(kWideHistSeg, m.num_bin - static_cast<int>(lo));
  const int p0 = static_cast<int>(static_cast<long long>(n) * blockIdx.x / active), p1 = static_cast<int>(static_cast<long long>(n) * (blockIdx.x + 1) / active);
  const int* __restrict__ idx = w.buf ? idx1 : idx0;
  const uint16_t* __restrict__ col = bins16 + static_cast<size_t>(blockIdx.y) * rows_stride;
  unsigned* pl0 = wplane; unsigned* pl1 = wplane + kWideHistSeg; unsigned* pl2 = wplane + 2 * kWideHistSeg; unsigned* pl3 = wplane + 3 * kWideHistSeg;
  for (int e = threadIdx.x; e < nb; e += kWideThreads) { pl0[e] = 0u; pl1[e] = 0u; pl2[e] = 0u; if (NATOM == 4) pl3[e] = 0u; }
  __syncthreads();
  for (int c0 = p0; c0 < p1; c0 += kFlushRows) {
    const int c1 = min(c0 + kFlushRows, p1);
    // four rows per thread in flight (index -> bin is a dependent pair of DRAM/L2 accesses; with one CTA per SM the loop is latency-bound)
    for (int p = c0 + threadIdx.x; p < c1; p += 4 * kWideThreads) {
      int4 q[4]; unsigned b[4]; size_t r[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int pj = p + j * kWideThreads;
        r[j] = 0;
        if (pj < c1) {
          if (w.use_idx) { r[j] = static_cast<size_t>(idx[w.begin + pj]); q[j] = qord[w.begin + pj]; }
          else { r[j] = static_cast<size_t>(w.begin + pj); q[j] = qgh[r[j]]; }
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = (p + j * kWideThreads < c1) ? static_cast<unsigned>(col[r[j]]) - lo : 0xffffffffu;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (b[j] >= static_cast<unsigned>(nb)) continue;           // another segment's bin (or past the end)
        atomicAdd(&pl0[b[j]], static_cast<unsigned>(q[j].x));
        atomicAdd(&pl1[b[j]], static_cast<unsigned>(q[j].y));
        atomicAdd(&pl2[b[j]], static_cast<unsigned>(q[j].z));
        if (NATOM == 4) atomicAdd(&pl3[b[j]], static_cast<unsigned>(q[j].w));
      }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < nb; e += kWideThreads) {
      const unsigned ghi = pl0[e], glo = pl1[e], hhi = pl2[e], hlo = (NATOM == 4) ? pl3[e] : 0u;
      if (ghi | glo | hhi | hlo) {
        const long long g = (static_cast<long long>(static_cast<int>(ghi)) << kLoBits) + static_cast<long long>(glo);
        const long long h = (NATOM == 4) ? (static_cast<long long>(static_cast<int>(hhi)) << kLoBits) + static_cast<long long>(hlo) : static_cast<long long>(hhi);
        const size_t o = (static_cast<size_t>(m.hist_off) + lo + e) * 2;
        if (g) atomicAdd(&hist[o], static_cast<unsigned long long>(g));
        if (h) atomicAdd(&hist[o + 1], static_cast<unsigned long long>(h));
        pl0[e] = 0u; pl1[e] = 0u; pl2[e] = 0u; if (NATOM == 4) pl3[e] = 0u;
      }
    }
    __syncthreads();
  }
}

// exclusive prefix (reverse == 0: over threads < t) or suffix (reverse == 1: over threads > t) sums of three int64 values across a 256-thread
// block, plus nothing else; sm = 3 * 8 long longs of shared scratch.  Exact integers: any association order gives the same result.
__device__ __forceinline__ void d_block_excl3(long long& a, long long& b, long long& c, int reverse, long long* sm) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long ia = a, ib = b, ic = c;
  for (int o = 1; o < 32; o <<= 1) {
    long long ta, tb, tc;
    if (reverse) { ta = __shfl_down_sync(0xffffffffu, ia, o); tb = __shfl_down_sync(0xffffffffu, ib, o); tc = __shfl_down_sync(0xffffffffu, ic, o); if (lane + o < 32) { ia += ta; ib += tb; ic += tc; } }
    else { ta = __shfl_up_sync(0xffffffffu, ia, o); tb = __shfl_up_sync(0xffffffffu, ib, o); tc = __shfl_up_sync(0xffffffffu, ic, o); if (lane >= o) { ia += ta; ib += tb; ic += tc; } }
  }
  __syncthreads();
  if (lane == (reverse ? 0 : 31)) { sm[warp] = ia; sm[8 + warp] = ib; sm[16 + warp] = ic; }
  __syncthreads();
  long long oa = 0, ob = 0, oc = 0;
  for (int w2 = 0; w2 < 8; ++w2) if (reverse ? w2 > warp : w2 < warp) { oa += sm[w2]; ob += sm[8 + w2]; oc += sm[16 + w2]; }
  a = oa + ia - a; b = ob + ib - b; c = oc + ic - c;
  __syncthreads();
}

// FeatureHistogram::FindBestThresholdSequentially for a WIDE numerical feature (max_bin > 255): the same two passes as d_scan_feature with the
// bins spread over a 256-thread block — thread t owns the contiguous bins [t*S, (t+1)*S) — exclusive block scans of the per-thread
// (g, h, count) sums, and a block argmax with the sequential scan's tie-breaks (reverse pass: the highest threshold wins, forward pass: the
// lowest).  hist = the leaf's reduced histogram of the feature in its pool slot.  Returns through *outp (thread 0) and *flag.
__device__ __noinline__ void d_scan_wide_numeric(const long long* __restrict__ hist, const WideMeta m, const LeafState& L, double inv_g, double inv_h,
                                                  const SplitParams& p, uint8_t* flag, SplitCand* outp) {
  __shared__ long long s_sc[24];
  __shared__ double s_bg[8], s_blg[8], s_blh[8];
  __shared__ int s_bt[8], s_blc[8], s_any;
  __shared__ long long s_tot[3];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double sum_g = L.sum_g, sum_h = L.sum_h + 2 * kEpsD;
  const int num_data = L.global_count;
  const double cnt_factor = num_data / sum_h;
  const double min_gain_shift = d_leaf_gain(sum_g, sum_h, p) + p.min_gain_to_split;
  const bool two_way = (m.num_bin > 2 && m.missing_type == 2);
  const int na = two_way ? 1 : 0;
  const int S = (m.num_bin + 255) / 256;
  const int b0 = threadIdx.x * S, b1 = min(b0 + S, m.num_bin);
  if (threadIdx.x == 0) s_any = 0;
  bool any_valid = false;
  // ---- reverse pass: bins hi .. 1, candidate threshold = b - 1
  double best_gain = kNegInf, best_lg = 0, best_lh = 0;
  int best_thr = -1, best_lc = 0, best_dl = 1;
  {
    const int hi = m.num_bin - 1 - na;
    long long lg = 0, lh = 0, lc = 0;
    for (int b = b0; b < b1; ++b)
      if (b >= 1 && b <= hi) { const long long qh = hist[b * 2 + 1]; lg += hist[b * 2]; lh += qh; lc += static_cast<int>(static_cast<double>(qh) * inv_h * cnt_factor + 0.5); }
    long long rg = lg, rh = lh, rc = lc;
    d_block_excl3(rg, rh, rc, 1, s_sc);
    for (int b = b1 - 1; b >= b0; --b) {
      if (b < 1 || b > hi) continue;
      const long long qg = hist[b * 2], qh = hist[b * 2 + 1];
      rg += qg; rh += qh; rc += static_cast<int>(static_cast<double>(qh) * inv_h * cnt_factor + 0.5);
      const double srg = static_cast<double>(rg) * inv_g;
      const double srh = kEpsD + static_cast<double>(rh) * inv_h;
      const int right_count = static_cast<int>(rc);
      if (right_count < p.min_data_in_leaf || srh < p.min_sum_hessian) continue;
      const int left_count = num_data - right_count;
      if (left_count < p.min_data_in_leaf) continue;
      const double slh = sum_h - srh;
      if (slh < p.min_sum_hessian) continue;
      const double slg = sum_g - srg;
      const double gain = d_leaf_gain(slg, slh, p) + d_leaf_gain(srg, srh, p);
      if (gain <= min_gain_shift) continue;
      any_valid = true;
      if (gain > best_gain) { best_gain = gain; best_lg = slg; best_lh = slh; best_thr = b - 1; best_lc = left_count; }
    }
    for (int o = 16; o; o >>= 1) {
      const double og = __shfl_xor_sync(0xffffffffu, best_gain, o);
      const int ot = __shfl_xor_sync(0xffffffffu, best_thr, o);
      const double olg = __shfl_xor_sync(0xffffffffu, best_lg, o), olh = __shfl_xor_sync(0xffffffffu, best_lh, o);
      const int olc = __shfl_xor_sync(0xffffffffu, best_lc, o);
      if (og > best_gain || (og == best_gain && ot > best_thr)) { best_gain = og; best_thr = ot; best_lg = olg; best_lh = olh; best_lc = olc; }
    }
    if (lane == 0) { s_bg[warp] = best_gain; s_bt[warp] = best_thr; s_blg[warp] = best_lg; s_blh[warp] = best_lh; s_blc[warp] = best_lc; }
    __syncthreads();
    for (int w2 = 0; w2 < 8; ++w2)
      if (s_bg[w2] > best_gain || (s_bg[w2] == best_gain && s_bt[w2] > best_thr)) { best_gain = s_bg[w2]; best_thr = s_bt[w2]; best_lg = s_blg[w2]; best_lh = s_blh[w2]; best_lc = s_blc[w2]; }
    __syncthreads();
  }
  // ---- forward pass (NaN-as-missing features only): bins 0 .. num_bin-2, threshold = b, NaN goes right
  if (two_way) {
    const int hi = m.num_bin - 2;
    long long ag = 0, ah = 0, ac = 0, lg = 0, lh = 0, lc = 0;
    for (int b = b0; b < b1; ++b) {
      const long long qg = hist[b * 2], qh = hist[b * 2 + 1];
      const int c = static_cast<int>(static_cast<double>(qh) * inv_h * cnt_factor + 0.5);
      if (b >= 1 && b < m.num_bin) { ag += qg; ah += qh; ac += c; }
      if (b >= m.offset && b <= hi) { lg += qg; lh += qh; lc += c; }
    }
    {   // block totals of (ag, ah, ac)
      long long ta = ag, tb = ah, tc = ac;
      for (int o = 16; o; o >>= 1) { ta += __shfl_xor_sync(0xffffffffu, ta, o); tb += __shfl_xor_sync(0xffffffffu, tb, o); tc += __shfl_xor_sync(0xffffffffu, tc, o); }
      if (lane == 0) { s_sc[warp] = ta; s_sc[8 + warp] = tb; s_sc[16 + warp] = tc; }
      __syncthreads();
      if (threadIdx.x == 0) { long long x = 0, y = 0, z = 0; for (int w2 = 0; w2 < 8; ++w2) { x += s_sc[w2]; y += s_sc[8 + w2]; z += s_sc[16 + w2]; } s_tot[0] = x; s_tot[1] = y; s_tot[2] = z; }
      __syncthreads();
      ag = s_tot[0]; ah = s_tot[1]; ac = s_tot[2];
    }
    long long pg = lg, ph = lh, pc = lc;
    d_block_excl3(pg, ph, pc, 0, s_sc);
    double base_g = 0.0, base_h = kEpsD; int base_c = 0;
    if (m.offset == 1) {   // implicit bin 0 = leaf total - everything stored  [UPSTREAM NA_AS_MISSING && offset==1]
      base_g = sum_g - static_cast<double>(ag) * inv_g;
      base_h = (sum_h - kEpsD) - static_cast<double>(ah) * inv_h;
      base_c = num_data - static_cast<int>(ac);
    }
    double f_gain = kNegInf, f_lg = 0, f_lh = 0; int f_thr = 1 << 30, f_lc = 0;
    for (int b = b0; b < b1; ++b) {
      if (b > hi) continue;
      if (b >= m.offset) { const long long qh = hist[b * 2 + 1]; pg += hist[b * 2]; ph += qh; pc += static_cast<int>(static_cast<double>(qh) * inv_h * cnt_factor + 0.5); }
      const double slg = base_g + static_cast<double>(pg) * inv_g;
      const double slh = base_h + static_cast<double>(ph) * inv_h;
      const int left_count = base_c + static_cast<int>(pc);
      if (left_count < p.min_data_in_leaf || slh < p.min_sum_hessian) continue;
      const int right_count = num_data - left_count;
      if (right_count < p.min_data_in_leaf) continue;
      const double srh = sum_h - slh;
      if (srh < p.min_sum_hessian) continue;
      const double srg = sum_g - slg;
      const double gain = d_leaf_gain(slg, slh, p) + d_leaf_gain(srg, srh, p);
      if (gain <= min_gain_shift) continue;
      any_valid = true;
      if (gain > f_gain) { f_gain = gain; f_lg = slg; f_lh = slh; f_thr = b; f_lc = left_count; }
    }
    for (int o = 16; o; o >>= 1) {
      const double og = __shfl_xor_sync(0xffffffffu, f_gain, o);
      const int ot = __shfl_xor_sync(0xffffffffu, f_thr, o);
      const double olg = __shfl_xor_sync(0xffffffffu, f_lg, o), olh = __shfl_xor_sync(0xffffffffu, f_lh, o);
      const int olc = __shfl_xor_sync(0xffffffffu, f_lc, o);
      if (og > f_gain || (og == f_gain && ot < f_thr)) { f_gain = og; f_thr = ot; f_lg = olg; f_lh = olh; f_lc = olc; }
    }
    if (lane == 0) { s_bg[warp] = f_gain; s_bt[warp] = f_thr; s_blg[warp] = f_lg; s_blh[warp] = f_lh; s_blc[warp] = f_lc; }
    __syncthreads();
    for (int w2 = 0; w2 < 8; ++w2)
      if (s_bg[w2] > f_gain || (s_bg[w2] == f_gain && s_bt[w2] < f_thr)) { f_gain = s_bg[w2]; f_thr = s_bt[w2]; f_lg = s_blg[w2]; f_lh = s_blh[w2]; f_lc = s_blc[w2]; }
    __syncthreads();
    if (f_gain > best_gain) { best_gain = f_gain; best_thr = f_thr; best_lg = f_lg; best_lh = f_lh; best_lc = f_lc; best_dl = 0; }
  } else if (m.missing_type == 2) {
    best_dl = 0;
  }
  if (any_valid) atomicOr(&s_any, 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    SplitCand& out = *outp;
    *flag = s_any ? 1 : 0;
    out.is_cat = 0; out.default_left = 1;
    if (s_any && best_gain > min_gain_shift) {
      out.gain = best_gain - min_gain_shift; out.left_g = best_lg; out.left_h = best_lh; out.threshold = best_thr;
      out.left_count = best_lc; out.default_left = best_dl;
    }
  }
}

// order of the wide categorical selection: side 0 ascending (key, bin), side 1 descending
__device__ __forceinline__ bool d_sel_prec(int side, double k, int b, double rk, int rb) {
  return side == 0 ? (k < rk || (k == rk && b < rb)) : (k > rk || (k == rk && b > rb));
}
constexpr int kSelList = 512;
// bitonic sort by 256 threads of TWO (key, id) arrays of n (power of two <= stride) entries: array 0 ascending, array 1 descending in
// (key, id); ends with a barrier
__device__ __noinline__ void d_block_bitonic2(double* k, int* id, int stride, int n) {
  for (int k2 = 2; k2 <= n; k2 <<= 1)
    for (int j = k2 >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int x = i ^ j;
        if (x <= i) continue;
        const bool up = (i & k2) == 0;
#pragma unroll
        for (int side = 0; side < 2; ++side) {
          double* kk = k + side * stride; int* ii = id + side * stride;
          const double ka = kk[i], kb = kk[x];
          const int ia = ii[i], ib = ii[x];
          const bool sw = up ? d_sel_prec(side, kb, ib, ka, ia) : d_sel_prec(side, ka, ia, kb, ib);
          if (sw) { kk[i] = kb; kk[x] = ka; ii[i] = ib; ii[x] = ia; }
        }
      }
    }
  __syncthreads();
}

// Split search of a WIDE categorical feature (FeatureHistogram::FindBestThresholdCategoricalInner, many-vs-many branch): one block per
// (smaller|larger, feature).  The histogram is reduced into the leaf's pool slot (parent - smaller for the larger child), the
// max_cat_threshold smallest and largest ctr = g / (h + cat_smooth) among the bins that hold >= cat_smooth rows are selected in the
// (ctr, bin) order of the reference's stable sort, and thread 0 accumulates from both ends exactly like the sequential code.
__global__ void __launch_bounds__(256)
k_scan_wide(const TreeCtrl* __restrict__ ctrl, const LeafState* __restrict__ leaves, const WideMeta* __restrict__ wm, const long long* __restrict__ H,
            long long* __restrict__ pool, size_t slot_elems, uint8_t* __restrict__ flags, SplitCand* __restrict__ cands, SplitParams p) {
  extern __shared__ __align__(16) unsigned char sw_smem[];
  double* s_key = reinterpret_cast<double*>(sw_smem);                          // [num_bin] ctr keys of the used bins, +inf otherwise
  __shared__ int s_used;
  const int which = blockIdx.y, w = blockIdx.x, u = p.nfn + w;
  const int leaf = which ? ctrl->larger : ctrl->smaller;
  if (!ctrl->go || leaf < 0) return;
  SplitCand out;
  out.gain = kNegInf; out.left_g = 0; out.left_h = 0; out.threshold = 0; out.left_count = 0; out.default_left = 0; out.feature = u;
  out.l2_extra = 0; out.is_cat = 1; out.cat_list_len = 0;
  for (int wd = 0; wd < 8; ++wd) out.cat_bits[wd] = 0u;
  uint8_t* flag = &flags[static_cast<size_t>(leaf) * p.nf_pad + u];
  if (!*flag) { if (threadIdx.x == 0) { cands[which * p.nf_pad + u] = out; __threadfence(); } return; }
  const WideMeta m = wm[w];
  const LeafState& L = leaves[leaf];
  const double inv_g = ctrl->inv_g, inv_h = ctrl->inv_h;
  long long* dst = pool + static_cast<size_t>(L.hist_slot) * slot_elems + static_cast<size_t>(m.hist_off) * 2;
  const long long* src = H + static_cast<size_t>(m.hist_off) * 2;
  const double sum_g = L.sum_g, sum_h = L.sum_h + 2 * kEpsD;
  const int num_data = L.global_count;
  const double cnt_factor = num_data / sum_h;
  if (!m.is_cat) {        // wide numerical feature (max_bin > 255): reduce into the pool slot, then the block-wide two-pass scan
    for (int b = threadIdx.x; b < m.num_bin; b += blockDim.x) {
      longlong2 sv = *reinterpret_cast<const longlong2*>(src + b * 2);
      if (which) { const longlong2 pr = *reinterpret_cast<const longlong2*>(dst + b * 2); sv.x = pr.x - sv.x; sv.y = pr.y - sv.y; }
      *reinterpret_cast<longlong2*>(dst + b * 2) = sv;
    }
    __syncthreads();      // every thread reads bins other threads reduced (same block: visible after the barrier)
    d_scan_wide_numeric(dst, m, L, inv_g, inv_h, p, flag, &out);
    if (threadIdx.x == 0) { cands[which * p.nf_pad + u] = out; __threadfence(); }
    return;
  }
  // ---- reduce into the pool slot and build the ctr keys (loads of 4 bins in flight per thread before the dependent stores)
  if (threadIdx.x == 0) s_used = 0;
  __syncthreads();
  int my_used = 0;
  const double kPosInf = __longlong_as_double(0x7ff0000000000000LL);      // unused bins: never selected
  for (int b0 = threadIdx.x; b0 < m.num_bin; b0 += 4 * blockDim.x) {
    longlong2 sv[4], pr[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int b = b0 + q * blockDim.x;
      if (b < m.num_bin) {
        sv[q] = *reinterpret_cast<const longlong2*>(src + b * 2);
        if (which) pr[q] = *reinterpret_cast<const longlong2*>(dst + b * 2);
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int b = b0 + q * blockDim.x;
      if (b >= m.num_bin) continue;
      longlong2 v = sv[q];
      if (which) { v.x = pr[q].x - v.x; v.y = pr[q].y - v.y; }
      *reinterpret_cast<longlong2*>(dst + b * 2) = v;
      const double g = static_cast<double>(v.x) * inv_g, h = static_cast<double>(v.y) * inv_h;
      const int cnt = static_cast<int>(h * cnt_factor + 0.5);
      double key = kPosInf;
      if (b >= 1 && cnt >= p.cat_smooth) { key = g / (h + p.cat_smooth); ++my_used; }
      s_key[b] = key;
    }
  }
  if (my_used) atomicAdd(&s_used, my_used);
  __syncthreads();
  const int used_bin = s_used;
  const int max_num_cat = min(min(p.max_cat_threshold, kCatListMax), (used_bin + 1) / 2);
  // ---- the reference sorts the used bins by (ctr, bin) and walks max_num_cat bins from either end; only those 2 * max_num_cat order
  // statistics are needed.  Sorting thousands of keys (first version: block-wide bitonic sort, ~600 us per launch) and selecting them
  // one per round (second version: 64 dependent rounds of a strided rescan, ~300 us — the rescan's latency is the same whether one
  // thread or all of them run it) both serialise on one SM.  Instead: (A) every thread takes the min and max of its own bins,
  // (B) the 256 per-thread minima (maxima) are sorted and the max_num_cat-th of them is a threshold that at least max_num_cat keys
  // reach, (C) the keys within the threshold are appended to a short list (typically max_num_cat + a few), (D) the list is sorted.
  // Three passes over the keys instead of 2 * max_num_cat.  The (key, bin) order is total, so the result equals the stable sort.
  __shared__ unsigned short s_sel[2][kCatListMax];
  __shared__ double s_selg[2][kCatListMax], s_selh[2][kCatListMax];
  __shared__ double s_rk[8];
  __shared__ int s_ri[8];
  __shared__ double s_tk[2][256], s_lk[2][kSelList];
  __shared__ int s_ti[2][256], s_li[2][kSelList];
  __shared__ int s_cnt[2];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  bool overflow = false;
  if (max_num_cat > 0) {
    double ak = kPosInf, zk = kNegInf; int ai = 0x7fffffff, zi = -1;
    for (int b = threadIdx.x; b < m.num_bin; b += blockDim.x) {
      const double k = s_key[b];
      if (!(k < kPosInf)) continue;
      if (k < ak) { ak = k; ai = b; }
      if (k >= zk) { zk = k; zi = b; }
    }
    s_tk[0][threadIdx.x] = ak; s_ti[0][threadIdx.x] = ai; s_tk[1][threadIdx.x] = zk; s_ti[1][threadIdx.x] = zi;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0;
    d_block_bitonic2(&s_tk[0][0], &s_ti[0][0], 256, 256);
    const double t0k = s_tk[0][max_num_cat - 1], t1k = s_tk[1][max_num_cat - 1];
    const int t0i = s_ti[0][max_num_cat - 1], t1i = s_ti[1][max_num_cat - 1];
    for (int b = threadIdx.x; b < m.num_bin; b += blockDim.x) {
      const double k = s_key[b];
      if (!(k < kPosInf)) continue;
      if (!d_sel_prec(0, t0k, t0i, k, b)) { const int pos = atomicAdd(&s_cnt[0], 1); if (pos < kSelList) { s_lk[0][pos] = k; s_li[0][pos] = b; } }
      if (!d_sel_prec(1, t1k, t1i, k, b)) { const int pos = atomicAdd(&s_cnt[1], 1); if (pos < kSelList) { s_lk[1][pos] = k; s_li[1][pos] = b; } }
    }
    __syncthreads();
    const int n0 = s_cnt[0], n1 = s_cnt[1];
    overflow = n0 > kSelList || n1 > kSelList;      // e.g. all small keys on bins congruent mod 256: fall back to the round-based selection
    if (!overflow) {
      int n2 = 2;
      while (n2 < n0 || n2 < n1) n2 <<= 1;
      for (int i = threadIdx.x; i < n2; i += blockDim.x) {
        if (i >= n0) { s_lk[0][i] = kPosInf; s_li[0][i] = 0x7fffffff; }
        if (i >= n1) { s_lk[1][i] = kNegInf; s_li[1][i] = -1; }
      }
      d_block_bitonic2(&s_lk[0][0], &s_li[0][0], kSelList, n2);
      if (threadIdx.x < 2 * max_num_cat) {
        const int side = threadIdx.x / max_num_cat, i = threadIdx.x - side * max_num_cat;
        s_sel[side][i] = static_cast<unsigned short>(s_li[side][i]);
      }
    }
  }
  // fallback (list overflow): tournament — every thread keeps the best remaining key of ITS bins (b = tid + 256 j); a round reduces the
  // 256 cached candidates and only the winner's owner rescans its own bins
  if (overflow)
  for (int side = 0; side < 2; ++side) {
    auto better = [&](double k, int b, double rk, int rb) -> bool {      // (k, b) precedes (rk, rb) on this side; rb sentinel = nothing yet
      if (side == 0) return rb == 0x7fffffff || k < rk || (k == rk && b < rb);
      return rb == -1 || k > rk || (k == rk && b > rb);
    };
    auto own_next = [&](double pk, int pi, double* ok, int* oi) {         // best own key strictly beyond (pk, pi)
      double bk = 0.0; int bi = side == 0 ? 0x7fffffff : -1;
      for (int b = threadIdx.x; b < m.num_bin; b += blockDim.x) {
        const double k = s_key[b];
        if (!(k < kPosInf)) continue;
        const bool beyond = side == 0 ? (k > pk || (k == pk && b > pi)) : (k < pk || (k == pk && b < pi));
        if (beyond && better(k, b, bk, bi)) { bk = k; bi = b; }
      }
      *ok = bk; *oi = bi;
    };
    const int none = side == 0 ? 0x7fffffff : -1;
    double ck; int ci;
    own_next(side == 0 ? kNegInf : kPosInf, side == 0 ? -1 : 0x7fffffff, &ck, &ci);
    for (int r = 0; r < max_num_cat; ++r) {
      double bk = ck; int bi = ci;
      for (int o = 16; o; o >>= 1) {
        const double ok = __shfl_xor_sync(0xffffffffu, bk, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi != none && better(ok, oi, bk, bi)) { bk = ok; bi = oi; }
      }
      if (lane == 0) { s_rk[warp] = bk; s_ri[warp] = bi; }
      __syncthreads();
      bk = s_rk[0]; bi = s_ri[0];
      for (int w2 = 1; w2 < 8; ++w2) if (s_ri[w2] != none && better(s_rk[w2], s_ri[w2], bk, bi)) { bk = s_rk[w2]; bi = s_ri[w2]; }
      __syncthreads();
      if (threadIdx.x == 0) s_sel[side][r] = static_cast<unsigned short>(bi);      // exists: r < max_num_cat <= used_bin
      if (bi != none && (bi & 255) == static_cast<int>(threadIdx.x)) own_next(bk, bi, &ck, &ci);      // only the owner of the winner moves on
    }
  }
  __syncthreads();
  if (threadIdx.x < 2 * max_num_cat) {
    const int side = threadIdx.x / max_num_cat, i = threadIdx.x - side * max_num_cat;
    const int t = s_sel[side][i];
    s_selg[side][i] = static_cast<double>(dst[t * 2]) * inv_g;
    s_selh[side][i] = static_cast<double>(dst[t * 2 + 1]) * inv_h;
  }
  __syncthreads();
  // the walk from either end is sequential only in its cheap state (running sums, the min_data_per_group counter, continue / break); lane 0
  // of warps 0 and 1 run it for one direction each and mark the prefixes the reference evaluates, the gains (fp64 divisions) are then
  // computed one prefix per thread, and thread 0 takes the first maximum in the reference's (direction, i) order
  __shared__ double s_plg[2][kCatListMax], s_plh[2][kCatListMax], s_pgain[2][kCatListMax];
  __shared__ int s_plc[2][kCatListMax];
  if (threadIdx.x < 2 * kCatListMax) s_pgain[threadIdx.x / kCatListMax][threadIdx.x % kCatListMax] = kNegInf;
  __syncthreads();
  if (lane == 0 && warp < 2) {
    const int d = warp;
    int cnt_cur_group = 0, left_count = 0;
    double slg = 0.0, slh = kEpsD;
    for (int i = 0; i < used_bin && i < max_num_cat; ++i) {
      const double g = s_selg[d][i], h = s_selh[d][i];
      const int cnt = static_cast<int>(h * cnt_factor + 0.5);
      slg += g; slh += h; left_count += cnt; cnt_cur_group += cnt;
      if (left_count < p.min_data_in_leaf || slh < p.min_sum_hessian) continue;
      const int right_count = num_data - left_count;
      if (right_count < p.min_data_in_leaf || right_count < p.min_data_per_group) break;
      const double srh = sum_h - slh;
      if (srh < p.min_sum_hessian) break;
      if (cnt_cur_group < p.min_data_per_group) continue;
      cnt_cur_group = 0;
      s_plg[d][i] = slg; s_plh[d][i] = slh; s_plc[d][i] = left_count; s_pgain[d][i] = 0.0;      // 0.0 = "evaluate me"
    }
  }
  __syncthreads();
  SplitParams pshift = p;
  if (!(p.max_delta_step > 0)) pshift.max_delta_step = 0;
  const double min_gain_shift = d_leaf_gain(sum_g, sum_h, pshift) + p.min_gain_to_split;
  if (threadIdx.x < 2 * kCatListMax) {
    const int d = threadIdx.x / kCatListMax, i = threadIdx.x % kCatListMax;
    if (s_pgain[d][i] == 0.0) {
      SplitParams pc = p;
      pc.l2 += p.cat_l2;
      const double slg = s_plg[d][i], slh = s_plh[d][i];
      s_pgain[d][i] = d_leaf_gain(slg, slh, pc) + d_leaf_gain(sum_g - slg, sum_h - slh, pc);
    }
  }
  __syncthreads();
  if (threadIdx.x != 0) return;
  bool any_valid = false;
  double best_gain = kNegInf, best_lg = 0, best_lh = 0;
  int best_i = -1, best_dir = 1, best_lc = 0;
  for (int d = 0; d < 2; ++d)
    for (int i = 0; i < max_num_cat; ++i) {
      const double gain = s_pgain[d][i];
      if (!(gain > min_gain_shift)) continue;      // also skips the -inf of the prefixes the walk did not evaluate
      any_valid = true;
      if (gain > best_gain) { best_gain = gain; best_lg = s_plg[d][i]; best_lh = s_plh[d][i]; best_lc = s_plc[d][i]; best_i = i; best_dir = d == 0 ? 1 : -1; }
    }
  *flag = any_valid ? 1 : 0;
  if (any_valid) {
    out.gain = best_gain - min_gain_shift; out.left_g = best_lg; out.left_h = best_lh; out.threshold = 0; out.left_count = best_lc;
    out.default_left = 0; out.is_cat = 1; out.l2_extra = p.cat_l2;
    out.cat_list_len = best_i + 1;
    for (int i = 0; i <= best_i && i < kCatListMax; ++i) out.cat_list[i] = s_sel[best_dir == 1 ? 0 : 1][i];
  }
  cands[which * p.nf_pad + u] = out;
  __threadfence();
}

// ---------------------------------------------------------------- K5/K6 for the tile features: one BLOCK per (smaller|larger, feature)
// Thread t = bin t.  The block reduces the feature into the leaf's pool slot (larger child: parent - smaller, exact int64), then runs the
// same block-wide two-pass scan as the wide numerical features (d_scan_wide_numeric with one bin per thread: exclusive block scans of
// (g, h, count), one candidate per thread and direction, block argmax with the sequential tie-breaks) — the dependent chain of software
// fp64 divisions per thread is 2 long instead of 16 as in the round-1 warp-per-feature scan, and the code is shared and small (the old
// kernel was instruction-fetch bound).  Categorical tile features keep the warp-level search (d_scan_feature_cat) on warp 0.  The block that
// finishes last picks the best candidate per leaf and the next leaf to split.
__global__ void __launch_bounds__(256, 4)
k_scan(TreeCtrl* ctrl, LeafState* leaves, const FeatMeta* __restrict__ meta,
       const long long* __restrict__ H, long long* __restrict__ pool, size_t slot_elems, uint8_t* __restrict__ flags,
       SplitCand* cands, SplitParams p) {
  const int which = blockIdx.y;
  const int leaf = which ? ctrl->larger : ctrl->smaller;
  const int u = blockIdx.x;
  if (ctrl->go && leaf >= 0 && u < p.nfn) {
    SplitCand out;
    out.gain = kNegInf; out.left_g = 0; out.left_h = 0; out.threshold = 0; out.left_count = 0; out.default_left = 1; out.feature = u;
    out.l2_extra = 0; out.is_cat = 0; out.cat_list_len = 0;
    for (int wd = 0; wd < 8; ++wd) out.cat_bits[wd] = 0u;
    uint8_t* flag = &flags[static_cast<size_t>(leaf) * p.nf_pad + u];
    if (*flag) {
      const LeafState& L = leaves[leaf];
      const FeatMeta fm = meta[u];
      long long* dst = pool + static_cast<size_t>(L.hist_slot) * slot_elems + static_cast<size_t>(u) * 512;
      const long long* src = H + static_cast<size_t>(u) * 512;
      {
        const int b = threadIdx.x;
        longlong2 sv = *reinterpret_cast<const longlong2*>(src + b * 2);
        if (which) { const longlong2 pr = *reinterpret_cast<const longlong2*>(dst + b * 2); sv.x = pr.x - sv.x; sv.y = pr.y - sv.y; }
        *reinterpret_cast<longlong2*>(dst + b * 2) = sv;
      }
      __syncthreads();      // the scan reads bins other threads of this block reduced
      if (!fm.is_categorical) {
        const WideMeta wm{fm.num_bin, 0, 0, 0, fm.default_bin, fm.missing_type, fm.real_index, 0, fm.offset, 0, 0, 0};
        d_scan_wide_numeric(dst, wm, L, ctrl->inv_g, ctrl->inv_h, p, flag, &out);
      } else if (threadIdx.x < 32) {
        extern __shared__ double scan_ws[];      // (3*256 doubles + 2*256 bytes) of scratch for the categorical search
        long long qg[8], qh[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) { const int b = threadIdx.x * 8 + j; qg[j] = dst[b * 2]; qh[j] = dst[b * 2 + 1]; }
        d_scan_feature_cat(qg, qh, threadIdx.x, fm, L, ctrl->inv_g, ctrl->inv_h, p, flag, &out, scan_ws);
      }
    }
    if (threadIdx.x == 0) { cands[which * p.nf_pad + u] = out; __threadfence(); }      // visible to the block that runs the pick step
  }
  __shared__ int s_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned t = atomicAdd(&ctrl->scan_ticket, 1u);
    s_last = (t == gridDim.x * gridDim.y - 1) ? 1 : 0;
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    d_pick_block(ctrl, leaves, meta, cands, p);
    if (threadIdx.x == 0) ctrl->scan_ticket = 0u;
  }
}

// ---------------------------------------------------------------- K8/K9 leaf values -> scores
// score[row] += shrinkage * leaf_value[leaf(row)], via the final data partition
__global__ void __launch_bounds__(256)
k_add_score(const TreeCtrl* __restrict__ ctrl, const LeafState* __restrict__ leaves, TreeDev tree, const int* __restrict__ idx0,
            const int* __restrict__ idx1, double* __restrict__ score, double shrinkage) {
  const int nl = ctrl->num_leaves;
  if (nl <= 1) return;
  for (int l = 0; l < nl; ++l) {
    const LeafState& L = leaves[l];
    double v = tree.leaf_value[l] * shrinkage;
    if (!(fabs(v) > 1e-35)) v = 0.0;
    const int* src = L.buf ? idx1 : idx0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L.count; i += gridDim.x * blockDim.x) {
      const int r = L.identity ? (L.begin + i) : src[L.begin + i];
      score[r] += v;
    }
  }
}
__global__ void k_add_const(double* __restrict__ score, int n, double v) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) score[i] += v;
}
// score of a (validation) dataset += shrinkage * tree(row), traversing by bin thresholds
__global__ void __launch_bounds__(256)
k_add_tree_binned(TreeDev tree, const FeatMeta* __restrict__ meta, BinView bv, int n,
                  double* __restrict__ score, double shrinkage, double bias = 0.0, double pre_mul = 1.0, double post_mul = 1.0) {
  const int nl = *tree.num_leaves;
  if (nl <= 1) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int node = 0;
    while (node >= 0) {
      const int f = tree.split_feature_inner[node];
      const unsigned bin = bv.at(f, static_cast<size_t>(i));
      const int dt = tree.decision_type[node];
      bool left;
      if (dt & 1) {
        if (f >= bv.nfn) {      // wide feature: short list of bins
          left = false;
          const int len = tree.cat_list_len[node];
          for (int k = 0; k < len; ++k) left |= (bin == tree.cat_list[node * kCatListMax + k]);
        } else {
          left = (tree.cat_bits[node * 8 + (bin >> 5)] >> (bin & 31u)) & 1u;
        }
      }
      else if (((dt >> 2) & 3) == 2 && bin == static_cast<unsigned>(meta[f].num_bin - 1)) left = dt & 2;
      else left = bin <= static_cast<unsigned>(tree.threshold_bin[node]);
      node = left ? tree.left_child[node] : tree.right_child[node];
    }
    double v = tree.leaf_value[~node] * shrinkage;
    if (!(fabs(v) > 1e-35)) v = 0.0;
    score[i] = (score[i] * pre_mul + (v + bias)) * post_mul;      // rf: running average of (tree + init score); gbdt: pre = post = 1, bias = 0
  }
}
__global__ void k_scale_add(double* __restrict__ score, int n, double pre_mul, double add, double post_mul) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) score[i] = (score[i] * pre_mul + add) * post_mul;
}

// ---------------------------------------------------------------- row subsampling: bagging / GOSS  (SURVEY §8f-3)
// [LightGBM src/boosting/gbdt.cpp GBDT::BaggingHelper, goss.hpp GOSS::BaggingHelper] Rows are drawn per 1024-row block, every block
// owning an LCG (x <- 214013 x + 2531011, float = ((x >> 16) & 0x7fff) / 32768) seeded bagging_seed + block. One CUDA block per
// 1024-row block. The draw of row j of a block is the (j+1)-th LCG output, which the jump table gives directly:
// x_{j+1} = mulA[j] * x0 + addC[j], so plain bagging is embarrassingly parallel and still bit-identical to the sequential draw.
constexpr int kBagBlock = 1024;
struct LcgJump { unsigned mul[kBagBlock]; unsigned add[kBagBlock]; };
__device__ __forceinline__ float d_lcg_float(unsigned x) { return static_cast<float>((x >> 16) & 0x7FFFu) / 32768.0f; }

__global__ void __launch_bounds__(256)
k_bag_draw(unsigned* __restrict__ lcg_state, const LcgJump* __restrict__ jump, int n, double fraction, uint8_t* __restrict__ in_bag,
           int* __restrict__ block_count, const float* __restrict__ label = nullptr, double pos_fraction = 1.0, double neg_fraction = 1.0) {
  const int b = blockIdx.x, base = b * kBagBlock, cnt = min(kBagBlock, n - base);
  const unsigned x0 = lcg_state[b];
  int mine = 0;
  for (int j = threadIdx.x; j < cnt; j += blockDim.x) {
    const unsigned x = jump->mul[j] * x0 + jump->add[j];
    // balanced bagging (label given): positives and negatives are kept with their own fractions [LightGBM BalancedBaggingHelper]
    const double frac = label ? (label[base + j] > 0 ? pos_fraction : neg_fraction) : fraction;
    const int take = static_cast<double>(d_lcg_float(x)) < frac;
    in_bag[base + j] = static_cast<uint8_t>(take);
    mine += take;
  }
  __shared__ int s_cnt;
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  for (int o = 16; o; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
  if ((threadIdx.x & 31) == 0) atomicAdd(&s_cnt, mine);
  __syncthreads();
  if (threadIdx.x == 0) { block_count[b] = s_cnt; lcg_state[b] = jump->mul[cnt - 1] * x0 + jump->add[cnt - 1]; }
}

// GOSS: keep the top_rate share of rows by sum_k |g*h| and sample other_rate of the rest, amplifying the sampled gradients by
// (cnt - top_k) / other_k.  The running probability depends on how many rows were sampled so far, so the draw is sequential inside
// a 1024-row chunk (thread 0); threshold selection (bitonic sort) and the gradient scaling are parallel.
__global__ void __launch_bounds__(256)
k_goss_draw(unsigned* __restrict__ lcg_state, int n, int K, double top_rate, double other_rate, float* __restrict__ grad,
            float* __restrict__ hess, uint8_t* __restrict__ in_bag, int* __restrict__ block_count) {
  __shared__ float s_tg[kBagBlock];
  __shared__ float s_sorted[kBagBlock];
  __shared__ uint8_t s_flag[kBagBlock];      // 0 out, 1 top, 2 sampled (amplified)
  __shared__ int s_left;
  const int b = blockIdx.x, base = b * kBagBlock, cnt = min(kBagBlock, n - base);
  for (int j = threadIdx.x; j < kBagBlock; j += blockDim.x) {
    float t = -1.0f;        // padding sorts last (real values are >= 0)
    if (j < cnt) {
      t = 0.0f;
      for (int k = 0; k < K; ++k) { const size_t id = static_cast<size_t>(k) * n + base + j; t = __fadd_rn(t, fabsf(__fmul_rn(grad[id], hess[id]))); }
    }
    s_tg[j] = t; s_sorted[j] = t;
  }
  __syncthreads();
  for (int k = 2; k <= kBagBlock; k <<= 1)            // bitonic sort, descending
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < kBagBlock; i += blockDim.x) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const float a = s_sorted[i], c = s_sorted[ixj];
          const bool desc = (i & k) == 0;
          if (desc ? (a < c) : (a > c)) { s_sorted[i] = c; s_sorted[ixj] = a; }
        }
      }
      __syncthreads();
    }
  const int top_k = max(1, static_cast<int>(cnt * top_rate));
  const int other_k = static_cast<int>(cnt * other_rate);
  const float multiply = static_cast<float>(cnt - top_k) / other_k;
  if (threadIdx.x == 0) {
    const float threshold = s_sorted[top_k - 1];
    unsigned x = lcg_state[b];
    int left = 0, big = 0;
    for (int i = 0; i < cnt; ++i) {
      uint8_t f = 0;
      if (s_tg[i] >= threshold) { f = 1; ++left; ++big; }
      else {
        const int rest_need = other_k - (left - big), rest_all = (cnt - i) - (top_k - big);
        const double prob = rest_need / static_cast<double>(rest_all);
        x = 214013u * x + 2531011u;
        if (static_cast<double>(d_lcg_float(x)) < prob) { f = 2; ++left; }
      }
      s_flag[i] = f;
    }
    lcg_state[b] = x;
    s_left = left;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < cnt; j += blockDim.x) {
    const uint8_t f = s_flag[j];
    in_bag[base + j] = f ? 1 : 0;
    if (f == 2)
      for (int k = 0; k < K; ++k) { const size_t id = static_cast<size_t>(k) * n + base + j; grad[id] = __fmul_rn(grad[id], multiply); hess[id] = __fmul_rn(hess[id], multiply); }
  }
  if (threadIdx.x == 0) block_count[b] = s_left;
}

// exclusive scan of the per-block in-bag counts (single CTA), total -> *bag_total
__global__ void __launch_bounds__(1024)
k_bag_scan(int* __restrict__ block_count, int nblocks, int* __restrict__ bag_total) {
  __shared__ int s_warp[32];
  __shared__ int s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  for (int base = 0; base < nblocks; base += 1024) {
    const int i = base + threadIdx.x;
    const int v = i < nblocks ? block_count[i] : 0;
    int incl = v;
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if ((threadIdx.x & 31) >= o) incl += t; }
    if ((threadIdx.x & 31) == 31) s_warp[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
      int w = s_warp[threadIdx.x];
      for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, w, o); if (threadIdx.x >= o) w += t; }
      s_warp[threadIdx.x] = w;
    }
    __syncthreads();
    const int warp_off = (threadIdx.x >> 5) ? s_warp[(threadIdx.x >> 5) - 1] : 0;
    const int carry = s_carry;
    if (i < nblocks) block_count[i] = carry + warp_off + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) s_carry = carry + warp_off + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) *bag_total = s_carry;
}
// ordered compaction: bag_idx[offset(block) + rank-in-block] = row
__global__ void __launch_bounds__(256)
k_bag_compact(const uint8_t* __restrict__ in_bag, const int* __restrict__ block_offset, int n, int* __restrict__ bag_idx) {
  __shared__ int s_warp[8];
  __shared__ int s_base;
  const int b = blockIdx.x, base = b * kBagBlock, cnt = min(kBagBlock, n - base);
  if (threadIdx.x == 0) s_base = block_offset[b];
  __syncthreads();
  for (int j0 = 0; j0 < cnt; j0 += blockDim.x) {
    const int j = j0 + threadIdx.x;
    const int take = (j < cnt) ? in_bag[base + j] : 0;
    const unsigned m = __ballot_sync(0xffffffffu, take);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) s_warp[warp] = __popc(m);
    __syncthreads();
    int off = s_base;
    for (int w = 0; w < warp; ++w) off += s_warp[w];
    if (take) bag_idx[off + __popc(m & ((1u << lane) - 1u))] = base + j;
    __syncthreads();
    if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 8; ++w) t += s_warp[w]; s_base += t; }
    __syncthreads();
  }
}

// ---------------------------------------------------------------- batched prediction (SURVEY §8f-2)
// Flattened forest on the device; one thread per (row, class) walks the trees of its class in model order, so the raw
// score is the same sequence of fp64 additions as the host predictor (HostModel::PredictRow) => bit-identical.
struct ForestDev {
  const int* tree_offset;        // [num_trees+1] node offset of each tree (a tree with L leaves has L-1 nodes)
  const int* leaf_offset;        // [num_trees+1]
  const int* num_leaves;         // [num_trees]
  const int* split_feature;      // per node: real feature index
  const double* threshold;
  const int* decision_type;
  const int* left_child;
  const int* right_child;
  const double* leaf_value;
  const int* cat_begin;          // per node: categorical nodes index their category bitset in cat_words
  const int* cat_len;
  const unsigned* cat_words;
  const double* node_count;      // per node: rows that reached it in training (TreeSHAP cover)
  const double* leaf_count;      // per leaf
  const double* expected;        // per tree: count-weighted mean leaf value
};
// child of global node g for this row (Tree::Decision: numerical with missing handling, or categorical bitset)
template <typename T>
__device__ __forceinline__ int d_node_child(const ForestDev& f, int g, const T* __restrict__ row) {
  double fval = static_cast<double>(row[f.split_feature[g]]);
  const int dt = f.decision_type[g];
  const int mt = (dt >> 2) & 3;
  bool left;
  if (dt & 1) {                 // categorical decision
    left = false;
    if (!(isnan(fval) && mt == 2)) {
      const int iv = isnan(fval) ? 0 : static_cast<int>(fval);
      const int w = iv >> 5;
      if (iv >= 0 && w < f.cat_len[g]) left = (f.cat_words[f.cat_begin[g] + w] >> (iv & 31)) & 1u;
    }
    return left ? f.left_child[g] : f.right_child[g];
  }
  if (isnan(fval) && mt != 2) fval = 0.0;
  if ((mt == 1 && fabs(fval) <= 1e-35) || (mt == 2 && isnan(fval))) left = (dt & 2) != 0;
  else left = fval <= f.threshold[g];
  return left ? f.left_child[g] : f.right_child[g];
}
template <typename T>
__device__ __forceinline__ int d_tree_leaf(const ForestDev& f, int t, const T* __restrict__ row) {
  if (f.num_leaves[t] <= 1) return 0;
  const int nb = f.tree_offset[t];
  int node = 0;
  while (node >= 0) node = d_node_child(f, nb + node, row);
  return ~node;
}
template <typename T>
__global__ void __launch_bounds__(256)
k_predict_raw(ForestDev f, const T* __restrict__ X, long long nrow, int ncol, int K, int t0, int t1, double* __restrict__ out) {
  const long long total = nrow * K;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total; e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = e / K;
    const int k = static_cast<int>(e - r * K);
    const T* row = X + r * ncol;
    double acc = 0.0;
    for (int t = t0 + k; t < t1; t += K) acc += f.leaf_value[f.leaf_offset[t] + d_tree_leaf(f, t, row)];
    out[e] = acc;
  }
}
template <typename T>
__global__ void __launch_bounds__(256)
k_predict_leaf(ForestDev f, const T* __restrict__ X, long long nrow, int ncol, int t0, int t1, double* __restrict__ out) {
  const int nt = t1 - t0;
  const long long total = nrow * nt;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total; e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long r = e / nt;
    const int t = t0 + static_cast<int>(e - r * nt);
    out[e] = static_cast<double>(d_tree_leaf(f, t, X + r * ncol));
  }
}

// histogram int64 -> fp64 (debug / parity export)
// ---------------------------------------------------------------- batched TreeSHAP (C_API_PREDICT_CONTRIB)
// One thread per row walks every tree of the model in model order with the path-dependent TreeSHAP recursion of Lundberg et al.
// (the algorithm behind [UPSTREAM] Tree::PredictContrib), turned into an explicit stack: a frame = (node, unique depth, parent
// path offset, zero/one fractions, feature).  The hot child is expanded before the cold one, children write their paths
// behind the parent's, so the parent's path is still intact when the cold frame is popped.  Same fp64 operation order as the host
// predictor (HostTree::ShapRecurse) => identical contributions.  Scratch per thread: path_stride PathElem + frame_stride frames.
struct ShapPathElem { int feature; int pad; double zf, of, pw; };
struct ShapFrame { int node, depth, parent_off, feature; double pzf, pof; };

__device__ __forceinline__ void d_shap_extend(ShapPathElem* p, int depth, double zf, double of, int fi) {
  p[depth].feature = fi; p[depth].zf = zf; p[depth].of = of; p[depth].pw = depth == 0 ? 1.0 : 0.0;
  for (int i = depth - 1; i >= 0; --i) {
    p[i + 1].pw += of * p[i].pw * (i + 1) / static_cast<double>(depth + 1);
    p[i].pw = zf * p[i].pw * (depth - i) / static_cast<double>(depth + 1);
  }
}
__device__ __forceinline__ void d_shap_unwind(ShapPathElem* p, int depth, int pi) {
  const double of = p[pi].of, zf = p[pi].zf;
  double next = p[depth].pw;
  for (int i = depth - 1; i >= 0; --i) {
    if (of != 0) {
      const double tmp = p[i].pw;
      p[i].pw = next * (depth + 1) / static_cast<double>((i + 1) * of);
      next = tmp - p[i].pw * zf * (depth - i) / static_cast<double>(depth + 1);
    } else {
      p[i].pw = (p[i].pw * (depth + 1)) / static_cast<double>(zf * (depth - i));
    }
  }
  for (int i = pi; i < depth; ++i) { p[i].feature = p[i + 1].feature; p[i].zf = p[i + 1].zf; p[i].of = p[i + 1].of; }
}
__device__ __forceinline__ double d_shap_unwound_sum(const ShapPathElem* p, int depth, int pi) {
  const double of = p[pi].of, zf = p[pi].zf;
  double next = p[depth].pw, total = 0;
  for (int i = depth - 1; i >= 0; --i) {
    if (of != 0) {
      const double tmp = next * (depth + 1) / static_cast<double>((i + 1) * of);
      total += tmp;
      next = p[i].pw - tmp * zf * ((depth - i) / static_cast<double>(depth + 1));
    } else {
      total += (p[i].pw / zf) / ((depth - i) / static_cast<double>(depth + 1));
    }
  }
  return total;
}
template <typename T>
__global__ void __launch_bounds__(128)
k_predict_contrib(ForestDev f, const T* __restrict__ X, long long nrow, int ncol, int K, int t0, int t1, int F1, ShapPathElem* __restrict__ path_scratch,
                  int path_stride, ShapFrame* __restrict__ frame_scratch, int frame_stride, double* __restrict__ out) {
  const long long tid = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
  ShapPathElem* const base = path_scratch + tid * path_stride;
  ShapFrame* const stack = frame_scratch + tid * frame_stride;
  for (long long r = tid; r < nrow; r += static_cast<long long>(gridDim.x) * blockDim.x) {
    const T* row = X + r * ncol;
    for (int t = t0; t < t1; ++t) {
      double* phi = out + (r * K + (t % K)) * F1;
      phi[F1 - 1] += f.expected[t];
      if (f.num_leaves[t] <= 1) continue;
      const int nb = f.tree_offset[t], lb = f.leaf_offset[t];
      int sp = 0;
      stack[sp++] = ShapFrame{0, 0, 0, -1, 1.0, 1.0};
      while (sp > 0) {
        const ShapFrame fr = stack[--sp];
        int depth = fr.depth;
        ShapPathElem* path = base + fr.parent_off + depth;
        const ShapPathElem* parent = base + fr.parent_off;
        for (int i = 0; i < depth; ++i) path[i] = parent[i];
        d_shap_extend(path, depth, fr.pzf, fr.pof, fr.feature);
        if (fr.node < 0) {
          const double lv = f.leaf_value[lb + ~fr.node];
          for (int i = 1; i <= depth; ++i) {
            const double w = d_shap_unwound_sum(path, depth, i);
            phi[path[i].feature] += w * (path[i].of - path[i].zf) * lv;
          }
          continue;
        }
        const int g = nb + fr.node;
        const int hot = d_node_child(f, g, row);
        const int cold = hot == f.left_child[g] ? f.right_child[g] : f.left_child[g];
        const double w = f.node_count[g];
        const double hot_zf = (hot >= 0 ? f.node_count[nb + hot] : f.leaf_count[lb + ~hot]) / w;
        const double cold_zf = (cold >= 0 ? f.node_count[nb + cold] : f.leaf_count[lb + ~cold]) / w;
        double inc_zf = 1, inc_of = 1;
        const int sf = f.split_feature[g];
        int pi = 0;
        for (; pi <= depth; ++pi) if (path[pi].feature == sf) break;
        if (pi != depth + 1) {
          inc_zf = path[pi].zf; inc_of = path[pi].of;
          d_shap_unwind(path, depth, pi);
          depth -= 1;
        }
        const int off = static_cast<int>(path - base);
        stack[sp++] = ShapFrame{cold, depth + 1, off, sf, cold_zf * inc_zf, 0.0};
        stack[sp++] = ShapFrame{hot, depth + 1, off, sf, hot_zf * inc_zf, inc_of};
      }
    }
  }
}

__global__ void k_hist_to_double(const long long* __restrict__ H, double* __restrict__ out, size_t elems, const TreeCtrl* ctrl) {
  const double ig = ctrl->inv_g, ih = ctrl->inv_h;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < elems; i += static_cast<size_t>(gridDim.x) * blockDim.x)
    out[i] = static_cast<double>(H[i]) * ((i & 1) ? ih : ig);
}

}  // namespace b200gbm
