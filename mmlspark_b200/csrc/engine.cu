// b200gbm engine implementation: network bootstrap, dataset ingestion/binning, GBDT driver and the
// device-resident leaf-wise tree learner.  See engine.h / kernels.cuh / hist_kernel.cuh.
#include "engine.h"
#include "objective.cuh"
#include "renew_kernel.cuh"
#include "metric_kernels.cuh"

#include <nvtx3/nvToolsExt.h>      // header-only NVTX v3: ranges are no-ops unless a profiler injects itself

#include <arpa/inet.h>
#include <netdb.h>
#include <netinet/in.h>
#include <netinet/tcp.h>
#include <sys/select.h>
#include <sys/socket.h>
#include <unistd.h>
#include <sys/types.h>

#include <algorithm>
#include <chrono>
#include <functional>
#include <mutex>
#include <omp.h>
#include <cstring>
#include <numeric>
#include <thread>

namespace b200gbm {

// NVTX ranges named after the kernel / collective numbering of SURVEY.md §2.5 (K1..K9, C1..C5): `nsys`/`ncu --nvtx` can filter on them
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
};

// =============================================================================== device / network
static thread_local int t_device = -1;
static thread_local Network t_net;
Network& Net() { return t_net; }

// Host-side OpenMP loops (bin finding on the sample, batch predict) must respect the container's CPU
// quota: the GPU box shows 128 logical CPUs behind a 16-core cgroup quota and oversubscribed OpenMP
// teams there are ~100x slower.
static void CapHostThreadsOnce() {
  static std::once_flag once;
  std::call_once(once, [] {
    int n = omp_get_max_threads();
    FILE* f = std::fopen("/sys/fs/cgroup/cpu.max", "r");
    if (f) {
      char q[64] = {0};
      long long period = 0;
      if (std::fscanf(f, "%63s %lld", q, &period) == 2 && std::strcmp(q, "max") != 0 && period > 0) {
        long long quota = std::atoll(q);
        n = static_cast<int>(std::max<long long>(1, std::min<long long>(n, quota / period)));
      }
      std::fclose(f);
    }
    omp_set_num_threads(n);
  });
}

static int DeviceCountOrDie() {
  CapHostThreadsOnce();
  int cnt = 0;
  cudaError_t e = cudaGetDeviceCount(&cnt);
  if (e != cudaSuccess || cnt <= 0)
    Fatal(std::string("b200gbm: no CUDA device available (") + cudaGetErrorString(e) +
          "). This engine is CUDA-only (sm_100a); there is no CPU fallback.");
  return cnt;
}
int CurrentDevice() {
  if (t_device < 0) {
    int cnt = DeviceCountOrDie();
    const char* lr = std::getenv("LOCAL_RANK");
    t_device = (lr ? std::atoi(lr) : 0) % cnt;
  }
  return t_device;
}
void SetThreadDevice(int ordinal) {
  int cnt = DeviceCountOrDie();
  if (ordinal < 0 || ordinal >= cnt) Fatal("b200gbm: device ordinal out of range");
  t_device = ordinal;
}
void EnsureDevice() { B200_CUDA(cudaSetDevice(CurrentDevice())); }

static void SendAll(int fd, const void* buf, size_t n) {
  const char* p = static_cast<const char*>(buf);
  while (n) { ssize_t k = ::send(fd, p, n, 0); if (k <= 0) Fatal("network bootstrap: send failed"); p += k; n -= k; }
}
static void RecvAll(int fd, void* buf, size_t n) {
  char* p = static_cast<char*>(buf);
  while (n) { ssize_t k = ::recv(fd, p, n, 0); if (k <= 0) Fatal("network bootstrap: recv failed"); p += k; n -= k; }
}

// Replaces LGBM_NetworkInit's TCP mesh (reference call site TrainUtils.scala:279-295): the machine list
// is only used to agree on ranks and to hand rank 0's ncclUniqueId to the others over one TCP
// connection each; all training traffic then goes over NCCL (NVLink / NVSwitch).
void NetworkInit(const char* machines, int local_listen_port, int listen_time_out_sec, int num_machines) {
  NetworkFree();
  if (num_machines <= 1) return;
  std::vector<std::pair<std::string, int>> nodes;
  {
    std::string s(machines ? machines : "");
    for (auto& c : s) if (c == ' ' || c == ';') c = ',';
    std::stringstream ss(s);
    std::string tok;
    while (std::getline(ss, tok, ',')) {
      if (tok.empty()) continue;
      size_t p = tok.rfind(':');
      if (p == std::string::npos) Fatal("machines should be a list of ip:port, got '" + tok + "'");
      nodes.emplace_back(tok.substr(0, p), std::atoi(tok.c_str() + p + 1));
    }
  }
  if (static_cast<int>(nodes.size()) < num_machines) Fatal("machine list shorter than num_machines");
  nodes.resize(num_machines);
  int rank = -1;
  for (int i = 0; i < num_machines; ++i) if (nodes[i].second == local_listen_port) { rank = i; break; }
  if (rank < 0) Fatal("local_listen_port " + std::to_string(local_listen_port) + " is not in the machine list");
  if (t_device < 0) {
    int cnt = DeviceCountOrDie();
    const char* lr = std::getenv("LOCAL_RANK");
    t_device = (lr ? std::atoi(lr) : rank) % cnt;
  }
  EnsureDevice();
  const auto deadline = std::chrono::steady_clock::now() + std::chrono::seconds(std::max(listen_time_out_sec, 1));
  ncclUniqueId id;
  if (rank == 0) {
    B200_NCCL(ncclGetUniqueId(&id));
    for (int r = 1; r < num_machines; ++r) {
      int fd = -1;
      while (true) {
        addrinfo hints{}, *res = nullptr;
        hints.ai_family = AF_INET; hints.ai_socktype = SOCK_STREAM;
        std::string port = std::to_string(nodes[r].second);
        if (getaddrinfo(nodes[r].first.c_str(), port.c_str(), &hints, &res) == 0 && res) {
          fd = ::socket(res->ai_family, res->ai_socktype, res->ai_protocol);
          if (fd >= 0 && ::connect(fd, res->ai_addr, res->ai_addrlen) == 0) { freeaddrinfo(res); break; }
          if (fd >= 0) ::close(fd);
          fd = -1;
          freeaddrinfo(res);
        }
        if (std::chrono::steady_clock::now() > deadline) Fatal("network bootstrap: cannot reach " + nodes[r].first + ":" + std::to_string(nodes[r].second));
        std::this_thread::sleep_for(std::chrono::milliseconds(20));
      }
      SendAll(fd, &id, sizeof(id));
      char ack = 0;
      RecvAll(fd, &ack, 1);
      ::close(fd);
    }
  } else {
    int ls = ::socket(AF_INET, SOCK_STREAM, 0);
    if (ls < 0) Fatal("network bootstrap: socket() failed");
    int one = 1;
    setsockopt(ls, SOL_SOCKET, SO_REUSEADDR, &one, sizeof(one));
    sockaddr_in addr{};
    addr.sin_family = AF_INET; addr.sin_addr.s_addr = htonl(INADDR_ANY); addr.sin_port = htons(static_cast<uint16_t>(local_listen_port));
    if (::bind(ls, reinterpret_cast<sockaddr*>(&addr), sizeof(addr)) != 0) { ::close(ls); Fatal("network bootstrap: cannot bind port " + std::to_string(local_listen_port)); }
    ::listen(ls, 4);
    fd_set fds;
    FD_ZERO(&fds); FD_SET(ls, &fds);
    timeval tv{std::max(listen_time_out_sec, 1), 0};
    if (::select(ls + 1, &fds, nullptr, nullptr, &tv) <= 0) { ::close(ls); Fatal("network bootstrap: timed out waiting for rank 0"); }
    int fd = ::accept(ls, nullptr, nullptr);
    if (fd < 0) { ::close(ls); Fatal("network bootstrap: accept failed"); }
    RecvAll(fd, &id, sizeof(id));
    char ack = 1;
    SendAll(fd, &ack, 1);
    ::close(fd);
    ::close(ls);
  }
  ncclComm_t comm;
  B200_NCCL(ncclCommInitRank(&comm, num_machines, id, rank));
  t_net.active = true; t_net.rank = rank; t_net.world = num_machines; t_net.comm = comm;
}
void NetworkFree() {
  if (t_net.active && t_net.comm) { ncclCommDestroy(t_net.comm); }
  t_net = Network();
}

// small host-value collectives (init scores, label statistics, bin mappers): stage through device memory
void AllReduceHost(double* v, int n, ncclRedOp_t op, cudaStream_t s) {
  if (!Net().active) return;
  DevBuf<double> d; d.Alloc(n);
  d.Upload(v, n, s);
  B200_NCCL(ncclAllReduce(d.p, d.p, n, ncclDouble, op, Net().comm, s));
  d.Download(v, n, s);
  B200_CUDA(cudaStreamSynchronize(s));
}

// =============================================================================== dataset
Dataset::~Dataset() {
  ReleaseIngestStaging();
  if (stream) cudaStreamDestroy(stream);
}

template <typename T>
__global__ void k_gather_rows(const T* __restrict__ X, long long nrow, int ncol, int row_major, const int* __restrict__ rows, int nsample,
                              double* __restrict__ out) {
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < static_cast<long long>(nsample) * ncol;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    int s = static_cast<int>(e / ncol), f = static_cast<int>(e % ncol);
    long long r = rows[s];
    out[e] = row_major ? static_cast<double>(X[r * ncol + f]) : static_cast<double>(X[static_cast<long long>(f) * nrow + r]);
  }
}

static bool IsDevicePointer(const void* p) {
  cudaPointerAttributes a;
  cudaError_t e = cudaPointerGetAttributes(&a, p);
  if (e != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

static void PackMapper(const FeatureBins& fb, double* r, int slots) {
  r[0] = fb.num_bin; r[1] = fb.missing_type; r[2] = fb.trivial; r[3] = fb.default_bin; r[4] = fb.most_freq_bin;
  r[5] = fb.sparse_rate; r[6] = fb.min_val; r[7] = fb.max_val; r[8] = fb.categorical; r[9] = 0;
  for (int i = 0; i < slots; ++i) {
    if (fb.categorical) r[10 + i] = i < static_cast<int>(fb.bin_to_cat.size()) ? fb.bin_to_cat[i] : 0.0;
    else r[10 + i] = i < static_cast<int>(fb.upper.size()) ? fb.upper[i] : 0.0;
  }
}
static FeatureBins UnpackMapper(const double* r) {
  FeatureBins fb;
  fb.num_bin = static_cast<int>(r[0]); fb.missing_type = static_cast<int>(r[1]); fb.trivial = r[2] != 0;
  fb.default_bin = static_cast<uint32_t>(r[3]); fb.most_freq_bin = static_cast<uint32_t>(r[4]);
  fb.sparse_rate = r[5]; fb.min_val = r[6]; fb.max_val = r[7]; fb.categorical = r[8] != 0;
  if (fb.categorical) {
    for (int b = 0; b < fb.num_bin; ++b) fb.bin_to_cat.push_back(static_cast<int>(r[10 + b]));
    std::vector<std::pair<int, int>> byc;
    for (int b = 1; b < fb.num_bin; ++b) byc.emplace_back(fb.bin_to_cat[b], b);
    std::sort(byc.begin(), byc.end());
    for (auto& p : byc) { fb.sorted_cats.push_back(p.first); fb.sorted_bins.push_back(p.second); }
  } else {
    fb.upper.assign(r + 10, r + 10 + fb.num_bin);
  }
  return fb;
}

void Dataset::FindBins(const void* data, bool on_device, int data_type, int is_row_major) {
  const int n = num_data, F = num_total_features;
  if (cfg.max_bin >= kWideMaxBins) Fatal("max_bin >= " + std::to_string(kWideMaxBins) + " is not supported");
  if (cfg.max_bin < 2) Fatal("max_bin should be >= 2");
  if (cfg.zero_as_missing) Fatal("zero_as_missing=true is not supported by this build");
  LcgRandom rnd(cfg.data_random_seed);
  int sample_cnt = n < cfg.bin_construct_sample_cnt ? n : cfg.bin_construct_sample_cnt;
  std::vector<int> rows = rnd.Sample(n, sample_cnt);
  sample_cnt = static_cast<int>(rows.size());
  std::vector<double> S(static_cast<size_t>(sample_cnt) * F);
  if (on_device) {
    DevBuf<int> d_rows; d_rows.Alloc(sample_cnt);
    DevBuf<double> d_S; d_S.Alloc(S.size());
    d_rows.Upload(rows.data(), sample_cnt, stream);
    int grid = static_cast<int>(std::min<size_t>((S.size() + 255) / 256, 148 * 32));
    if (data_type == 0) k_gather_rows<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(data), n, F, is_row_major, d_rows.p, sample_cnt, d_S.p);
    else k_gather_rows<double><<<grid, 256, 0, stream>>>(static_cast<const double*>(data), n, F, is_row_major, d_rows.p, sample_cnt, d_S.p);
    B200_CUDA(cudaGetLastError());
    d_S.Download(S.data(), S.size(), stream);
    B200_CUDA(cudaStreamSynchronize(stream));
  } else {
#pragma omp parallel for schedule(static)
    for (int s = 0; s < sample_cnt; ++s) {
      const long long r = rows[s];
      for (int f = 0; f < F; ++f) {
        double v;
        if (data_type == 0) v = is_row_major ? static_cast<const float*>(data)[r * F + f] : static_cast<const float*>(data)[static_cast<long long>(f) * n + r];
        else v = is_row_major ? static_cast<const double*>(data)[r * F + f] : static_cast<const double*>(data)[static_cast<long long>(f) * n + r];
        S[static_cast<size_t>(s) * F + f] = v;
      }
    }
  }
  std::vector<std::vector<double>> nz(F);
  {
    const int world = Net().active ? Net().world : 1, rank = Net().active ? Net().rank : 0;
    int step = std::max(1, (F + world - 1) / world);
    const int f0 = world == 1 ? 0 : std::min(F, rank * step), f1 = world == 1 ? F : std::min(F, f0 + step);
#pragma omp parallel for schedule(dynamic)
    for (int f = f0; f < f1; ++f) {
      nz[f].reserve(sample_cnt);
      for (int s = 0; s < sample_cnt; ++s) {
        double v = S[static_cast<size_t>(s) * F + f];
        if (std::fabs(v) > kZeroThr || std::isnan(v)) nz[f].push_back(v);
      }
    }
  }
  FindBinsFromColumns(&nz, sample_cnt);
}

// nz[f] = sampled values of feature f with |v| > 1e-35 or NaN (only this rank's slice needs filling)
void Dataset::FindBinsFromColumns(std::vector<std::vector<double>>* nzp, int sample_cnt) {
  NvtxRange nvtx("b200gbm:find bins (host) + C5 mapper all-gather");
  std::vector<std::vector<double>>& nz = *nzp;
  const int n = num_data, F = num_total_features;
  const int filter_cnt = static_cast<int>(static_cast<double>(cfg.min_data_in_leaf) * sample_cnt / n);
  // feature ownership for distributed bin finding (SURVEY.md fact 9, A.2): contiguous slices of ceil(F/R)
  const int world = Net().active ? Net().world : 1, rank = Net().active ? Net().rank : 0;
  int step = (F + world - 1) / world;
  if (step < 1) step = 1;
  const int f0 = world == 1 ? 0 : std::min(F, rank * step), f1 = world == 1 ? F : std::min(F, f0 + step);
  mappers.assign(F, FeatureBins());
#pragma omp parallel for schedule(dynamic)
  for (int f = f0; f < f1; ++f) {
    const bool is_cat = std::find(cfg.categorical_feature.begin(), cfg.categorical_feature.end(), f) != cfg.categorical_feature.end();
    if (is_cat) mappers[f] = FindCategoricalBins(&nz[f], sample_cnt, cfg.max_bin, cfg.min_data_in_bin, filter_cnt, cfg.feature_pre_filter);
    else mappers[f] = FindFeatureBins(&nz[f], sample_cnt, cfg.max_bin, cfg.min_data_in_bin, filter_cnt, cfg.feature_pre_filter, cfg.use_missing,
                                      cfg.zero_as_missing);
  }
  for (int f = f0; f < f1; ++f)
    if (mappers[f].num_bin > kWideMaxBins)
      Fatal("categorical feature " + std::to_string(f) + " needs " + std::to_string(mappers[f].num_bin) +
            " bins (a categorical feature keeps categories until 99% of its mass is covered); this build supports at most " + std::to_string(kWideMaxBins) + " bins per feature");
  if (world > 1) {   // C5: all-gather the serialized mappers (record = 10 header doubles + the largest bin count of any rank)
    double maxbins = 256;
    for (int f = f0; f < f1; ++f) maxbins = std::max(maxbins, static_cast<double>(mappers[f].num_bin));
    AllReduceHost(&maxbins, 1, ncclMax, stream);
    const int slots = static_cast<int>(maxbins);
    const size_t kMapperRecord = 10 + static_cast<size_t>(slots);
    std::vector<double> send(static_cast<size_t>(step) * kMapperRecord, 0.0), recv(static_cast<size_t>(world) * step * kMapperRecord);
    for (int f = f0; f < f1; ++f) PackMapper(mappers[f], &send[static_cast<size_t>(f - f0) * kMapperRecord], slots);
    DevBuf<double> ds, dr; ds.Alloc(send.size()); dr.Alloc(recv.size());
    ds.Upload(send.data(), send.size(), stream);
    B200_NCCL(ncclAllGather(ds.p, dr.p, send.size(), ncclDouble, Net().comm, stream));
    dr.Download(recv.data(), recv.size(), stream);
    B200_CUDA(cudaStreamSynchronize(stream));
    for (int f = 0; f < F; ++f) {
      int owner = f / step, off = f - owner * step;
      mappers[f] = UnpackMapper(&recv[(static_cast<size_t>(owner) * step + off) * kMapperRecord]);
    }
  }
}

void Dataset::UploadMeta() {
  // inner order: features with <= 256 bins first (uint8 tiles of 32), then the wide ones (uint16 columns), each group in real-index order
  used.clear();
  inner_of.assign(num_total_features, -1);
  std::vector<int> wide_real;
  for (int f = 0; f < num_total_features; ++f) {
    if (mappers[f].trivial) continue;
    if (mappers[f].num_bin > 256) wide_real.push_back(f);
    else { inner_of[f] = static_cast<int>(used.size()); used.push_back(f); }
  }
  nfn = static_cast<int>(used.size());
  for (int f : wide_real) { inner_of[f] = static_cast<int>(used.size()); used.push_back(f); }
  nf = static_cast<int>(used.size());
  nw = nf - nfn;
  sample_order.clear();
  for (int f = 0; f < num_total_features; ++f) if (inner_of[f] >= 0) sample_order.push_back(inner_of[f]);
  num_tiles = std::max(1, (nfn + 31) / 32);
  nf_pad = num_tiles * 32 + nw;
  meta_host.assign(nf_pad, FeatMeta{1, 0, 0, 0, 0, 0, 0, 0});
  std::vector<double> ubh(static_cast<size_t>(num_tiles) * 32 * 256, 0.0);
  std::vector<uint8_t> cbh(static_cast<size_t>(num_tiles) * 32 * 256, 0);
  has_categorical = false;
  hist_pairs = static_cast<size_t>(num_tiles) * 32 * 256;
  wide_host.clear();
  std::vector<int> wcats;
  std::vector<unsigned short> wbins;
  std::vector<double> wub;
  for (int u = 0; u < nf; ++u) {
    const FeatureBins& fb = mappers[used[u]];
    int hist_off = u * 256;
    if (u >= nfn) {
      hist_off = static_cast<int>(hist_pairs);
      WideMeta wm{fb.num_bin, hist_off, static_cast<int>(fb.categorical ? wcats.size() : wub.size()), static_cast<int>(fb.sorted_cats.size()),
                  static_cast<int>(fb.default_bin), fb.missing_type, used[u], fb.categorical ? 1 : 0, fb.most_freq_bin == 0 ? 1 : 0, 0, 0, 0};
      wide_host.push_back(wm);
      if (fb.categorical) for (size_t i = 0; i < fb.sorted_cats.size(); ++i) { wcats.push_back(fb.sorted_cats[i]); wbins.push_back(static_cast<unsigned short>(fb.sorted_bins[i])); }
      else wub.insert(wub.end(), fb.upper.begin(), fb.upper.end());
      hist_pairs += (static_cast<size_t>(fb.num_bin) + 255) / 256 * 256;
      if (hist_pairs > (1u << 30)) Fatal("histogram of the wide features is too large");
    }
    meta_host[u] = FeatMeta{fb.num_bin, fb.missing_type, static_cast<int>(fb.default_bin), fb.most_freq_bin == 0 ? 1 : 0, used[u],
                            fb.categorical ? 1 : 0, static_cast<int>(fb.sorted_cats.size()), hist_off};
    if (fb.categorical) has_categorical = true;
    if (u >= nfn) continue;
    if (fb.categorical) {
      for (size_t i = 0; i < fb.sorted_cats.size(); ++i) {
        ubh[static_cast<size_t>(u) * 256 + i] = fb.sorted_cats[i];
        cbh[static_cast<size_t>(u) * 256 + i] = static_cast<uint8_t>(fb.sorted_bins[i]);
      }
    } else {
      for (int b = 0; b < fb.num_bin; ++b) ubh[static_cast<size_t>(u) * 256 + b] = fb.upper[b];
    }
  }
  meta.Alloc(nf_pad); ub.Alloc(ubh.size()); catbin.Alloc(cbh.size());
  meta.Upload(meta_host.data(), nf_pad, stream);
  ub.Upload(ubh.data(), ubh.size(), stream);
  catbin.Upload(cbh.data(), cbh.size(), stream);
  if (nw > 0) {
    wide_meta.Alloc(nw); wide_meta.Upload(wide_host.data(), nw, stream);
    wide_cats.Alloc(std::max<size_t>(wcats.size(), 1)); wide_catbin.Alloc(std::max<size_t>(wbins.size(), 1));
    if (!wcats.empty()) { wide_cats.Upload(wcats.data(), wcats.size(), stream); wide_catbin.Upload(wbins.data(), wbins.size(), stream); }
    wide_ub.Alloc(std::max<size_t>(wub.size(), 1));
    if (!wub.empty()) wide_ub.Upload(wub.data(), wub.size(), stream);
  }
  B200_CUDA(cudaStreamSynchronize(stream));
}

// bins (tiles + wide columns) of a freshly created dataset
static void AllocBins(Dataset* d) {
  d->bins.Alloc(static_cast<size_t>(d->num_tiles) * d->rows_stride * 32);
  if (d->nw > 0) d->bins16.Alloc(static_cast<size_t>(d->nw) * d->rows_stride);
}

template <typename T>
static void LaunchBin(const T* X, long long nrow, int ncol, int row_major, long long ld, const Dataset& d, long long row_offset, cudaStream_t s) {
  // function attributes are per device/context: set on every call (rank-threads drive different GPUs)
  B200_CUDA(cudaFuncSetAttribute(k_bin_rows<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
  dim3 grid(static_cast<unsigned>(std::min<long long>((nrow + 7) / 8, 148 * 8)), d.num_tiles);
  if (grid.x == 0) grid.x = 1;
  k_bin_rows<T><<<grid, 256, 65536, s>>>(X, nrow, ncol, row_major, ld, d.meta.p, d.ub.p, d.catbin.p, d.nfn, d.bins.p, static_cast<long long>(d.rows_stride), row_offset);
  if (d.nw > 0)
    k_bin_wide<T><<<148 * 8, 256, 0, s>>>(X, nrow, row_major, ld, d.wide_meta.p, d.nw, d.wide_cats.p, d.wide_catbin.p, d.wide_ub.p, d.bins16.p, d.rows_stride, row_offset);
  B200_CUDA(cudaGetLastError());
}

void Dataset::BinBlock(const void* data, bool on_device, int data_type, int is_row_major, long long n, long long start_row) {
  NvtxRange nvtx("b200gbm:K0 bin rows (H2D + value->bin)");
  const int F = num_total_features;
  const size_t esz = data_type == 0 ? 4 : 8;
  if (start_row < 0 || start_row + n > num_data) Fatal("row block out of range");
  if (on_device) {
    const long long ld = is_row_major ? F : n;
    if (data_type == 0) LaunchBin<float>(static_cast<const float*>(data), n, F, is_row_major, ld, *this, start_row, stream);
    else LaunchBin<double>(static_cast<const double*>(data), n, F, is_row_major, ld, *this, start_row, stream);
    B200_CUDA(cudaStreamSynchronize(stream));
    return;
  }
  // host source: stream row chunks through two device buffers, copy of chunk i+1 overlaps binning of chunk i.  The staging
  // buffers, copy stream and events persist across LGBM_DatasetPushRows calls (a cudaMalloc/cudaFree pair per call costs as much
  // as the copy itself) and are released when the last row has arrived.
  const size_t kStageBytes = 256u << 20;
  long long chunk = std::max<long long>(1, std::min<long long>(n, static_cast<long long>(kStageBytes) / (static_cast<long long>(F) * esz)));
  const size_t need = static_cast<size_t>(chunk) * F * esz;
  if (!ingest_copy_stream_) {
    B200_CUDA(cudaStreamCreateWithFlags(&ingest_copy_stream_, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      B200_CUDA(cudaEventCreateWithFlags(&ingest_copied_[i], cudaEventDisableTiming));
      B200_CUDA(cudaEventCreateWithFlags(&ingest_binned_[i], cudaEventDisableTiming));
    }
  }
  for (int i = 0; i < 2; ++i) if (ingest_buf_[i].n < need) ingest_buf_[i].Alloc(std::max(need, std::min(kStageBytes, static_cast<size_t>(num_data) * F * esz)));
  cudaStream_t copy_stream = ingest_copy_stream_;
  int it = 0;
  for (long long r0 = 0; r0 < n; r0 += chunk, ++it) {
    const int b = it & 1;
    const long long rows = std::min(chunk, n - r0);
    if (it >= 2) B200_CUDA(cudaStreamWaitEvent(copy_stream, ingest_binned_[b], 0));
    if (is_row_major) {
      B200_CUDA(cudaMemcpyAsync(ingest_buf_[b].p, static_cast<const unsigned char*>(data) + static_cast<size_t>(r0) * F * esz, static_cast<size_t>(rows) * F * esz,
                                cudaMemcpyHostToDevice, copy_stream));
    } else {   // column-major: F column segments of `rows` elements, device chunk keeps ld = rows
      B200_CUDA(cudaMemcpy2DAsync(ingest_buf_[b].p, static_cast<size_t>(rows) * esz, static_cast<const unsigned char*>(data) + static_cast<size_t>(r0) * esz,
                                  static_cast<size_t>(n) * esz, static_cast<size_t>(rows) * esz, F, cudaMemcpyHostToDevice, copy_stream));
    }
    B200_CUDA(cudaEventRecord(ingest_copied_[b], copy_stream));
    B200_CUDA(cudaStreamWaitEvent(stream, ingest_copied_[b], 0));
    const long long ld = is_row_major ? F : rows;
    if (data_type == 0) LaunchBin<float>(reinterpret_cast<const float*>(ingest_buf_[b].p), rows, F, is_row_major, ld, *this, start_row + r0, stream);
    else LaunchBin<double>(reinterpret_cast<const double*>(ingest_buf_[b].p), rows, F, is_row_major, ld, *this, start_row + r0, stream);
    B200_CUDA(cudaEventRecord(ingest_binned_[b], stream));
  }
  B200_CUDA(cudaStreamSynchronize(stream));          // all copies are consumed: the caller may reuse its buffer
  ingest_rows_done_ += n;
  if (ingest_rows_done_ >= num_data) ReleaseIngestStaging();
}

void Dataset::ReleaseIngestStaging() {
  for (int i = 0; i < 2; ++i) {
    ingest_buf_[i].Free();
    if (ingest_copied_[i]) { cudaEventDestroy(ingest_copied_[i]); ingest_copied_[i] = nullptr; }
    if (ingest_binned_[i]) { cudaEventDestroy(ingest_binned_[i]); ingest_binned_[i] = nullptr; }
  }
  if (ingest_copy_stream_) { cudaStreamDestroy(ingest_copy_stream_); ingest_copy_stream_ = nullptr; }
}

Dataset* Dataset::CreateFromSampledColumn(double** sample_data, int** sample_indices, int ncol, const int* num_per_col, int num_sample_row,
                                          int num_total_row, const char* params) {
  (void)sample_indices;
  EnsureDevice();
  if (num_total_row <= 0 || ncol <= 0) Fatal("Dataset should have at least one row and one column");
  std::unique_ptr<Dataset> d(new Dataset());
  d->device = CurrentDevice();
  B200_CUDA(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
  d->num_data = num_total_row; d->num_total_features = ncol;
  d->cfg.Parse(params);
  if (d->cfg.max_bin >= kWideMaxBins) Fatal("max_bin >= " + std::to_string(kWideMaxBins) + " is not supported");
  std::vector<std::vector<double>> nz(ncol);
  for (int f = 0; f < ncol; ++f) nz[f].assign(sample_data[f], sample_data[f] + num_per_col[f]);
  d->FindBinsFromColumns(&nz, num_sample_row);
  d->feature_names.resize(ncol);
  for (int f = 0; f < ncol; ++f) d->feature_names[f] = "Column_" + std::to_string(f);
  d->UploadMeta();
  d->rows_stride = static_cast<size_t>(num_total_row);
  AllocBins(d.get());
  return d.release();
}

void Dataset::PushRows(const void* data, int data_type, int nrow, int ncol, int start_row) {
  EnsureDevice();
  if (ncol != num_total_features) Fatal("PushRows: wrong number of columns");
  if (data_type != 0 && data_type != 1) Fatal("PushRows: unknown data type");
  cudaEvent_t e0, e1;
  B200_CUDA(cudaEventCreate(&e0)); B200_CUDA(cudaEventCreate(&e1));
  B200_CUDA(cudaEventRecord(e0, stream));
  BinBlock(data, IsDevicePointer(data), data_type, 1, nrow, start_row);
  B200_CUDA(cudaEventRecord(e1, stream));
  B200_CUDA(cudaEventSynchronize(e1));
  float ms = 0;
  B200_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  ingest_ms += ms;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
}

void Dataset::GetBinsRowMajor(uint8_t* out) const {
  if (nw > 0) Fatal("this dataset has features with more than 256 bins: use B200GBM_DatasetGetBins16");
  std::vector<uint8_t> h(bins.n);
  B200_CUDA(cudaMemcpy(h.data(), bins.p, bins.n, cudaMemcpyDeviceToHost));
  std::memset(out, 0, static_cast<size_t>(num_data) * num_total_features);
  for (int u = 0; u < nfn; ++u) {
    const int f = used[u];
    const uint8_t* src = h.data() + (static_cast<size_t>(u >> 5) * rows_stride) * 32 + (u & 31);
    for (int i = 0; i < num_data; ++i) out[static_cast<size_t>(i) * num_total_features + f] = src[static_cast<size_t>(i) * 32];
  }
}
void Dataset::GetBinsRowMajor16(uint16_t* out) const {
  std::vector<uint8_t> h(bins.n);
  B200_CUDA(cudaMemcpy(h.data(), bins.p, bins.n, cudaMemcpyDeviceToHost));
  std::memset(out, 0, static_cast<size_t>(num_data) * num_total_features * sizeof(uint16_t));
  for (int u = 0; u < nfn; ++u) {
    const int f = used[u];
    const uint8_t* src = h.data() + (static_cast<size_t>(u >> 5) * rows_stride) * 32 + (u & 31);
    for (int i = 0; i < num_data; ++i) out[static_cast<size_t>(i) * num_total_features + f] = src[static_cast<size_t>(i) * 32];
  }
  if (nw > 0) {
    std::vector<uint16_t> hw(bins16.n);
    B200_CUDA(cudaMemcpy(hw.data(), bins16.p, bins16.n * sizeof(uint16_t), cudaMemcpyDeviceToHost));
    for (int w = 0; w < nw; ++w) {
      const int f = used[nfn + w];
      const uint16_t* src = hw.data() + static_cast<size_t>(w) * rows_stride;
      for (int i = 0; i < num_data; ++i) out[static_cast<size_t>(i) * num_total_features + f] = src[i];
    }
  }
}

__global__ void k_gather_bin_rows(BinView bv, int nf, const FeatMeta* __restrict__ meta, const int* __restrict__ rows, int nrows, int F,
                                  uint16_t* __restrict__ out) {
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < static_cast<long long>(nrows) * nf;
       e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(e / nf), u = static_cast<int>(e % nf);
    out[static_cast<size_t>(i) * F + meta[u].real_index] = static_cast<uint16_t>(bv.at(u, static_cast<size_t>(rows[i])));
  }
}
void Dataset::GetBinsOfRows(const int32_t* rows, int nrows, uint16_t* out) const {
  if (nrows <= 0) return;
  for (int i = 0; i < nrows; ++i) if (rows[i] < 0 || rows[i] >= num_data) Fatal("GetBinsOfRows: row index out of range");
  DevBuf<int> dr; dr.Alloc(nrows);
  DevBuf<uint16_t> dout; dout.Alloc(static_cast<size_t>(nrows) * num_total_features);
  dr.Upload(rows, nrows, stream);
  dout.Zero(stream);
  if (nf > 0) k_gather_bin_rows<<<148 * 4, 256, 0, stream>>>(View(), nf, meta.p, dr.p, nrows, num_total_features, dout.p);
  B200_CUDA(cudaGetLastError());
  dout.Download(out, dout.n, stream);
  B200_CUDA(cudaStreamSynchronize(stream));
}

void Dataset::Histogram(const float* grad, const float* hess, const int32_t* idx, int cnt, double* out) const {
  EnsureDevice();
  B200_CUDA(cudaFuncSetAttribute(k4_hist_build_ws<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWsSmemBytes));
  const int n = num_data;
  DevBuf<float> g, h; g.Alloc(n); h.Alloc(n);
  g.Upload(grad, n, stream); h.Upload(hess, n, stream);
  DevBuf<int4> q; q.Alloc(n);
  DevBuf<TreeCtrl> ctrl; ctrl.Alloc(1); ctrl.Zero(stream);
  DevBuf<int> didx; didx.Alloc(std::max(cnt, 1));
  if (idx) didx.Upload(idx, cnt, stream);
  const size_t elems = static_cast<size_t>(num_tiles) * 32 * 512;      // tile features only (wide features are covered by the model-level tests)
  DevBuf<long long> H; H.Alloc(elems); H.Zero(stream);
  DevBuf<double> D; D.Alloc(elems);
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
  k_absmax<<<sms * 4, 256, 0, stream>>>(g.p, h.p, n, ctrl.p);
  k_set_scale<<<1, 1, 0, stream>>>(ctrl.p, 0, 1.0);
  k_quantize<<<sms * 4, 256, 0, stream>>>(g.p, h.p, n, q.p, ctrl.p, 0, nullptr, 0);
  HistWork w{0, cnt, idx ? 1 : 0, 0};
  B200_CUDA(cudaMemcpyAsync(&ctrl.p->hist_work, &w, sizeof(w), cudaMemcpyHostToDevice, stream));
  DevBuf<int4> qo; qo.Alloc(std::max(cnt, 1));
  k_gather_q<<<sms * 4, 256, 0, stream>>>(&ctrl.p->hist_work, didx.p, didx.p, q.p, qo.p);
  k4_hist_build_ws<4><<<sms, kWsThreads, kWsSmemBytes, stream>>>(bins.p, rows_stride, num_tiles, q.p, qo.p, didx.p, didx.p, &ctrl.p->hist_work,
                                                                 reinterpret_cast<unsigned long long*>(H.p));
  k_hist_to_double<<<sms * 4, 256, 0, stream>>>(H.p, D.p, elems, ctrl.p);
  B200_CUDA(cudaGetLastError());
  std::vector<double> hd(elems);
  D.Download(hd.data(), elems, stream);
  B200_CUDA(cudaStreamSynchronize(stream));
  std::memset(out, 0, sizeof(double) * static_cast<size_t>(num_total_features) * 512);
  for (int u = 0; u < nfn; ++u) std::memcpy(out + static_cast<size_t>(used[u]) * 512, hd.data() + static_cast<size_t>(u) * 512, sizeof(double) * 512);
}

Dataset* Dataset::CreateFromMat(const void* data, int data_type, int nrow, int ncol, int is_row_major, const char* params,
                                const Dataset* reference) {
  EnsureDevice();
  if (data_type != 0 && data_type != 1) Fatal("Unknown data type in CreateFromMat (expect C_API_DTYPE_FLOAT32 or FLOAT64)");
  if (nrow <= 0 || ncol <= 0) Fatal("Dataset should have at least one row and one column");
  std::unique_ptr<Dataset> d(new Dataset());
  d->device = CurrentDevice();
  B200_CUDA(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
  d->num_data = nrow; d->num_total_features = ncol;
  d->cfg.Parse(params);
  cudaEvent_t e0, e1;
  B200_CUDA(cudaEventCreate(&e0)); B200_CUDA(cudaEventCreate(&e1));
  B200_CUDA(cudaEventRecord(e0, d->stream));
  const bool on_device = IsDevicePointer(data);
  if (reference) {
    if (reference->num_total_features != ncol) Fatal("Validation data has a different number of features than the reference dataset");
    d->mappers = reference->mappers;
    d->feature_names = reference->feature_names;
  } else {
    d->FindBins(data, on_device, data_type, is_row_major);
    d->feature_names.resize(ncol);
    for (int f = 0; f < ncol; ++f) d->feature_names[f] = "Column_" + std::to_string(f);
  }
  d->UploadMeta();
  d->rows_stride = static_cast<size_t>(nrow);
  AllocBins(d.get());
  d->BinBlock(data, on_device, data_type, is_row_major, nrow, 0);
  B200_CUDA(cudaEventRecord(e1, d->stream));
  B200_CUDA(cudaEventSynchronize(e1));
  float ms = 0;
  B200_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  d->ingest_ms = ms;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return d.release();
}

// ---- CSR ingestion without densifying (replaces LGBM_DatasetCreateFromCSR, reference call site DatasetAggregator.scala:438-459).
// Bin finding walks the nonzeros of the sampled rows only; binning fills every row of a tile with the features' zero bins and then
// scatters one thread per stored element.  Memory: O(nnz) + the uint8 bins, never nrow x num_col doubles.
__global__ void k_fill_default_wide(const WideMeta* __restrict__ wm, int nw, uint16_t* __restrict__ bins16, size_t rows_stride, long long nrow) {
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < nrow * nw; e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int w = static_cast<int>(e / nrow);
    bins16[static_cast<size_t>(w) * rows_stride + (e - static_cast<long long>(w) * nrow)] = static_cast<uint16_t>(wm[w].default_bin);
  }
}
__global__ void k_fill_default_bins(const FeatMeta* __restrict__ meta, int nf, uint8_t* __restrict__ bins, size_t rows_stride, long long nrow, int num_tiles) {
  const long long total = nrow * num_tiles * 32;
  for (long long e = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; e < total; e += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int lane = static_cast<int>(e & 31);
    const long long rt = e >> 5;
    const int tile = static_cast<int>(rt / nrow);
    const long long r = rt - static_cast<long long>(tile) * nrow;
    const int u = tile * 32 + lane;
    bins[(static_cast<size_t>(tile) * rows_stride + r) * 32 + lane] = u < nf ? static_cast<uint8_t>(meta[u].default_bin) : 0;
  }
}
template <typename TI, typename TV>
__global__ void k_bin_csr(const TI* __restrict__ indptr, const int* __restrict__ indices, const TV* __restrict__ vals, long long nrow, const int* __restrict__ inner_of,
                          const FeatMeta* __restrict__ meta, const double* __restrict__ ub, const uint8_t* __restrict__ catbin, uint8_t* __restrict__ bins,
                          size_t rows_stride, long long elem_base, int nfn, const WideMeta* __restrict__ wm, const int* __restrict__ wcats,
                          const unsigned short* __restrict__ wcatbin, const double* __restrict__ wub, uint16_t* __restrict__ bins16) {
  const int lane = threadIdx.x & 31;
  const long long warp = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5, nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  for (long long r = warp; r < nrow; r += nwarps) {
    const long long a = static_cast<long long>(indptr[r]) - elem_base, b = static_cast<long long>(indptr[r + 1]) - elem_base;
    for (long long k = a + lane; k < b; k += 32) {
      const int u = inner_of[indices[k]];
      if (u < 0) continue;
      const FeatMeta m = meta[u];
      double v = static_cast<double>(vals[k]);
      if (u >= nfn) {           // wide column (categorical with > 256 bins, or numerical with max_bin > 255)
        bins16[static_cast<size_t>(u - nfn) * rows_stride + r] = static_cast<uint16_t>(d_wide_bin(v, wm[u - nfn], wcats, wcatbin, wub));
        continue;
      }
      const double* myub = ub + static_cast<size_t>(u) * 256;
      unsigned bin = 0;
      if (m.is_categorical) {
        if (!isnan(v)) {
          const int iv = static_cast<int>(v);
          if (iv >= 0) {
            int lo = 0, hi = m.num_sorted_cats;
            while (lo < hi) { int mid = (lo + hi) >> 1; if (static_cast<int>(myub[mid]) < iv) lo = mid + 1; else hi = mid; }
            if (lo < m.num_sorted_cats && static_cast<int>(myub[lo]) == iv) bin = catbin[static_cast<size_t>(u) * 256 + lo];
          }
        }
      } else {
        if (isnan(v)) { if (m.missing_type == 2) bin = m.num_bin - 1; else v = 0.0; }
        if (!isnan(v)) {
          int lo = 0, hi = m.num_bin - 1 - (m.missing_type == 2 ? 1 : 0);
          while (lo < hi) { int mid = (hi + lo - 1) / 2; if (v <= myub[mid]) hi = mid; else lo = mid + 1; }
          bin = lo;
        }
      }
      bins[(static_cast<size_t>(u >> 5) * rows_stride + r) * 32 + (u & 31)] = static_cast<uint8_t>(bin);
    }
  }
}

Dataset* Dataset::CreateFromCSR(const void* indptr, int indptr_type, const int32_t* indices, const void* data, int data_type,
                                int64_t nindptr, int64_t nelem, int64_t num_col, const char* params, const Dataset* reference) {
  EnsureDevice();
  if (num_col <= 0) Fatal("CreateFromCSR: num_col must be given");
  if (num_col > std::numeric_limits<int>::max()) Fatal("CreateFromCSR: too many columns");
  if (indptr_type != 2 && indptr_type != 3) Fatal("CreateFromCSR: indptr must be int32 or int64");
  if (data_type != 0 && data_type != 1) Fatal("Unknown data type in CreateFromCSR (expect C_API_DTYPE_FLOAT32 or FLOAT64)");
  const int64_t nrow = nindptr - 1;
  if (nrow <= 0) Fatal("Dataset should have at least one row and one column");
  if (nrow > std::numeric_limits<int>::max()) Fatal("CreateFromCSR: too many rows for one partition");
  auto ip = [&](int64_t r) -> int64_t { return indptr_type == 2 ? static_cast<const int32_t*>(indptr)[r] : static_cast<const int64_t*>(indptr)[r]; };
  auto val = [&](int64_t k) -> double { return data_type == 0 ? static_cast<double>(static_cast<const float*>(data)[k]) : static_cast<const double*>(data)[k]; };
  if (ip(0) < 0 || ip(nrow) > nelem) Fatal("CreateFromCSR: indptr does not match the number of elements");
  {
    int bad = 0;
#pragma omp parallel for schedule(static) reduction(| : bad)
    for (int64_t r = 0; r < nrow; ++r) {
      if (ip(r) > ip(r + 1)) bad |= 1;
      else for (int64_t k = ip(r); k < ip(r + 1); ++k) if (indices[k] < 0 || indices[k] >= num_col) bad |= 2;
    }
    if (bad & 1) Fatal("CreateFromCSR: indptr is not non-decreasing");
    if (bad & 2) Fatal("CreateFromCSR: a column index is negative or >= num_col");
  }
  std::unique_ptr<Dataset> d(new Dataset());
  d->device = CurrentDevice();
  B200_CUDA(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
  d->num_data = static_cast<int>(nrow); d->num_total_features = static_cast<int>(num_col);
  d->cfg.Parse(params);
  cudaEvent_t e0, e1;
  B200_CUDA(cudaEventCreate(&e0)); B200_CUDA(cudaEventCreate(&e1));
  B200_CUDA(cudaEventRecord(e0, d->stream));
  const int F = d->num_total_features;
  if (reference) {
    if (reference->num_total_features != F) Fatal("Validation data has a different number of features than the reference dataset");
    d->mappers = reference->mappers;
    d->feature_names = reference->feature_names;
  } else {
    if (d->cfg.max_bin >= kWideMaxBins) Fatal("max_bin >= " + std::to_string(kWideMaxBins) + " is not supported");
    if (d->cfg.max_bin < 2) Fatal("max_bin should be >= 2");
    if (d->cfg.zero_as_missing) Fatal("zero_as_missing=true is not supported by this build");
    LcgRandom rnd(d->cfg.data_random_seed);
    int sample_cnt = d->num_data < d->cfg.bin_construct_sample_cnt ? d->num_data : d->cfg.bin_construct_sample_cnt;
    std::vector<int> rows = rnd.Sample(d->num_data, sample_cnt);
    sample_cnt = static_cast<int>(rows.size());
    std::vector<std::vector<double>> nz(F);
    for (int r : rows)
      for (int64_t k = ip(r); k < ip(r + 1); ++k) {
        const double v = val(k);
        if (std::fabs(v) > kZeroThr || std::isnan(v)) nz[indices[k]].push_back(v);
      }
    d->FindBinsFromColumns(&nz, sample_cnt);
    d->feature_names.resize(F);
    for (int f = 0; f < F; ++f) d->feature_names[f] = "Column_" + std::to_string(f);
  }
  d->UploadMeta();
  d->rows_stride = static_cast<size_t>(nrow);
  AllocBins(d.get());
  k_fill_default_bins<<<148 * 8, 256, 0, d->stream>>>(d->meta.p, d->nfn, d->bins.p, d->rows_stride, nrow, d->num_tiles);
  if (d->nw > 0) k_fill_default_wide<<<148 * 8, 256, 0, d->stream>>>(d->wide_meta.p, d->nw, d->bins16.p, d->rows_stride, nrow);
  B200_CUDA(cudaGetLastError());
  if (d->nf > 0) {
    DevBuf<int> d_inner; d_inner.Alloc(F); d_inner.Upload(d->inner_of.data(), F, d->stream);
    // row blocks of bounded element count: the stored elements are staged through one device buffer per block
    const size_t isz = indptr_type == 2 ? 4 : 8, vsz = data_type == 0 ? 4 : 8;
    const int64_t kBlockElems = 64LL << 20;
    DevBuf<unsigned char> d_ip, d_ix, d_v;
    int64_t r0 = 0;
    while (r0 < nrow) {
      int64_t r1 = r0 + 1;
      while (r1 < nrow && ip(r1 + 1) - ip(r0) <= kBlockElems) ++r1;
      const int64_t e0k = ip(r0), ne = ip(r1) - e0k, nr = r1 - r0;
      if (d_ip.n < static_cast<size_t>(nr + 1) * isz) d_ip.Alloc(static_cast<size_t>(nr + 1) * isz);
      if (ne > 0) {
        if (d_ix.n < static_cast<size_t>(ne) * 4) d_ix.Alloc(static_cast<size_t>(ne) * 4);
        if (d_v.n < static_cast<size_t>(ne) * vsz) d_v.Alloc(static_cast<size_t>(ne) * vsz);
        B200_CUDA(cudaMemcpyAsync(d_ix.p, indices + e0k, static_cast<size_t>(ne) * 4, cudaMemcpyHostToDevice, d->stream));
        B200_CUDA(cudaMemcpyAsync(d_v.p, static_cast<const unsigned char*>(data) + static_cast<size_t>(e0k) * vsz, static_cast<size_t>(ne) * vsz, cudaMemcpyHostToDevice, d->stream));
      }
      B200_CUDA(cudaMemcpyAsync(d_ip.p, static_cast<const unsigned char*>(indptr) + static_cast<size_t>(r0) * isz, static_cast<size_t>(nr + 1) * isz, cudaMemcpyHostToDevice, d->stream));
      if (ne > 0) {
        const int grid = static_cast<int>(std::min<int64_t>((nr + 7) / 8, 148 * 8));
        uint8_t* base = d->bins.p + static_cast<size_t>(r0) * 32;       // row offset inside every tile
#define B200_CSR_LAUNCH(TI, TV)                                                                                                              \
        k_bin_csr<TI, TV><<<grid, 256, 0, d->stream>>>(reinterpret_cast<const TI*>(d_ip.p), reinterpret_cast<const int*>(d_ix.p),               \
                                                      reinterpret_cast<const TV*>(d_v.p), nr, d_inner.p, d->meta.p, d->ub.p, d->catbin.p, base,  \
                                                      d->rows_stride, e0k, d->nfn, d->wide_meta.p, d->wide_cats.p, d->wide_catbin.p, d->wide_ub.p,  \
                                                      d->bins16.p ? d->bins16.p + r0 : nullptr)
        if (indptr_type == 2 && data_type == 0) B200_CSR_LAUNCH(int32_t, float);
        else if (indptr_type == 2) B200_CSR_LAUNCH(int32_t, double);
        else if (data_type == 0) B200_CSR_LAUNCH(int64_t, float);
        else B200_CSR_LAUNCH(int64_t, double);
#undef B200_CSR_LAUNCH
        B200_CUDA(cudaGetLastError());
      }
      B200_CUDA(cudaStreamSynchronize(d->stream));      // the staging buffers are reused by the next block
      r0 = r1;
    }
  }
  B200_CUDA(cudaEventRecord(e1, d->stream));
  B200_CUDA(cudaEventSynchronize(e1));
  float ms = 0;
  B200_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  d->ingest_ms = ms;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return d.release();
}

void Dataset::SetField(const char* name, const void* data, int n, int type) {
  EnsureDevice();
  std::string s(name);
  auto to_f32 = [&](std::vector<float>* out) {
    out->resize(n);
    if (type == 0) std::memcpy(out->data(), data, sizeof(float) * n);
    else if (type == 1) for (int i = 0; i < n; ++i) (*out)[i] = static_cast<float>(static_cast<const double*>(data)[i]);
    else Fatal("Input type error for field " + s + " (expect float32)");
  };
  if (s == "label" || s == "target") {
    if (n != num_data) Fatal("Length of label is not same with #data");
    to_f32(&label);
    d_label.Alloc(n); d_label.Upload(label.data(), n, stream);
  } else if (s == "weight" || s == "weights") {
    if (n == 0 || data == nullptr) { weight.clear(); d_weight.Free(); return; }
    if (n != num_data) Fatal("Length of weights is not same with #data");
    to_f32(&weight);
    d_weight.Alloc(n); d_weight.Upload(weight.data(), n, stream);
  } else if (s == "init_score") {
    if (n == 0 || data == nullptr) { init_score.clear(); return; }
    if (n % num_data != 0) Fatal("Initial score size doesn't match data size");
    init_score.resize(n);
    if (type == 1) std::memcpy(init_score.data(), data, sizeof(double) * n);
    else if (type == 0) for (int i = 0; i < n; ++i) init_score[i] = static_cast<const float*>(data)[i];
    else Fatal("Input type error for init_score (expect float64)");
  } else if (s == "group" || s == "query") {
    if (type != 2) Fatal("Input type error for group (expect int32)");
    const int32_t* g = static_cast<const int32_t*>(data);
    group_sizes.assign(g, g + n);
    query_boundaries.assign(1, 0);
    for (int i = 0; i < n; ++i) query_boundaries.push_back(query_boundaries.back() + g[i]);
    if (query_boundaries.back() != num_data) Fatal("Sum of query counts is not same with #data");
    d_qb.Alloc(query_boundaries.size()); d_qb.Upload(query_boundaries.data(), query_boundaries.size(), stream);
  } else {
    Fatal("Unknown field name: " + s);
  }
  B200_CUDA(cudaStreamSynchronize(stream));
}

void Dataset::GetField(const char* name, int* out_len, const void** out_ptr, int* out_type) const {
  std::string s(name);
  if (s == "label" || s == "target") { *out_len = static_cast<int>(label.size()); *out_ptr = label.data(); *out_type = 0; }
  else if (s == "weight" || s == "weights") { *out_len = static_cast<int>(weight.size()); *out_ptr = weight.empty() ? nullptr : weight.data(); *out_type = 0; }
  else if (s == "init_score") { *out_len = static_cast<int>(init_score.size()); *out_ptr = init_score.empty() ? nullptr : init_score.data(); *out_type = 1; }
  else if (s == "group" || s == "query") { *out_len = static_cast<int>(query_boundaries.size()); *out_ptr = query_boundaries.empty() ? nullptr : query_boundaries.data(); *out_type = 2; }
  else Fatal("Unknown field name: " + s);
}

void Dataset::SetFeatureNames(const char** names, int n) {
  if (n != num_total_features) Fatal("Size of feature_names error, should equal with total number of features");
  feature_names.assign(n, "");
  for (int i = 0; i < n; ++i) {
    feature_names[i] = names[i];
    for (auto& c : feature_names[i]) if (c == ' ') c = '_';
  }
}

// =============================================================================== booster
static size_t Align16(size_t x) { return (x + 15) & ~static_cast<size_t>(15); }
constexpr int kScanSmem = (768 + 64) * 8;         // k_scan: scratch of the categorical split search (one warp per block runs it)

Booster::Booster(const std::string& model_text) {
  std::unique_ptr<HostModel> m = HostModel::FromString(model_text);
  model = std::move(*m);
  K = model.num_tree_per_iteration;
  num_init_iteration = model.NumIterations();
}

Booster::Booster(const Dataset* tr, const char* params) : train(tr) {
  EnsureDevice();
  device_ = CurrentDevice();
  cfg.Parse(params);
  if (cfg.boosting != "gbdt" && cfg.boosting != "rf" && cfg.boosting != "goss" && cfg.boosting != "dart")
    Fatal("Unknown boosting type " + cfg.boosting);
  is_rf_ = cfg.boosting == "rf"; is_goss_ = cfg.boosting == "goss"; is_dart_ = cfg.boosting == "dart";
  drop_rand_ = LcgRandom(cfg.drop_seed);
  obj_.reset(new Objective(cfg, train));
  balanced_bagging_ = cfg.bagging_freq > 0 && (cfg.pos_bagging_fraction < 1.0 || cfg.neg_bagging_fraction < 1.0) && obj_->IsBinary();
  bagging_ = cfg.bagging_freq > 0 && (cfg.bagging_fraction < 1.0 || balanced_bagging_);
  if (bagging_ && !(cfg.bagging_fraction > 0.0)) Fatal("bagging_fraction should be in (0, 1]");
  if (is_goss_) {      // [LightGBM goss.hpp ResetGoss]
    if (!(cfg.top_rate + cfg.other_rate <= 1.0)) Fatal("Check failed: (config_->top_rate + config_->other_rate) <= (1.0f)");
    if (!(cfg.top_rate > 0.0 && cfg.other_rate > 0.0)) Fatal("Check failed: config_->top_rate > 0.0f && config_->other_rate > 0.0f");
    if (bagging_) Fatal("Cannot use bagging in GOSS");
  }
  if (is_rf_) {        // [LightGBM rf.hpp RF::Init]
    const bool ff = cfg.feature_fraction < 1.0 && cfg.feature_fraction > 0.0;
    if (!(bagging_ || ff)) Fatal("Check failed: (config->bagging_freq > 0 && config->bagging_fraction < 1.0f && config->bagging_fraction > 0.0f) || (config->feature_fraction < 1.0f && config->feature_fraction > 0.0f)");
  }
  if (cfg.num_leaves < 2) Fatal("num_leaves should be >= 2");
  ValidateMetrics();      // an unknown metric must fail LGBM_BoosterCreate, not the first LGBM_BoosterGetEval inside the training loop
  obj_->CheckData();
  CheckMetricLabels(train, cfg);
  K = obj_->NumModelPerIteration();
  parallel_ = Net().active && Net().world > 1;
  cfg.num_machines = parallel_ ? Net().world : 1;
  if (balanced_bagging_) {      // [LightGBM GBDT::ResetBaggingConfig] needs (globally) at least one positive row
    double npos = static_cast<double>(std::count_if(train->label.begin(), train->label.end(), [](float v) { return v > 0; }));
    if (parallel_) {
      cudaStream_t ts;
      B200_CUDA(cudaStreamCreateWithFlags(&ts, cudaStreamNonBlocking));
      AllReduceHost(&npos, 1, ncclSum, ts);
      B200_CUDA(cudaStreamDestroy(ts));
    }
    if (!(npos > 0)) { balanced_bagging_ = false; bagging_ = cfg.bagging_freq > 0 && cfg.bagging_fraction < 1.0; }
  }
  shrinkage_ = is_rf_ ? 1.0 : cfg.learning_rate;      // "no shrinkage rate for the RF"
  model.average_output = is_rf_;
  model.num_class = K;
  model.num_tree_per_iteration = K;
  model.label_index = 0;
  model.max_feature_idx = train->num_total_features - 1;
  model.feature_names = train->feature_names;
  for (int f = 0; f < train->num_total_features; ++f) model.feature_infos.push_back(train->mappers[f].InfoString());
  InitTraining();
  model.objective_str = obj_->ToString();
}

Booster::~Booster() {
  if (split_op_trees_ > 0) {
    double tot = 0; for (auto& kv : split_op_ms_) tot += kv.second;
    fprintf(stderr, "[b200gbm split timing] %d trees, %.3f ms per tree in split operations:", split_op_trees_, tot / split_op_trees_);
    for (auto& kv : split_op_ms_) fprintf(stderr, " %s=%.1fus", kv.first.c_str(), 1000.0 * kv.second / split_op_trees_ / std::max(cfg.num_leaves - 1, 1));
    fprintf(stderr, " (per split)\n");
  }
  for (auto* v : valids_) delete v;
  for (void* p : ipc_opened_) cudaIpcCloseMemHandle(p);
  if (tree_host_) cudaFreeHost(tree_host_);
  if (ctrl_host_) cudaFreeHost(ctrl_host_);
  if (leaves_host_) cudaFreeHost(leaves_host_);
  if (ev_a_) cudaEventDestroy(ev_a_);
  if (ev_b_) cudaEventDestroy(ev_b_);
  if (stream_) cudaStreamDestroy(stream_);
}

void Booster::GetInfo(int* out4) const {
  out4[0] = parallel_ ? Net().world : 1;
  out4[1] = parallel_ ? Net().rank : 0;
  out4[2] = fused_ ? 1 : (p2p_allreduce_ ? 2 : 0);
  out4[3] = obj_ && obj_->IsConstantHessian() && !is_goss_ ? 1 : 0;      // GOSS amplifies hessians [LightGBM goss.hpp GetIsConstHessian -> false]
}

void Booster::InitTraining() {
  const int n = train->num_data;
  const int L = cfg.num_leaves;
  cudaDeviceProp prop;
  B200_CUDA(cudaGetDeviceProperties(&prop, device_));
  num_sms_ = prop.multiProcessorCount;
  B200_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  B200_CUDA(cudaEventCreate(&ev_a_)); B200_CUDA(cudaEventCreate(&ev_b_));
  // leaf passes gather single 32-byte sectors: ask L2 not to fetch the neighbouring sector from DRAM on a miss (default 64 B).
  // A hint; measured +3.7 % on a 10 %-density leaf, neutral on streamed passes (profiles/r01_k4v4_cost_model.json)
  cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, 32);
  cudaGetLastError();
  B200_CUDA(cudaFuncSetAttribute(k4_hist_build_ws<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWsSmemBytes));
  B200_CUDA(cudaFuncSetAttribute(k4_hist_build_ws<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWsSmemBytes));
  B200_CUDA(cudaFuncSetAttribute(k_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, kScanSmem));

  sp_.l1 = cfg.lambda_l1; sp_.l2 = cfg.lambda_l2; sp_.max_delta_step = cfg.max_delta_step;
  sp_.min_gain_to_split = cfg.min_gain_to_split; sp_.min_sum_hessian = cfg.min_sum_hessian_in_leaf;
  sp_.min_data_in_leaf = cfg.min_data_in_leaf; sp_.max_depth = cfg.max_depth; sp_.num_leaves = L; sp_.parallel = parallel_ ? 1 : 0;
  sp_.nf = train->nf; sp_.nf_pad = train->nf_pad; sp_.num_tiles = train->num_tiles; sp_.nfn = train->nfn;
  {   // categorical split search parameters: native defaults unless given (SURVEY.md B.2)
    auto gd = [&](const char* k, double d) { auto it = cfg.raw.find(k); return (it != cfg.raw.end() && !it->second.empty()) ? std::atof(it->second.c_str()) : d; };
    sp_.cat_l2 = gd("cat_l2", 10.0); sp_.cat_smooth = gd("cat_smooth", 10.0);
    sp_.max_cat_threshold = static_cast<int>(gd("max_cat_threshold", 32)); sp_.max_cat_to_onehot = static_cast<int>(gd("max_cat_to_onehot", 4));
    sp_.min_data_per_group = static_cast<int>(gd("min_data_per_group", 100)); sp_.pad3 = 0;
    if (train->nw > 0) {
      if (sp_.max_cat_threshold > kCatListMax) Fatal("max_cat_threshold > " + std::to_string(kCatListMax) + " is not supported together with categorical features of more than 256 bins");
      if (sp_.max_cat_to_onehot > 256) Fatal("max_cat_to_onehot > 256 is not supported together with categorical features of more than 256 bins");
      B200_CUDA(cudaFuncSetAttribute(k4_hist_wide<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * kWideHistSeg * 4));
      B200_CUDA(cudaFuncSetAttribute(k4_hist_wide<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * kWideHistSeg * 4));
      B200_CUDA(cudaFuncSetAttribute(k_scan_wide, cudaFuncAttributeMaxDynamicSharedMemorySize, kWideMaxBins * 8));
    }
  }

  score_.Alloc(static_cast<size_t>(K) * n); score_.Zero(stream_);
  grad_.Alloc(static_cast<size_t>(K) * n); hess_.Alloc(static_cast<size_t>(K) * n);
  qgh_.Alloc(n); qord_.Alloc(n); idx0_.Alloc(n); idx1_.Alloc(n);
  slot_elems_ = train->hist_pairs * 2;
  H_.Alloc(slot_elems_); H_.Zero(stream_); pool_.Alloc(slot_elems_ * L);
  {
    int per_sm = 0;
    B200_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_partition, 256, 0));
    int coop = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device_);
    if (!coop || per_sm < 1) Fatal("this device cannot launch the cooperative partition kernel");
    part_max_blocks_ = per_sm * num_sms_;
  }
  flags_.Alloc(static_cast<size_t>(L) * train->nf_pad);
  cands_.Alloc(2 * static_cast<size_t>(train->nf_pad));
  leaves_.Alloc(L); ctrl_.Alloc(1); ctrl_.Zero(stream_);
  const int chunks = n / kPartChunk + 2;
  part_bits_.Alloc(static_cast<size_t>(chunks) * (kPartChunk / 32)); part_chunks_.Alloc(static_cast<size_t>(chunks) + chunks / kPartLocalScan + 8); part_chunks_.Zero(stream_);      // + the super-chunk totals of the two-level scan
  // SoA tree blob
  {
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += Align16(bytes); return o; };
    size_t o_lc = take(4 * (L - 1)), o_rc = take(4 * (L - 1)), o_sf = take(4 * (L - 1)), o_tb = take(4 * (L - 1)), o_dt = take(4 * (L - 1));
    size_t o_sg = take(4 * (L - 1)), o_lv = take(8 * L), o_lw = take(8 * L), o_lcn = take(4 * L), o_iv = take(8 * (L - 1)), o_iw = take(8 * (L - 1));
    size_t o_ic = take(4 * (L - 1)), o_lp = take(4 * L), o_ld = take(4 * L), o_nl = take(16), o_cb = take(32 * (L - 1));
    size_t o_cl = take(2 * kCatListMax * (L - 1)), o_cn = take(4 * (L - 1));
    tree_blob_bytes_ = off;
    tree_blob_.Alloc(off);
    unsigned char* b = tree_blob_.p;
    tree_dev_.left_child = reinterpret_cast<int*>(b + o_lc); tree_dev_.right_child = reinterpret_cast<int*>(b + o_rc);
    tree_dev_.split_feature_inner = reinterpret_cast<int*>(b + o_sf); tree_dev_.threshold_bin = reinterpret_cast<int*>(b + o_tb);
    tree_dev_.decision_type = reinterpret_cast<int*>(b + o_dt); tree_dev_.split_gain = reinterpret_cast<float*>(b + o_sg);
    tree_dev_.leaf_value = reinterpret_cast<double*>(b + o_lv); tree_dev_.leaf_weight = reinterpret_cast<double*>(b + o_lw);
    tree_dev_.leaf_count = reinterpret_cast<int*>(b + o_lcn); tree_dev_.internal_value = reinterpret_cast<double*>(b + o_iv);
    tree_dev_.internal_weight = reinterpret_cast<double*>(b + o_iw); tree_dev_.internal_count = reinterpret_cast<int*>(b + o_ic);
    tree_dev_.leaf_parent = reinterpret_cast<int*>(b + o_lp); tree_dev_.leaf_depth = reinterpret_cast<int*>(b + o_ld);
    tree_dev_.num_leaves = reinterpret_cast<int*>(b + o_nl);
    tree_dev_.cat_bits = reinterpret_cast<unsigned*>(b + o_cb);
    tree_dev_.cat_list = reinterpret_cast<unsigned short*>(b + o_cl);
    tree_dev_.cat_list_len = reinterpret_cast<int*>(b + o_cn);
    B200_CUDA(cudaMemsetAsync(b, 0, off, stream_));
    B200_CUDA(cudaMallocHost(reinterpret_cast<void**>(&tree_host_), off));
    B200_CUDA(cudaMallocHost(reinterpret_cast<void**>(&ctrl_host_), sizeof(TreeCtrl)));
    B200_CUDA(cudaMallocHost(reinterpret_cast<void**>(&leaves_host_), sizeof(LeafState) * L));
  }
  // init score from the dataset
  if (!train->init_score.empty()) {
    if (train->init_score.size() != static_cast<size_t>(K) * n) Fatal("Initial score size doesn't match data size");
    has_init_score_ = true;
    score_.Upload(train->init_score.data(), train->init_score.size(), stream_);
  }
  // ---- objective set-up
  obj_->Init(stream_, num_sms_);
  if (obj_->IsRenewTreeOutput()) {
    // sort buffers of the renewal pass (renew_kernel.cuh)
    rn_keys_a_.Alloc(n); rn_keys_b_.Alloc(n); rn_pos_a_.Alloc(n); rn_pos_b_.Alloc(n); rn_leaf_of_pos_.Alloc(n); rn_leaf_a_.Alloc(n); rn_leaf_b_.Alloc(n);
    rn_res_.Alloc(n); rn_row_.Alloc(n); rn_seg_.Alloc(L + 1); rn_out_.Alloc(2 * static_cast<size_t>(L));
    if (obj_->RenewWeights()) rn_cdf_.Alloc(n);
    size_t t1 = 0, t2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, rn_keys_a_.p, rn_keys_b_.p, rn_pos_a_.p, rn_pos_b_.p, n, 0, 64, stream_);
    cub::DeviceRadixSort::SortPairs(nullptr, t2, rn_leaf_a_.p, rn_leaf_b_.p, rn_pos_b_.p, rn_pos_a_.p, n, 0, 32, stream_);
    rn_tmp_bytes_ = std::max(t1, t2);
    rn_tmp_.Alloc(rn_tmp_bytes_ + 16);
  }
  if (parallel_) SetupPeerReduce();
  // ColSampler: one draw at init, then one per tree ([UPSTREAM] ColSampler::SetTrainingData / ResetByTree)
  col_rand_ = LcgRandom(cfg.feature_fraction_seed);
  feature_used_host_.assign(train->nf_pad, 0);
  for (int u = 0; u < train->nf; ++u) feature_used_host_[u] = 1;
  feature_used_.Alloc(train->nf_pad);
  feature_used_.Upload(feature_used_host_.data(), train->nf_pad, stream_);
  ResetFeaturesByTree();
  if (bagging_ || is_goss_) {
    bag_blocks_ = (n + kBagBlock - 1) / kBagBlock;
    std::vector<unsigned> st(bag_blocks_);
    for (int i = 0; i < bag_blocks_; ++i) st[i] = static_cast<unsigned>(cfg.bagging_seed + i);     // bagging_rands_[i] = Random(bagging_seed + i)
    bag_lcg_.Alloc(bag_blocks_); bag_lcg_.Upload(st.data(), st.size(), stream_);
    std::unique_ptr<LcgJump> jt(new LcgJump());
    unsigned a = 1, c = 0;
    for (int j = 0; j < kBagBlock; ++j) { a = a * 214013u; c = c * 214013u + 2531011u; jt->mul[j] = a; jt->add[j] = c; }
    bag_jump_.Alloc(1); bag_jump_.Upload(jt.get(), 1, stream_);
    in_bag_.Alloc(n); bag_block_cnt_.Alloc(bag_blocks_); bag_idx_.Alloc(n); bag_total_.Alloc(1);
    need_re_bagging_ = bagging_;
    B200_CUDA(cudaStreamSynchronize(stream_));
  }
  if (is_rf_) {        // [LightGBM rf.hpp RF::Boosting] gradients are taken once, at the constant init score
    if (!train->init_score.empty()) Fatal("Check failed: train_data->metadata().init_score() == nullptr");
    rf_init_scores_.assign(K, 0.0);
    DevBuf<double> tmp;
    tmp.Alloc(static_cast<size_t>(K) * n); tmp.Zero(stream_);
    for (int k = 0; k < K; ++k) {
      double init = (cfg.boost_from_average && !has_init_score_) ? obj_->BoostFromScore(k) : 0.0;
      if (!(std::fabs(init) > kEps)) init = 0.0;
      rf_init_scores_[k] = init;
      if (init != 0.0) k_add_const<<<num_sms_ * 4, 256, 0, stream_>>>(tmp.p + static_cast<size_t>(k) * n, n, init);
    }
    ComputeGradientsAt(tmp.p);
    B200_CUDA(cudaStreamSynchronize(stream_));
  }
  B200_CUDA(cudaStreamSynchronize(stream_));
}

// ---- DART [LightGBM src/boosting/dart.hpp]
TreeDev Booster::RebasedTree(unsigned char* base) const {
  TreeDev t = tree_dev_;
  auto mv = [&](auto*& p) { p = reinterpret_cast<std::remove_reference_t<decltype(p)>>(base + (reinterpret_cast<unsigned char*>(p) - tree_blob_.p)); };
  mv(t.left_child); mv(t.right_child); mv(t.split_feature_inner); mv(t.threshold_bin); mv(t.decision_type); mv(t.split_gain);
  mv(t.leaf_value); mv(t.leaf_weight); mv(t.leaf_count); mv(t.internal_value); mv(t.internal_weight); mv(t.internal_count);
  mv(t.leaf_parent); mv(t.leaf_depth); mv(t.num_leaves); mv(t.cat_bits); mv(t.cat_list); mv(t.cat_list_len);
  return t;
}
// ScoreUpdater::AddScore(models_[tree], class): the tree's CURRENT host leaf values (after the Shrinkage calls) are pushed into
// its stored device blob and every row walks the tree on its bins.
void Booster::AddStoredTree(int iter_index, int k, bool to_train, bool to_valid) {
  const size_t ti = static_cast<size_t>(num_init_iteration + iter_index) * K + k;
  const HostTree& ht = *model.trees[ti];
  cudaStream_t s = stream_;
  const int n = train->num_data;
  if (ht.num_leaves <= 1) {
    const double v = ht.leaf_value[0];
    if (v != 0.0) {
      if (to_train) k_add_const<<<num_sms_ * 4, 256, 0, s>>>(score_.p + static_cast<size_t>(k) * n, n, v);
      if (to_valid) for (auto* vs : valids_) k_add_const<<<num_sms_ * 4, 256, 0, s>>>(vs->score.p + static_cast<size_t>(k) * vs->ds->num_data, vs->ds->num_data, v);
    }
    return;
  }
  DevBuf<unsigned char>& blob = *tree_store_.at(static_cast<size_t>(iter_index) * K + k);
  TreeDev td = RebasedTree(blob.p);
  B200_CUDA(cudaMemcpyAsync(td.leaf_value, ht.leaf_value.data(), sizeof(double) * ht.num_leaves, cudaMemcpyHostToDevice, s));
  const int egrid = num_sms_ * 8;
  if (to_train) k_add_tree_binned<<<egrid, 256, 0, s>>>(td, train->meta.p, train->View(), n, score_.p + static_cast<size_t>(k) * n, 1.0);
  if (to_valid)
    for (auto* vs : valids_)
      k_add_tree_binned<<<egrid, 256, 0, s>>>(td, vs->ds->meta.p, vs->ds->View(), vs->ds->num_data,
                                              vs->score.p + static_cast<size_t>(k) * vs->ds->num_data, 1.0);
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaStreamSynchronize(s));        // the pageable host leaf values must stay put until the copy is done
  timing.launches += (to_train ? 1 : 0) + (to_valid ? static_cast<long long>(valids_.size()) : 0);
}
void Booster::DroppingTrees() {
  drop_index_.clear();
  const bool is_skip = drop_rand_.NextFloat() < cfg.skip_drop;
  if (!is_skip) {
    double drop_rate = cfg.drop_rate;
    if (!cfg.uniform_drop) {
      const double inv_average_weight = static_cast<double>(tree_weight_.size()) / sum_weight_;
      if (cfg.max_drop > 0) drop_rate = std::min(drop_rate, cfg.max_drop * inv_average_weight / sum_weight_);
      for (int i = 0; i < iter; ++i)
        if (drop_rand_.NextFloat() < drop_rate * tree_weight_[i] * inv_average_weight) {
          drop_index_.push_back(i);
          if (drop_index_.size() >= static_cast<size_t>(cfg.max_drop)) break;
        }
    } else {
      if (cfg.max_drop > 0) drop_rate = std::min(drop_rate, cfg.max_drop / static_cast<double>(iter));
      for (int i = 0; i < iter; ++i)
        if (drop_rand_.NextFloat() < drop_rate) {
          drop_index_.push_back(i);
          if (drop_index_.size() >= static_cast<size_t>(cfg.max_drop)) break;
        }
    }
  }
  for (int i : drop_index_)
    for (int k = 0; k < K; ++k) {
      model.trees[static_cast<size_t>(num_init_iteration + i) * K + k]->Shrink(-1.0);
      AddStoredTree(i, k, true, false);
    }
  if (!cfg.xgboost_dart_mode) shrinkage_ = cfg.learning_rate / (1.0f + static_cast<double>(drop_index_.size()));
  else if (drop_index_.empty()) shrinkage_ = cfg.learning_rate;
  else shrinkage_ = cfg.learning_rate / (cfg.learning_rate + static_cast<double>(drop_index_.size()));
  if (!drop_index_.empty()) forest_.reset();
  dart_dropped_this_iter_ = true;
}
void Booster::DartNormalize() {
  const double k = static_cast<double>(drop_index_.size());
  for (int i : drop_index_) {
    for (int c = 0; c < K; ++c) {
      HostTree& t = *model.trees[static_cast<size_t>(num_init_iteration + i) * K + c];
      if (!cfg.xgboost_dart_mode) {
        t.Shrink(1.0f / (k + 1.0f)); AddStoredTree(i, c, false, true);
        t.Shrink(-k); AddStoredTree(i, c, true, false);
      } else {
        t.Shrink(shrinkage_); AddStoredTree(i, c, false, true);
        t.Shrink(-k / cfg.learning_rate); AddStoredTree(i, c, true, false);
      }
    }
    if (!cfg.uniform_drop) {
      if (!cfg.xgboost_dart_mode) { sum_weight_ -= tree_weight_[i] * (1.0f / (k + 1.0f)); tree_weight_[i] *= (k / (k + 1.0f)); }
      else { sum_weight_ -= tree_weight_[i] * (1.0f / (k + cfg.learning_rate)); tree_weight_[i] *= (k / (k + cfg.learning_rate)); }
    }
  }
  if (!drop_index_.empty()) forest_.reset();        // leaf values of earlier trees changed: the device forest for predict is stale
}

// [LightGBM gbdt.cpp GBDT::Bagging / goss.hpp GOSS::Bagging] draws the in-bag flags on the device, compacts the in-bag rows
// (ascending) into bag_idx_; the tree's root leaf is that list.  One small D2H (the bag size) per re-bagging.
void Booster::Bagging(int it) {
  const int n = train->num_data;
  cudaStream_t s = stream_;
  if (is_goss_) {
    use_bag_ = false;
    if (it < static_cast<int>(1.0f / cfg.learning_rate)) return;
    k_goss_draw<<<bag_blocks_, 256, 0, s>>>(bag_lcg_.p, n, K, cfg.top_rate, cfg.other_rate, grad_.p, hess_.p, in_bag_.p, bag_block_cnt_.p);
  } else {
    if (!bagging_) return;
    if (!((use_bag_ && it % cfg.bagging_freq == 0) || need_re_bagging_)) return;
    need_re_bagging_ = false;
    k_bag_draw<<<bag_blocks_, 256, 0, s>>>(bag_lcg_.p, bag_jump_.p, n, cfg.bagging_fraction, in_bag_.p, bag_block_cnt_.p,
                                           balanced_bagging_ ? train->d_label.p : nullptr, cfg.pos_bagging_fraction, cfg.neg_bagging_fraction);
  }
  k_bag_scan<<<1, 1024, 0, s>>>(bag_block_cnt_.p, bag_blocks_, bag_total_.p);
  k_bag_compact<<<bag_blocks_, 256, 0, s>>>(in_bag_.p, bag_block_cnt_.p, n, bag_idx_.p);
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaMemcpyAsync(&bag_count_, bag_total_.p, sizeof(int), cudaMemcpyDeviceToHost, s));
  B200_CUDA(cudaStreamSynchronize(s));
  timing.launches += 3;
  use_bag_ = true;
}

// Peer-memory set-up for the fused reduce+scan (k_scan_dp / k_pick_dp): every rank publishes its scratch histogram, mailbox and
// flag block; ranks in the same process exchange raw pointers (peer access), ranks in other processes CUDA-IPC handles.
struct PeerInfo {
  long long pid;
  int device, ok;
  unsigned long long ptr[3];
  cudaIpcMemHandle_t ipc[3];
};
void Booster::SetupPeerReduce() {
  const char* env = std::getenv("B200GBM_FUSED_REDUCE");
  const int R = Net().world, me = Net().rank;
  mailbox_.Alloc(static_cast<size_t>(kMaxPeers) * 2); mailbox_.Zero(stream_);
  peer_flags_.Alloc(64); peer_flags_.Zero(stream_);      // [0,16) "histogram ready" epochs by rank, [16,32) "second barrier" epochs, [48] block ticket
  peer_error_.Alloc(1); peer_error_.Zero(stream_);
  B200_CUDA(cudaStreamSynchronize(stream_));
  PeerInfo mine{};
  mine.pid = static_cast<long long>(getpid()); mine.device = device_;
  // Default = NCCL: measured on 8xB200 (100M x 512, profiles/r01_fused_vs_nccl_8gpu.md) the in-switch ncclAllReduce of the 2 MB
  // histogram is ~3 % faster end to end than the fused peer-memory reduce-scatter (two cross-GPU flag barriers per split).
  int mode = env ? std::atoi(env) : 0;      // 0 NCCL, 1 fused reduce-scatter + scan of the owned slice, 2 two-shot P2P all-reduce + replicated scan
  if (mode == 1 && train->has_categorical) mode = 0;      // the fused scan handles numerical tile features only (same decision on every rank)
  mine.ok = (R <= kMaxPeers && (mode == 1 || mode == 2)) ? 1 : 0;
  void* bufs[3] = {H_.p, mailbox_.p, peer_flags_.p};
  for (int i = 0; i < 3; ++i) {
    mine.ptr[i] = reinterpret_cast<unsigned long long>(bufs[i]);
    if (cudaIpcGetMemHandle(&mine.ipc[i], bufs[i]) != cudaSuccess) { cudaGetLastError(); mine.ok = 0; }
  }
  std::vector<PeerInfo> all(R);
  {
    DevBuf<unsigned char> ds, dr; ds.Alloc(sizeof(PeerInfo)); dr.Alloc(sizeof(PeerInfo) * R);
    B200_CUDA(cudaMemcpyAsync(ds.p, &mine, sizeof(PeerInfo), cudaMemcpyHostToDevice, stream_));
    B200_NCCL(ncclAllGather(ds.p, dr.p, sizeof(PeerInfo), ncclChar, Net().comm, stream_));
    B200_CUDA(cudaMemcpyAsync(all.data(), dr.p, sizeof(PeerInfo) * R, cudaMemcpyDeviceToHost, stream_));
    B200_CUDA(cudaStreamSynchronize(stream_));
  }
  int ok = 1;
  for (int r = 0; r < R; ++r) ok &= all[r].ok;
  PeerTables pt{};
  if (ok) {
    for (int r = 0; r < R && ok; ++r) {
      void* p3[3];
      if (r == me) { for (int i = 0; i < 3; ++i) p3[i] = bufs[i]; }
      else if (all[r].pid == mine.pid) {          // rank-thread of the same process (the reference's local mode)
        int can = 0;
        cudaDeviceCanAccessPeer(&can, device_, all[r].device);
        if (!can) { ok = 0; break; }
        cudaError_t e = cudaDeviceEnablePeerAccess(all[r].device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); ok = 0; break; }
        cudaGetLastError();
        for (int i = 0; i < 3; ++i) p3[i] = reinterpret_cast<void*>(all[r].ptr[i]);
      } else {                                    // one process per GPU (torchrun): CUDA IPC
        for (int i = 0; i < 3; ++i) {
          if (cudaIpcOpenMemHandle(&p3[i], all[r].ipc[i], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { cudaGetLastError(); ok = 0; break; }
          ipc_opened_.push_back(p3[i]);
        }
        if (!ok) break;
      }
      pt.H[r] = static_cast<const long long*>(p3[0]); pt.mail[r] = static_cast<SplitCand*>(p3[1]); pt.flags[r] = static_cast<unsigned*>(p3[2]);
    }
  }
  // every rank must take the same path: agree on `ok`
  double okd = ok ? 1.0 : 0.0;
  AllReduceHost(&okd, 1, ncclMin, stream_);
  const bool peers_ok = okd > 0.5;
  fused_ = peers_ok && mode == 1;
  p2p_allreduce_ = peers_ok && mode == 2;
  if (p2p_allreduce_) { pt.rank = me; pt.world = R; pt.feat0 = 0; pt.feat1 = 0; pt.error = peer_error_.p; peers_ = pt; return; }
  if (!fused_) return;
  const int tiles_per_rank = (train->num_tiles + R - 1) / R;
  pt.rank = me; pt.world = R;
  pt.feat0 = std::min(train->nf_pad, me * tiles_per_rank * 32);
  pt.feat1 = std::min(train->nf_pad, (me + 1) * tiles_per_rank * 32);
  pt.error = peer_error_.p;
  peers_ = pt;
}

void Booster::ResetFeaturesByTree() {
  if (cfg.feature_fraction >= 1.0) return;
  const int total = train->nf;
  int cnt = std::max(static_cast<int>(total * cfg.feature_fraction + 0.5), std::min(2, total));
  std::fill(feature_used_host_.begin(), feature_used_host_.end(), 0);
  for (int i : col_rand_.Sample(total, cnt)) feature_used_host_[train->sample_order[i]] = 1;      // the draw indexes the used features in real-index order
  // no host sync: the copy is ordered after the previous tree's kernels on the same stream, and a copy from pageable memory is staged
  // by the driver before the call returns, so the host vector may be rewritten for the next tree
  feature_used_.Upload(feature_used_host_.data(), train->nf_pad, stream_);
}

double Booster::BoostFromAverage(int k) {
  if (model.trees.empty() && !has_init_score_ && cfg.boost_from_average) {
    double init = obj_->BoostFromScore(k);
    if (std::fabs(init) > kEps) {
      const int n = train->num_data;
      k_add_const<<<num_sms_ * 4, 256, 0, stream_>>>(score_.p + static_cast<size_t>(k) * n, n, init);
      for (auto* v : valids_) k_add_const<<<num_sms_ * 4, 256, 0, stream_>>>(v->score.p + static_cast<size_t>(k) * v->ds->num_data, v->ds->num_data, init);
      B200_CUDA(cudaGetLastError());
      return init;
    }
  }
  return 0.0;
}

void Booster::ComputeGradients() { ComputeGradientsAt(score_.p); }
void Booster::ComputeGradientsAt(const double* score_p) {
  NvtxRange nvtx("b200gbm:K1/K2 gradients");
  obj_->GetGradients(score_p, grad_.p, hess_.p);
  B200_CUDA(cudaGetLastError());
  timing.launches += 1;
}

// [LightGBM SerialTreeLearner::RenewTreeOutput] device pass described in renew_kernel.cuh; patches tree_dev_.leaf_value in place
void Booster::RenewTreeOutput(int k, double rf_pred) {
  const int n = train->num_data;
  const int total = use_bag_ ? bag_count_ : n;
  const int L = cfg.num_leaves;
  cudaStream_t s = stream_;
  TreeCtrl* ctrl = ctrl_.p;
  const int egrid = num_sms_ * 8;
  const float* wptr = obj_->RenewWeights();
  const bool weighted = wptr != nullptr;
  const double alpha = obj_->RenewAlpha();
  k_renew_gather<<<egrid, 256, 0, s>>>(ctrl, leaves_.p, idx0_.p, idx1_.p, train->d_label.p, is_rf_ ? nullptr : score_.p + static_cast<size_t>(k) * n, rf_pred,
                                       rn_keys_a_.p, rn_pos_a_.p, rn_res_.p, rn_leaf_of_pos_.p, rn_row_.p);
  size_t tb = rn_tmp_bytes_;
  B200_CUDA(cub::DeviceRadixSort::SortPairs(rn_tmp_.p, tb, rn_keys_a_.p, rn_keys_b_.p, rn_pos_a_.p, rn_pos_b_.p, total, 0, 64, s));
  k_renew_leaf_keys<<<egrid, 256, 0, s>>>(rn_pos_b_.p, rn_leaf_of_pos_.p, total, rn_leaf_a_.p);
  int leaf_bits = 1;
  while ((1 << leaf_bits) < L) ++leaf_bits;
  tb = rn_tmp_bytes_;
  B200_CUDA(cub::DeviceRadixSort::SortPairs(rn_tmp_.p, tb, rn_leaf_a_.p, rn_leaf_b_.p, rn_pos_b_.p, rn_pos_a_.p, total, 0, leaf_bits, s));
  k_renew_offsets<<<1, 32, 0, s>>>(ctrl, leaves_.p, rn_seg_.p);
  double* out = rn_out_.p;
  double* has = rn_out_.p + L;
  const int lgrid = (L + 127) / 128;
  if (!weighted) {
    k_renew_unweighted<<<lgrid, 128, 0, s>>>(ctrl, rn_seg_.p, rn_pos_a_.p, rn_res_.p, alpha, out, has);
  } else {
    k_renew_cdf<<<L, 1024, 0, s>>>(ctrl, rn_seg_.p, rn_pos_a_.p, rn_row_.p, wptr, rn_cdf_.p);
    k_renew_weighted<<<lgrid, 128, 0, s>>>(ctrl, rn_seg_.p, rn_pos_a_.p, rn_res_.p, rn_cdf_.p, alpha, out, has);
  }
  if (parallel_) B200_NCCL(ncclAllReduce(out, out, 2 * static_cast<size_t>(L), ncclDouble, ncclSum, Net().comm, s));
  k_renew_apply<<<lgrid, 128, 0, s>>>(ctrl, tree_dev_, out, has, parallel_ ? 1 : 0);
  B200_CUDA(cudaGetLastError());
  timing.launches += weighted ? 7 : 6;
}

// k_partition is launched cooperatively: its software grid barriers need every block resident
// Column-major copy of the training tiles for k_partition (kernels.cuh: k_tiles_to_columns).  Built once, before the first tree, after every
// other buffer of the booster exists, and only if it leaves a reserve of device memory (validation scores, metric and prediction scratch
// come later); B200GBM_COLUMN_COPY=0 disables it.  Without it the partition reads one 32-byte sector per row — same results.
void Booster::EnsureColumnCopy() {
  if (cols_tried_) return;
  cols_tried_ = true;
  const Dataset& d = *train;
  const char* env = std::getenv("B200GBM_COLUMN_COPY");
  if ((env && std::atoi(env) == 0) || d.nfn == 0 || d.num_data == 0) return;
  const size_t stride = (static_cast<size_t>(d.num_data) + 255) & ~static_cast<size_t>(255);
  const size_t need = static_cast<size_t>(d.num_tiles) * 32 * stride;
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return; }
  const size_t reserve = std::max<size_t>(static_cast<size_t>(8) << 30, total_b / 10);
  if (free_b < need + reserve) return;
  uint8_t* p = nullptr;
  if (cudaMalloc(reinterpret_cast<void**>(&p), need) != cudaSuccess) { cudaGetLastError(); return; }
  bins_cols_.p = p; bins_cols_.n = need;
  cols_stride_ = stride;
  const long long work = ((static_cast<long long>(d.num_data) + 255) / 256) * d.num_tiles;
  k_tiles_to_columns<<<static_cast<unsigned>(std::min<long long>(work, static_cast<long long>(num_sms_) * 16)), 256, 0, stream_>>>(
      d.bins.p, d.rows_stride, d.num_tiles, d.num_data, bins_cols_.p, stride);
  B200_CUDA(cudaGetLastError());
}

void Booster::GetMemoryInfo(int64_t* out2) {
  EnsureDevice();
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); free_b = 0; }
  out2[0] = static_cast<int64_t>(bins_cols_.n);
  out2[1] = static_cast<int64_t>(free_b);
}

void Booster::LaunchPartition(int grid, int last) {
  const Dataset& d = *train;
  TreeCtrl* ctrl = ctrl_.p;
  LeafState* leaves = leaves_.p;
  TreeDev tree = tree_dev_;
  uint8_t* flags = flags_.p;
  const FeatMeta* meta = d.meta.p;
  SplitParams sp = sp_;
  const uint8_t* bins = d.bins.p;
  size_t rows_stride = d.rows_stride;
  int* i0 = idx0_.p; int* i1 = idx1_.p;
  unsigned* bits = part_bits_.p;
  int* chunks = part_chunks_.p;
  const int4* qgh = qgh_.p;
  int4* qord = qord_.p;
  long long* H = H_.p;
  size_t h_elems = slot_elems_;
  const uint16_t* bins16 = d.bins16.p;
  static const int tickets = [] { const char* e = std::getenv("B200GBM_PART_TICKETS"); return e ? std::atoi(e) : 8; }();      // 0: one chunk per ticket
  int tickets_per_block = tickets;
  const uint8_t* cols = bins_cols_.p;
  size_t cols_stride = cols_stride_;
  int* super_tot = part_chunks_.p + (train->num_data / kPartChunk + 2);
  void* args[] = {&ctrl, &leaves, &tree, &flags, &meta, &sp, &last, &bins, &rows_stride, &i0, &i1, &bits, &chunks, &qgh, &qord, &H, &h_elems, &bins16, &tickets_per_block,
                  &cols, &cols_stride, &super_tot};
  B200_CUDA(cudaLaunchCooperativeKernel(reinterpret_cast<void*>(k_partition), dim3(grid), dim3(256), args, 0, stream_));
}

// One tree: the whole leaf-wise growth is enqueued without a host sync; leaf choice, smaller/larger
// selection, partition sizes all live in TreeCtrl / LeafState on the device.
void Booster::TrainOneTree(int k, HostTree* out, bool const_hessian) {
  NvtxRange nvtx_tree("b200gbm:tree");
  EnsureColumnCopy();
  const Dataset& d = *train;
  const int n = d.num_data;
  const int L = cfg.num_leaves;
  const float* g = grad_.p + static_cast<size_t>(k) * n;
  const float* h = hess_.p + static_cast<size_t>(k) * n;
  TreeCtrl* ctrl = ctrl_.p;
  cudaStream_t s = stream_;
  const int egrid = num_sms_ * 8;
  nvtxRangePushA("b200gbm:K3 quantize + C1 root sums");
  B200_CUDA(cudaMemsetAsync(&ctrl->absmax_bits[0], 0, 8, s));
  k_absmax<<<egrid, 256, 0, s>>>(g, h, n, ctrl);
  if (parallel_) B200_NCCL(ncclAllReduce(&ctrl->absmax_bits[0], &ctrl->absmax_bits[0], 2, ncclUint32, ncclMax, Net().comm, s));
  k_set_scale<<<1, 1, 0, s>>>(ctrl, const_hessian ? 1 : 0, 1.0);
  k_quantize<<<egrid, 256, 0, s>>>(g, h, n, qgh_.p, ctrl, const_hessian ? 1 : 0, use_bag_ ? in_bag_.p : nullptr, bag_count_);
  if (parallel_) B200_NCCL(ncclAllReduce(&ctrl->root_q[0], &ctrl->root_q[0], 3, ncclInt64, ncclSum, Net().comm, s));
  ResetFeaturesByTree();
  if (use_bag_)      // the root leaf is the ascending in-bag row list (SetBaggingData); partitions then ping-pong idx0/idx1 as usual
    B200_CUDA(cudaMemcpyAsync(idx0_.p, bag_idx_.p, static_cast<size_t>(bag_count_) * sizeof(int), cudaMemcpyDeviceToDevice, s));
  k_tree_init<<<1, 256, 0, s>>>(ctrl, leaves_.p, tree_dev_, flags_.p, sp_, use_bag_ ? bag_count_ : n, feature_used_.p, use_bag_ ? 1 : 0);
  nvtxRangePop();
  timing.launches += 4;
  const int pgrid = std::max(1, std::min(n / kPartChunk + 1, part_max_blocks_));
  const dim3 sgrid(std::max(1, d.nfn), 2);      // one block per (leaf, tile feature); the pick step in the last block also sees the wide features' candidates
  std::vector<cudaEvent_t> evs;
  // B200GBM_SPLIT_TIMING=1 (debug): an event after every operation of a split; per-operation averages go to stderr when the booster is freed
  static const bool split_timing = getenv("B200GBM_SPLIT_TIMING") != nullptr;
  std::vector<cudaEvent_t> sev;
  auto mark = [&]() { if (split_timing) { cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s); sev.push_back(e); } };
  // round 0's controller is its own launch; every later round's runs in the tail of the previous round's partition kernel
  k_round_ctl<<<1, 256, 0, s>>>(ctrl, leaves_.p, tree_dev_, flags_.p, d.meta.p, sp_, 0);
  timing.launches += 1;
  for (int split = 0; split < L - 1; ++split) {
    mark();
    if (profile_hist) { cudaEvent_t a, b; B200_CUDA(cudaEventCreate(&a)); B200_CUDA(cudaEventCreate(&b)); evs.push_back(a); evs.push_back(b); B200_CUDA(cudaEventRecord(a, s)); }
    // leaf order of the (g,h) words: written by the previous split's partition kernel; only a bagged root needs its own pass
    if (split == 0 && use_bag_) k_gather_q<<<egrid, 256, 0, s>>>(&ctrl->hist_work, idx0_.p, idx1_.p, qgh_.p, qord_.p);
    mark();
    // the scratch histogram H is zero here: zeroed at set-up and by every partition kernel after the scan consumed it
    nvtxRangePushA("b200gbm:K4 histogram");
    if (const_hessian)
      k4_hist_build_ws<3><<<num_sms_, kWsThreads, kWsSmemBytes, s>>>(d.bins.p, d.rows_stride, d.num_tiles, qgh_.p, qord_.p, idx0_.p, idx1_.p, &ctrl->hist_work,
                                                                     reinterpret_cast<unsigned long long*>(H_.p));
    else
      k4_hist_build_ws<4><<<num_sms_, kWsThreads, kWsSmemBytes, s>>>(d.bins.p, d.rows_stride, d.num_tiles, qgh_.p, qord_.p, idx0_.p, idx1_.p, &ctrl->hist_work,
                                                                     reinterpret_cast<unsigned long long*>(H_.p));
    if (d.nw > 0) {      // the features with more than 256 bins: own sub-histogram layout (k4_hist_wide)
      int max_nb = 0;
      for (const WideMeta& wm : d.wide_host) max_nb = std::max(max_nb, wm.num_bin);
      const int segs = (max_nb + kWideHistSeg - 1) / kWideHistSeg;      // z: 8192-bin segments of the largest feature
      // x: row parts, chosen so that the CTAs that have work (a (feature, segment) pair past the feature's last bin exits at once) make
      // about four waves of one CTA per SM (128 KB of shared memory each)
      int units = 0;
      for (const WideMeta& wm : d.wide_host) units += (wm.num_bin + kWideHistSeg - 1) / kWideHistSeg;
      const dim3 wgrid(static_cast<unsigned>(std::max(1, std::min(64, 4 * num_sms_ / std::max(1, units)))), static_cast<unsigned>(d.nw), static_cast<unsigned>(segs));
      if (const_hessian)
        k4_hist_wide<3><<<wgrid, kWideThreads, 4 * kWideHistSeg * 4, s>>>(d.bins16.p, d.rows_stride, d.wide_meta.p, qgh_.p, qord_.p, idx0_.p, idx1_.p, &ctrl->hist_work,
                                                                         reinterpret_cast<unsigned long long*>(H_.p));
      else
        k4_hist_wide<4><<<wgrid, kWideThreads, 4 * kWideHistSeg * 4, s>>>(d.bins16.p, d.rows_stride, d.wide_meta.p, qgh_.p, qord_.p, idx0_.p, idx1_.p, &ctrl->hist_work,
                                                                         reinterpret_cast<unsigned long long*>(H_.p));
      timing.launches += 1;
    }
    nvtxRangePop();
    if (profile_hist) B200_CUDA(cudaEventRecord(evs.back(), s));
    mark();
    nvtxRangePushA(parallel_ ? "b200gbm:C2 histogram reduce + K5 scan + pick" : "b200gbm:K5 scan + pick");
    if (fused_) {
      // C2+K5+C3 fused over NVLink peer memory: signal "histogram ready", then the scan reduces its owned slice from all peers
      ++epoch_;
      const dim3 dgrid(std::max(1, (peers_.feat1 - peers_.feat0 + 7) / 8), 2);
      k_scan_dp<<<dgrid, 256, 0, s>>>(ctrl, leaves_.p, d.meta.p, peers_, pool_.p, slot_elems_, flags_.p, cands_.p, sp_, epoch_);
      k_pick_dp<<<1, 256, 0, s>>>(ctrl, leaves_.p, d.meta.p, cands_.p, sp_, peers_, epoch_);
      mark();
    } else {
      if (p2p_allreduce_) {       // C2 as one kernel over NVLink peer memory (k_allreduce_p2p)
        ++epoch_;
        const int agrid = static_cast<int>(std::max<size_t>(1, std::min<size_t>(64, slot_elems_ / 2 / Net().world / 256 + 1)));
        k_allreduce_p2p<<<agrid, 256, 0, s>>>(ctrl, peers_, slot_elems_, epoch_, peer_flags_.p + 48);
        timing.launches += 1;
      } else if (parallel_) {
        B200_NCCL(ncclAllReduce(H_.p, H_.p, slot_elems_, ncclInt64, ncclSum, Net().comm, s));   // C2
      }
      mark();
      if (d.nw > 0) {
        k_scan_wide<<<dim3(d.nw, 2), 256, kWideMaxBins * 8, s>>>(ctrl, leaves_.p, d.wide_meta.p, H_.p, pool_.p, slot_elems_, flags_.p, cands_.p, sp_);
        timing.launches += 1;
      }
      // scan + (last block) pick; the dynamic scratch is only touched by categorical features
      k_scan<<<sgrid, 256, d.has_categorical ? kScanSmem : 0, s>>>(ctrl, leaves_.p, d.meta.p, H_.p, pool_.p, slot_elems_, flags_.p, cands_.p, sp_);
    }
    nvtxRangePop();
    mark();
    nvtxRangePushA("b200gbm:K7 partition + controller");
    LaunchPartition(pgrid, split == L - 2 ? 1 : 0);
    nvtxRangePop();
    mark();
    timing.launches += fused_ ? 4 : 3; timing.hist_launches += 1;
  }
  if (obj_->IsRenewTreeOutput()) RenewTreeOutput(k, is_rf_ ? rf_init_scores_[k] : 0.0);
  // rf keeps scores as the running average of (tree + init score) over the iterations [LightGBM rf.hpp MultiplyScore / UpdateScore]
  const double bias = is_rf_ ? rf_init_scores_[k] : 0.0, pre = is_rf_ ? static_cast<double>(iter + num_init_iteration) : 1.0;
  const double post = is_rf_ ? 1.0 / (iter + num_init_iteration + 1) : 1.0;
  if (use_bag_ || is_rf_)      // out-of-bag rows are scored by walking the tree on the binned data, so walk it for every row
    k_add_tree_binned<<<egrid, 256, 0, s>>>(tree_dev_, d.meta.p, d.View(), n, score_.p + static_cast<size_t>(k) * n, shrinkage_, bias, pre, post);
  else
    k_add_score<<<egrid, 256, 0, s>>>(ctrl, leaves_.p, tree_dev_, idx0_.p, idx1_.p, score_.p + static_cast<size_t>(k) * n, shrinkage_);
  for (auto* v : valids_)
    k_add_tree_binned<<<egrid, 256, 0, s>>>(tree_dev_, v->ds->meta.p, v->ds->View(), v->ds->num_data,
                                            v->score.p + static_cast<size_t>(k) * v->ds->num_data, shrinkage_, bias, pre, post);
  timing.launches += 2 + static_cast<long long>(valids_.size());
  B200_CUDA(cudaGetLastError());
  B200_CUDA(cudaMemcpyAsync(tree_host_, tree_blob_.p, tree_blob_bytes_, cudaMemcpyDeviceToHost, s));
  B200_CUDA(cudaMemcpyAsync(ctrl_host_, ctrl, sizeof(TreeCtrl), cudaMemcpyDeviceToHost, s));
  B200_CUDA(cudaStreamSynchronize(s));
  if (split_timing && !fused_ && !sev.empty()) {
    static const char* kOps[] = {"gather_q(bagged root)", "K4", "allreduce", "scan+pick", "partition+zeroH+ctl"};
    const int per = 6;       // marks per split
    for (size_t b0 = 0; b0 + per <= sev.size(); b0 += per)
      for (int o = 0; o < per - 1; ++o) { float ms = 0; cudaEventElapsedTime(&ms, sev[b0 + o], sev[b0 + o + 1]); split_op_ms_[kOps[o]] += ms; }
    split_op_trees_ += 1;
    for (auto e : sev) cudaEventDestroy(e);
  }
  if (profile_hist) {
    for (size_t i = 0; i + 1 < evs.size(); i += 2) { float ms = 0; cudaEventElapsedTime(&ms, evs[i], evs[i + 1]); timing.hist_ms += ms; }
    for (auto e : evs) cudaEventDestroy(e);
  }
  timing.hist_rows += ctrl_host_->trace_rows;
  if (fused_ || p2p_allreduce_) {
    int err = 0;
    B200_CUDA(cudaMemcpy(&err, peer_error_.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (err) Fatal("data-parallel training: a peer rank stopped responding (peer-memory barrier timed out)");
  }
  // ---- host copy of the tree
  const unsigned char* hb = tree_host_;
  auto at = [&](const void* devp) { return hb + (static_cast<const unsigned char*>(devp) - tree_blob_.p); };
  const int nl = *reinterpret_cast<const int*>(at(tree_dev_.num_leaves));
  out->Resize(nl);
  if (nl > 1) {
    const int* lc = reinterpret_cast<const int*>(at(tree_dev_.left_child));
    const int* rc = reinterpret_cast<const int*>(at(tree_dev_.right_child));
    const int* sf = reinterpret_cast<const int*>(at(tree_dev_.split_feature_inner));
    const int* tb = reinterpret_cast<const int*>(at(tree_dev_.threshold_bin));
    const int* dt = reinterpret_cast<const int*>(at(tree_dev_.decision_type));
    const float* sg = reinterpret_cast<const float*>(at(tree_dev_.split_gain));
    const double* lv = reinterpret_cast<const double*>(at(tree_dev_.leaf_value));
    const double* lw = reinterpret_cast<const double*>(at(tree_dev_.leaf_weight));
    const int* lcn = reinterpret_cast<const int*>(at(tree_dev_.leaf_count));
    const double* iv = reinterpret_cast<const double*>(at(tree_dev_.internal_value));
    const double* iw = reinterpret_cast<const double*>(at(tree_dev_.internal_weight));
    const int* ic = reinterpret_cast<const int*>(at(tree_dev_.internal_count));
    const int* ld = reinterpret_cast<const int*>(at(tree_dev_.leaf_depth));
    const unsigned* cb = reinterpret_cast<const unsigned*>(at(tree_dev_.cat_bits));
    const unsigned short* cl = reinterpret_cast<const unsigned short*>(at(tree_dev_.cat_list));
    const int* cln = reinterpret_cast<const int*>(at(tree_dev_.cat_list_len));
    for (int i = 0; i < nl - 1; ++i) {
      out->left_child[i] = lc[i]; out->right_child[i] = rc[i]; out->split_feature_inner[i] = sf[i];
      out->split_feature[i] = d.used[sf[i]]; out->threshold_in_bin[i] = static_cast<uint32_t>(tb[i]);
      out->decision_type[i] = static_cast<int8_t>(dt[i]); out->split_gain[i] = sg[i];
      const FeatureBins& fbm = d.mappers[d.used[sf[i]]];
      if (dt[i] & 1) {          // categorical node: bins of the inner bitset -> category values ([UPSTREAM] RealThreshold per bin)
        std::vector<int> cats;
        if (sf[i] >= d.nfn) { for (int k = 0; k < cln[i]; ++k) cats.push_back(fbm.bin_to_cat[cl[i * kCatListMax + k]]); }
        else for (int b = 0; b < fbm.num_bin; ++b) if ((cb[i * 8 + (b >> 5)] >> (b & 31)) & 1u) cats.push_back(fbm.bin_to_cat[b]);
        out->AddCategoricalNode(i, cats);
      } else {
        double thr = fbm.upper[tb[i]];
        if (std::isnan(thr)) thr = 0.0; else if (thr >= 1e300) thr = 1e300; else if (thr <= -1e300) thr = -1e300;
        out->threshold[i] = thr;
      }
      out->internal_value[i] = iv[i]; out->internal_weight[i] = iw[i]; out->internal_count[i] = ic[i];
    }
    for (int i = 0; i < nl; ++i) { out->leaf_value[i] = lv[i]; out->leaf_weight[i] = lw[i]; out->leaf_count[i] = lcn[i]; out->leaf_depth[i] = ld[i]; }
  } else {
    out->leaf_value[0] = 0.0;
  }
}

bool Booster::TrainTrees(const float* custom_g, const float* custom_h) {
  NvtxRange nvtx("b200gbm:iteration (LGBM_BoosterUpdateOneIter)");
  if (!train) Fatal("this booster was loaded from a model string and cannot be trained");
  EnsureDevice();
  cudaStream_t s = stream_;
  const int n = train->num_data;
  B200_CUDA(cudaEventRecord(ev_a_, s));
  std::vector<double> init_scores(K, 0.0);
  const bool const_hessian = obj_->IsConstantHessian() && !is_goss_ && !custom_g;      // GOSS amplifies hessians; custom ones are arbitrary
  if (is_rf_) {
    if (custom_g) Fatal("RF mode do not support custom objective function, please use built-in objectives.");
    init_scores = rf_init_scores_;
  } else if (!custom_g) {
    for (int k = 0; k < K; ++k) init_scores[k] = BoostFromAverage(k);
    if (is_dart_ && !dart_dropped_this_iter_) DroppingTrees();      // GetTrainingScore() in GBDT::Boosting: "only drop one time in one iteration"
    ComputeGradients();
  } else {
    grad_.Upload(custom_g, static_cast<size_t>(K) * n, s);
    hess_.Upload(custom_h, static_cast<size_t>(K) * n, s);
  }
  Bagging(iter);
  bool should_continue = is_rf_;        // a random forest never stops early
  for (int k = 0; k < K; ++k) {
    std::unique_ptr<HostTree> t(new HostTree());
    t->Resize(1);
    t->leaf_value[0] = 0;
    if (obj_->ClassNeedTrain(k) && train->nf > 0) TrainOneTree(k, t.get(), const_hessian);
    if (t->num_leaves > 1) {
      should_continue = true;
      t->Shrink(shrinkage_);
      if (std::fabs(init_scores[k]) > kEps) t->AddBias(init_scores[k]);
    } else if (static_cast<int>(model.trees.size()) < K) {
      double output = obj_->ClassNeedTrain(k) ? init_scores[k] : obj_->BoostFromScore(k);
      t->MakeConstant(output);
      const double pre = is_rf_ ? static_cast<double>(iter + num_init_iteration) : 1.0, post = is_rf_ ? 1.0 / (iter + num_init_iteration + 1) : 1.0;
      k_scale_add<<<num_sms_ * 4, 256, 0, s>>>(score_.p + static_cast<size_t>(k) * n, n, pre, output, post);
      for (auto* v : valids_) k_scale_add<<<num_sms_ * 4, 256, 0, s>>>(v->score.p + static_cast<size_t>(k) * v->ds->num_data, v->ds->num_data, pre, output, post);
    } else {
      t->MakeConstant(0.0);
    }
    model.trees.push_back(std::move(t));
    if (is_dart_) {       // keep the device form of the tree (bin thresholds, inner bitsets) for later drops
      tree_store_.emplace_back(new DevBuf<unsigned char>());
      tree_store_.back()->Alloc(tree_blob_bytes_);
      B200_CUDA(cudaMemcpyAsync(tree_store_.back()->p, tree_blob_.p, tree_blob_bytes_, cudaMemcpyDeviceToDevice, s));
    }
  }
  B200_CUDA(cudaEventRecord(ev_b_, s));
  B200_CUDA(cudaEventSynchronize(ev_b_));
  float ms = 0;
  B200_CUDA(cudaEventElapsedTime(&ms, ev_a_, ev_b_));
  timing.total_ms += ms;
  dart_dropped_this_iter_ = false;
  if (!should_continue) {
    if (static_cast<int>(model.trees.size()) > K) for (int k = 0; k < K; ++k) { model.trees.pop_back(); if (is_dart_) tree_store_.pop_back(); }
    return true;
  }
  ++iter;
  if (is_dart_) {
    DartNormalize();
    if (!cfg.uniform_drop) { tree_weight_.push_back(shrinkage_); sum_weight_ += shrinkage_; }
  }
  return false;
}

bool Booster::UpdateOneIter() { return TrainTrees(nullptr, nullptr); }
bool Booster::UpdateOneIterCustom(const float* grad, const float* hess) { return TrainTrees(grad, hess); }

void Booster::ResetParameter(const char* params) {
  Config nc;
  nc.Parse(params);
  Config next = cfg;
  for (auto& kv : nc.raw) next.raw[kv.first] = kv.second;
  next.Refresh();
  next.num_machines = cfg.num_machines;
  if (train) {      // checked before the change is applied: a refused reset leaves the booster as it was
    CheckMetricLabels(train, next);
    for (auto* v : valids_) CheckMetricLabels(v->ds, next);
  }
  cfg = next;       // in place: the objective keeps a reference to cfg
  shrinkage_ = is_rf_ ? 1.0 : cfg.learning_rate;
  if (is_dart_) { drop_rand_ = LcgRandom(cfg.drop_seed); sum_weight_ = 0.0; }      // [LightGBM dart.hpp DART::ResetConfig]
  sp_.l1 = cfg.lambda_l1; sp_.l2 = cfg.lambda_l2; sp_.max_delta_step = cfg.max_delta_step; sp_.min_gain_to_split = cfg.min_gain_to_split;
  sp_.min_sum_hessian = cfg.min_sum_hessian_in_leaf; sp_.min_data_in_leaf = cfg.min_data_in_leaf; sp_.max_depth = cfg.max_depth;
}

void Booster::AddValidData(const Dataset* valid) {
  EnsureDevice();
  if (!train) Fatal("cannot add validation data to a prediction-only booster");
  if (valid->nf != train->nf) Fatal("validation data must be created with reference=train");
  CheckMetricLabels(valid, cfg);
  ValidSet* v = new ValidSet();
  v->ds = valid;
  v->score.Alloc(static_cast<size_t>(K) * valid->num_data);
  v->score.Zero(stream_);
  if (!valid->init_score.empty() && valid->init_score.size() == static_cast<size_t>(K) * valid->num_data)
    v->score.Upload(valid->init_score.data(), valid->init_score.size(), stream_);
  B200_CUDA(cudaStreamSynchronize(stream_));
  valids_.push_back(v);
}

void Booster::MergeFrom(const Booster* other) {
  // [UPSTREAM GBDT::MergeFrom] other's trees first, then ours; scores are NOT replayed
  std::vector<std::unique_ptr<HostTree>> mine = std::move(model.trees);
  model.trees.clear();
  for (auto& t : other->model.trees) model.trees.emplace_back(new HostTree(*t));
  num_init_iteration = static_cast<int>(model.trees.size()) / std::max(K, 1);
  for (auto& t : mine) model.trees.push_back(std::move(t));
}

std::string Booster::SaveModelToString(int start_iteration, int num_iteration, int importance_type) const {
  std::string pb = train ? cfg.ToString() : std::string();
  return model.ToString(start_iteration, num_iteration, importance_type, pb);
}

std::string Booster::DumpModelJson(int start_iteration, int num_iteration) const {
  std::ostringstream s;
  int t0, t1;
  model.IterRange(start_iteration, num_iteration, &t0, &t1);
  s << "{\"name\":\"tree\",\"version\":\"v3\",\"num_class\":" << model.num_class << ",\"num_tree_per_iteration\":" << model.num_tree_per_iteration
    << ",\"label_index\":" << model.label_index << ",\"max_feature_idx\":" << model.max_feature_idx << ",\"objective\":\"" << model.objective_str
    << "\",\"average_output\":" << (model.average_output ? "true" : "false") << ",\"feature_names\":[";
  for (size_t i = 0; i < model.feature_names.size(); ++i) s << (i ? "," : "") << '"' << model.feature_names[i] << '"';
  s << "],\"tree_info\":[";
  char buf[64];
  auto num = [&](double v) { snprintf(buf, sizeof(buf), "%.17g", v); return std::string(buf); };
  for (int t = t0; t < t1; ++t) {
    const HostTree& tr = *model.trees[t];
    s << (t > t0 ? "," : "") << "{\"tree_index\":" << (t - t0) << ",\"num_leaves\":" << tr.num_leaves << ",\"num_cat\":" << (tr.cat_boundaries.empty() ? 0 : static_cast<int>(tr.cat_boundaries.size()) - 1)
      << ",\"shrinkage\":" << num(tr.shrinkage)
      << ",\"tree_structure\":";
    struct Rec { static void node(std::ostringstream& o, const HostTree& tr, int idx, const std::function<std::string(double)>& num) {
      if (idx >= 0) {
        int mt = (tr.decision_type[idx] >> 2) & 3;
        const bool is_cat = (tr.decision_type[idx] & 1) != 0;
        std::string thr = num(tr.threshold[idx]);
        if (is_cat) {       // [UPSTREAM Tree::NodeToJSON]: the categories that go left, joined by "||"
          const int ci = static_cast<int>(tr.threshold[idx]);
          thr = "\"";
          bool first = true;
          for (int wd = tr.cat_boundaries[ci]; wd < tr.cat_boundaries[ci + 1]; ++wd)
            for (int bit = 0; bit < 32; ++bit)
              if ((tr.cat_threshold[wd] >> bit) & 1u) { thr += (first ? "" : "||") + std::to_string((wd - tr.cat_boundaries[ci]) * 32 + bit); first = false; }
          thr += "\"";
        }
        o << "{\"split_index\":" << idx << ",\"split_feature\":" << tr.split_feature[idx] << ",\"split_gain\":" << num(tr.split_gain[idx])
          << ",\"threshold\":" << thr << ",\"decision_type\":\"" << (is_cat ? "==" : "<=") << "\",\"default_left\":" << ((tr.decision_type[idx] & 2) ? "true" : "false")
          << ",\"missing_type\":\"" << (mt == 0 ? "None" : mt == 1 ? "Zero" : "NaN") << "\",\"internal_value\":" << num(tr.internal_value[idx])
          << ",\"internal_weight\":" << num(tr.internal_weight[idx]) << ",\"internal_count\":" << tr.internal_count[idx] << ",\"left_child\":";
        node(o, tr, tr.left_child[idx], num);
        o << ",\"right_child\":";
        node(o, tr, tr.right_child[idx], num);
        o << "}";
      } else {
        int l = ~idx;
        o << "{\"leaf_index\":" << l << ",\"leaf_value\":" << num(tr.leaf_value[l]) << ",\"leaf_weight\":" << num(tr.leaf_weight[l]) << ",\"leaf_count\":" << tr.leaf_count[l] << "}";
      }
    } };
    if (tr.num_leaves <= 1) s << "{\"leaf_value\":" << num(tr.leaf_value[0]) << "}";
    else Rec::node(s, tr, 0, num);
    s << "}";
  }
  s << "],\"feature_importances\":{";
  std::vector<double> imp = model.FeatureImportance(num_iteration, 0);
  bool first = true;
  for (size_t i = 0; i < imp.size() && i < model.feature_names.size(); ++i)
    if (imp[i] > 0) { s << (first ? "" : ",") << '"' << model.feature_names[i] << "\":" << static_cast<long long>(imp[i]); first = false; }
  s << "}}";
  return s.str();
}

// ---- evaluation (host side: metrics are not on the hot path; scores are read back) -------------
std::vector<std::string> Booster::EvalNames() const {
  std::vector<std::string> names;
  for (auto& m : cfg.metric) {
    if (m == "ndcg" || m == "map") for (int k : cfg.eval_at) names.push_back(m + "@" + std::to_string(k));
    else names.push_back(m);
  }
  return names;
}
int64_t Booster::NumPredict(int data_idx) const {
  if (!train) Fatal("this booster was loaded from a model string: it holds no training/validation data (use the predict entry points)");
  if (data_idx == 0) return static_cast<int64_t>(K) * train->num_data;
  if (data_idx - 1 >= static_cast<int>(valids_.size())) Fatal("data_idx out of range");
  return static_cast<int64_t>(K) * valids_[data_idx - 1]->ds->num_data;
}
void Booster::GetPredict(int data_idx, int64_t* out_len, double* out) {
  if (!train) Fatal("this booster was loaded from a model string: it holds no training/validation data (use the predict entry points)");
  EnsureDevice();
  if (is_dart_ && data_idx == 0 && !dart_dropped_this_iter_) DroppingTrees();      // DART::GetTrainingScore
  const Dataset* ds = data_idx == 0 ? train : valids_.at(data_idx - 1)->ds;
  const DevBuf<double>& sc = data_idx == 0 ? score_ : valids_[data_idx - 1]->score;
  const int n = ds->num_data;
  std::vector<double> raw(static_cast<size_t>(K) * n);
  sc.Download(raw.data(), raw.size(), stream_);
  B200_CUDA(cudaStreamSynchronize(stream_));
  std::vector<double> r(K), o(K);
  for (int i = 0; i < n; ++i) {
    for (int k = 0; k < K; ++k) r[k] = raw[static_cast<size_t>(k) * n + i];
    model.Convert(r.data(), o.data());
    for (int k = 0; k < K; ++k) out[static_cast<size_t>(k) * n + i] = o[k];
  }
  *out_len = static_cast<int64_t>(K) * n;
}

// ---- evaluation on the device (metric_kernels.cuh): only the reduced sums cross PCIe
static int MetricKindOf(const std::string& m) {
  static const std::map<std::string, int> kinds = {
      {"l2", kMetL2}, {"rmse", kMetL2}, {"l1", kMetL1}, {"huber", kMetHuber}, {"fair", kMetFair}, {"poisson", kMetPoisson}, {"gamma", kMetGamma},
      {"gamma_deviance", kMetGammaDeviance}, {"tweedie", kMetTweedie}, {"quantile", kMetQuantile}, {"mape", kMetMape},
      {"binary_logloss", kMetBinLogloss}, {"binary_error", kMetBinError}, {"multi_logloss", kMetMultiLogloss}, {"multi_error", kMetMultiError},
      {"cross_entropy", kMetXent}};
  auto it = kinds.find(m);
  return it == kinds.end() ? -1 : it->second;
}
// [LightGBM NDCGMetric::Init -> DCGCalculator::CheckLabel]: k_metric_rank indexes label_gain with the labels of every evaluated set
void Booster::CheckMetricLabels(const Dataset* ds, const Config& c) const {
  if (std::find(c.metric.begin(), c.metric.end(), "ndcg") != c.metric.end()) CheckRankLabels(ds->label, RankLabelGain(c).size());
}
void Booster::ValidateMetrics() const {
  for (auto& m : cfg.metric)
    if (MetricKindOf(m) < 0 && m != "auc" && m != "ndcg" && m != "map") Fatal("Unknown metric type name: " + m);
  if (cfg.eval_at.size() > static_cast<size_t>(kMaxEvalAt)) Fatal("eval_at: at most " + std::to_string(kMaxEvalAt) + " positions are supported");
}

std::vector<double> Booster::GetEval(int data_idx) {
  NvtxRange nvtx("b200gbm:eval metrics (LGBM_BoosterGetEval)");
  if (!train) Fatal("this booster was loaded from a model string: it holds no training/validation data to evaluate");
  EnsureDevice();
  if (is_dart_ && data_idx == 0 && !dart_dropped_this_iter_) DroppingTrees();      // DART::GetTrainingScore
  const Dataset* ds = data_idx == 0 ? train : valids_.at(data_idx - 1)->ds;
  const DevBuf<double>& sc = data_idx == 0 ? score_ : valids_[data_idx - 1]->score;
  const int n = ds->num_data;
  cudaStream_t s = stream_;
  if (ds->label.empty()) Fatal("label should not be empty for evaluation");
  const float* d_y = ds->d_label.p;
  const float* d_w = ds->weight.empty() ? nullptr : ds->d_weight.p;
  const int grid = std::max(1, std::min((n + kMetricBlock - 1) / kMetricBlock, num_sms_ * 8));
  if (met_partial_.n < static_cast<size_t>(grid) * 2 * kMaxEvalAt) met_partial_.Alloc(static_cast<size_t>(grid) * 2 * kMaxEvalAt);
  if (met_out_.n < 2 * kMaxEvalAt) met_out_.Alloc(2 * kMaxEvalAt);
  std::vector<double> out;
  auto avg = [&](double loss, double sw) {
    double v[2] = {loss, sw};
    AllReduceHost(v, 2, ncclSum, s);     // averaged metrics are global in distributed mode (B.5)
    return v[0] / v[1];
  };
  auto fetch = [&](int count, double* host) {
    met_out_.Download(host, count, s);
    B200_CUDA(cudaStreamSynchronize(s));
  };
  bool rank_done = false;
  std::vector<double> ndcg_vals, map_vals;
  for (auto& m : cfg.metric) {
    const int kind = MetricKindOf(m);
    if (kind >= 0) {
      MetricParams mp{kind, K, obj_->IsOva() ? 1 : 0, 0, cfg.alpha, cfg.fair_c, cfg.tweedie_variance_power, cfg.sigmoid};
      if ((kind == kMetMultiLogloss || kind == kMetMultiError) && K < 2) Fatal("metric " + m + " needs a multiclass objective");
      k_metric_pointwise<<<grid, kMetricBlock, 0, s>>>(sc.p, d_y, d_w, n, mp, met_partial_.p);
      k_metric_finish<<<1, 32, 0, s>>>(met_partial_.p, grid, 2, met_out_.p);
      B200_CUDA(cudaGetLastError());
      double v[2];
      fetch(2, v);
      const double a = avg(v[0], v[1]);
      out.push_back(m == "rmse" ? std::sqrt(a) : a);
    } else if (m == "auc") {
      // [UPSTREAM AUCMetric::Eval] is rank-local (no network sync), like the reference's per-task evaluation
      if (auc_keys_a_.n < static_cast<size_t>(n)) {
        auc_keys_a_.Alloc(n); auc_keys_b_.Alloc(n); auc_rows_a_.Alloc(n); auc_rows_b_.Alloc(n); auc_wpos_.Alloc(n); auc_wneg_.Alloc(n);
        auc_ppos_.Alloc(n); auc_pneg_.Alloc(n); auc_head_.Alloc(n); auc_start_.Alloc(n);
        size_t t1 = 0, t2 = 0, t3 = 0;
        cub::DeviceRadixSort::SortPairsDescending(nullptr, t1, auc_keys_a_.p, auc_keys_b_.p, auc_rows_a_.p, auc_rows_b_.p, n, 0, 64, s);
        cub::DeviceScan::InclusiveSum(nullptr, t2, auc_wpos_.p, auc_ppos_.p, n, s);
        cub::DeviceScan::InclusiveScan(nullptr, t3, auc_head_.p, auc_start_.p, cub::Max(), n, s);
        auc_tmp_.Alloc(std::max(t1, std::max(t2, t3)) + 16);
      }
      size_t tb = auc_tmp_.n;
      const int eg = num_sms_ * 8;
      k_auc_keys<<<eg, 256, 0, s>>>(sc.p, n, auc_keys_a_.p, auc_rows_a_.p);
      B200_CUDA(cub::DeviceRadixSort::SortPairsDescending(auc_tmp_.p, tb, auc_keys_a_.p, auc_keys_b_.p, auc_rows_a_.p, auc_rows_b_.p, n, 0, 64, s));
      k_auc_weights<<<eg, 256, 0, s>>>(auc_keys_b_.p, auc_rows_b_.p, d_y, d_w, n, auc_wpos_.p, auc_wneg_.p, auc_head_.p);
      tb = auc_tmp_.n; B200_CUDA(cub::DeviceScan::InclusiveSum(auc_tmp_.p, tb, auc_wpos_.p, auc_ppos_.p, n, s));
      tb = auc_tmp_.n; B200_CUDA(cub::DeviceScan::InclusiveSum(auc_tmp_.p, tb, auc_wneg_.p, auc_pneg_.p, n, s));
      tb = auc_tmp_.n; B200_CUDA(cub::DeviceScan::InclusiveScan(auc_tmp_.p, tb, auc_head_.p, auc_start_.p, cub::Max(), n, s));
      k_auc_terms<<<grid, kMetricBlock, 0, s>>>(auc_keys_b_.p, auc_start_.p, auc_ppos_.p, auc_pneg_.p, n, met_partial_.p);
      k_metric_finish<<<1, 32, 0, s>>>(met_partial_.p, grid, 2, met_out_.p);
      B200_CUDA(cudaGetLastError());
      double v[2], tot[2];
      fetch(2, v);
      B200_CUDA(cudaMemcpyAsync(&tot[0], auc_ppos_.p + (n - 1), sizeof(double), cudaMemcpyDeviceToHost, s));
      B200_CUDA(cudaMemcpyAsync(&tot[1], auc_pneg_.p + (n - 1), sizeof(double), cudaMemcpyDeviceToHost, s));
      B200_CUDA(cudaStreamSynchronize(s));
      out.push_back((tot[0] > 0 && tot[1] > 0) ? v[0] / (tot[0] * tot[1]) : 1.0);
    } else if (m == "ndcg" || m == "map") {
      if (!rank_done) {
        const int nq = static_cast<int>(ds->query_boundaries.size()) - 1;
        if (nq <= 0) Fatal("The " + std::string(m == "ndcg" ? "NDCG" : "MAP") + " metric requires query information");
        const std::vector<double> lg = RankLabelGain(cfg);
        int max_q = 1;
        for (int q = 0; q < nq; ++q) max_q = std::max(max_q, ds->query_boundaries[q + 1] - ds->query_boundaries[q]);
        std::vector<double> disc(static_cast<size_t>(max_q) + 1);
        for (size_t i = 0; i < disc.size(); ++i) disc[i] = 1.0 / std::log2(2.0 + i);
        DevBuf<double> d_lg, d_disc;
        d_lg.Alloc(lg.size()); d_lg.Upload(lg.data(), lg.size(), s);
        d_disc.Alloc(disc.size()); d_disc.Upload(disc.data(), disc.size(), s);
        RankEvalParams rp{};
        std::vector<int> ks = cfg.eval_at;      // evaluated in ascending order ([UPSTREAM] Config sorts eval_at); reported in the given order
        std::sort(ks.begin(), ks.end());
        rp.nk = static_cast<int>(ks.size());
        for (int e = 0; e < rp.nk; ++e) rp.ks[e] = ks[e];
        rp.want_ndcg = std::find(cfg.metric.begin(), cfg.metric.end(), "ndcg") != cfg.metric.end();
        rp.want_map = std::find(cfg.metric.begin(), cfg.metric.end(), "map") != cfg.metric.end();
        const size_t smem = RankMetricSmem(max_q, static_cast<int>(lg.size()));
        if (smem > 200 * 1024) Fatal("a query group is too large for the ranking metric kernel");
        B200_CUDA(cudaFuncSetAttribute(k_metric_rank, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(std::max<size_t>(smem, 1024))));
        const int rgrid = std::max(1, std::min(nq, num_sms_ * 8));
        if (met_partial_.n < static_cast<size_t>(rgrid) * 2 * kMaxEvalAt) met_partial_.Alloc(static_cast<size_t>(rgrid) * 2 * kMaxEvalAt);
        k_metric_rank<<<rgrid, 128, std::max<size_t>(smem, 1024), s>>>(sc.p, d_y, ds->d_qb.p, nq, d_lg.p, static_cast<int>(lg.size()), d_disc.p, rp, max_q, met_partial_.p);
        k_metric_finish<<<1, 32, 0, s>>>(met_partial_.p, rgrid, 2 * kMaxEvalAt, met_out_.p);
        B200_CUDA(cudaGetLastError());
        double v[2 * kMaxEvalAt];
        fetch(2 * kMaxEvalAt, v);
        for (size_t e = 0; e < cfg.eval_at.size(); ++e) {
          const size_t pos = std::find(ks.begin(), ks.end(), cfg.eval_at[e]) - ks.begin();
          ndcg_vals.push_back(avg(v[pos], nq));
          map_vals.push_back(avg(v[kMaxEvalAt + pos], nq));
        }
        rank_done = true;
      }
      const std::vector<double>& vals = m == "ndcg" ? ndcg_vals : map_vals;
      out.insert(out.end(), vals.begin(), vals.end());
    } else {
      Fatal("Unknown metric type name: " + m);
    }
  }
  return out;
}

// Gradients and hessians of the objective at the current training scores, into scratch buffers: grad_ / hess_ (which random
// forest reuses across iterations) and the timing counters are left alone, so calling this changes nothing the training sees
void Booster::GetGradients(float* out_g, float* out_h) {
  if (!train || !obj_) Fatal("this booster was loaded from a model string: it has no objective to take gradients of");
  EnsureDevice();
  const size_t len = static_cast<size_t>(K) * train->num_data;
  DevBuf<float> g, h;
  g.Alloc(len); h.Alloc(len);
  g.Zero(stream_); h.Zero(stream_);      // classes the objective skips stay 0
  obj_->GetGradients(score_.p, g.p, h.p);
  B200_CUDA(cudaGetLastError());
  g.Download(out_g, len, stream_); h.Download(out_h, len, stream_);
  B200_CUDA(cudaStreamSynchronize(stream_));
}

void Booster::GetRawScores(int data_idx, double* out) {
  if (!train) Fatal("this booster was loaded from a model string: it holds no training/validation data");
  EnsureDevice();
  const Dataset* ds = data_idx == 0 ? train : valids_.at(data_idx - 1)->ds;
  const DevBuf<double>& sc = data_idx == 0 ? score_ : valids_[data_idx - 1]->score;
  sc.Download(out, static_cast<size_t>(K) * ds->num_data, stream_);
  B200_CUDA(cudaStreamSynchronize(stream_));
}

void Booster::UploadForest() {
  if (forest_ && forest_->trees == model.trees.size()) return;
  forest_.reset(new ForestBufs());
  ForestBufs& f = *forest_;
  const size_t T = model.trees.size();
  std::vector<int> toff(T + 1, 0), loff(T + 1, 0), nl(T), sf, dt, lc, rc, cbeg, clen;
  std::vector<unsigned> cwords;
  std::vector<double> thr, lv, ncnt, lcnt, expv(T, 0.0);
  for (size_t t = 0; t < T; ++t) {
    const HostTree& tr = *model.trees[t];
    nl[t] = tr.num_leaves;
    expv[t] = tr.ExpectedValue();
    if (tr.num_leaves > 1) f.max_depth = std::max(f.max_depth, tr.MaxDepth());
    toff[t + 1] = toff[t] + std::max(tr.num_leaves - 1, 0);
    loff[t + 1] = loff[t] + tr.num_leaves;
    for (int i = 0; i < tr.num_leaves - 1; ++i) {
      sf.push_back(tr.split_feature[i]); dt.push_back(tr.decision_type[i]); lc.push_back(tr.left_child[i]); rc.push_back(tr.right_child[i]);
      thr.push_back(tr.threshold[i]); ncnt.push_back(tr.internal_count[i]);
      if (tr.decision_type[i] & 1) {
        const int ci = static_cast<int>(tr.threshold[i]);
        cbeg.push_back(static_cast<int>(cwords.size())); clen.push_back(tr.cat_boundaries[ci + 1] - tr.cat_boundaries[ci]);
        for (int w = tr.cat_boundaries[ci]; w < tr.cat_boundaries[ci + 1]; ++w) cwords.push_back(tr.cat_threshold[w]);
      } else { cbeg.push_back(0); clen.push_back(0); }
    }
    for (int i = 0; i < tr.num_leaves; ++i) { lv.push_back(tr.leaf_value[i]); lcnt.push_back(tr.leaf_count[i]); }
  }
  if (!stream_) B200_CUDA(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  auto up_i = [&](DevBuf<int>& d, std::vector<int>& h) { d.Alloc(std::max<size_t>(h.size(), 1)); if (!h.empty()) d.Upload(h.data(), h.size(), stream_); };
  auto up_d = [&](DevBuf<double>& d, std::vector<double>& h) { d.Alloc(std::max<size_t>(h.size(), 1)); if (!h.empty()) d.Upload(h.data(), h.size(), stream_); };
  up_i(f.tree_offset, toff); up_i(f.leaf_offset, loff); up_i(f.num_leaves, nl); up_i(f.split_feature, sf); up_i(f.decision_type, dt);
  up_i(f.left_child, lc); up_i(f.right_child, rc); up_d(f.threshold, thr); up_d(f.leaf_value, lv); up_i(f.cat_begin, cbeg); up_i(f.cat_len, clen);
  up_d(f.node_count, ncnt); up_d(f.leaf_count, lcnt); up_d(f.expected, expv);
  f.cat_words.Alloc(std::max<size_t>(cwords.size(), 1));
  if (!cwords.empty()) f.cat_words.Upload(cwords.data(), cwords.size(), stream_);
  B200_CUDA(cudaStreamSynchronize(stream_));
  f.trees = T;
}

int64_t Booster::PredictBatch(const void* data, int data_type, int64_t nrow, int ncol, int predict_type, int start_iteration, int num_iteration,
                              double* out) {
  EnsureDevice();
  if (data_type != 0 && data_type != 1) Fatal("PredictBatch: unknown data type");
  if (predict_type < 0 || predict_type > 3) Fatal("PredictBatch: unknown predict type");
  if (ncol < model.max_feature_idx + 1) Fatal("PredictBatch: the matrix has fewer columns than the model has features");
  UploadForest();
  const ForestBufs& fb = *forest_;
  ForestDev f{fb.tree_offset.p, fb.leaf_offset.p, fb.num_leaves.p, fb.split_feature.p, fb.threshold.p, fb.decision_type.p, fb.left_child.p, fb.right_child.p, fb.leaf_value.p,
              fb.cat_begin.p, fb.cat_len.p, fb.cat_words.p, fb.node_count.p, fb.leaf_count.p, fb.expected.p};
  int t0, t1;
  model.IterRange(start_iteration, num_iteration, &t0, &t1);
  const int Kc = model.num_tree_per_iteration;
  const int F1 = model.max_feature_idx + 2;            // contributions: one per feature + the expected value
  const int64_t per_row = predict_type == 2 ? (t1 - t0) : predict_type == 3 ? static_cast<int64_t>(Kc) * F1 : Kc;
  const size_t esz = data_type == 0 ? 4 : 8;
  const bool on_device = IsDevicePointer(data);
  int64_t chunk = on_device ? nrow : std::max<int64_t>(1, std::min<int64_t>(nrow, (512LL << 20) / (static_cast<int64_t>(ncol) * esz)));
  chunk = std::max<int64_t>(1, std::min<int64_t>(chunk, (1024LL << 20) / (per_row * 8)));      // bound the device output buffer too (contributions are wide)
  // TreeSHAP scratch: per thread (depth+2)(depth+3)/2 path elements + depth+3 stack frames (kernels.cuh k_predict_contrib)
  const int shap_threads = 128;
  int shap_grid = 0, path_stride = 0, frame_stride = 0;
  DevBuf<ShapPathElem> shap_paths;
  DevBuf<ShapFrame> shap_frames;
  if (predict_type == 3) {
    const int md = fb.max_depth + 2;
    path_stride = md * (md + 1) / 2 + md;
    frame_stride = md + 2;
    shap_grid = static_cast<int>(std::min<int64_t>((std::min(chunk, nrow) + shap_threads - 1) / shap_threads, static_cast<int64_t>(num_sms_ > 0 ? num_sms_ : 148) * 4));
    shap_paths.Alloc(static_cast<size_t>(shap_grid) * shap_threads * path_stride);
    shap_frames.Alloc(static_cast<size_t>(shap_grid) * shap_threads * frame_stride);
  }
  DevBuf<unsigned char> xin;
  if (!on_device) xin.Alloc(static_cast<size_t>(chunk) * ncol * esz);
  DevBuf<double> dout; dout.Alloc(static_cast<size_t>(std::min(chunk, nrow)) * per_row);
  cudaEvent_t e0, e1;
  B200_CUDA(cudaEventCreate(&e0)); B200_CUDA(cudaEventCreate(&e1));
  B200_CUDA(cudaEventRecord(e0, stream_));
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, CurrentDevice());
  for (int64_t r0 = 0; r0 < nrow; r0 += chunk) {
    const int64_t rows = std::min(chunk, nrow - r0);
    const void* x = static_cast<const unsigned char*>(data) + static_cast<size_t>(r0) * ncol * esz;
    if (!on_device) { B200_CUDA(cudaMemcpyAsync(xin.p, x, static_cast<size_t>(rows) * ncol * esz, cudaMemcpyHostToDevice, stream_)); x = xin.p; }
    const int grid = static_cast<int>(std::min<int64_t>((rows * per_row + 255) / 256, static_cast<int64_t>(sms) * 16));
    if (predict_type == 3) {
      B200_CUDA(cudaMemsetAsync(dout.p, 0, static_cast<size_t>(rows) * per_row * sizeof(double), stream_));
      if (data_type == 0) k_predict_contrib<float><<<shap_grid, shap_threads, 0, stream_>>>(f, static_cast<const float*>(x), rows, ncol, Kc, t0, t1, F1, shap_paths.p, path_stride, shap_frames.p, frame_stride, dout.p);
      else k_predict_contrib<double><<<shap_grid, shap_threads, 0, stream_>>>(f, static_cast<const double*>(x), rows, ncol, Kc, t0, t1, F1, shap_paths.p, path_stride, shap_frames.p, frame_stride, dout.p);
    } else if (predict_type == 2) {
      if (data_type == 0) k_predict_leaf<float><<<grid, 256, 0, stream_>>>(f, static_cast<const float*>(x), rows, ncol, t0, t1, dout.p);
      else k_predict_leaf<double><<<grid, 256, 0, stream_>>>(f, static_cast<const double*>(x), rows, ncol, t0, t1, dout.p);
    } else {
      if (data_type == 0) k_predict_raw<float><<<grid, 256, 0, stream_>>>(f, static_cast<const float*>(x), rows, ncol, Kc, t0, t1, dout.p);
      else k_predict_raw<double><<<grid, 256, 0, stream_>>>(f, static_cast<const double*>(x), rows, ncol, Kc, t0, t1, dout.p);
    }
    B200_CUDA(cudaGetLastError());
    B200_CUDA(cudaMemcpyAsync(out + r0 * per_row, dout.p, static_cast<size_t>(rows) * per_row * sizeof(double), cudaMemcpyDeviceToHost, stream_));
    B200_CUDA(cudaStreamSynchronize(stream_));
  }
  B200_CUDA(cudaEventRecord(e1, stream_));
  B200_CUDA(cudaEventSynchronize(e1));
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  last_predict_ms = ms;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  const bool avg = model.average_output && t1 > t0 && predict_type < 2;       // rf: raw score = mean over the iterations
  if (avg && predict_type == 1)
    for (int64_t i = 0; i < nrow * Kc; ++i) out[i] /= ((t1 - t0) / Kc);
  if (predict_type == 0) {          // objective transform on the host, identical to the single-row predictor
    std::vector<double> r(Kc), o(Kc);
    for (int64_t i = 0; i < nrow; ++i) {
      double* p = out + i * Kc;
      if (avg) for (int k = 0; k < Kc; ++k) p[k] /= ((t1 - t0) / Kc);
      for (int k = 0; k < Kc; ++k) r[k] = p[k];
      model.Convert(r.data(), o.data());
      for (int k = 0; k < Kc; ++k) p[k] = o[k];
    }
  }
  return nrow * per_row;
}

}  // namespace b200gbm
