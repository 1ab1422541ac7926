// ksched.cu — sm_100a kernels and the C-ABI of include/ksched.h.
//
//  K0  sort_keys / gather_rows   FFD order of the queue (queue.go:35-110) and the dense, FFD-ordered
//                                P x 256 B pod-row matrix the feasibility kernel streams.
//  K1  class_feasibility_kernel + feasibility_kernel: dense pods x (template, instance type) bitmask F, bit-sliced over columns:
//                                Requirements.Compatible/Intersects (requirements.go:123-206), fits /
//                                hasOffering (node.go:143-159), Taints.Tolerates (taints.go:28) as AND/OR of
//                                precomputed column bitsets; warp ballot/ffs gives the per-pod best column.
//  K2  pack_kernel               the sequential first-fit of Scheduler.add (scheduler.go:174-219) with
//                                Node.Add / ExistingNode.Add (node.go:62-107, existingnode.go:77-130),
//                                topology domains (topology.go:120-167, topologygroup.go:88-243), queue
//                                requeue / relaxation (scheduler.go:104-124, queue.go:44-68) in ONE persistent
//                                CTA: candidate nodes are examined in parallel, the reference's scan order is
//                                recovered with a block-wide argmin on (pod count, stable tie-break).
// Integer / bitmask work only — no tensor cores by design (BASELINE.json north_star).
#include <cuda_runtime.h>
#include <nccl.h>
#include <stdint.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cub/cub.cuh>
#include <string>
#include <mutex>
#include <vector>

#include "ksched.h"
#include "reqmask.cuh"
#include "launch.cuh"

using ksched::KeyMeta;
using ksched::Req;

#define CUDA_TRY(h, expr)                                                                         \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) {                                                                      \
      (h)->err = std::string(#expr) + ": " + cudaGetErrorString(_e);                              \
      return KSCHED_ERR_CUDA;                                                                     \
    }                                                                                             \
  } while (0)

namespace {

constexpr int kMaxCG = 8;        // topology groups that may constrain one pod class
constexpr int kMaxTouched = 8;   // requirement keys one Add may touch (pod keys + topology keys)
constexpr int kPackThreads = 512;
constexpr int kFreshMemoSlots = 8192;  // PackState::fd_*
constexpr uint64_t kNoBest = ~0ull;

#include "catalog.cuh"
#include "feasibility_kernel.cuh"
#include "topology.cuh"

}  // namespace

#include "pack_kernel.cuh"
#include "cluster.cuh"

namespace {

// Launch choice per finished new node (launch.cuh): one warp per node, lanes over the words of its final option set.
__global__ void launch_choice_kernel(DevCatalog c, const long long* counters, const uint64_t* nn_vals, const uint64_t* nn_meta,
                                     const uint32_t* nn_opts, int max_new, ksched_launch_choice* out) {
  const int n_new = (int)counters[0];
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int n = warp; n < n_new; n += nwarps) {
    // zones / capacity types the node's requirements admit (Offerings.Requirements, types.go:120-126)
    uint32_t zmask = 0xFFFF, cmask = 0xF;
    const uint64_t meta = nn_meta[n];
    if (c.zone_key >= 0) {
      const Req z = load_soa(nn_vals, meta, max_new, n, c.zone_key);
      if (z.present) zmask = (uint32_t)ksched::req_allowed(z, c.keys[c.zone_key].dict_mask, key_meta(c, c.zone_key));
    }
    if (c.ct_key >= 0) {
      const Req ct = load_soa(nn_vals, meta, max_new, n, c.ct_key);
      if (ct.present) cmask = (uint32_t)ksched::req_allowed(ct, c.keys[c.ct_key].dict_mask, key_meta(c, c.ct_key));
    }
    unsigned long long best = ~0ull, best_off = ksched::kNoOffering;
    int best_col = -1;
    for (int w = lane; w < c.W32; w += 32) {
      uint32_t m = nn_opts[(size_t)w * max_new + n];
      while (m) {
        const int t = w * 32 + __ffs(m) - 1;
        m &= m - 1;
        const uint64_t ok = ksched::offering_min_key(c.offer_keys + (size_t)t * 64, zmask, cmask);
        if (ok == ksched::kNoOffering) continue;
        const unsigned long long key = ksched::option_key(ok, c.input_index[t]);
        if (key < best) { best = key; best_off = ok; best_col = t; }
      }
    }
    const unsigned long long wbest = warp_min_u64(best);
    const unsigned owner = __ballot_sync(0xffffffffu, best == wbest && best != ~0ull);  // keys are unique per option
    if (owner) {
      const int src = __ffs(owner) - 1;
      best_col = __shfl_sync(0xffffffffu, best_col, src);
      best_off = __shfl_sync(0xffffffffu, best_off, src);
    } else {
      best_col = -1;
    }
    if (lane == 0) {
      ksched_launch_choice o;
      o.type_column = best_col;
      o.offering_slot = best_col >= 0 ? (int32_t)(best_off & 0xFF) : -1;
      o.price_rank = best_col >= 0 ? (uint32_t)(best_off >> 16) : 0;
      o.offering_index = best_col >= 0 ? (uint32_t)((best_off >> 8) & 0xFF) : 0;
      out[n] = o;
    }
  }
}

// L2 flush helper: write a buffer larger than L2 between timed iterations
__global__ void flush_kernel(uint32_t* buf, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) buf[i] = (uint32_t)i;
}

template <class T>
struct DevBuf {
  T* ptr = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t n) {
    if (n <= cap && ptr) return cudaSuccess;
    if (ptr) cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    size_t want = n ? n : 1;
    cudaError_t e = cudaMalloc(&ptr, want * sizeof(T));
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() { if (ptr) cudaFree(ptr); ptr = nullptr; cap = 0; }
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
};

}  // namespace

struct ksched_handle {
  K1Params k1_host;  // staging copies of the kernels' constant-memory parameters (must outlive the async copies)
  K2Params k2_host;  // staging copy of the pack kernel's constant-memory parameters (must outlive the async copy)
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  // catalog
  bool have_catalog = false;
  DevCatalog cat{};
  int W64 = 0;
  DevBuf<ksched_keyinfo> d_keys;
  DevBuf<int64_t> d_key_int, d_capacity, d_alloc_sorted;
  DevBuf<ksched_key_regions> d_key_regions;
  DevBuf<ksched_class_volumes> d_cls_vol;
  DevBuf<int32_t> d_cls_cursor;
  // device-resident cluster snapshot (ksched_load_cluster)
  bool have_cluster = false;
  int stop_new_nodes = 0;
  int sup_pods = 0, sup_pending = 0;
  std::vector<int32_t> h_node_first, h_node_count;   // per existing slot: first superset pod bound to it, how many
  DevBuf<int32_t> d_sup_pod_node, d_node_first, d_node_dst, d_set_nodes, d_pod_src;
  DevBuf<uint32_t> d_sup_class, d_sup_uid, d_sim_types;
  DevBuf<int64_t> d_sup_ts, d_sim_remaining;
  DevBuf<uint8_t> d_in_set;
  DevBuf<SimResultDev> d_sim_results;
  bool cluster_topology = false;
  int filt_words = 0;
  DevBuf<uint32_t> d_cc_begin, d_filt;
  DevBuf<ksched_count_rel> d_cc;
  DevBuf<int8_t> d_node_dom;
  DevBuf<uint8_t> d_node_hostlabel;
  DevBuf<uint8_t> d_gather_send, d_gather_recv;
  DevBuf<int32_t> d_rk_off, d_rk_prio, d_rk_order, d_rk_n;
  DevBuf<double> d_rk_dc, d_rk_age, d_rk_ttl, d_rk_cost_in, d_rk_cost, d_rk_cost_out;
  DevBuf<uint8_t> d_rk_flags, d_rk_elig_in, d_rk_elig;
  DevBuf<ksched_node_volumes> d_ex_vol, d_ex_vol0;
  bool have_volumes = false;
  uint64_t vol_mask[KSCHED_MAX_VOLUME_DRIVERS] = {};
  DevBuf<ksched_template> d_templates;
  DevBuf<ksched_type_row> d_types;
  DevBuf<float> d_price32;
  DevBuf<int16_t> d_valrow, d_offrow;
  DevBuf<uint32_t> d_valset, d_absent, d_negempty, d_offset, d_anyoffer, d_member, d_fitset, d_domset, d_input_index;
  DevBuf<uint64_t> d_offer_keys;
  DevBuf<ksched_launch_choice> d_launch;
  std::vector<ksched_template> h_templates;
  std::vector<unsigned char> catalog_blob;  // host copy of the resident catalog's inputs (ksched_load_catalog early-out)
  int n_valrows = 1, n_offrows = 1;
  // problem
  bool uploaded = false;
  bool sorted = false;  // the FFD-ordered pod-row matrix of the uploaded problem exists
  int n_pods = 0, n_classes = 0, n_existing = 0, n_groups = 0, max_new = 0, n_hostgroups = 0;
  DevBuf<ksched_pod_row> d_classes;
  DevBuf<uint32_t> d_pod_pos, d_pod_class0, d_pod_class, d_uid_rank, d_order, d_idx_tmp, d_itype_sets, d_queue, d_last_epoch;
  DevBuf<int64_t> d_ts;
  DevBuf<uint64_t> d_k_cpu, d_k_mem, d_k_tie, d_k_tmp, d_rows;
  DevBuf<uint8_t> d_cub_tmp, d_itype_comp, d_ex_closed, d_nn_tmpl;
  DevBuf<ksched_topo_group> d_groups;
  DevBuf<ksched_class_topo> d_class_topo;
  DevBuf<RelX> d_relx;
  DevBuf<ksched_reqset> d_filter_terms;
  DevBuf<int32_t> d_hostname_reqs, d_relax, d_assign, d_place_seq, d_last_len, d_nn_count, d_nn_tb, d_ov_node, d_perm_desc, d_grp_cnt,
      d_grp_cnt0, d_grp_host_row, d_grp_host_total, d_grp_host_total0;
  DevBuf<uint32_t> d_F, d_Fclass;
  DevBuf<unsigned long long> d_best_class;
  DevBuf<unsigned long long> d_best;
  DevBuf<int64_t> d_ex_req, d_ex_req0, d_ex_avail, d_nn_req, d_remaining, d_alloc_rt;
  DevBuf<long long> d_ov_q, d_ov_bound, d_ov_bound2, d_fc_bound, d_fc_bound2;
  DevBuf<unsigned long long> d_ov_key;
  DevBuf<unsigned short> d_ov_flags;
  DevBuf<uint8_t> d_fc_state, d_fc_dom, d_fc_front_state, d_grp_active, d_grp_active0;
  DevBuf<int32_t> d_grp_min_slot;
  DevBuf<uint32_t> d_fc_opts, d_fc_qp, d_ov_absorbed, d_ov_rejected;
  DevBuf<uint64_t> d_fc_vals, d_fc_meta;
  DevBuf<long long> d_fc_q;
  DevBuf<uint8_t> d_fd_state, d_fd_dom;
  DevBuf<uint32_t> d_fd_fc, d_fd_opts;
  DevBuf<uint64_t> d_fd_meta, d_fd_vals;
  DevBuf<long long> d_fd_bound, d_fd_bound2;
  int count_visited = 1;
  DevBuf<uint32_t> d_ex_req_present, d_ex_req_present0, d_ex_avail_present, d_ex_taintset, d_ex_itype, d_nn_req_present, d_nn_opts;
  DevBuf<uint64_t> d_ex_vals, d_ex_vals0, d_ex_meta, d_ex_meta0, d_ex_hp, d_ex_hp0, d_nn_vals, d_nn_meta, d_nn_hp, d_grp_registered,
      d_grp_registered0;
  DevBuf<uint16_t> d_grp_host, d_grp_host0;
  DevBuf<long long> d_counters, d_k1dbg;
  DevBuf<uint32_t> d_flush;
  size_t cub_tmp_bytes = 0;
  // one-pass queue order (feasibility_kernel.cuh: sort_key1_kernel): total key bits, 0 = the three-key path
  int sort1_bits = 0, sort1_ts_bits = 0, sort1_uid_bits = 0;
  long long sort1_ts_min = 0;
  DevBuf<uint32_t> d_cls_rank;
  int64_t min_req[KSCHED_MAX_RES] = {0};
  // sharding / nccl
  int rank = 0, world = 1;
  ncclComm_t comm = nullptr;
  // timings
  ksched_timings tm{};
  cudaEvent_t ev[8] = {nullptr};
};

template <class T>
static cudaError_t upload(ksched_handle* h, DevBuf<T>& buf, const T* src, size_t n) {
  cudaError_t e = buf.ensure(n);
  if (e != cudaSuccess) return e;
  if (n == 0) return cudaSuccess;
  h->tm.h2d_bytes += (int64_t)(n * sizeof(T));
  return cudaMemcpyAsync(buf.ptr, src, n * sizeof(T), cudaMemcpyHostToDevice, h->stream);
}
template <class T>
static cudaError_t upload_vec(ksched_handle* h, DevBuf<T>& buf, const std::vector<T>& v) { return upload(h, buf, v.data(), v.size()); }

static int type_words64(int n_types) { int w = (n_types + 63) / 64; return w ? w : 1; }

extern "C" {

int ksched_abi_version(void) { return KSCHED_ABI_VERSION; }
int ksched_type_words(int n_types) { return type_words64(n_types); }

int ksched_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) return KSCHED_ERR_NO_DEVICE;
  return n;
}

int ksched_create(int device_ordinal, ksched_handle** out) {
  if (!out) return KSCHED_ERR_INVALID;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0 || device_ordinal >= n) return KSCHED_ERR_NO_DEVICE;
  ksched_handle* h = new ksched_handle();
  h->device = device_ordinal;
  if (cudaSetDevice(device_ordinal) != cudaSuccess || cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
    delete h;
    return KSCHED_ERR_CUDA;
  }
  for (auto& e : h->ev) cudaEventCreate(&e);
  {
    // CUDA loads kernels lazily on first launch: pull ours in here, not inside the first Solve
    cudaFuncAttributes fa;
    cudaFuncGetAttributes(&fa, pack_kernel);
    cudaFuncGetAttributes(&fa, feasibility_kernel);
    cudaFuncGetAttributes(&fa, class_feasibility_kernel);
    cudaFuncGetAttributes(&fa, finalize_options_kernel);
    cudaFuncGetAttributes(&fa, gather_rows_kernel);
    cudaFuncGetAttributes(&fa, sort_keys_kernel);
    cudaFuncGetAttributes(&fa, gather_u64_kernel);
  }
  *out = h;
  return KSCHED_OK;
}

void ksched_destroy(ksched_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  if (h->comm) ncclCommDestroy(h->comm);
  for (auto& e : h->ev) if (e) cudaEventDestroy(e);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;  // every DevBuf frees its allocation
}

const char* ksched_last_error(const ksched_handle* h) { return h ? h->err.c_str() : "null handle"; }


int ksched_load_catalog(ksched_handle* h, const ksched_catalog* cat) {
  if (!h || !cat) return KSCHED_ERR_INVALID;
  if (cat->n_keys > KSCHED_MAX_KEYS || cat->n_res > KSCHED_MAX_RES || cat->n_templates > KSCHED_MAX_TEMPLATES || cat->n_templates < 1 ||
      cat->n_types < 0) { h->err = "catalog dimensions out of range"; return KSCHED_ERR_INVALID; }
  // Gt/Lt cross the ABI in region form (ksched_key_regions): a requirement set that still carries gt / lt is a caller bug
  if (cat->type_bounds || cat->template_bounds) { h->err = "bounds arrays must be NULL: Gt/Lt requirements are passed in region form (ksched_key_regions)"; return KSCHED_ERR_INVALID; }
  for (int v = 0; v < cat->n_templates; ++v)
    if (cat->templates[v].reqs.meta >> KSCHED_META_HASGT_SHIFT) { h->err = "template requirement with HASGT/HASLT set: pass Gt/Lt in region form"; return KSCHED_ERR_INVALID; }
  for (int t = 0; t < cat->n_types; ++t)
    if (cat->types[t].meta >> KSCHED_META_HASGT_SHIFT) { h->err = "instance-type requirement with HASGT/HASLT set: pass Gt/Lt in region form"; return KSCHED_ERR_INVALID; }
  if (cat->key_regions)
    for (int k = 0; k < cat->n_keys; ++k) {
      const ksched_key_regions& g = cat->key_regions[k];
      if (!g.region_mask) continue;
      const uint64_t want = (g.n_thresholds + 1 >= 64 ? ~0ull : ((1ull << (g.n_thresholds + 1)) - 1)) << g.region_shift;
      if (g.n_thresholds < 0 || g.n_thresholds > KSCHED_MAX_THRESHOLDS || g.region_shift < 0 || g.region_shift + g.n_thresholds + 1 > 63 ||
          g.region_mask != want || (g.region_mask & cat->keys[k].dict_mask)) { h->err = "inconsistent ksched_key_regions"; return KSCHED_ERR_INVALID; }
    }
  CUDA_TRY(h, cudaSetDevice(h->device));
  const int T = cat->n_types, NK = cat->n_keys, V = cat->n_templates, R = cat->n_res;
  const int W64 = type_words64(T), W32 = W64 * 2;
  {
    // Instance types change rarely: when the byte-identical catalog is already resident there is nothing to do (exact
    // comparison against a host copy; the O(T^2) dominance table alone is milliseconds of host time at T = 1000).
    std::vector<unsigned char> blob;
    auto put = [&](const void* p, size_t n) { const unsigned char* b = (const unsigned char*)p; blob.insert(blob.end(), b, b + n); };
    int dims[4] = {NK, R, T, V};
    put(dims, sizeof dims);
    put(cat->keys, sizeof(ksched_keyinfo) * (size_t)NK);
    unsigned char has_int = cat->key_int_values != nullptr, has_off = cat->offering_keys != nullptr, has_reg = cat->key_regions != nullptr;
    put(&has_int, 1); put(&has_off, 1); put(&has_reg, 1);
    if (has_reg) put(cat->key_regions, sizeof(ksched_key_regions) * (size_t)NK);
    if (has_int) put(cat->key_int_values, sizeof(int64_t) * (size_t)NK * 64);
    put(cat->types, sizeof(ksched_type_row) * (size_t)T);
    put(cat->type_capacity, sizeof(int64_t) * (size_t)T * KSCHED_MAX_RES);
    if (has_off) put(cat->offering_keys, sizeof(uint64_t) * (size_t)T * 64);
    if (h->have_catalog && blob == h->catalog_blob) {
      // same instance types: only the templates can differ (remaining provisioner limits move between solves, daemonset
      // overhead with the daemonsets) - they are small, re-upload them when they changed
      if (h->h_templates.size() != (size_t)V || std::memcmp(h->h_templates.data(), cat->templates, sizeof(ksched_template) * (size_t)V) != 0) {
        CUDA_TRY(h, upload(h, h->d_templates, cat->templates, (size_t)V));
        CUDA_TRY(h, cudaStreamSynchronize(h->stream));
        h->cat.templates = h->d_templates.ptr;
        h->h_templates.assign(cat->templates, cat->templates + V);
      }
      return KSCHED_OK;
    }
    h->catalog_blob.swap(blob);
  }
  h->W64 = W64;
  // ---- bit-sliced tables, built on the host (amortised: instance types change rarely)
  std::vector<int16_t> valrow((size_t)NK * 64, -1), offrow(64, -1);
  std::vector<uint32_t> valset, absent((size_t)std::max(NK, 1) * W32, 0), negempty((size_t)std::max(NK, 1) * W32, 0), offset, anyoffer(W32, 0),
      member((size_t)V * W32, 0);
  uint32_t type_relevant = 0;
  int zone_key = -1, ct_key = -1;
  for (int k = 0; k < NK; ++k) {
    if (cat->keys[k].is_zone) zone_key = k;
    if (cat->keys[k].is_capacity_type) ct_key = k;
  }
  std::vector<float> price32(std::max(T, 1), 0.f);
  for (int t = 0; t < T; ++t) {
    const ksched_type_row& row = cat->types[t];
    if (t > 0 && row.min_price < cat->types[t - 1].min_price) { h->err = "instance types must be in ascending price order"; return KSCHED_ERR_INVALID; }
    price32[t] = (float)row.min_price;
    const int w = t >> 5;
    const uint32_t bit = 1u << (t & 31);
    for (int k = 0; k < NK; ++k) {
      bool present = (row.meta >> (KSCHED_META_PRESENT_SHIFT + k)) & 1;
      if (!present) { absent[(size_t)k * W32 + w] |= bit; continue; }
      type_relevant |= 1u << k;
      uint64_t v = row.values[k];
      if ((row.meta >> (KSCHED_META_COMPLEMENT_SHIFT + k)) & 1) {
        // complement requirement (NotIn / Exists / Gt / Lt, region form): the type admits every value and region it does not
        // exclude; its operator is negative (NotIn) when it really excludes a value (requirement.go:186-197)
        const uint64_t region_mask = cat->key_regions ? cat->key_regions[k].region_mask : 0;
        if (!region_mask) { h->err = "instance type with a complement requirement on a key without region bits"; return KSCHED_ERR_INVALID; }
        ksched::Req r{v, 0, 0, true, true, false, false};
        if (ksched::req_excluded(r, KeyMeta{0, nullptr, cat->key_regions + k}) != 0) negempty[(size_t)k * W32 + w] |= bit;
        v = ~v & (cat->keys[k].dict_mask | region_mask);
      } else if (!v) { negempty[(size_t)k * W32 + w] |= bit; continue; }
      while (v) {
        int b = __builtin_ctzll(v);
        v &= v - 1;
        int16_t& r = valrow[(size_t)k * 64 + b];
        if (r < 0) { r = (int16_t)(valset.size() / W32); valset.resize(valset.size() + W32, 0); }
        valset[(size_t)r * W32 + w] |= bit;
      }
    }
    uint64_t o = row.offerings;
    if (o) anyoffer[w] |= bit;
    while (o) {
      int b = __builtin_ctzll(o);
      o &= o - 1;
      int16_t& r = offrow[b];
      if (r < 0) { r = (int16_t)(offset.size() / W32); offset.resize(offset.size() + W32, 0); }
      offset[(size_t)r * W32 + w] |= bit;
    }
    for (int v = 0; v < V; ++v) if ((row.template_members >> v) & 1) member[(size_t)v * W32 + w] |= bit;
  }
  if (valset.empty()) valset.resize(W32, 0);
  if (offset.empty()) offset.resize(W32, 0);
  std::vector<int32_t> perm_desc((size_t)std::max(R, 1) * std::max(T, 1), 0);
  std::vector<int64_t> alloc_rt((size_t)std::max(R, 1) * std::max(T, 1), 0);
  std::vector<int64_t> alloc_sorted((size_t)std::max(R, 1) * std::max(T, 1), 0);
  std::vector<uint32_t> fitset((size_t)std::max(R, 1) * (T + 1) * W32, 0);
  {
    std::vector<int> perm(T);
    for (int r = 0; r < R; ++r) {
      for (int t = 0; t < T; ++t) perm[t] = t;
      std::stable_sort(perm.begin(), perm.end(), [&](int a, int b) { return cat->types[a].allocatable[r] < cat->types[b].allocatable[r]; });
      for (int i = 0; i < T; ++i) {
        alloc_sorted[(size_t)r * T + i] = cat->types[perm[i]].allocatable[r];
        perm_desc[(size_t)r * T + (T - 1 - i)] = perm[i];
        alloc_rt[(size_t)r * T + i] = cat->types[i].allocatable[r];
      }
      uint32_t* base = &fitset[(size_t)r * (T + 1) * W32];
      for (int i = T - 1; i >= 0; --i) {
        uint32_t* cur = base + (size_t)i * W32;
        std::memcpy(cur, base + (size_t)(i + 1) * W32, W32 * sizeof(uint32_t));
        cur[perm[i] >> 5] |= 1u << (perm[i] & 31);
      }
    }
  }
  {
    // the device's dict_mask includes the region bits: "every admissible value" of a complement requirement then covers the
    // regions a complement instance type shares with it (catalog.cuh: key_typeset_word walks the admitted bits)
    std::vector<ksched_keyinfo> dev_keys(cat->keys, cat->keys + NK);
    if (cat->key_regions) for (int k = 0; k < NK; ++k) dev_keys[k].dict_mask |= cat->key_regions[k].region_mask;
    CUDA_TRY(h, upload_vec(h, h->d_keys, dev_keys));
    if (cat->key_regions) CUDA_TRY(h, upload(h, h->d_key_regions, cat->key_regions, (size_t)NK));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // dev_keys is a stack vector
  }
  if (cat->key_int_values) CUDA_TRY(h, upload(h, h->d_key_int, cat->key_int_values, (size_t)NK * 64));
  CUDA_TRY(h, upload(h, h->d_templates, cat->templates, (size_t)V));
  CUDA_TRY(h, upload(h, h->d_types, cat->types, (size_t)T));
  CUDA_TRY(h, upload(h, h->d_capacity, cat->type_capacity, (size_t)T * KSCHED_MAX_RES));
  CUDA_TRY(h, upload_vec(h, h->d_price32, price32));
  CUDA_TRY(h, upload_vec(h, h->d_valrow, valrow));
  CUDA_TRY(h, upload_vec(h, h->d_offrow, offrow));
  CUDA_TRY(h, upload_vec(h, h->d_valset, valset));
  CUDA_TRY(h, upload_vec(h, h->d_absent, absent));
  CUDA_TRY(h, upload_vec(h, h->d_negempty, negempty));
  CUDA_TRY(h, upload_vec(h, h->d_offset, offset));
  CUDA_TRY(h, upload_vec(h, h->d_anyoffer, anyoffer));
  CUDA_TRY(h, upload_vec(h, h->d_member, member));
  CUDA_TRY(h, upload_vec(h, h->d_alloc_sorted, alloc_sorted));
  CUDA_TRY(h, upload_vec(h, h->d_perm_desc, perm_desc));
  CUDA_TRY(h, upload_vec(h, h->d_alloc_rt, alloc_rt));
  {
    // dominance bitsets over the first min(R,4) resources (pack kernel: Pareto front of a node's options)
    const int RH = std::min(R, 4);
    std::vector<uint32_t> domset((size_t)std::max(T, 1) * W32, 0);
    for (int a = 0; a < T; ++a)
      for (int b = 0; b < T; ++b) {
        bool dom = true;
        for (int r = 0; r < RH && dom; ++r) dom = cat->types[a].allocatable[r] >= cat->types[b].allocatable[r];
        if (dom) domset[(size_t)a * W32 + (b >> 5)] |= 1u << (b & 31);
      }
    CUDA_TRY(h, upload_vec(h, h->d_domset, domset));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  }
  CUDA_TRY(h, upload_vec(h, h->d_fitset, fitset));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->h_templates.assign(cat->templates, cat->templates + V);
  h->n_valrows = (int)(valset.size() / W32);
  h->n_offrows = (int)(offset.size() / W32);
  DevCatalog& c = h->cat;
  c.n_keys = NK; c.n_res = R; c.n_types = T; c.n_templates = V; c.W32 = W32;
  c.keys = h->d_keys.ptr;
  c.key_int_values = cat->key_int_values ? h->d_key_int.ptr : nullptr;
  c.key_regions = cat->key_regions ? h->d_key_regions.ptr : nullptr;
  c.templates = h->d_templates.ptr;
  c.types = h->d_types.ptr;
  c.capacity = h->d_capacity.ptr;
  c.price32 = h->d_price32.ptr;
  c.valrow = h->d_valrow.ptr; c.valset = h->d_valset.ptr; c.absent = h->d_absent.ptr; c.negempty = h->d_negempty.ptr;
  c.type_relevant = type_relevant;
  c.offrow = h->d_offrow.ptr; c.offset = h->d_offset.ptr; c.anyoffer = h->d_anyoffer.ptr; c.member = h->d_member.ptr;
  c.alloc_sorted = h->d_alloc_sorted.ptr; c.fitset = h->d_fitset.ptr;
  c.perm_desc = h->d_perm_desc.ptr; c.alloc_rt = h->d_alloc_rt.ptr; c.domset = h->d_domset.ptr;
  c.offer_keys = nullptr;
  c.input_index = nullptr;
  if (cat->offering_keys && T > 0) {
    std::vector<uint32_t> input_index(T);
    for (int t = 0; t < T; ++t) input_index[t] = cat->types[t].input_index;
    CUDA_TRY(h, upload(h, h->d_offer_keys, cat->offering_keys, (size_t)T * 64));
    CUDA_TRY(h, upload_vec(h, h->d_input_index, input_index));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // input_index is a stack vector
    c.offer_keys = h->d_offer_keys.ptr;
    c.input_index = h->d_input_index.ptr;
  }
  c.zone_key = zone_key; c.ct_key = ct_key;
  {
    // pin_neutral (catalog.cuh): U = union of every template's member types
    std::vector<uint32_t> U(W32, 0);
    for (int v = 0; v < V; ++v) for (int w = 0; w < W32; ++w) U[w] |= member[(size_t)v * W32 + w];
    auto covers = [&](const std::vector<uint32_t>& set) { for (int w = 0; w < W32; ++w) if (U[w] & ~set[w]) return false; return true; };
    auto offer_rows = [&](int ct, int z, std::vector<uint32_t>& acc) {
      const int16_t r = offrow[ct * 16 + z];
      if (r >= 0) for (int w = 0; w < W32; ++w) acc[w] |= offset[(size_t)r * W32 + w];
    };
    for (int k = 0; k < KSCHED_MAX_KEYS; ++k) c.pin_neutral[k] = 0;
    for (int k = 0; k < NK; ++k) {
      for (int b = 0; b < 64; ++b) {
        if (!((cat->keys[k].dict_mask >> b) & 1)) continue;
        std::vector<uint32_t> set(W32, 0);
        for (int w = 0; w < W32; ++w) set[w] = absent[(size_t)k * W32 + w];
        if (valrow[(size_t)k * 64 + b] >= 0) for (int w = 0; w < W32; ++w) set[w] |= valset[(size_t)valrow[(size_t)k * 64 + b] * W32 + w];
        bool ok = covers(set);
        if (ok && k == zone_key) {
          if (b >= 16) ok = false;
          else if (ct_key >= 0) {
            for (int ct = 0; ct < 4 && ok; ++ct) {
              if (!((cat->keys[ct_key].dict_mask >> ct) & 1)) continue;
              std::vector<uint32_t> acc(W32, 0);
              offer_rows(ct, b, acc);
              ok = covers(acc);
            }
            if (cat->keys[ct_key].dict_mask >> 4) ok = false;
          } else {
            std::vector<uint32_t> acc(W32, 0);
            for (int ct = 0; ct < 4; ++ct) offer_rows(ct, b, acc);
            ok = covers(acc);
          }
        }
        if (ok && k == ct_key) {
          if (b >= 4) ok = false;
          else if (zone_key >= 0) {
            for (int z = 0; z < 16 && ok; ++z) {
              if (!((cat->keys[zone_key].dict_mask >> z) & 1)) continue;
              std::vector<uint32_t> acc(W32, 0);
              offer_rows(b, z, acc);
              ok = covers(acc);
            }
            if (cat->keys[zone_key].dict_mask >> 16) ok = false;
          } else {
            std::vector<uint32_t> acc(W32, 0);
            for (int z = 0; z < 16; ++z) offer_rows(b, z, acc);
            ok = covers(acc);
          }
        }
        if (ok) c.pin_neutral[k] |= 1ull << b;
      }
    }
  }
  h->have_catalog = true;
  h->uploaded = false;
  return KSCHED_OK;
}

int ksched_set_shard(ksched_handle* h, int rank, int world) {
  if (!h || world < 1 || rank < 0 || rank >= world) return KSCHED_ERR_INVALID;
  h->rank = rank;
  h->world = world;
  return KSCHED_OK;
}

int ksched_shard_range(int n_words32, int rank, int world, int* begin, int* end) {
  if (n_words32 < 0 || world < 1 || rank < 0 || rank >= world || !begin || !end) return KSCHED_ERR_INVALID;
  const int per = (n_words32 + world - 1) / world;
  *begin = std::min(n_words32, rank * per);
  *end = std::min(n_words32, *begin + per);
  return KSCHED_OK;
}

int ksched_nccl_unique_id(void* out128) {
  ncclUniqueId id;
  if (ncclGetUniqueId(&id) != ncclSuccess) return KSCHED_ERR_NCCL;
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  std::memcpy(out128, &id, 128);
  return KSCHED_OK;
}
int ksched_nccl_init(ksched_handle* h, const void* id128, int rank, int world) {
  if (!h || !id128) return KSCHED_ERR_INVALID;
  if (cudaSetDevice(h->device) != cudaSuccess) return KSCHED_ERR_CUDA;
  ncclUniqueId id;
  std::memcpy(&id, id128, 128);
  ncclResult_t r = ncclCommInitRank(&h->comm, world, id, rank);
  if (r != ncclSuccess) { h->err = std::string("ncclCommInitRank: ") + ncclGetErrorString(r); return KSCHED_ERR_NCCL; }
  h->rank = rank;
  h->world = world;
  return KSCHED_OK;
}

// One ncclAllGather of `bytes` bytes per rank on the handle's communicator (consolidation: the verdicts of the simulations
// each rank ran, SURVEY.md 8e). Host buffers in and out; recv holds world * bytes.
int ksched_allgather(ksched_handle* h, const void* send, size_t bytes, void* recv) {
  if (!h || !send || !recv) return KSCHED_ERR_INVALID;
  if (!h->comm) { h->err = "ksched_nccl_init must be called first"; return KSCHED_ERR_INVALID; }
  CUDA_TRY(h, cudaSetDevice(h->device));
  int world = 0;
  if (ncclCommCount(h->comm, &world) != ncclSuccess) return KSCHED_ERR_NCCL;
  CUDA_TRY(h, h->d_gather_send.ensure(std::max<size_t>(bytes, 1)));
  CUDA_TRY(h, h->d_gather_recv.ensure(std::max<size_t>(bytes * (size_t)world, 1)));
  CUDA_TRY(h, cudaMemcpyAsync(h->d_gather_send.ptr, send, bytes, cudaMemcpyHostToDevice, h->stream));
  ncclResult_t r = ncclAllGather(h->d_gather_send.ptr, h->d_gather_recv.ptr, bytes, ncclUint8, h->comm, h->stream);
  if (r != ncclSuccess) { h->err = std::string("ncclAllGather: ") + ncclGetErrorString(r); return KSCHED_ERR_NCCL; }
  CUDA_TRY(h, cudaMemcpyAsync(recv, h->d_gather_recv.ptr, bytes * (size_t)world, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return KSCHED_OK;
}

// ---- upload one problem (pods / nodes / topology) and keep pristine copies of everything the pack kernel mutates
int ksched_upload(ksched_handle* h, const ksched_problem* pb) {
  if (!h || !pb) return KSCHED_ERR_INVALID;
  if (!h->have_catalog) { h->err = "ksched_load_catalog must be called first"; return KSCHED_ERR_INVALID; }
  if (pb->class_bounds || pb->existing_bounds) { h->err = "bounds arrays must be NULL: Gt/Lt requirements are passed in region form (ksched_key_regions)"; return KSCHED_ERR_INVALID; }
  for (int i = 0; i < pb->n_classes; ++i)
    if (pb->classes[i].meta >> KSCHED_META_HASGT_SHIFT) { h->err = "requirement with HASGT/HASLT set: pass Gt/Lt in region form"; return KSCHED_ERR_INVALID; }
  for (int i = 0; i < pb->n_existing; ++i)
    if (pb->existing[i].reqs.meta >> KSCHED_META_HASGT_SHIFT) { h->err = "requirement with HASGT/HASLT set: pass Gt/Lt in region form"; return KSCHED_ERR_INVALID; }
  for (int i = 0; i < pb->n_filter_terms; ++i)
    if (pb->filter_terms[i].meta >> KSCHED_META_HASGT_SHIFT) { h->err = "requirement with HASGT/HASLT set: pass Gt/Lt in region form"; return KSCHED_ERR_INVALID; }
  CUDA_TRY(h, cudaSetDevice(h->device));
  h->tm.h2d_bytes = 0;
  const DevCatalog& c = h->cat;
  const int P = pb->n_pods, NC = pb->n_classes, NE = pb->n_existing, NG = pb->n_groups, W32 = c.W32, V = c.n_templates;
  const int MAXN = std::max(1, std::min(pb->max_new_nodes > 0 ? pb->max_new_nodes : P, std::max(P, 1)));
  h->n_pods = P; h->n_classes = NC; h->n_existing = NE; h->n_groups = NG; h->max_new = MAXN;
  h->count_visited = pb->count_nodes_visited;
  for (int c2 = 0; c2 < NC; ++c2) {
    const ksched_pod_row& row = pb->classes[c2];
    if (row.relax_next != KSCHED_NONE && row.relax_next >= (uint32_t)NC) { h->err = "relax_next out of range"; return KSCHED_ERR_INVALID; }
    if (row.topo_end < row.topo_begin || row.topo_end > (uint32_t)pb->n_class_topo) { h->err = "class_topo range out of bounds"; return KSCHED_ERR_INVALID; }
    int ncg = 0, touched = __builtin_popcountll((row.meta >> KSCHED_META_PRESENT_SHIFT) & 0xFFFF);
    for (uint32_t e = row.topo_begin; e < row.topo_end; ++e) {
      if (pb->class_topo[e].group >= (uint32_t)NG) { h->err = "class_topo group out of range"; return KSCHED_ERR_INVALID; }
      if (pb->class_topo[e].flags & KSCHED_TOPO_CONSTRAINS) { ++ncg; if (pb->groups[pb->class_topo[e].group].key != KSCHED_KEY_HOSTNAME) ++touched; }
    }
    if (ncg > kMaxCG || touched > kMaxTouched) { h->err = "a pod class is constrained by more topology groups / label keys than the pack kernel carries"; return KSCHED_ERR_UNSUPPORTED; }
  }
  // min request per resource over all classes (node closing rule)
  for (int r = 0; r < KSCHED_MAX_RES; ++r) {
    int64_t mn = INT64_MAX;
    for (int c2 = 0; c2 < NC; ++c2) {
      const ksched_pod_row& row = pb->classes[c2];
      int64_t v = ((row.res_present >> r) & 1) ? row.requests[r] : 0;
      mn = std::min(mn, v);
    }
    h->min_req[r] = (NC == 0 || mn == INT64_MAX || mn < 0) ? 0 : mn;
  }
  CUDA_TRY(h, upload(h, h->d_classes, pb->classes, (size_t)NC));
  {
    // queue.go:82-108 orders by cpu desc, memory desc, timestamp asc, UID asc. (cpu, memory) is a property of the class: rank
    // the classes once here, and the whole order is one packed key when rank, timestamp span and UID rank fit 64 bits.
    std::vector<uint32_t> by((size_t)NC), rank((size_t)std::max(NC, 1), 0);
    for (int i = 0; i < NC; ++i) by[(size_t)i] = (uint32_t)i;
    auto cpu = [&](uint32_t c) { return pb->classes[c].requests[0]; };
    auto mem = [&](uint32_t c) { return pb->classes[c].requests[1]; };
    std::sort(by.begin(), by.end(), [&](uint32_t a, uint32_t b) { return cpu(a) != cpu(b) ? cpu(a) > cpu(b) : mem(a) > mem(b); });
    uint32_t r = 0;
    for (int i = 0; i < NC; ++i) {
      if (i > 0 && (cpu(by[(size_t)i]) != cpu(by[(size_t)i - 1]) || mem(by[(size_t)i]) != mem(by[(size_t)i - 1]))) ++r;
      rank[by[(size_t)i]] = r;
    }
    auto bits = [](unsigned long long v) { int b = 0; while (v) { ++b; v >>= 1; } return std::max(b, 1); };
    long long ts_min = 0, ts_max = 0;
    uint32_t uid_max = 0;
    for (int i = 0; i < P; ++i) {
      const long long t = pb->pod_timestamp[i];
      if (i == 0 || t < ts_min) ts_min = t;
      if (i == 0 || t > ts_max) ts_max = t;
      uid_max = std::max(uid_max, pb->pod_uid_rank[i]);
    }
    const unsigned long long span = (unsigned long long)(ts_max - ts_min);
    h->sort1_ts_bits = bits(span);
    h->sort1_uid_bits = bits(uid_max);
    h->sort1_ts_min = ts_min;
    const int total = bits(r) + h->sort1_ts_bits + h->sort1_uid_bits;
    h->sort1_bits = (span < (1ull << 62) && total <= 64 && !std::getenv("KSCHED_SORT3")) ? total : 0;
    CUDA_TRY(h, upload_vec(h, h->d_cls_rank, rank));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // rank is a stack vector
  }
  CUDA_TRY(h, upload(h, h->d_pod_class0, pb->pod_class, (size_t)P));
  CUDA_TRY(h, h->d_pod_class.ensure(P));
  CUDA_TRY(h, upload(h, h->d_ts, pb->pod_timestamp, (size_t)P));
  CUDA_TRY(h, upload(h, h->d_uid_rank, pb->pod_uid_rank, (size_t)P));
  CUDA_TRY(h, upload(h, h->d_groups, pb->groups, (size_t)NG));
  CUDA_TRY(h, upload(h, h->d_class_topo, pb->class_topo, (size_t)pb->n_class_topo));
  CUDA_TRY(h, upload(h, h->d_filter_terms, pb->filter_terms, (size_t)pb->n_filter_terms));
  CUDA_TRY(h, upload(h, h->d_hostname_reqs, pb->hostname_reqs, (size_t)pb->n_hostname_reqs * 2));
  CUDA_TRY(h, upload(h, h->d_itype_comp, pb->itype_req_complement, (size_t)pb->n_itype_reqs));
  CUDA_TRY(h, upload(h, h->d_itype_sets, reinterpret_cast<const uint32_t*>(pb->itype_req_sets), (size_t)pb->n_itype_reqs * W32));
  // existing nodes -> SoA
  {
    std::vector<int64_t> req((size_t)8 * std::max(NE, 1), 0), avail((size_t)8 * std::max(NE, 1), 0);
    std::vector<uint32_t> reqp(std::max(NE, 1), 0), availp(std::max(NE, 1), 0), ts(std::max(NE, 1), 0), it(std::max(NE, 1), 0);
    std::vector<uint64_t> vals((size_t)16 * std::max(NE, 1), 0), meta(std::max(NE, 1), 0), hp(std::max(NE, 1), 0);
    for (int e = 0; e < NE; ++e) {
      const ksched_existing_node& n = pb->existing[e];
      for (int r = 0; r < 8; ++r) { req[(size_t)r * NE + e] = n.requests[r]; avail[(size_t)r * NE + e] = n.available[r]; }
      for (int k = 0; k < 16; ++k) vals[(size_t)k * NE + e] = n.reqs.values[k];
      meta[e] = n.reqs.meta & 0xFFFFFFFFull;
      reqp[e] = n.requests_present; availp[e] = n.available_present; ts[e] = n.taintset; it[e] = n.itype; hp[e] = n.hostport_entries;
    }
    CUDA_TRY(h, upload_vec(h, h->d_ex_req0, req));
    CUDA_TRY(h, upload_vec(h, h->d_ex_avail, avail));
    CUDA_TRY(h, upload_vec(h, h->d_ex_req_present0, reqp));
    CUDA_TRY(h, upload_vec(h, h->d_ex_avail_present, availp));
    CUDA_TRY(h, upload_vec(h, h->d_ex_taintset, ts));
    CUDA_TRY(h, upload_vec(h, h->d_ex_itype, it));
    CUDA_TRY(h, upload_vec(h, h->d_ex_vals0, vals));
    CUDA_TRY(h, upload_vec(h, h->d_ex_meta0, meta));
    CUDA_TRY(h, upload_vec(h, h->d_ex_hp0, hp));
    h->have_volumes = pb->class_volumes != nullptr && pb->existing_volumes != nullptr && NE > 0;
    if (h->have_volumes) {
      CUDA_TRY(h, upload(h, h->d_cls_vol, pb->class_volumes, (size_t)NC));
      CUDA_TRY(h, upload(h, h->d_ex_vol0, pb->existing_volumes, (size_t)NE));
      CUDA_TRY(h, h->d_ex_vol.ensure((size_t)NE));
      for (int d = 0; d < KSCHED_MAX_VOLUME_DRIVERS; ++d) h->vol_mask[d] = pb->volume_driver_mask[d];
    }
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // host vectors go out of scope
    size_t ne = (size_t)std::max(NE, 1);
    CUDA_TRY(h, h->d_ex_req.ensure(8 * ne));
    CUDA_TRY(h, h->d_ex_req_present.ensure(ne));
    CUDA_TRY(h, h->d_ex_vals.ensure(16 * ne));
    CUDA_TRY(h, h->d_ex_meta.ensure(ne));
    CUDA_TRY(h, h->d_ex_hp.ensure(ne));
    CUDA_TRY(h, h->d_ex_closed.ensure(ne));
  }
  // topology counters
  {
    std::vector<int32_t> host_row(std::max(NG, 1), -1), host_total(std::max(NG, 1), 0), cnt((size_t)std::max(NG, 1) * 64, 0);
    std::vector<uint64_t> registered(std::max(NG, 1), 0);
    int nh = 0;
    for (int g = 0; g < NG; ++g) {
      if (pb->groups[g].key == KSCHED_KEY_HOSTNAME) host_row[g] = nh++;
      else if (pb->groups[g].key >= c.n_keys) { h->err = "topology group key out of range"; return KSCHED_ERR_INVALID; }
      registered[g] = pb->groups[g].registered;
      for (int d = 0; d < 64; ++d) cnt[(size_t)g * 64 + d] = pb->group_domain_counts[(size_t)g * 64 + d];
    }
    h->n_hostgroups = nh;
    const size_t stride = (size_t)NE + MAXN;
    // [hostname group][existing node | new node slot] counters: only the existing-node columns carry initial values, the
    // rest of the (up to 40 MB) matrix is zeroed on the device instead of being built and shipped from the host
    std::vector<uint16_t> host((size_t)std::max(nh, 1) * std::max(NE, 1), 0);
    for (int g = 0; g < NG; ++g) {
      if (host_row[g] < 0) continue;
      int total = pb->groups[g].extra_nonzero_domains;
      for (int e = 0; e < NE; ++e) {
        int32_t v = pb->group_existing_counts[(size_t)g * std::max(NE, 1) + e];
        host[(size_t)host_row[g] * NE + e] = (uint16_t)std::min(v, 0xFFFF);
        if (v > 0) ++total;
      }
      host_total[g] = total;
    }
    std::vector<uint8_t> active(std::max(NG, 1), 1);
    for (int g = 0; g < NG; ++g) active[g] = pb->groups[g].dormant ? 0 : 1;
    CUDA_TRY(h, upload_vec(h, h->d_grp_active0, active));
    CUDA_TRY(h, h->d_grp_active.ensure(std::max(NG, 1)));
    CUDA_TRY(h, h->d_grp_min_slot.ensure(std::max(NG, 1)));
    CUDA_TRY(h, upload_vec(h, h->d_grp_host_row, host_row));
    {
      std::vector<RelX> relx((size_t)std::max(pb->n_class_topo, 1));
      for (int e = 0; e < pb->n_class_topo; ++e) {
        const ksched_class_topo& ct = pb->class_topo[e];
        if ((int)ct.group >= NG) { h->err = "class_topo names a group out of range"; return KSCHED_ERR_INVALID; }
        const ksched_topo_group& g = pb->groups[ct.group];
        RelX x{};
        x.group = ct.group; x.flags = ct.flags; x.key = g.key; x.type = g.type; x.has_filter = g.filter_begin != g.filter_end;
        // a term without any requirement is Compatible with every node (topologynodefilter.go:57-70): such a filter always matches
        for (uint32_t f = g.filter_begin; f < g.filter_end && f < (uint32_t)pb->n_filter_terms; ++f)
          if (((pb->filter_terms[f].meta >> KSCHED_META_PRESENT_SHIFT) & 0xFFFF) == 0) x.has_filter = 0;
        x.max_skew = g.max_skew; x.host_row = host_row[ct.group];
        relx[e] = x;
      }
      CUDA_TRY(h, upload_vec(h, h->d_relx, relx));
    }
    CUDA_TRY(h, upload_vec(h, h->d_grp_host_total0, host_total));
    CUDA_TRY(h, upload_vec(h, h->d_grp_cnt0, cnt));
    CUDA_TRY(h, upload_vec(h, h->d_grp_registered0, registered));
    CUDA_TRY(h, h->d_grp_host0.ensure((size_t)std::max(nh, 1) * stride));
    CUDA_TRY(h, cudaMemsetAsync(h->d_grp_host0.ptr, 0, (size_t)std::max(nh, 1) * stride * sizeof(uint16_t), h->stream));
    if (NE > 0 && nh > 0) {
      CUDA_TRY(h, cudaMemcpy2DAsync(h->d_grp_host0.ptr, stride * sizeof(uint16_t), host.data(), (size_t)NE * sizeof(uint16_t), (size_t)NE * sizeof(uint16_t),
                                    (size_t)nh, cudaMemcpyHostToDevice, h->stream));
      h->tm.h2d_bytes += (int64_t)nh * NE * 2;
    }
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    CUDA_TRY(h, h->d_grp_host_total.ensure(std::max(NG, 1)));
    CUDA_TRY(h, h->d_grp_cnt.ensure((size_t)std::max(NG, 1) * 64));
    CUDA_TRY(h, h->d_grp_registered.ensure(std::max(NG, 1)));
    CUDA_TRY(h, h->d_grp_host.ensure((size_t)std::max(nh, 1) * stride));
  }
  // scratch / state
  const size_t p1 = (size_t)std::max(P, 1);
  CUDA_TRY(h, h->d_order.ensure(p1)); CUDA_TRY(h, h->d_idx_tmp.ensure(p1)); CUDA_TRY(h, h->d_pod_pos.ensure(p1));
  CUDA_TRY(h, h->d_k_cpu.ensure(p1)); CUDA_TRY(h, h->d_k_mem.ensure(p1)); CUDA_TRY(h, h->d_k_tie.ensure(p1)); CUDA_TRY(h, h->d_k_tmp.ensure(p1));
  CUDA_TRY(h, h->d_rows.ensure(p1 * KSCHED_ROW_WORDS));
  CUDA_TRY(h, h->d_F.ensure(p1 * V * W32));
  CUDA_TRY(h, h->d_best.ensure(p1));
  CUDA_TRY(h, h->d_Fclass.ensure((size_t)std::max(NC, 1) * V * W32));
  CUDA_TRY(h, h->d_best_class.ensure((size_t)std::max(NC, 1)));
  CUDA_TRY(h, h->d_relax.ensure(p1)); CUDA_TRY(h, h->d_assign.ensure(p1)); CUDA_TRY(h, h->d_place_seq.ensure(p1));
  CUDA_TRY(h, h->d_queue.ensure(p1 + 1)); CUDA_TRY(h, h->d_last_len.ensure(p1)); CUDA_TRY(h, h->d_last_epoch.ensure(p1));
  const size_t mn = (size_t)MAXN;
  CUDA_TRY(h, h->d_nn_tmpl.ensure(mn)); CUDA_TRY(h, h->d_nn_count.ensure(mn)); CUDA_TRY(h, h->d_nn_tb.ensure(mn));
  CUDA_TRY(h, h->d_nn_req.ensure(8 * mn)); CUDA_TRY(h, h->d_nn_req_present.ensure(mn));
  CUDA_TRY(h, h->d_nn_vals.ensure(16 * mn)); CUDA_TRY(h, h->d_nn_meta.ensure(mn));
  CUDA_TRY(h, h->d_nn_opts.ensure((size_t)W32 * mn)); CUDA_TRY(h, h->d_nn_hp.ensure(mn));
  CUDA_TRY(h, h->d_ov_key.ensure(mn)); CUDA_TRY(h, h->d_ov_q.ensure(4 * mn)); CUDA_TRY(h, h->d_ov_bound.ensure(4 * mn)); CUDA_TRY(h, h->d_ov_bound2.ensure(4 * mn));
  CUDA_TRY(h, h->d_ov_node.ensure(mn)); CUDA_TRY(h, h->d_ov_flags.ensure(mn));
  CUDA_TRY(h, h->d_ov_absorbed.ensure(mn)); CUDA_TRY(h, h->d_ov_rejected.ensure(mn));
  {
    const size_t nfc = (size_t)std::max(NC, 1) * V;
    CUDA_TRY(h, h->d_fc_state.ensure(nfc)); CUDA_TRY(h, h->d_fc_dom.ensure(nfc)); CUDA_TRY(h, h->d_fc_front_state.ensure(nfc)); CUDA_TRY(h, h->d_fc_bound.ensure(nfc * 4)); CUDA_TRY(h, h->d_fc_bound2.ensure(nfc * 4));
    CUDA_TRY(h, h->d_fc_opts.ensure(nfc * W32));
    CUDA_TRY(h, h->d_fc_vals.ensure(nfc * KSCHED_MAX_KEYS)); CUDA_TRY(h, h->d_fc_meta.ensure(nfc)); CUDA_TRY(h, h->d_fc_q.ensure(nfc * KSCHED_MAX_RES));
    CUDA_TRY(h, h->d_fc_qp.ensure(nfc));
    const size_t nfd = kFreshMemoSlots;
    CUDA_TRY(h, h->d_fd_state.ensure(nfd)); CUDA_TRY(h, h->d_fd_dom.ensure(nfd)); CUDA_TRY(h, h->d_fd_fc.ensure(nfd)); CUDA_TRY(h, h->d_fd_meta.ensure(nfd));
    CUDA_TRY(h, h->d_fd_vals.ensure(nfd * KSCHED_MAX_KEYS)); CUDA_TRY(h, h->d_fd_opts.ensure(nfd * W32));
    CUDA_TRY(h, h->d_fd_bound.ensure(nfd * 4)); CUDA_TRY(h, h->d_fd_bound2.ensure(nfd * 4));
  }
  CUDA_TRY(h, h->d_remaining.ensure((size_t)V * KSCHED_MAX_RES));
  CUDA_TRY(h, h->d_counters.ensure(80));
  {
    size_t need = 0, n2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, need, (uint64_t*)nullptr, (uint64_t*)nullptr, (uint32_t*)nullptr, (uint32_t*)nullptr, (int)p1, 0, 64, h->stream);
    n2 = need;
    CUDA_TRY(h, h->d_cub_tmp.ensure(n2 + 256));
    h->cub_tmp_bytes = n2 + 256;
  }
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->uploaded = true;
  h->sorted = false;
  return KSCHED_OK;
}

static int run_sort(ksched_handle* h) {
  const int P = h->n_pods;
  if (P == 0) return KSCHED_OK;
  const int threads = 256, blocks = (P + threads - 1) / threads;
  if (h->sort1_bits > 0) {  // one packed key, only its significant bits sorted
    sort_key1_kernel<<<blocks, threads, 0, h->stream>>>(P, h->d_cls_rank.ptr, h->d_pod_class.ptr, h->d_ts.ptr, h->d_uid_rank.ptr, h->sort1_ts_min,
                                                        h->sort1_ts_bits, h->sort1_uid_bits, h->d_k_tie.ptr, h->d_idx_tmp.ptr);
    size_t tmp1 = h->cub_tmp_bytes;
    CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(h->d_cub_tmp.ptr, tmp1, h->d_k_tie.ptr, h->d_k_tmp.ptr, h->d_idx_tmp.ptr, h->d_order.ptr, P, 0, h->sort1_bits,
                                                h->stream));
    const int gblocks1 = std::min((P + 7) / 8, 148 * 8);
    gather_rows_kernel<<<gblocks1, 256, 0, h->stream>>>(P, h->d_classes.ptr, h->d_pod_class.ptr, h->d_order.ptr, h->d_rows.ptr);
    h->tm.sort_launches = 3;
    h->sorted = true;
    return KSCHED_OK;
  }
  sort_keys_kernel<<<blocks, threads, 0, h->stream>>>(P, h->d_classes.ptr, h->d_pod_class.ptr, h->d_ts.ptr, h->d_uid_rank.ptr, h->d_k_cpu.ptr,
                                                      h->d_k_mem.ptr, h->d_k_tie.ptr, h->d_order.ptr);
  // LSD over three 64-bit keys with a stable radix sort: tie-break key first, cpu last
  size_t tmp = h->cub_tmp_bytes;
  uint32_t *ia = h->d_order.ptr, *ib = h->d_idx_tmp.ptr;
  CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(h->d_cub_tmp.ptr, tmp, h->d_k_tie.ptr, h->d_k_tmp.ptr, ia, ib, P, 0, 64, h->stream));
  gather_u64_kernel<<<blocks, threads, 0, h->stream>>>(P, h->d_k_mem.ptr, ib, h->d_k_tie.ptr);
  tmp = h->cub_tmp_bytes;
  CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(h->d_cub_tmp.ptr, tmp, h->d_k_tie.ptr, h->d_k_tmp.ptr, ib, ia, P, 0, 64, h->stream));
  gather_u64_kernel<<<blocks, threads, 0, h->stream>>>(P, h->d_k_cpu.ptr, ia, h->d_k_tie.ptr);
  tmp = h->cub_tmp_bytes;
  CUDA_TRY(h, cub::DeviceRadixSort::SortPairs(h->d_cub_tmp.ptr, tmp, h->d_k_tie.ptr, h->d_k_tmp.ptr, ia, ib, P, 0, 64, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(h->d_order.ptr, ib, (size_t)P * sizeof(uint32_t), cudaMemcpyDeviceToDevice, h->stream));
  const int gblocks = std::min((P + 7) / 8, 148 * 8);
  gather_rows_kernel<<<gblocks, 256, 0, h->stream>>>(P, h->d_classes.ptr, h->d_pod_class.ptr, h->d_order.ptr, h->d_rows.ptr);
  h->tm.sort_launches = 7;
  h->sorted = true;
  return KSCHED_OK;
}

static void fill_k1(ksched_handle* h, K1Params& k1) {
  // the row evaluation runs over the class table (every class once); feasibility_kernel replicates the rows per pod
  k1.cat = h->cat;
  k1.rows = reinterpret_cast<const uint64_t*>(h->d_classes.ptr);
  k1.n_pods = h->n_classes;
  k1.itype_sets = h->d_itype_sets.ptr;
  k1.F = h->d_Fclass.ptr;
  k1.best = h->d_best_class.ptr;
  const int W32 = h->cat.W32;
  if (h->world > 1) {
    ksched_shard_range(W32, h->rank, h->world, &k1.word_begin, &k1.word_end);
  } else {
    k1.word_begin = 0;
    k1.word_end = W32;
  }
}

static std::mutex g_k1_mu;
static cudaEvent_t g_k1_done[64] = {};

// K1, class pass: every distinct pod row evaluated once (class_feasibility_kernel over the class table).
static int run_class_feasibility(ksched_handle* h) {
  if (h->n_pods == 0 || h->n_classes == 0) return KSCHED_OK;
  K1Params k1;
  fill_k1(h, k1);
  const DevCatalog& c = h->cat;
  const size_t alloc_bytes = (size_t)c.n_res * c.n_types * sizeof(int64_t);
  k1.alloc_in_smem = alloc_bytes <= (size_t)(128 << 10) ? 1 : 0;
  size_t smem = sizeof(ksched_template) * c.n_templates + sizeof(ksched_keyinfo) * KSCHED_MAX_KEYS + (k1.alloc_in_smem ? alloc_bytes : 0) +
                sizeof(int16_t) * KSCHED_MAX_KEYS * 64 + sizeof(int16_t) * 64;
  k1.n_valrows = h->n_valrows;
  k1.n_offrows = h->n_offrows;
  const size_t table_bytes = (size_t)(h->n_valrows + 2 * c.n_keys + h->n_offrows + 1 + c.n_templates) * c.W32 * sizeof(uint32_t);
  k1.tables_in_smem = smem + table_bytes <= (size_t)(160 << 10) ? 1 : 0;
  if (k1.tables_in_smem) smem += table_bytes;
  // one warp per class row (a row evaluation is ~10k cycles of dependent work: no chunking)
  const int warps_per_block = kK1Threads / 32;
  const int blocks = std::max(1, std::min(148 * 2, (h->n_classes + warps_per_block - 1) / warps_per_block));
  k1.dbg = nullptr;
#ifdef KSCHED_PROFILE_K1
  CUDA_TRY(h, h->d_k1dbg.ensure(8));
  CUDA_TRY(h, cudaMemsetAsync(h->d_k1dbg.ptr, 0, 8 * sizeof(long long), h->stream));
  k1.dbg = h->d_k1dbg.ptr;
#endif
  {
    std::lock_guard<std::mutex> lock(g_k1_mu);  // one __constant__ parameter block per device: see run_pack
    if (h->device < 0 || h->device >= 64) { h->err = "device ordinal out of range"; return KSCHED_ERR_INVALID; }
    cudaEvent_t& done = g_k1_done[h->device];
    if (!done) CUDA_TRY(h, cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
    CUDA_TRY(h, cudaStreamWaitEvent(h->stream, done, 0));
    h->k1_host = k1;
    CUDA_TRY(h, cudaMemcpyToSymbolAsync(g_k1, &h->k1_host, sizeof(K1Params), 0, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaFuncSetAttribute(class_feasibility_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  // per function: under the launch lock
    if (h->world > 1)  // column words of the other shards read as 0
      CUDA_TRY(h, cudaMemsetAsync(h->d_Fclass.ptr, 0, (size_t)std::max(h->n_classes, 1) * c.n_templates * c.W32 * 4, h->stream));
    class_feasibility_kernel<<<blocks, kK1Threads, smem, h->stream>>>();
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaEventRecord(done, h->stream));
  }
#ifdef KSCHED_PROFILE_K1
  {
    long long dbg[8];
    cudaMemcpyAsync(dbg, h->d_k1dbg.ptr, sizeof dbg, cudaMemcpyDeviceToHost, h->stream);
    cudaStreamSynchronize(h->stream);
    fprintf(stderr, "[k1 profile] blocks=%d max cycles: stage=%lld compute=%lld total=%lld max_computes_per_warp=%lld | total computes=%lld avg compute cycles=%lld\n",
            blocks, dbg[0], dbg[1], dbg[2], dbg[3], dbg[4], dbg[4] ? dbg[5] / dbg[4] : 0);
  }
#endif
  return KSCHED_OK;
}

// K1 proper: the dense pods x (template, instance type) matrix and the per-pod best column, streamed from the class rows.
static int run_feasibility(ksched_handle* h) {
  if (h->n_pods == 0) return KSCHED_OK;
  const int RW = h->cat.n_templates * h->cat.W32;
  const int nblk = (h->n_pods + 31) / 32;
  const int blocks = std::max(1, std::min(148 * 8, (nblk + 7) / 8));  // 8 warps per CTA, one 32-row block per warp and iteration
  feasibility_kernel<<<blocks, 256, 0, h->stream>>>(h->d_rows.ptr, h->n_pods, h->n_classes, RW, h->d_Fclass.ptr, h->d_best_class.ptr, h->d_F.ptr,
                                                    h->d_best.ptr);
  CUDA_TRY(h, cudaGetLastError());
  h->tm.feasibility_launches = 2;
  const long long C = (long long)h->cat.n_templates * h->cat.n_types;
  h->tm.feasibility_bytes = (long long)h->n_pods * 256 + C * 256 + (long long)h->n_pods * C / 8;
  return KSCHED_OK;
}

// Every array a Solve mutates goes back to its pristine copy (or to zero) in ONE launch: a table of (dst, src, bytes)
// segments passed by value. (Round 1 issued ~20 cudaMemcpyAsync / cudaMemsetAsync calls per Solve; a consolidation
// simulation is so short that those launches were most of it.)
struct ResetSeg { void* dst; const void* src; unsigned long long bytes; };
struct ResetTable { int n; ResetSeg seg[30]; };
__global__ void reset_kernel(ResetTable t) {
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (size_t)gridDim.x * blockDim.x;
  for (int q = 0; q < t.n; ++q) {
    const ResetSeg sg = t.seg[q];
    const size_t n16 = sg.bytes / 16;
    uint4* d = static_cast<uint4*>(sg.dst);
    const uint4* sv = static_cast<const uint4*>(sg.src);
    for (size_t i = tid; i < n16; i += nth) d[i] = sv ? sv[i] : make_uint4(0, 0, 0, 0);
    unsigned char* db = static_cast<unsigned char*>(sg.dst);
    const unsigned char* sb = static_cast<const unsigned char*>(sg.src);
    for (size_t i = n16 * 16 + tid; i < sg.bytes; i += nth) db[i] = sb ? sb[i] : 0;
  }
}

static int reset_state(ksched_handle* h, const int64_t* d_remaining_src = nullptr, void* also_zero = nullptr, size_t also_zero_bytes = 0) {
  const int P = h->n_pods, NE = std::max(h->n_existing, 1), NG = std::max(h->n_groups, 1);
  CUDA_TRY(h, h->d_cls_cursor.ensure((size_t)std::max(h->n_classes, 1)));
  ResetTable t{};
  auto add = [&](void* dst, const void* src, size_t bytes) { if (bytes) t.seg[t.n++] = ResetSeg{dst, src, (unsigned long long)bytes}; };
  add(h->d_pod_class.ptr, h->d_pod_class0.ptr, (size_t)P * 4);
  add(h->d_relax.ptr, nullptr, (size_t)std::max(P, 1) * 4);
  add(h->d_ex_req.ptr, h->d_ex_req0.ptr, (size_t)8 * NE * 8);
  add(h->d_ex_req_present.ptr, h->d_ex_req_present0.ptr, (size_t)NE * 4);
  add(h->d_ex_vals.ptr, h->d_ex_vals0.ptr, (size_t)16 * NE * 8);
  add(h->d_ex_meta.ptr, h->d_ex_meta0.ptr, (size_t)NE * 8);
  add(h->d_ex_hp.ptr, h->d_ex_hp0.ptr, (size_t)NE * 8);
  add(h->d_ex_closed.ptr, nullptr, (size_t)NE);
  add(h->d_cls_cursor.ptr, nullptr, (size_t)std::max(h->n_classes, 1) * 4);
  if (h->have_volumes) add(h->d_ex_vol.ptr, h->d_ex_vol0.ptr, (size_t)h->n_existing * sizeof(ksched_node_volumes));
  add(h->d_grp_cnt.ptr, h->d_grp_cnt0.ptr, (size_t)NG * 64 * 4);
  add(h->d_grp_registered.ptr, h->d_grp_registered0.ptr, (size_t)NG * 8);
  add(h->d_grp_host_total.ptr, h->d_grp_host_total0.ptr, (size_t)NG * 4);
  add(h->d_grp_active.ptr, h->d_grp_active0.ptr, (size_t)NG);
  add(h->d_grp_min_slot.ptr, nullptr, (size_t)NG * 4);
  const size_t hs = (size_t)std::max(h->n_hostgroups, 1) * ((size_t)h->n_existing + h->max_new);
  add(h->d_grp_host.ptr, h->d_grp_host0.ptr, hs * 2);
  if (d_remaining_src)  // simulation on the cluster snapshot: limits with the removed nodes' capacity given back, already on the device
    add(h->d_remaining.ptr, d_remaining_src, (size_t)h->cat.n_templates * KSCHED_MAX_RES * 8);
  add(h->d_counters.ptr, nullptr, 80 * sizeof(long long));
  add(h->d_fc_state.ptr, nullptr, (size_t)std::max(h->n_classes, 1) * h->cat.n_templates);
  add(h->d_fc_front_state.ptr, nullptr, (size_t)std::max(h->n_classes, 1) * h->cat.n_templates);
  add(h->d_fd_state.ptr, nullptr, (size_t)kFreshMemoSlots);
  add(also_zero, nullptr, also_zero_bytes);
  if (!d_remaining_src) {
    std::vector<int64_t> rem((size_t)h->cat.n_templates * KSCHED_MAX_RES);
    for (int v = 0; v < h->cat.n_templates; ++v)
      for (int r = 0; r < KSCHED_MAX_RES; ++r) rem[(size_t)v * KSCHED_MAX_RES + r] = h->h_templates[v].remaining[r];
    CUDA_TRY(h, cudaMemcpyAsync(h->d_remaining.ptr, rem.data(), rem.size() * 8, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));  // rem is a stack vector
  }
  reset_kernel<<<148 * 2, 256, 0, h->stream>>>(t);
  CUDA_TRY(h, cudaGetLastError());
  return KSCHED_OK;
}

// g_k2 is one __constant__ object per device: a launch may only overwrite it after the previous pack kernel on that
// device (possibly of another handle, on another stream) has finished. Ordered on the device, never on the host.
static std::mutex g_k2_mu;
static cudaEvent_t g_k2_done[64] = {};

static int run_pack(ksched_handle* h) {
  K2Params& k2 = h->k2_host;
  k2.cat = h->cat;
  PackState& s = k2.st;
  s.relx = h->d_relx.ptr;
  s.classes = h->d_classes.ptr; s.groups = h->d_groups.ptr; s.class_topo = h->d_class_topo.ptr; s.filter_terms = h->d_filter_terms.ptr;
  s.itype_sets = h->d_itype_sets.ptr; s.itype_complement = h->d_itype_comp.ptr; s.hostname_reqs = h->d_hostname_reqs.ptr;
  s.order = h->d_order.ptr; s.rows = h->d_rows.ptr; s.F = h->d_F.ptr; s.best = h->d_best.ptr;
  s.pod_pos = h->d_pod_pos.ptr; s.use_F = h->world == 1 ? 1 : 0;
  s.n_pods = h->n_pods; s.n_classes = h->n_classes; s.n_existing = h->n_existing; s.n_groups = h->n_groups; s.max_new = h->max_new;
  for (int r = 0; r < KSCHED_MAX_RES; ++r) s.min_req[r] = h->min_req[r];
  s.pod_class = h->d_pod_class.ptr; s.relax_level = h->d_relax.ptr; s.assign = h->d_assign.ptr; s.place_seq = h->d_place_seq.ptr;
  s.queue = h->d_queue.ptr; s.last_len = h->d_last_len.ptr; s.last_epoch = h->d_last_epoch.ptr;
  s.ex_req = h->d_ex_req.ptr; s.ex_avail = h->d_ex_avail.ptr; s.ex_req_present = h->d_ex_req_present.ptr; s.ex_avail_present = h->d_ex_avail_present.ptr;
  s.ex_vals = h->d_ex_vals.ptr; s.ex_meta = h->d_ex_meta.ptr; s.ex_taintset = h->d_ex_taintset.ptr; s.ex_itype = h->d_ex_itype.ptr;
  s.ex_hp = h->d_ex_hp.ptr; s.ex_closed = h->d_ex_closed.ptr;
  s.cls_cursor = h->d_cls_cursor.ptr;
  s.cls_vol = h->have_volumes ? h->d_cls_vol.ptr : nullptr; s.ex_vol = h->have_volumes ? h->d_ex_vol.ptr : nullptr;
  for (int d = 0; d < KSCHED_MAX_VOLUME_DRIVERS; ++d) s.vol_mask[d] = h->vol_mask[d];
  s.nn_tmpl = h->d_nn_tmpl.ptr; s.nn_count = h->d_nn_count.ptr; s.nn_tb = h->d_nn_tb.ptr; s.nn_req = h->d_nn_req.ptr;
  s.nn_req_present = h->d_nn_req_present.ptr;
  s.nn_vals = h->d_nn_vals.ptr; s.nn_meta = h->d_nn_meta.ptr; s.nn_opts = h->d_nn_opts.ptr; s.nn_hp = h->d_nn_hp.ptr;
  s.ov_key = h->d_ov_key.ptr; s.ov_q = h->d_ov_q.ptr; s.ov_bound = h->d_ov_bound.ptr; s.ov_bound2 = h->d_ov_bound2.ptr; s.ov_node = h->d_ov_node.ptr; s.ov_flags = h->d_ov_flags.ptr;
  s.fc_state = h->d_fc_state.ptr; s.fc_opts = h->d_fc_opts.ptr; s.fc_bound = h->d_fc_bound.ptr; s.fc_bound2 = h->d_fc_bound2.ptr; s.fc_dom = h->d_fc_dom.ptr; s.fc_front_state = h->d_fc_front_state.ptr;
  s.fc_vals = h->d_fc_vals.ptr; s.fc_meta = h->d_fc_meta.ptr; s.fc_q = h->d_fc_q.ptr; s.fc_qp = h->d_fc_qp.ptr;
  s.ov_absorbed = h->d_ov_absorbed.ptr; s.ov_rejected = h->d_ov_rejected.ptr;
  s.fd_cap = kFreshMemoSlots; s.fd_state = h->d_fd_state.ptr; s.fd_fc = h->d_fd_fc.ptr; s.fd_meta = h->d_fd_meta.ptr; s.fd_vals = h->d_fd_vals.ptr;
  s.fd_opts = h->d_fd_opts.ptr; s.fd_bound = h->d_fd_bound.ptr; s.fd_bound2 = h->d_fd_bound2.ptr; s.fd_dom = h->d_fd_dom.ptr;
  s.count_visited = h->count_visited;
  s.stop_new_nodes = h->stop_new_nodes;
  s.grp_cnt = h->d_grp_cnt.ptr; s.grp_registered = h->d_grp_registered.ptr; s.grp_host = h->d_grp_host.ptr;
  s.grp_host_row = h->d_grp_host_row.ptr; s.grp_host_total = h->d_grp_host_total.ptr; s.remaining = h->d_remaining.ptr;
  s.grp_active = h->d_grp_active.ptr; s.grp_min_slot = h->d_grp_min_slot.ptr;
  s.counters = h->d_counters.ptr;
  const size_t alloc_bytes = (size_t)h->cat.n_res * h->cat.n_types * sizeof(int64_t);
  // 227 KB per CTA on sm_100a: the hot node window + ~4 KB of static shared memory come first
  const size_t static_smem = (size_t)(14 << 10);  // file-scope __shared__ objects (pod row, PodTopo, RunCtx with its variants, scratch)
  const size_t smem_left = (size_t)(227 << 10) - sizeof(HotSmem) - kRunArrayBytes - static_smem;
  s.alloc_in_smem = alloc_bytes <= smem_left ? 1 : 0;
  s.run_off = s.alloc_in_smem ? (int)((alloc_bytes + 15) & ~(size_t)15) : 0;
  const size_t smem = sizeof(HotSmem) + (size_t)s.run_off + kRunArrayBytes;
  s.any_limits = 0;
  for (const ksched_template& tm : h->h_templates) if (tm.has_limits && tm.limit_present) s.any_limits = 1;
  s.use_warp_loop = getenv("KSCHED_WARPLOOP") ? 1 : 0;  // superseded by the class-run loop (kept for A/B timing: 18 ms vs 8 ms on C2 when both are on)
  s.use_class_run = getenv("KSCHED_NO_CLASSRUN") ? 0 : 1;
  s.use_level_step = std::getenv("KSCHED_NO_LEVELSTEP") ? 0 : 1;
  s.use_level_run = std::getenv("KSCHED_NO_LEVELRUN") ? 0 : 1;
  s.use_mask_run = std::getenv("KSCHED_NO_MASKRUN") ? 0 : 1;
  s.use_level_warp = std::getenv("KSCHED_NO_LEVELWARP") ? 0 : 1;
  // block size: the chain is latency-bound on ONE thread's commit; more warps only help when there are many candidate
  // nodes to examine per pod (existing nodes, large in-flight sets)
  int threads = h->n_existing >= 2048 ? kPackThreads : (h->n_existing >= 256 ? 256 : 128);
  if (const char* e = getenv("KSCHED_PACK_THREADS")) { int v = atoi(e); if (v >= 32 && v <= kPackThreads && v % 32 == 0) threads = v; }
  {
    std::lock_guard<std::mutex> lock(g_k2_mu);
    if (h->device < 0 || h->device >= 64) { h->err = "device ordinal out of range"; return KSCHED_ERR_INVALID; }
    cudaEvent_t& done = g_k2_done[h->device];
    if (!done) CUDA_TRY(h, cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
    CUDA_TRY(h, cudaStreamWaitEvent(h->stream, done, 0));  // no-op for an event that was never recorded
    CUDA_TRY(h, cudaMemcpyToSymbolAsync(g_k2, &k2, sizeof(K2Params), 0, cudaMemcpyHostToDevice, h->stream));
    // the attribute belongs to the function, not to the handle: set it under the same lock as the launch
    CUDA_TRY(h, cudaFuncSetAttribute(pack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    pack_kernel<<<1, threads, smem, h->stream>>>();
    CUDA_TRY(h, cudaGetLastError());
    CUDA_TRY(h, cudaEventRecord(done, h->stream));
  }
  finalize_options_kernel<<<148, 256, 0, h->stream>>>(h->cat, h->d_counters.ptr, h->d_nn_req.ptr, h->d_nn_req_present.ptr, h->d_nn_opts.ptr, h->max_new);
  h->tm.pack_launches = 2;
  return KSCHED_OK;
}

static int flush_l2(ksched_handle* h) {
  const size_t n = (size_t)64 << 20;  // 256 MiB of u32 > 126 MB L2
  CUDA_TRY(h, h->d_flush.ensure(n));
  flush_kernel<<<148 * 4, 512, 0, h->stream>>>(h->d_flush.ptr, n);
  return KSCHED_OK;
}

static float ev_us(cudaEvent_t a, cudaEvent_t b) {
  float ms = 0;
  cudaEventElapsedTime(&ms, a, b);
  return ms * 1000.f;
}

int ksched_run_resident(ksched_handle* h, int do_flush) {
  if (!h || !h->uploaded) return KSCHED_ERR_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  int rc;
  if ((rc = reset_state(h)) != KSCHED_OK) return rc;
  if (do_flush && (rc = flush_l2(h)) != KSCHED_OK) return rc;
  CUDA_TRY(h, cudaEventRecord(h->ev[0], h->stream));
  if ((rc = run_sort(h)) != KSCHED_OK) return rc;
  CUDA_TRY(h, cudaEventRecord(h->ev[1], h->stream));
  if ((rc = run_class_feasibility(h)) != KSCHED_OK) return rc;
  if ((rc = run_feasibility(h)) != KSCHED_OK) return rc;
  CUDA_TRY(h, cudaEventRecord(h->ev[2], h->stream));
  h->tm.allreduce_us = 0;
  if (h->world > 1 && h->comm) {
    ncclResult_t r = ncclAllReduce(h->d_best.ptr, h->d_best.ptr, (size_t)h->n_pods, ncclUint64, ncclMin, h->comm, h->stream);
    if (r != ncclSuccess) { h->err = std::string("ncclAllReduce: ") + ncclGetErrorString(r); return KSCHED_ERR_NCCL; }
  }
  CUDA_TRY(h, cudaEventRecord(h->ev[3], h->stream));
  if ((rc = run_pack(h)) != KSCHED_OK) return rc;
  CUDA_TRY(h, cudaEventRecord(h->ev[4], h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  CUDA_TRY(h, cudaGetLastError());
  h->tm.sort_us = ev_us(h->ev[0], h->ev[1]);
  h->tm.feasibility_us = ev_us(h->ev[1], h->ev[2]);
  h->tm.allreduce_us = ev_us(h->ev[2], h->ev[3]);
  h->tm.pack_us = ev_us(h->ev[3], h->ev[4]);
  h->tm.total_us = ev_us(h->ev[0], h->ev[4]);
  return KSCHED_OK;
}

int ksched_run_feasibility_only(ksched_handle* h, int do_flush, float* elapsed_us) {
  if (!h || !h->uploaded) return KSCHED_ERR_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  int rc;
  if (!h->sorted) {  // K0 first: the kernel streams the FFD-ordered pod-row matrix
    CUDA_TRY(h, cudaMemcpyAsync(h->d_pod_class.ptr, h->d_pod_class0.ptr, (size_t)h->n_pods * 4, cudaMemcpyDeviceToDevice, h->stream));
    if ((rc = run_sort(h)) != KSCHED_OK) return rc;
  }
  CUDA_TRY(h, cudaEventRecord(h->ev[7], h->stream));
  if ((rc = run_class_feasibility(h)) != KSCHED_OK) return rc;  // n_classes row evaluations (timed on their own)
  if (do_flush && (rc = flush_l2(h)) != KSCHED_OK) return rc;
  CUDA_TRY(h, cudaEventRecord(h->ev[5], h->stream));
  if ((rc = run_feasibility(h)) != KSCHED_OK) return rc;
  CUDA_TRY(h, cudaEventRecord(h->ev[6], h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  CUDA_TRY(h, cudaGetLastError());
  if (elapsed_us) *elapsed_us = ev_us(h->ev[5], h->ev[6]);
  h->tm.feasibility_us = ev_us(h->ev[5], h->ev[6]);
  h->tm.class_feasibility_us = ev_us(h->ev[7], h->ev[5]);  // includes the L2 flush when one was asked for
  return KSCHED_OK;
}

#ifdef KSCHED_PROFILE_PACK
static void print_pack_profile(const long long* counters) {
  fprintf(stderr, "[pack profile] generic: topo=%lld existing=%lld eval=%lld commit=%lld fresh=%lld fail=%lld | fastblock=%lld genericcall=%lld | "
                  "n_generic=%lld inflight_placed=%lld fresh_steps=%lld failures=%lld paths[rej,cached,row,dyn,cachedempty]=%lld,%lld,%lld,%lld,%lld steps=%lld\n",
          counters[8], counters[9], counters[10], counters[11], counters[12], counters[13], counters[14], counters[15], counters[17], counters[18],
          counters[19], counters[20], counters[21], counters[22], counters[23], counters[24], counters[25], counters[5]);
  fprintf(stderr, "[pack profile] fresh: decide=%lld words=%lld commit=%lld rest=%lld | in-flight verify=%lld\n", counters[26], counters[27], counters[28],
          counters[12], counters[29]);
  fprintf(stderr, "[pack profile] in-flight commit: winner+barrier=%lld record=%lld rest=%lld\n", counters[30], counters[31], counters[11]);
  fprintf(stderr, "[pack profile] class_run: calls=%lld pods=%lld bails=%lld ineligible=%lld cycles=%lld\n", counters[40], counters[41], counters[42], counters[43],
          counters[14]);
  fprintf(stderr, "[pack profile] mask run steps=%lld with >1 admissible domain=%lld round-able=%lld (counters shared with generic n/fresh: ignore there)\n", counters[18], counters[19], counters[17]);
  fprintf(stderr, "[pack profile] mask run: build cycles=%lld (refused %lld) loop cycles=%lld pods=%lld entries=%lld\n", counters[38], counters[47], counters[6], counters[7], counters[16]);
  fprintf(stderr, "[pack profile] class_run without mask-key spread: cycles=%lld pods=%lld level+fill iterations=%lld (fill %lld) fresh=%lld per-pod=%lld | with: cycles=%lld pods=%lld fresh=%lld per-pod=%lld\n",
          counters[32], counters[33], counters[34], counters[46], counters[35], counters[44], counters[36], counters[37], counters[39], counters[45]);
  static const char* kinds[6] = {"round pinned", "round fresh", "round unpinned", "single pinned", "single pin", "single fresh"};
  for (int k = 0; k < 6; ++k)
    fprintf(stderr, "[pack profile] mask run %-14s: iterations=%lld pods=%lld cycles=%lld\n", kinds[k], counters[48 + 3 * k], counters[49 + 3 * k],
            counters[50 + 3 * k]);
  fprintf(stderr, "[pack profile] mask run declined rounds: na<=1=%lld staged<na=%lld unpinned-first=%lld room-slow=%lld level=%lld no-fresh=%lld "
                  "unpinned-few=%lld unpinned-pin=%lld\n",
          counters[66], counters[67], counters[68], counters[69], counters[70], counters[71], counters[72], counters[73]);
}
#endif

int ksched_download(ksched_handle* h, const ksched_problem* pb, ksched_result* res) {
  if (!h || !pb || !res || !h->uploaded) return KSCHED_ERR_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  const int P = h->n_pods, NE = h->n_existing, MAXN = h->max_new, W32 = h->cat.W32, W64 = h->W64, V = h->cat.n_templates;
  long long counters[80];
  CUDA_TRY(h, cudaMemcpyAsync(counters, h->d_counters.ptr, sizeof counters, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
#ifdef KSCHED_PROFILE_PACK
  print_pack_profile(counters);
#endif
  if (counters[4] != 0) {
    h->err = counters[4] == KSCHED_ERR_OVERFLOW ? "new-node capacity exceeded" : "a pod is constrained by more topology groups than the kernel supports";
    return (int)counters[4];
  }
  const int n_new = (int)counters[0];
  h->tm.d2h_bytes = (int64_t)sizeof counters + (int64_t)P * 4 * ((res->assign != nullptr) + (res->relax_level != nullptr) + (res->place_seq != nullptr)) +
                    (int64_t)n_new * (1 + 4 + 4 + 8 + 64 + 128 + (int64_t)W32 * 4) + (res->existing_reqs ? (int64_t)NE * 136 : 0) +
                    (res->launch ? (int64_t)n_new * (int64_t)sizeof(ksched_launch_choice) : 0) +
                    (res->feasibility ? (int64_t)P * V * W32 * 4 + (int64_t)P * 4 : 0) + (res->best_column ? (int64_t)P * 12 : 0);
  res->n_new_nodes = n_new;
  res->n_unscheduled = (int)counters[1];
  res->nodes_visited = counters[2];
  res->add_calls = counters[3];
  h->tm.pack_steps = counters[5];
  if (res->assign) CUDA_TRY(h, cudaMemcpyAsync(res->assign, h->d_assign.ptr, (size_t)P * 4, cudaMemcpyDeviceToHost, h->stream));
  if (res->relax_level) CUDA_TRY(h, cudaMemcpyAsync(res->relax_level, h->d_relax.ptr, (size_t)P * 4, cudaMemcpyDeviceToHost, h->stream));
  if (res->place_seq) CUDA_TRY(h, cudaMemcpyAsync(res->place_seq, h->d_place_seq.ptr, (size_t)P * 4, cudaMemcpyDeviceToHost, h->stream));
  if (n_new > 0 && res->new_nodes && res->new_node_types) {
    std::vector<uint8_t> tmpl(n_new);
    std::vector<int32_t> count(n_new);
    std::vector<int64_t> req((size_t)8 * n_new);
    std::vector<uint32_t> reqp(n_new), opts((size_t)W32 * n_new);
    std::vector<uint64_t> vals((size_t)16 * n_new), meta(n_new);
    CUDA_TRY(h, cudaMemcpyAsync(tmpl.data(), h->d_nn_tmpl.ptr, n_new, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(count.data(), h->d_nn_count.ptr, (size_t)n_new * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(reqp.data(), h->d_nn_req_present.ptr, (size_t)n_new * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(meta.data(), h->d_nn_meta.ptr, (size_t)n_new * 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpy2DAsync(req.data(), (size_t)n_new * 8, h->d_nn_req.ptr, (size_t)MAXN * 8, (size_t)n_new * 8, 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpy2DAsync(vals.data(), (size_t)n_new * 8, h->d_nn_vals.ptr, (size_t)MAXN * 8, (size_t)n_new * 8, 16, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpy2DAsync(opts.data(), (size_t)n_new * 4, h->d_nn_opts.ptr, (size_t)MAXN * 4, (size_t)n_new * 4, W32, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (int n = 0; n < n_new; ++n) {
      ksched_new_node& o = res->new_nodes[n];
      std::memset(&o, 0, sizeof o);
      o.template_index = tmpl[n];
      o.pod_count = count[n];
      o.requests_present = reqp[n];
      for (int r = 0; r < 8; ++r) o.requests[r] = req[(size_t)r * n_new + n];
      for (int k = 0; k < 16; ++k) o.reqs.values[k] = vals[(size_t)k * n_new + n];
      o.reqs.meta = meta[n];
      uint32_t* dst = reinterpret_cast<uint32_t*>(res->new_node_types + (size_t)n * W64);
      for (int w = 0; w < W32; ++w) dst[w] = opts[(size_t)w * n_new + n];
      if (W32 & 1) dst[W32] = 0;  // the row is W64 64-bit words: the caller's buffer need not be cleared
    }
  }
  if (res->launch && n_new > 0) {
    if (!h->cat.offer_keys) { h->err = "ksched_result.launch needs ksched_catalog.offering_keys"; return KSCHED_ERR_INVALID; }
    CUDA_TRY(h, h->d_launch.ensure((size_t)n_new));
    launch_choice_kernel<<<148, 256, 0, h->stream>>>(h->cat, h->d_counters.ptr, h->d_nn_vals.ptr, h->d_nn_meta.ptr, h->d_nn_opts.ptr, MAXN,
                                                     h->d_launch.ptr);
    CUDA_TRY(h, cudaMemcpyAsync(res->launch, h->d_launch.ptr, (size_t)n_new * sizeof(ksched_launch_choice), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  }
  if (res->existing_reqs && NE > 0) {
    std::vector<uint64_t> vals((size_t)16 * NE), meta(NE);
    CUDA_TRY(h, cudaMemcpyAsync(vals.data(), h->d_ex_vals.ptr, vals.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(meta.data(), h->d_ex_meta.ptr, meta.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (int e = 0; e < NE; ++e) {
      for (int k = 0; k < 16; ++k) res->existing_reqs[e].values[k] = vals[(size_t)k * NE + e];
      res->existing_reqs[e].meta = meta[e];
    }
  }
  if (res->feasibility) {
    // device rows are in FFD (queue) order; the caller gets them in its own pod order
    std::vector<uint32_t> order(P), F((size_t)P * V * W32);
    CUDA_TRY(h, cudaMemcpyAsync(order.data(), h->d_order.ptr, (size_t)P * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(F.data(), h->d_F.ptr, F.size() * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    const size_t rowb = (size_t)V * W32;
    for (int j = 0; j < P; ++j) std::memcpy(reinterpret_cast<uint32_t*>(res->feasibility) + (size_t)order[j] * rowb, &F[(size_t)j * rowb], rowb * 4);
  }
  if (res->best_column) {
    std::vector<uint32_t> order(P);
    std::vector<unsigned long long> best(P);
    CUDA_TRY(h, cudaMemcpyAsync(order.data(), h->d_order.ptr, (size_t)P * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(best.data(), h->d_best.ptr, (size_t)P * 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    for (int j = 0; j < P; ++j) res->best_column[order[j]] = best[j];
  }
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  return KSCHED_OK;
}

int ksched_solve(ksched_handle* h, const ksched_problem* pb, ksched_result* res) {
  if (!h || !pb || !res) return KSCHED_ERR_INVALID;
  auto t0 = std::chrono::steady_clock::now();
  int rc = ksched_upload(h, pb);
  if (rc != KSCHED_OK) return rc;
  auto t1 = std::chrono::steady_clock::now();
  rc = ksched_run_resident(h, 0);
  if (rc != KSCHED_OK) return rc;
  auto t2 = std::chrono::steady_clock::now();
  rc = ksched_download(h, pb, res);
  auto t3 = std::chrono::steady_clock::now();
  h->tm.upload_us = std::chrono::duration<double, std::micro>(t1 - t0).count();
  h->tm.download_us = std::chrono::duration<double, std::micro>(t3 - t2).count();
  return rc;
}

// ---- consolidation simulator on a device-resident cluster snapshot (cluster.cuh)
int ksched_load_cluster(ksched_handle* h, const ksched_cluster* cl) {
  if (!h || !cl || !cl->problem || (!cl->pod_node && cl->problem->n_pods > 0)) return KSCHED_ERR_INVALID;
  const ksched_problem* pb = cl->problem;
  h->have_cluster = false;
  const bool topo = pb->n_groups != 0;
  if (topo && (!cl->class_count_begin || !cl->node_domain || !cl->node_has_hostname_label || !cl->group_filter_match)) {
    h->err = "unsupported: a cluster with topology groups needs the counting tables of ksched_cluster";
    return KSCHED_ERR_UNSUPPORTED;
  }
  const int P = pb->n_pods, NE = pb->n_existing;
  // pods: the pending ones first, then node by node (every node's pods contiguous)
  std::vector<int32_t> first((size_t)std::max(NE, 1), -1), count((size_t)std::max(NE, 1), 0);
  int pending = 0;
  for (int i = 0; i < P; ++i) {
    const int nd = cl->pod_node[i];
    if (nd >= NE) { h->err = "pod_node out of range"; return KSCHED_ERR_INVALID; }
    if (nd < 0) { if (i != pending) { h->err = "pending pods must come first"; return KSCHED_ERR_INVALID; } ++pending; continue; }
    if (first[nd] < 0) first[nd] = i;
    else if (cl->pod_node[i - 1] != nd) { h->err = "the pods of one node must be contiguous"; return KSCHED_ERR_INVALID; }
    ++count[nd];
  }
  int rc = ksched_upload(h, pb);  // the superset problem: buffers sized for the largest batch, existing-node state, class tables
  if (rc != KSCHED_OK) return rc;
  CUDA_TRY(h, upload(h, h->d_sup_pod_node, cl->pod_node, (size_t)P));
  CUDA_TRY(h, upload(h, h->d_sup_class, pb->pod_class, (size_t)P));
  CUDA_TRY(h, upload(h, h->d_sup_ts, pb->pod_timestamp, (size_t)P));
  CUDA_TRY(h, upload(h, h->d_sup_uid, pb->pod_uid_rank, (size_t)P));
  CUDA_TRY(h, upload_vec(h, h->d_node_first, first));
  CUDA_TRY(h, h->d_node_dst.ensure((size_t)std::max(NE, 1)));
  CUDA_TRY(h, h->d_in_set.ensure((size_t)std::max(NE, 1)));
  CUDA_TRY(h, h->d_pod_src.ensure((size_t)std::max(P, 1)));
  h->cluster_topology = topo;
  if (topo) {
    const int NC = pb->n_classes, NK = h->cat.n_keys;
    h->filt_words = (NE + 31) / 32;
    const uint32_t n_rel = cl->class_count_begin[NC];
    for (uint32_t q = 0; q < n_rel; ++q)
      if (cl->class_count[q].group >= (uint32_t)pb->n_groups) { h->err = "class_count group out of range"; return KSCHED_ERR_INVALID; }
    CUDA_TRY(h, upload(h, h->d_cc_begin, cl->class_count_begin, (size_t)NC + 1));
    CUDA_TRY(h, upload(h, h->d_cc, cl->class_count, (size_t)std::max<uint32_t>(n_rel, 1)));
    CUDA_TRY(h, upload(h, h->d_node_dom, cl->node_domain, (size_t)std::max(NK, 1) * std::max(NE, 1)));
    CUDA_TRY(h, upload(h, h->d_node_hostlabel, cl->node_has_hostname_label, (size_t)std::max(NE, 1)));
    CUDA_TRY(h, upload(h, h->d_filt, cl->group_filter_match, (size_t)pb->n_groups * std::max(h->filt_words, 1)));
  }
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  h->h_node_first.swap(first);
  h->h_node_count.swap(count);
  h->sup_pods = P;
  h->sup_pending = pending;
  h->have_cluster = true;
  return KSCHED_OK;
}

int ksched_simulate_batch(ksched_handle* h, const ksched_candidate_set* sets, int n_sets, ksched_sim_result* results, uint64_t* node0_types) {
  if (!h || !sets || n_sets < 0 || (n_sets > 0 && !results)) return KSCHED_ERR_INVALID;
  if (!h->have_cluster) { h->err = "ksched_load_cluster must be called first"; return KSCHED_ERR_INVALID; }
  if (n_sets == 0) return KSCHED_OK;
  CUDA_TRY(h, cudaSetDevice(h->device));
  const int NE = h->n_existing, V = h->cat.n_templates, W32 = h->cat.W32, W64 = h->W64;
  // stage every set's node list, per-node batch offsets and limits in one upload each
  std::vector<int32_t> all_nodes, all_dst((size_t)n_sets * std::max(NE, 1), 0), batch((size_t)n_sets, 0), node_off((size_t)n_sets + 1, 0);
  std::vector<int64_t> all_rem((size_t)n_sets * V * KSCHED_MAX_RES, 0);
  std::vector<uint8_t> seen((size_t)std::max(NE, 1), 0);
  for (int q = 0; q < n_sets; ++q) {
    const ksched_candidate_set& cs = sets[q];
    if (cs.n_nodes < 0 || (cs.n_nodes > 0 && !cs.nodes)) { h->err = "bad candidate set"; return KSCHED_ERR_INVALID; }
    std::vector<int32_t> nodes(cs.nodes, cs.nodes + cs.n_nodes);
    std::sort(nodes.begin(), nodes.end());  // the batch lists the removed nodes' pods in slot order (the queue sorts them anyway, queue.go:35-110)
    int pos = h->sup_pending;
    for (size_t i = 0; i < nodes.size(); ++i) {
      const int nd = nodes[i];
      if (nd < 0 || nd >= NE || (i > 0 && nodes[i - 1] == nd)) { h->err = "candidate set: existing slot out of range or repeated"; return KSCHED_ERR_INVALID; }
      all_dst[(size_t)q * NE + nd] = pos;
      pos += h->h_node_count[(size_t)nd];
    }
    batch[(size_t)q] = pos;
    all_nodes.insert(all_nodes.end(), nodes.begin(), nodes.end());
    node_off[(size_t)q + 1] = (int32_t)all_nodes.size();
    for (int v = 0; v < V; ++v)
      for (int r = 0; r < KSCHED_MAX_RES; ++r)
        all_rem[((size_t)q * V + v) * KSCHED_MAX_RES + r] = cs.remaining ? cs.remaining[(size_t)v * KSCHED_MAX_RES + r] : h->h_templates[(size_t)v].remaining[r];
  }
  (void)seen;
  if (all_nodes.empty()) all_nodes.push_back(0);
  CUDA_TRY(h, upload_vec(h, h->d_set_nodes, all_nodes));
  CUDA_TRY(h, upload_vec(h, h->d_node_dst, all_dst));
  CUDA_TRY(h, upload_vec(h, h->d_sim_remaining, all_rem));
  CUDA_TRY(h, h->d_sim_results.ensure((size_t)n_sets));
  CUDA_TRY(h, h->d_sim_types.ensure((size_t)n_sets * W32));
  CUDA_TRY(h, cudaEventRecord(h->ev[0], h->stream));
  int rc = KSCHED_OK;
  // nothing computeConsolidation can return depends on what happens after a second new node is opened
  // (consolidation.go:214-224: len(newNodes) != 1 -> do nothing): the simulation stops there
  h->stop_new_nodes = 2;
  for (int q = 0; q < n_sets && rc == KSCHED_OK; ++q) {
    const int n_nodes = node_off[(size_t)q + 1] - node_off[(size_t)q];
    h->n_pods = batch[(size_t)q];
    rc = reset_state(h, h->d_sim_remaining.ptr + (size_t)q * V * KSCHED_MAX_RES, h->d_in_set.ptr, (size_t)std::max(NE, 1));
    if (rc != KSCHED_OK) break;
    if (n_nodes > 0)
      cluster_mark_kernel<<<(n_nodes + 255) / 256, 256, 0, h->stream>>>(h->d_set_nodes.ptr + node_off[(size_t)q], n_nodes, h->d_in_set.ptr, h->d_ex_closed.ptr);
    if (h->sup_pods > 0)
      cluster_select_kernel<<<(h->sup_pods + 255) / 256, 256, 0, h->stream>>>(h->sup_pods, h->d_sup_pod_node.ptr, h->d_in_set.ptr, h->d_node_dst.ptr + (size_t)q * NE,
                                                                              h->d_node_first.ptr, h->sup_pending, h->d_sup_class.ptr, h->d_sup_ts.ptr, h->d_sup_uid.ptr,
                                                                              h->d_pod_class0.ptr, h->d_ts.ptr, h->d_uid_rank.ptr, h->d_pod_src.ptr);
    if (h->cluster_topology && h->sup_pods > 0)
      cluster_topology_kernel<<<(h->sup_pods + 255) / 256, 256, 0, h->stream>>>(
          h->sup_pods, h->d_sup_pod_node.ptr, h->d_in_set.ptr, h->d_sup_class.ptr, h->d_cc_begin.ptr, h->d_cc.ptr, h->d_groups.ptr, h->d_node_dom.ptr,
          h->d_node_hostlabel.ptr, h->d_filt.ptr, h->filt_words, NE, NE + h->max_new, h->d_grp_host_row.ptr, h->d_grp_cnt.ptr,
          reinterpret_cast<unsigned long long*>(h->d_grp_registered.ptr), h->d_grp_host.ptr, h->d_grp_host_total.ptr);
    // the working copy of the pod classes (reset_state copied the previous batch's): refresh it from the new batch
    if (h->n_pods > 0) CUDA_TRY(h, cudaMemcpyAsync(h->d_pod_class.ptr, h->d_pod_class0.ptr, (size_t)h->n_pods * 4, cudaMemcpyDeviceToDevice, h->stream));
    if ((rc = run_sort(h)) != KSCHED_OK) break;
    // the class rows of the feasibility matrix depend on the classes and the catalog only: once per batch
    if (q == 0 && (rc = run_class_feasibility(h)) != KSCHED_OK) break;
    if ((rc = run_feasibility(h)) != KSCHED_OK) break;
    if ((rc = run_pack(h)) != KSCHED_OK) break;
    cluster_collect_kernel<<<1, 64, 0, h->stream>>>(h->d_counters.ptr, h->n_pods, h->d_nn_tmpl.ptr, h->d_nn_count.ptr, h->d_nn_req.ptr, h->d_nn_req_present.ptr,
                                                    h->d_nn_vals.ptr, h->d_nn_meta.ptr, h->d_nn_opts.ptr, h->max_new, W32, h->d_sim_results.ptr + q,
                                                    h->d_sim_types.ptr + (size_t)q * W32);
  }
  h->n_pods = h->sup_pods;
  h->stop_new_nodes = 0;
  if (rc != KSCHED_OK) return rc;
  CUDA_TRY(h, cudaEventRecord(h->ev[4], h->stream));
#ifdef KSCHED_PROFILE_PACK
  {
    long long counters[48];
    CUDA_TRY(h, cudaMemcpyAsync(counters, h->d_counters.ptr, sizeof counters, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
    print_pack_profile(counters);  // the last simulation of the batch
  }
#endif
  std::vector<SimResultDev> dev((size_t)n_sets);
  std::vector<uint32_t> types((size_t)n_sets * W32);
  CUDA_TRY(h, cudaMemcpyAsync(dev.data(), h->d_sim_results.ptr, dev.size() * sizeof(SimResultDev), cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaMemcpyAsync(types.data(), h->d_sim_types.ptr, types.size() * 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  CUDA_TRY(h, cudaGetLastError());
  h->tm.total_us = ev_us(h->ev[0], h->ev[4]);
  for (int q = 0; q < n_sets; ++q) {
    const SimResultDev& d = dev[(size_t)q];
    ksched_sim_result& o = results[q];
    std::memset(&o, 0, sizeof o);
    o.n_pods = d.n_pods; o.n_unscheduled = d.n_unscheduled; o.n_new_nodes = d.n_new_nodes; o.error = d.error;
    if (d.n_new_nodes >= 1) {
      o.node0.template_index = d.template_index; o.node0.pod_count = d.pod_count; o.node0.requests_present = d.requests_present;
      std::memcpy(o.node0.requests, d.requests, sizeof d.requests);
      std::memcpy(o.node0.reqs.values, d.values, sizeof d.values);
      o.node0.reqs.meta = d.meta;
    }
    if (node0_types) {
      std::memset(node0_types + (size_t)q * W64, 0, (size_t)W64 * 8);
      if (d.n_new_nodes >= 1) std::memcpy(node0_types + (size_t)q * W64, &types[(size_t)q * W32], (size_t)W32 * 4);
    }
  }
  return KSCHED_OK;
}

int ksched_rank_candidates(ksched_handle* h, const ksched_rank_input* in, int32_t* order, double* cost, int32_t* n_candidates) {
  if (!h || !in || !order || !cost || !n_candidates || in->n_nodes < 0 || in->n_pods < 0) return KSCHED_ERR_INVALID;
  *n_candidates = 0;
  const int N = in->n_nodes, NP = in->n_pods;
  if (N == 0) return KSCHED_OK;
  if (!in->node_eligible || (!in->node_cost && (!in->pod_offsets || !in->node_age_seconds || !in->node_ttl_seconds ||
                                                (NP > 0 && (!in->pod_deletion_cost || !in->pod_priority || !in->pod_flags))))) return KSCHED_ERR_INVALID;
  CUDA_TRY(h, cudaSetDevice(h->device));
  CUDA_TRY(h, upload(h, h->d_rk_elig_in, in->node_eligible, (size_t)N));
  if (in->node_cost) {
    CUDA_TRY(h, upload(h, h->d_rk_cost_in, in->node_cost, (size_t)N));
  } else {
    CUDA_TRY(h, upload(h, h->d_rk_off, in->pod_offsets, (size_t)N + 1));
    CUDA_TRY(h, upload(h, h->d_rk_age, in->node_age_seconds, (size_t)N));
    CUDA_TRY(h, upload(h, h->d_rk_ttl, in->node_ttl_seconds, (size_t)N));
    if (NP > 0) {
      CUDA_TRY(h, upload(h, h->d_rk_dc, in->pod_deletion_cost, (size_t)NP));
      CUDA_TRY(h, upload(h, h->d_rk_prio, in->pod_priority, (size_t)NP));
      CUDA_TRY(h, upload(h, h->d_rk_flags, in->pod_flags, (size_t)NP));
    }
  }
  CUDA_TRY(h, h->d_rk_cost.ensure((size_t)N));
  CUDA_TRY(h, h->d_rk_cost_out.ensure((size_t)N));
  CUDA_TRY(h, h->d_rk_elig.ensure((size_t)N));
  CUDA_TRY(h, h->d_rk_order.ensure((size_t)N));
  CUDA_TRY(h, h->d_rk_n.ensure(1));
  const int blocks = (N + 255) / 256;
  rank_cost_kernel<<<blocks, 256, 0, h->stream>>>(N, h->d_rk_off.ptr, h->d_rk_dc.ptr, h->d_rk_prio.ptr, h->d_rk_flags.ptr, h->d_rk_elig_in.ptr, h->d_rk_age.ptr,
                                                  h->d_rk_ttl.ptr, in->node_cost ? h->d_rk_cost_in.ptr : nullptr, h->d_rk_cost.ptr, h->d_rk_elig.ptr);
  rank_position_kernel<<<blocks, 256, 0, h->stream>>>(N, h->d_rk_cost.ptr, h->d_rk_elig.ptr, h->d_rk_order.ptr, h->d_rk_cost_out.ptr, h->d_rk_n.ptr);
  CUDA_TRY(h, cudaGetLastError());
  int32_t n = 0;
  CUDA_TRY(h, cudaMemcpyAsync(&n, h->d_rk_n.ptr, 4, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  if (n > 0) {
    CUDA_TRY(h, cudaMemcpyAsync(order, h->d_rk_order.ptr, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaMemcpyAsync(cost, h->d_rk_cost_out.ptr, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(h, cudaStreamSynchronize(h->stream));
  }
  *n_candidates = n;
  return KSCHED_OK;
}

int ksched_get_timings(const ksched_handle* h, ksched_timings* out) {
  if (!h || !out) return KSCHED_ERR_INVALID;
  *out = h->tm;
  return KSCHED_OK;
}

}  // extern "C"
