// K2 — pack_kernel: Scheduler.add's sequential first-fit (scheduler.go:174-219) in one persistent CTA.
//
// Design (B200-first, latency-bound integer work; DESIGN.md section 4 has the long form):
//  * one CTA (128..512 threads), one pod per iteration, three speeds: a register-resident warp loop when at most 32
//    nodes are open and the pod cannot change any requirement (warp_resident_loop), a block-wide fast path over the
//    shared-memory window of open nodes, and the out-of-line generic step (existing nodes, requirement / topology
//    evaluation, fresh nodes, relaxation);
//  * candidate nodes are examined one per thread and the reference's scan order is recovered by an argmin over
//    (pod count, stable tie-break) = the position under sort.Slice(newNodes, len(Pods)<) treated as a stable sort;
//  * the state every candidate check needs (order key, request vector, Pareto front of the allocatable vectors of the
//    node's surviving instance types) lives in SHARED MEMORY for the first kActCap open nodes; everything colder
//    (requirement masks, instance-type bitsets, host ports) stays in global memory / L2;
//  * the instance-type bitset of a node is filtered LAZILY by resources: Fits() is monotone in the request vector, so
//    options_true = options_stored AND FIT(requests) and the AND is applied once, by finalize_options_kernel;
//  * generic step: cheap per-candidate filter -> block argmin -> full evaluation of the winner only -> the whole CTA
//    checks / narrows the winner's instance-type words (exclude + retry when it fails);
//  * parameters come from __constant__ memory (g_k2), the per-CTA working set is file-scope __shared__: out-of-line
//    functions reach both with immediate addresses.
#pragma once

namespace {

constexpr int kActCap = 1280;  // open in-flight nodes whose hot state is held in shared memory
constexpr int kHotRes = 4;     // resources covered by the hot request / bound vectors (cpu, memory, pods, +1)

struct HotSmem {
  unsigned long long key[kActCap];     // (pod count << 32) | biased tie-break  == position under a stable sort
  long long q[kHotRes][kActCap];       // node.Requests
  // Exact resource test without touching the option bitsets: when the Pareto front of the allocatable vectors of a
  // node's stored options has one or two members (flags bit0 "exact"; bit5 "two members"), a request vector fits some
  // option iff it fits a front member. Otherwise bound holds per-resource maxima (a necessary test only).
  long long bound[kHotRes][kActCap];
  long long bound2[kHotRes][kActCap];
  int node[kActCap];
  unsigned short flags[kActCap];       // bit0 dominant option exists; bits 1..4 request-map keys; bits 8.. template
  // Requirement verdict memo per open node, valid for topology-free pod classes without host ports:
  //  absorbed: the node's requirements already contain this class's requirements (a further pod of the class changes
  //            nothing: Compatible holds, the merge is the identity, the stored options are untouched);
  //  rejected: the last requirement / instance-type evaluation of this class against the node failed and nothing has
  //            been committed to the node since.
  unsigned absorbed[kActCap];
  unsigned rejected[kActCap];
  unsigned long long nn_last[kActCap];  // class_run: the key a tombstoned node had when it left the active set
};

struct Hot {
  HotSmem* sm;
  unsigned long long* ov_key;
  long long* ov_q;      // [kHotRes][ov_stride]
  long long* ov_bound;  // [kHotRes][ov_stride]
  long long* ov_bound2;
  int* ov_node;
  unsigned short* ov_flags;
  unsigned* ov_absorbed;
  unsigned* ov_rejected;
  int ov_stride;
  __device__ __forceinline__ unsigned long long& key(int a) const { return a < kActCap ? sm->key[a] : ov_key[a - kActCap]; }
  __device__ __forceinline__ long long& q(int r, int a) const { return a < kActCap ? sm->q[r][a] : ov_q[(size_t)r * ov_stride + (a - kActCap)]; }
  __device__ __forceinline__ long long& bound(int r, int a) const { return a < kActCap ? sm->bound[r][a] : ov_bound[(size_t)r * ov_stride + (a - kActCap)]; }
  __device__ __forceinline__ long long& bound2(int r, int a) const { return a < kActCap ? sm->bound2[r][a] : ov_bound2[(size_t)r * ov_stride + (a - kActCap)]; }
  __device__ __forceinline__ int& node(int a) const { return a < kActCap ? sm->node[a] : ov_node[a - kActCap]; }
  __device__ __forceinline__ unsigned short& flags(int a) const { return a < kActCap ? sm->flags[a] : ov_flags[a - kActCap]; }
  __device__ __forceinline__ unsigned& absorbed(int a) const { return a < kActCap ? sm->absorbed[a] : ov_absorbed[a - kActCap]; }
  __device__ __forceinline__ unsigned& rejected(int a) const { return a < kActCap ? sm->rejected[a] : ov_rejected[a - kActCap]; }
  __device__ void move(int dst, int src) const {
    key(dst) = key(src);
    for (int r = 0; r < kHotRes; ++r) { q(r, dst) = q(r, src); bound(r, dst) = bound(r, src); bound2(r, dst) = bound2(r, src); }
    node(dst) = node(src);
    flags(dst) = flags(src);
    absorbed(dst) = absorbed(src);
    rejected(dst) = rejected(src);
  }
};

__device__ __forceinline__ unsigned long long order_key(int count, int tb) {
  return ((unsigned long long)(unsigned)count << 32) | (unsigned)(tb ^ 0x80000000);
}

constexpr unsigned short kFlExact = 1, kFlTwo = 0x20;

// Pareto front (size <= 2) of the allocatable vectors of a node's stored options, or per-resource maxima when the front
// is larger. Candidates are the per-resource arg-max types (found by probing each resource's descending order); a
// candidate pair is a front iff every stored option is dominated by one of the two.
__device__ __noinline__ void compute_front(const uint32_t* opts, int stride, int n, long long* b1, long long* b2, unsigned short* bits) {
  KS_K2
  const int R = c.n_res < kHotRes ? c.n_res : kHotRes;
  const int T = c.n_types;
  int arg[kHotRes];
  for (int r = 0; r < kHotRes; ++r) { b1[r] = INT64_MIN; b2[r] = INT64_MIN; arg[r] = -1; }
  *bits = 0;
  for (int r = 0; r < R; ++r) {
    const int32_t* perm = c.perm_desc + (size_t)r * T;
    for (int i = 0; i < T; ++i) {
      const int t = perm[i];
      if ((opts[(size_t)(t >> 5) * stride + n] >> (t & 31)) & 1) { arg[r] = t; b1[r] = c.alloc_rt[(size_t)r * T + t]; break; }
    }
  }
  if (arg[0] < 0 || c.n_res > kHotRes) return;  // no option left / resources beyond the hot vectors: necessary test only
  auto dominates = [&](int a, const long long* v) {  // alloc(a) >= v in every hot resource
    for (int r = 0; r < R; ++r) if (c.alloc_rt[(size_t)r * T + a] < v[r]) return false;
    return true;
  };
  if (dominates(arg[0], b1)) { *bits = kFlExact; return; }  // one option is maximal in every resource
  // distinct candidates
  int cand[kHotRes], nc = 0;
  for (int r = 0; r < R; ++r) {
    bool seen = false;
    for (int i = 0; i < nc; ++i) seen = seen || cand[i] == arg[r];
    if (!seen) cand[nc++] = arg[r];
  }
  // which candidate pairs cover every option?  opts ⊆ domset[ci] ∪ domset[cj], word by word
  unsigned pair_ok = 0;  // bit (i*4+j), i<j
  for (int i = 0; i < nc; ++i) for (int j = i + 1; j < nc; ++j) pair_ok |= 1u << (i * 4 + j);
  const int W32 = c.W32;
  for (int w = 0; w < W32 && pair_ok; ++w) {
    const uint32_t m = opts[(size_t)w * stride + n];
    if (!m) continue;
    uint32_t d[kHotRes];
    for (int i = 0; i < nc; ++i) d[i] = c.domset[(size_t)cand[i] * W32 + w];
    for (int i = 0; i < nc; ++i) for (int j = i + 1; j < nc; ++j)
      if (m & ~(d[i] | d[j])) pair_ok &= ~(1u << (i * 4 + j));
  }
  if (!pair_ok) return;  // front larger than two: b1 keeps the per-resource maxima
  const int pi = (__ffs(pair_ok) - 1) / 4, pj = (__ffs(pair_ok) - 1) % 4;
  for (int r = 0; r < R; ++r) { b1[r] = c.alloc_rt[(size_t)r * T + cand[pi]]; b2[r] = c.alloc_rt[(size_t)r * T + cand[pj]]; }
  *bits = kFlExact | kFlTwo;
}

// 0 = no option can hold the requests, 1 = some option holds them (exact), 2 = unknown (per-resource maxima pass)
__device__ __forceinline__ int quick_fit(const long long* q, uint32_t qp, int RH, const long long* b1, const long long* b2, unsigned short fl) {
  bool f1 = true, f2 = true;
#pragma unroll
  for (int r = 0; r < kHotRes; ++r)
    if (r < RH && ((qp >> r) & 1)) { f1 = f1 && q[r] <= b1[r]; f2 = f2 && q[r] <= b2[r]; }
  if (fl & kFlExact) return (f1 || ((fl & kFlTwo) && f2)) ? 1 : 0;
  return f1 ? 2 : 0;
}
// no pod of the batch can ever fit again (min_req: per-resource minimum request over all pod classes)
__device__ __forceinline__ bool node_closed(const long long* q, const long long* min_req, int RH, const long long* b1, const long long* b2, unsigned short fl) {
  bool o1 = false, o2 = false;
#pragma unroll
  for (int r = 0; r < kHotRes; ++r)
    if (r < RH && min_req[r] > 0) { o1 = o1 || q[r] + min_req[r] > b1[r]; o2 = o2 || q[r] + min_req[r] > b2[r]; }
  return (fl & kFlTwo) ? (o1 && o2) : o1;
}

// 64-bit min over a warp with two 32-bit REDUX operations (hi word first, then lo word among the hi-minimal lanes)
__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long v) {
  const unsigned hi = (unsigned)(v >> 32), lo = (unsigned)v;
  const unsigned mhi = __reduce_min_sync(0xffffffffu, hi);
  const unsigned mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xffffffffu);
  return ((unsigned long long)mhi << 32) | mlo;
}
// single-sync block argmin (double-buffered scratch)
__device__ __forceinline__ unsigned long long block_min_u64_db(unsigned long long v, unsigned long long (*red)[32], int& parity) {
  v = warp_min_u64(v);
  if (blockDim.x == 32) return v;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned long long* buf = red[parity];
  parity ^= 1;
  if (lane == 0) buf[warp] = v;
  __syncthreads();
  const unsigned long long r = lane < (int)(blockDim.x >> 5) ? buf[lane] : ~0ull;
  return warp_min_u64(r);
}

// two independent u32 minima with one barrier (double-buffered scratch, same protocol as block_min_u64_db)
__device__ __forceinline__ void block_min2_u32_db(unsigned a, unsigned b, unsigned long long (*red)[32], int& parity, unsigned* ra, unsigned* rb) {
  a = __reduce_min_sync(0xffffffffu, a);
  b = __reduce_min_sync(0xffffffffu, b);
  if (blockDim.x == 32) { *ra = a; *rb = b; return; }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned long long* buf = red[parity];
  parity ^= 1;
  if (lane == 0) buf[warp] = ((unsigned long long)a << 32) | b;
  __syncthreads();
  const unsigned long long r = lane < (int)(blockDim.x >> 5) ? buf[lane] : ~0ull;
  *ra = __reduce_min_sync(0xffffffffu, (unsigned)(r >> 32));
  *rb = __reduce_min_sync(0xffffffffu, (unsigned)r);
}

// compute_front with the whole CTA (same result, every thread calls it): the per-resource arg-max types are found by
// probing each resource's descending order T positions at a time (block minimum of the first hit), the pair coverage test
// runs one option word per thread. The serial version walks the orders and the words through dependent L2 loads - 30 000
// cycles per fresh node of a new shape on the 1 000-type catalog (profiles/README.md, round 2).
__shared__ unsigned g_front_pairs;
__device__ __noinline__ void compute_front_block(const uint32_t* opts, int stride, int n, long long* b1, long long* b2, unsigned short* bits,
                                                 unsigned long long (*red)[32], int& parity) {
  KS_K2
  const int R = c.n_res < kHotRes ? c.n_res : kHotRes;
  const int T = c.n_types, tid = threadIdx.x, NT = blockDim.x, W32 = c.W32;
  unsigned pos[kHotRes] = {~0u, ~0u, ~0u, ~0u};
  for (int r = 0; r < R; ++r) {
    const int32_t* perm = c.perm_desc + (size_t)r * T;
    for (int i = tid; i < T; i += NT) {
      const int t = perm[i];
      if ((opts[(size_t)(t >> 5) * stride + n] >> (t & 31)) & 1) { pos[r] = (unsigned)i; break; }
    }
  }
  unsigned pm[kHotRes];
  block_min2_u32_db(pos[0], pos[1], red, parity, &pm[0], &pm[1]);
  block_min2_u32_db(pos[2], pos[3], red, parity, &pm[2], &pm[3]);
  if (tid == 0) g_front_pairs = ~0u;
  int arg[kHotRes];
  long long m1v[kHotRes];
  for (int r = 0; r < kHotRes; ++r) {
    arg[r] = (r < R && pm[r] != ~0u) ? c.perm_desc[(size_t)r * T + pm[r]] : -1;
    m1v[r] = arg[r] >= 0 ? c.alloc_rt[(size_t)r * T + arg[r]] : INT64_MIN;
  }
  bool done = arg[0] < 0 || c.n_res > kHotRes;  // no option left / resources beyond the hot vectors: necessary test only
  unsigned short fb = 0;
  if (!done) {
    bool dom0 = true;  // one option is maximal in every resource
    for (int r = 0; r < R; ++r) dom0 = dom0 && c.alloc_rt[(size_t)r * T + arg[0]] >= m1v[r];
    if (dom0) { fb = kFlExact; done = true; }
  }
  if (done) {
    if (tid == 0) {
      for (int r = 0; r < kHotRes; ++r) { b1[r] = m1v[r]; b2[r] = INT64_MIN; }
      *bits = fb;
    }
    return;  // (uniform: every thread holds the same values)
  }
  int cand[kHotRes], nc = 0;
  for (int r = 0; r < R; ++r) {
    bool seen = false;
    for (int i = 0; i < nc; ++i) seen = seen || cand[i] == arg[r];
    if (!seen) cand[nc++] = arg[r];
  }
  unsigned pair_ok = 0;  // bit (i*4+j), i<j: every option is dominated by candidate i or j
  for (int i = 0; i < nc; ++i) for (int j = i + 1; j < nc; ++j) pair_ok |= 1u << (i * 4 + j);
  unsigned mine = pair_ok;
  for (int w = tid; w < W32; w += NT) {
    const uint32_t m = opts[(size_t)w * stride + n];
    if (!m) continue;
    uint32_t d[kHotRes];
    for (int i = 0; i < nc; ++i) d[i] = c.domset[(size_t)cand[i] * W32 + w];
    for (int i = 0; i < nc; ++i) for (int j = i + 1; j < nc; ++j)
      if (m & ~(d[i] | d[j])) mine &= ~(1u << (i * 4 + j));
  }
  mine = __reduce_and_sync(0xffffffffu, mine);
  __syncthreads();  // g_front_pairs initialised
  if ((tid & 31) == 0) atomicAnd(&g_front_pairs, mine);
  __syncthreads();
  pair_ok &= g_front_pairs;
  if (tid == 0) {
    for (int r = 0; r < kHotRes; ++r) { b1[r] = m1v[r]; b2[r] = INT64_MIN; }
    *bits = 0;
    if (pair_ok) {
      const int pi = (__ffs(pair_ok) - 1) / 4, pj = (__ffs(pair_ok) - 1) % 4;
      for (int r = 0; r < R; ++r) { b1[r] = c.alloc_rt[(size_t)r * T + cand[pi]]; b2[r] = c.alloc_rt[(size_t)r * T + cand[pj]]; }
      *bits = kFlExact | kFlTwo;
    }
  }
}

struct StepShared {
  int placed_closed;   // commit outcome: 1 = the accepting node became full and left the active set
  int path;            // fresh-node path
  unsigned any;
  long long q[KSCHED_MAX_RES];
  unsigned qp;
  long long bound[kHotRes], bound2[kHotRes];
  unsigned short front_bits;
  long long visited;
  // in-flight winner posted for the cooperative instance-type check / commit
  int win_a, win_n, win_need, win_commit, win_fail;
  int excl[16];        // nodes that won the argmin of this step but failed the instance-type check
  // fresh node of a topology-constrained class: slot of the outcome memo (PackState::fd_*), new node's requirement meta
  int fd_slot;
  uint64_t meta;
};
constexpr int kMaxExcl = 16;

enum { kPathReject = 0, kPathCached = 1, kPathRow = 2, kPathDynamic = 3, kPathCachedEmpty = 4, kPathDynCached = 5, kPathDynEmpty = 6 };

// The words of a pod row every candidate check needs. Loaded RAW one iteration ahead for first-pass pods (anything
// derived from them is computed by the consuming iteration, so the prefetch never waits on its own loads).
struct PodRegs {
  const ksched_pod_row* row;
  uint32_t pod, res, itype, hostname, topo_begin, topo_end;
  long long req[kHotRes];
  uint64_t tol, hpc, hpe, meta, cls64;
};
__device__ __forceinline__ PodRegs load_pod_regs(const ksched_pod_row* row, uint32_t pod) {
  PodRegs r;
  r.row = row;
  r.pod = pod;
  r.res = row->res_present;
#pragma unroll
  for (int i = 0; i < kHotRes; ++i) r.req[i] = row->requests[i];  // 0 where the resource is absent
  r.tol = row->tolerated_taintsets;
  r.hpc = row->hostport_conflicts;
  r.hpe = row->hostport_entries;
  r.meta = row->meta;
  r.itype = row->itype_req;
  r.hostname = row->hostname_req;
  r.topo_begin = row->topo_begin;
  r.topo_end = row->topo_end;
  r.cls64 = row->reserved;
  return r;
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Slow part of a candidate check (requirement keys / topology / instance-type words), kept out of line so that the
// common path (no requirement can change, dominant option fits) stays in registers.
struct SlowEval {
  Touched t;
  TypeCtx x;
  long long q[KSCHED_MAX_RES];
  uint32_t qp;
  bool changed;
  bool need_types;  // with_types == false: the instance-type options still have to be checked (by the whole CTA, for the winner only)
};
// `t` receives the touched requirement keys: the thread's own e.t, or the CTA's shared Touched when the caller is the argmin winner
__device__ __noinline__ bool evaluate_slow(bool plain,
                                           int n, unsigned short fl, const long long* q_hot, const int64_t* alloc_sorted, bool with_types, Touched& t,
                                           SlowEval& e) {
  KS_K2
  KS_ROW
  const int MAXN = s.max_new, NE = s.n_existing, R = c.n_res, W32 = c.W32;
  const uint32_t p_res = row.res_present;
  t.n = 0;
  e.changed = false;
  bool need_types = !(fl & 1) || row.itype_req != KSCHED_NONE;
  if (!plain) {
    if (!requirements_phase(s.nn_vals, s.nn_meta[n], MAXN, n, NE + n, false, t)) return false;
    for (int i = 0; i < t.n; ++i) e.changed = e.changed || t.changed[i];
    need_types = need_types || e.changed;
  }
  for (int r = 0; r < kHotRes; ++r) e.q[r] = q_hot[r];
  for (int r = kHotRes; r < R; ++r) e.q[r] = s.nn_req[(size_t)r * MAXN + n] + (((p_res >> r) & 1) ? row.requests[r] : 0);
  e.qp = s.nn_req_present[n] | p_res;
  e.need_types = need_types && !with_types;
  if (!need_types || !with_types) return true;  // the dominant option fits and no requirement changed / checked later
  build_type_ctx(t, e.q, e.qp, s.nn_vals, s.nn_meta[n], MAXN, n, false, alloc_sorted, e.x);
  for (int w = 0; w < W32; ++w) {
    const uint32_t base = s.nn_opts[(size_t)w * MAXN + n];
    if (base && type_word(c, s, e.x, base, w)) return true;
  }
  return false;
}
// Requirement part of a commit: the node's new masks.
__device__ __forceinline__ uint64_t commit_reqs(int n, const Touched& t) {
  KS_K2
  const int MAXN = s.max_new;
  uint64_t meta = s.nn_meta[n];
  for (int i = 0; i < t.n; ++i) {
    const int k = t.key[i];
    const Req& f = t.fin[i];
    const uint64_t bit = 1ull << k;
    meta &= ~((bit << KSCHED_META_PRESENT_SHIFT) | (bit << KSCHED_META_COMPLEMENT_SHIFT));
    if (f.present) meta |= bit << KSCHED_META_PRESENT_SHIFT;
    if (f.present && f.complement) meta |= bit << KSCHED_META_COMPLEMENT_SHIFT;
    s.nn_vals[(size_t)k * MAXN + n] = f.values;
  }
  s.nn_meta[n] = meta;
  return meta;
}
// Requirement-changing commit done by ONE thread (fallback mode): new masks, requirement-driven narrowing of the stored
// options, new bounds.
__device__ __noinline__ void commit_slow(int n, SlowEval& e, long long* bound,
                                         long long* bound2, unsigned short* front_bits, uint64_t* meta_out) {
  KS_K2
  KS_ROW
  const int MAXN = s.max_new, W32 = c.W32;
  *meta_out = commit_reqs(n, e.t);
  e.x.res_mask = 0;  // resources stay lazy (finalize_options_kernel)
  for (int w = 0; w < W32; ++w) {
    const uint32_t base = s.nn_opts[(size_t)w * MAXN + n];
    if (base) s.nn_opts[(size_t)w * MAXN + n] = type_word(c, s, e.x, base, w);
  }
  compute_front(s.nn_opts, MAXN, n, bound, bound2, front_bits);
}

// per-CTA objects of the generic step (file scope: see g_row / g_pt in ksched.cu)
__shared__ Touched g_fresh_t;
__shared__ TypeCtx g_fresh_x;
__shared__ unsigned long long g_red[2][32];
__shared__ StepShared g_sh;
__shared__ uint32_t g_tmpl_taintset[KSCHED_MAX_TEMPLATES];
extern __shared__ __align__(16) unsigned char dyn_smem[];  // HotSmem, then (optionally) the sorted allocatable arrays
__device__ __forceinline__ Hot make_hot(const PackState& s) {
  return Hot{reinterpret_cast<HotSmem*>(dyn_smem), s.ov_key, s.ov_q, s.ov_bound, s.ov_bound2, s.ov_node, s.ov_flags, s.ov_absorbed, s.ov_rejected, s.max_new};
}
__device__ __forceinline__ const int64_t* alloc_table(const DevCatalog& c, const PackState& s) {
  return s.alloc_in_smem ? reinterpret_cast<const int64_t*>(dyn_smem + sizeof(HotSmem)) : c.alloc_sorted;
}
struct LoopVars {
  int head, qlen, n_new, n_active, tick, seq, parity, fatal;
  uint32_t epoch;
  bool pt_nonempty;
  long long nodes_visited;
  uint32_t pt_class;   // class the shared PodTopo was built for (KSCHED_NONE: none)
  uint32_t row_class;  // class whose row g_row holds
  // the step has just opened node slot fresh_a for a pod of class fresh_cls and the node is still open (class_run captures it)
  int fresh_valid, fresh_a;
  uint32_t fresh_cls;
  // the step failed and depends on nothing but (class, placements so far, relaxations so far): no topology relation of
  // any kind, no relaxation left. pack_kernel requeues the following pods of the class without evaluating them again.
  int fail_memo;
};

// ---- existing-node run ("water-fill") --------------------------------------------------------------------------------
// A run of consecutive first-pass pods of ONE plain class (no requirement key, no topology relation, no host port, no
// volume, no instance-type / hostname requirement) is placed on the existing nodes in one pass. First fit over existing
// nodes in slice order (scheduler.go:176-180) sends identical pods to the first node that still fits one, until it does not:
// node e takes K_e = min over requested resources of floor((available - requests) / request) of them, so the run is an
// exclusive prefix sum of K over the nodes from the class's cursor on. Every effect of the sequential commits is reproduced
// (requests, closed flag, assign, place_seq); what the existing nodes cannot take is left to the generic step.
constexpr int kExRunMax = 1 << 20;
__device__ __forceinline__ bool class_has_volumes(const PackState& s, unsigned cls) {
  if (!s.cls_vol) return false;
  const ksched_class_volumes v = s.cls_vol[cls];
  return (v.shared | v.priv[0] | v.priv[1] | v.priv[2] | v.priv[3]) != 0;
}
struct ExRunIO { int qi, head, qlen, seq, parity, placed; long long add_calls; };
__shared__ ExRunIO g_xio;
__shared__ int g_xscan[2][8];
__device__ __forceinline__ int block_scan_incl(int v, int* total, int& xpar) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
  int* buf = g_xscan[xpar];
  xpar ^= 1;
  if (lane == 31) buf[warp] = x;
  __syncthreads();
  int base = 0, tot = 0;
  for (int w = 0; w < nw; ++w) { const int t = buf[w]; if (w < warp) base += t; tot += t; }
  *total = tot;
  return x + base;
}
__device__ __noinline__ void existing_run(const PodRegs& first) {
  KS_K2
  const int tid = threadIdx.x, T = blockDim.x, NE = s.n_existing, R = c.n_res;
  ExRunIO& io = g_xio;
  const unsigned cls = (unsigned)first.cls64;
  const ksched_pod_row* ffd_rows = reinterpret_cast<const ksched_pod_row*>(s.rows);
  const int qi = io.qi, seq0 = io.seq;
  int parity = io.parity, xpar = 0;
  __syncthreads();  // everybody has read g_xio
  // run length: consecutive queue entries of this class
  const int lim = min(s.n_pods - qi, kExRunMax);
  unsigned long long stop = ~0ull;
  for (int j = tid; j < lim; j += T)
    if ((unsigned)ffd_rows[qi + j].reserved != cls) { stop = (unsigned long long)j; break; }
  const unsigned long long st = block_min_u64_db(stop, g_red, parity);
  const int m = st == ~0ull ? lim : (int)st;
  int e0 = s.cls_cursor[cls], placed = 0, last_used = -1;
  while (placed < m && e0 < NE) {
    const int e = e0 + tid;
    int k = 0;
    if (e < NE && !s.ex_closed[e] && ((first.tol >> s.ex_taintset[e]) & 1)) {
      long long K = m - placed;
      const uint32_t qp = s.ex_req_present[e] | first.res, ap = s.ex_avail_present[e];
      for (int r = 0; r < R && K > 0; ++r) {
        if (!((qp >> r) & 1)) continue;
        const long long a = ((ap >> r) & 1) ? s.ex_avail[(size_t)r * NE + e] : 0;
        const long long q = s.ex_req[(size_t)r * NE + e];
        const long long pr = (r < kHotRes && ((first.res >> r) & 1)) ? first.req[r] : 0;
        if (q + pr > a) { K = 0; break; }  // Fits(requests + pod, available) fails for the very next pod (existingnode.go:98-102)
        if (pr > 0) { const long long kk = (a - q) / pr; if (kk < K) K = kk; }
      }
      k = (int)K;
    }
    int total;
    const int incl = block_scan_incl(k, &total, xpar);
    const int excl = incl - k, want = m - placed;
    const int take = excl < want ? min(k, want - excl) : 0;
    if (take > 0) {
      bool closed = false;
      for (int r = 0; r < R; ++r) {
        if (r < kHotRes && ((first.res >> r) & 1)) s.ex_req[(size_t)r * NE + e] += (long long)take * first.req[r];
        const long long a = ((s.ex_avail_present[e] >> r) & 1) ? s.ex_avail[(size_t)r * NE + e] : 0;
        if (s.min_req[r] > 0 && s.ex_req[(size_t)r * NE + e] + s.min_req[r] > a) closed = true;
      }
      s.ex_req_present[e] |= first.res;
      s.ex_closed[e] = closed;
      for (int j = 0; j < take; ++j) {
        const uint32_t pod = s.order[qi + placed + excl + j];
        s.assign[pod] = e;
        s.place_seq[pod] = seq0 + placed + excl + j;
      }
    }
    const unsigned long long lu = block_min_u64_db(take > 0 ? (unsigned long long)(0x7fffffff - e) : ~0ull, g_red, parity);  // max e that took pods
    if (lu != ~0ull) last_used = 0x7fffffff - (int)lu;
    placed += min(total, want);
    if (placed < m) e0 += T;
  }
  if (tid == 0) {
    // nodes passed over took nothing for a monotone reason (closed, taint, requests), nodes filled are full for this class
    s.cls_cursor[cls] = placed < m ? NE : (last_used >= 0 ? last_used : s.cls_cursor[cls]);
    const int qcap = s.n_pods + 1;
    io.qi = qi + placed;
    io.head = (io.head + placed) % qcap;
    io.qlen -= placed;
    io.seq = seq0 + placed;
    io.add_calls += placed;
    io.placed = placed;
    io.parity = parity;
  }
  __syncthreads();
}

// One full Scheduler.add for one pod (existing nodes -> in-flight nodes -> new node -> relax/requeue). Every thread of
// the CTA calls it together. Kept out of line: the steady-state path in pack_kernel must stay a few KB of code, because a
// single resident CTA runs straight out of the instruction cache hierarchy (L0 ~6 KB, L1.5 32 KB).
__device__ __noinline__ void generic_step(const PodRegs& cur, bool first_pass, int fpos_first, LoopVars& L) {
  KS_K2
  const int tid = threadIdx.x, lane = tid & 31;
  const int W32 = c.W32, V = c.n_templates, NE = s.n_existing, MAXN = s.max_new;
  const int R = c.n_res, RH = R < kHotRes ? R : kHotRes;
  const int qcap = s.n_pods + 1;
  PodTopo& pt = g_pt;
  Touched& fresh_t = g_fresh_t;
  TypeCtx& fresh_x = g_fresh_x;
  unsigned long long (*red)[32] = g_red;
  StepShared& sh = g_sh;
  const uint32_t* tmpl_taintset = g_tmpl_taintset;
  const Hot H = make_hot(s);
  const int64_t* alloc_sorted = alloc_table(c, s);
  int &head = L.head, &qlen = L.qlen, &n_new = L.n_new, &n_active = L.n_active, &tick = L.tick, &seq = L.seq, &parity = L.parity, &fatal = L.fatal;
  uint32_t& epoch = L.epoch;
  bool& pt_nonempty = L.pt_nonempty;
  long long& nodes_visited = L.nodes_visited;
  uint32_t& pt_class = L.pt_class;
#ifdef KSCHED_PROFILE_PACK
  long long gk_last = clock64();
#define GK_T(i) { if (tid == 0) { long long _n = clock64(); s.counters[8 + (i)] += _n - gk_last; gk_last = _n; } }
#define GK_C(i) { if (tid == 0) s.counters[8 + (i)] += 1; }
#else
#define GK_T(i)
#define GK_C(i)
#endif
    const uint32_t pod = cur.pod, cls = (uint32_t)cur.cls64;
    L.fresh_valid = 0;
    L.fail_memo = 0;
    const ksched_pod_row& row = g_row;
    const uint32_t p_res = cur.res;
    long long preq[kHotRes];
#pragma unroll
    for (int r = 0; r < kHotRes; ++r) preq[r] = cur.req[r];
    const uint64_t p_tol = cur.tol, p_hpc = cur.hpc, p_hpe = cur.hpe;
    const uint32_t p_keys = (uint32_t)(cur.meta >> KSCHED_META_PRESENT_SHIFT) & 0xFFFF, p_itype = cur.itype, p_hostname = cur.hostname;
    const bool has_topo = cur.topo_begin != cur.topo_end;
    // The pod's 256-byte row lives in shared memory (everything below reads it with immediate addresses); rows of one
    // class are identical, so it is copied on a class change only.
    const bool new_row = L.row_class != cls;
    const bool topo_step = has_topo || pt_nonempty;
    if (new_row || topo_step) {
      __syncthreads();  // previous step's readers of g_row / g_pt are done
      if (tid < 32) {
        if (new_row) {
          reinterpret_cast<uint64_t*>(&g_row)[tid] = reinterpret_cast<const uint64_t*>(cur.row)[tid];
          __syncwarp();
        }
        if (topo_step) {
          if (pt_class == cls && !pt.overflow) refresh_pod_topo();  // same relations as the previous step, new counters
          else build_pod_topo();
        }
      }
      L.row_class = cls;
      if (topo_step) pt_class = cls;
      __syncthreads();
      if (topo_step) {
        pt_nonempty = pt.n != 0;
        if (pt.overflow) { fatal = KSCHED_ERR_UNSUPPORTED; return; }
      }
    }
    const bool plain = p_keys == 0 && !pt_nonempty && p_itype == KSCHED_NONE && p_hostname == KSCHED_NONE;  // no requirement can change
    const bool simple = !has_topo && p_hpc == 0 && p_hpe == 0;  // the requirement verdict memo (HotSmem::absorbed/rejected) applies

    bool placed = false;
    ksched_class_volumes p_vol{};
    bool has_vol = false;
    if (s.cls_vol) {
      p_vol = s.cls_vol[cls];
      has_vol = (p_vol.shared | p_vol.priv[0] | p_vol.priv[1] | p_vol.priv[2] | p_vol.priv[3]) != 0;
    }
    GK_T(0)
    // ------------------------------------------------------------ 1) existing nodes in caller order (scheduler.go:176-180)
    if (NE > 0) {
      // Every existing node below the class's cursor refuses this class for good: it is closed, its taints are not
      // tolerated, a host port or a volume limit is taken, or the requests no longer fit - all of which only get worse as
      // pods are added (existingnode.go:79-102). Rejections by requirements / topology can be lifted later and stop the cursor.
      const int start = s.cls_cursor[cls];
      unsigned mine = ~0u, soft = ~0u;  // first node this thread accepts / first node it did not refuse for good
      Touched t;
      t.n = 0;
      for (int e = start + tid; e < NE; e += blockDim.x) {
        if (s.ex_closed[e]) continue;
        if (!((p_tol >> s.ex_taintset[e]) & 1)) continue;
        if (p_hpc && (s.ex_hp[e] & p_hpc)) continue;
        if (has_vol) {  // volumeUsage.Validate(pod).Exceeds(volumeLimits) existingnode.go:88-96
          const ksched_node_volumes nv = s.ex_vol[e];
          const uint64_t all = nv.mounted | p_vol.shared;
          bool over = false;
#pragma unroll
          for (int d = 0; d < KSCHED_MAX_VOLUME_DRIVERS; ++d)
            over = over || (nv.limit[d] >= 0 && nv.used[d] + __popcll(all & s.vol_mask[d]) + (int)p_vol.priv[d] > nv.limit[d]);
          if (over) continue;
        }
        bool ok = true;  // Fits(requests, available) comes first (existingnode.go:98-102)
        const uint32_t qp = s.ex_req_present[e] | p_res;
        for (int r = 0; r < R && ok; ++r) {
          if (!((qp >> r) & 1)) continue;
          long long q = s.ex_req[(size_t)r * NE + e] + (((p_res >> r) & 1) ? row.requests[r] : 0);
          long long a = ((s.ex_avail_present[e] >> r) & 1) ? s.ex_avail[(size_t)r * NE + e] : 0;
          ok = q <= a;
        }
        if (!ok) continue;
        if (soft == ~0u) soft = (unsigned)e;
        if (p_itype != KSCHED_NONE) {
          const uint32_t it = s.ex_itype[e];
          bool allowed = it == KSCHED_NONE ? (s.itype_complement[p_itype] != 0) : ((s.itype_sets[(size_t)p_itype * W32 + (it >> 5)] >> (it & 31)) & 1);
          if (!allowed) continue;
        }
        if (!plain && !requirements_phase(s.ex_vals, s.ex_meta[e], NE, e, e, true, t)) continue;
        mine = (unsigned)e;
        break;  // this thread's remaining nodes have larger indices
      }
      unsigned w32, soft_min;
      block_min2_u32_db(mine, soft, red, parity, &w32, &soft_min);
      if (tid == 0) s.cls_cursor[cls] = soft_min == ~0u ? NE : (int)soft_min;  // read again only after the next step's barriers
      const unsigned long long w = w32 == ~0u ? ~0ull : (unsigned long long)w32;
      if (w != ~0ull) {
        const int e = (int)w;
        nodes_visited += e + 1;
        if (mine == w32) {  // the winning thread commits its own candidate
          uint64_t meta = s.ex_meta[e];
          if (!plain) {
            for (int i = 0; i < t.n; ++i) {
              const int k = t.key[i];
              const Req& f = t.fin[i];
              const uint64_t bit = 1ull << k;
              meta &= ~((bit << KSCHED_META_PRESENT_SHIFT) | (bit << KSCHED_META_COMPLEMENT_SHIFT));
              if (f.present) meta |= bit << KSCHED_META_PRESENT_SHIFT;
              if (f.present && f.complement) meta |= bit << KSCHED_META_COMPLEMENT_SHIFT;
              s.ex_vals[(size_t)k * NE + e] = f.values;
            }
            s.ex_meta[e] = meta;
          }
          bool closed = false;
          for (int r = 0; r < R; ++r) {
            if ((p_res >> r) & 1) s.ex_req[(size_t)r * NE + e] += row.requests[r];
            long long a = ((s.ex_avail_present[e] >> r) & 1) ? s.ex_avail[(size_t)r * NE + e] : 0;
            if (s.min_req[r] > 0 && s.ex_req[(size_t)r * NE + e] + s.min_req[r] > a) closed = true;
          }
          s.ex_req_present[e] |= p_res;
          if (p_hpe) s.ex_hp[e] |= p_hpe;
          if (has_vol) {  // volumeUsage.Add existingnode.go:128
            ksched_node_volumes nv = s.ex_vol[e];
            nv.mounted |= p_vol.shared;
#pragma unroll
            for (int d = 0; d < KSCHED_MAX_VOLUME_DRIVERS; ++d) nv.used[d] += (int)p_vol.priv[d];
            s.ex_vol[e] = nv;
          }
          s.ex_closed[e] = closed;
          s.assign[pod] = e;
          s.place_seq[pod] = seq;
        }
        ++seq;
        placed = true;
        __syncthreads();  // the commit is read by every thread in the next step
        if (has_topo) topo_record_block(s.ex_vals, s.ex_meta[e], NE, e, e);
      } else {
        nodes_visited += NE;
      }
    }
    GK_T(1)
    // ------------------------------------------------------------ 2) in-flight nodes, fewest pods first (scheduler.go:183-190)
    // Every thread checks candidates for everything except the instance-type options (requirements, topology, the
    // resource pre-test); the block argmin picks the first such node in the reference's order; the whole CTA then
    // verifies the winner's instance-type options word-parallel and, if they survive, narrows them in place. A winner
    // whose options do not survive is excluded and the argmin is repeated (after kMaxExcl such failures every candidate is
    // checked in full by its own thread, which needs no verification).
    if (!placed && n_active > 0) {
      int n_excl = 0;
      bool full_eval = false;
      const bool two_stage = pt_nonempty;  // topology-constrained pod
      while (true) {
        unsigned long long mine = ~0ull;
        int best_a = -1, last_slow = -1;
        long long bq[kHotRes] = {0, 0, 0, 0};
        SlowEval ev;
        bool best_slow = false;
        for (int a = tid; a < n_active; a += blockDim.x) {
          const unsigned long long key = H.key(a);
          if (key >= mine) continue;  // cannot beat this thread's current candidate
          if (n_excl) {
            bool excluded = false;
            for (int i = 0; i < n_excl && i < kMaxExcl; ++i) excluded = excluded || sh.excl[i] == a;
            if (excluded) continue;
          }
          const unsigned short fl = H.flags(a);
          if (!((p_tol >> tmpl_taintset[fl >> 8]) & 1)) continue;  // Taints.Tolerates
          const uint32_t qp = ((fl >> 1) & 0xF) | p_res;
          long long q[kHotRes], b1[kHotRes], b2[kHotRes];
#pragma unroll
          for (int r = 0; r < kHotRes; ++r) { q[r] = H.q(r, a) + preq[r]; b1[r] = H.bound(r, a); b2[r] = H.bound2(r, a); }
          const int qf = quick_fit(q, qp, RH, b1, b2, fl);
          if (qf == 0) continue;
          if (p_hpc && (s.nn_hp[H.node(a)] & p_hpc)) continue;
          if (simple && H.rejected(a) == cls) continue;  // memo: same class, node untouched since it was refused
          const bool fast = (plain || (simple && H.absorbed(a) == cls)) && qf == 1;  // nothing can change and an option holds the requests
          if (!fast) {
            if (two_stage && !full_eval) {  // necessary condition only; the winner is checked in full
              const int n = H.node(a);
              if (!topo_prefilter(s.nn_vals, s.nn_meta[n], MAXN, n, NE + n)) continue;
            } else {
              last_slow = a;
              if (!evaluate_slow(plain, H.node(a), fl, q, alloc_sorted, full_eval, ev.t, ev)) {
                if (simple) H.rejected(a) = cls;
                continue;
              }
            }
          }
          mine = key;
          best_a = a;
          best_slow = !fast;
#pragma unroll
          for (int r = 0; r < kHotRes; ++r) bq[r] = q[r];
        }
        GK_T(2)
        const unsigned long long wkey = block_min_u64_db(mine, red, parity);
        if (wkey == ~0ull) {
          nodes_visited += n_new;
          break;
        }
        const bool winner = mine == wkey;
        if (winner) {  // post the candidate for the cooperative instance-type check
          const int a = best_a;
          bool okw = true, in_shared = false;
          if (best_slow && last_slow != a) {
            // without the instance-type part the touched keys go straight into the CTA's shared Touched
            in_shared = !full_eval;
            okw = evaluate_slow(plain, H.node(a), H.flags(a), bq, alloc_sorted, full_eval, in_shared ? fresh_t : ev.t, ev);
          }
          sh.win_a = a;
          sh.win_n = H.node(a);
          sh.win_fail = okw ? 0 : 1;
          sh.win_need = (okw && best_slow && ev.need_types) ? 1 : 0;
          sh.win_commit = (okw && best_slow && (ev.changed || p_itype != KSCHED_NONE)) ? 1 : 0;
          if (sh.win_need) {
            if (!in_shared) fresh_t = ev.t;
            for (int r = 0; r < KSCHED_MAX_RES; ++r) sh.q[r] = r < R ? ev.q[r] : 0;
            sh.qp = ev.qp;
          }
        }
        __syncthreads();
        const int wa = sh.win_a, wn = sh.win_n;
        if (sh.win_fail) {  // the prefilter let through a node the full requirement check refuses
          if (tid == 0) {
            if (n_excl < kMaxExcl) sh.excl[n_excl] = wa;
            if (simple) H.rejected(wa) = cls;
          }
          ++n_excl;
          if (n_excl >= kMaxExcl) full_eval = true;
          __syncthreads();
          continue;
        }
        const bool coop = sh.win_need != 0;
        bool opts_changed = false;
        if (coop) {
          // TypeCtx of the winner: requirement part by thread 0, one Fits rank per resource by the first lanes of warp 1
          const int rbase = blockDim.x >= 64 ? 32 : 0;
          if (tid == 0) build_type_ctx(fresh_t, sh.q, sh.qp, s.nn_vals, s.nn_meta[wn], MAXN, wn, false, alloc_sorted, fresh_x, rbase == 0);
          if (rbase && tid >= rbase && tid < rbase + R) {
            const int r = tid - rbase;
            fresh_x.rank[r] = ((sh.qp >> r) & 1) ? fit_rank(alloc_sorted, c.n_types, r, sh.q[r]) : 0;
          }
          __syncthreads();
          // one pass: requirement-narrowed word kept in a register, resource test on top of it
          uint32_t keep_base = 0, keep = 0;
          int local_any = 0;
          for (int w = tid; w < W32; w += blockDim.x) {
            const uint32_t base = s.nn_opts[(size_t)w * MAXN + wn];
            if (!base) continue;
            const uint32_t sw = type_word_keys(c, s, fresh_x, base, w);
            if (w == tid) { keep_base = base; keep = sw; }
            if (sw && type_word_res(c, fresh_x, sw, w)) local_any = 1;
          }
          if (!__syncthreads_or(local_any)) {  // no option survives: Node.Add fails on this node (node.go:92-95)
            if (tid == 0) {
              if (n_excl < kMaxExcl) sh.excl[n_excl] = wa;
              if (simple) H.rejected(wa) = cls;
            }
            ++n_excl;
            if (n_excl >= kMaxExcl) full_eval = true;
            __syncthreads();
            continue;
          }
          if (sh.win_commit) {  // requirement-driven narrowing of the stored options; resources stay lazy
            int local_changed = 0;
            if (tid < W32 && keep != keep_base) { s.nn_opts[(size_t)tid * MAXN + wn] = keep; local_changed = 1; }
            for (int w = tid + blockDim.x; w < W32; w += blockDim.x) {
              const uint32_t base = s.nn_opts[(size_t)w * MAXN + wn];
              if (!base) continue;
              const uint32_t sw = type_word_keys(c, s, fresh_x, base, w);
              if (sw != base) { s.nn_opts[(size_t)w * MAXN + wn] = sw; local_changed = 1; }
            }
            opts_changed = __syncthreads_or(local_changed) != 0;
          }
        }
        GK_T(21)
        GK_C(10)
        if (s.count_visited) {  // rank of the winner among ALL in-flight nodes (the reference also walks the full ones)
          int less = 0;
          for (int i = tid; i < n_new; i += blockDim.x) less += order_key(s.nn_count[i], s.nn_tb[i]) < wkey;
          for (int o = 16; o; o >>= 1) less += __shfl_xor_sync(0xffffffffu, less, o);
          __syncthreads();
          if (tid == 0) sh.visited = 0;
          __syncthreads();
          if (lane == 0 && less) atomicAdd((unsigned long long*)&sh.visited, (unsigned long long)less);
          __syncthreads();
          nodes_visited += sh.visited + 1;
        }
        if (winner) {  // the winning thread commits its own candidate
          const int a = best_a;
          const int n = wn;
          unsigned short fl = H.flags(a);
#pragma unroll
          for (int r = 0; r < kHotRes; ++r) H.q(r, a) = bq[r];
          for (int r = kHotRes; r < R; ++r)
            if ((p_res >> r) & 1) s.nn_req[(size_t)r * MAXN + n] += row.requests[r];
          if ((p_res >> kHotRes) || ((p_res & 0xF) & ~((fl >> 1) & 0xF))) s.nn_req_present[n] |= p_res;
          fl |= (unsigned short)((p_res & 0xF) << 1);
          if (p_hpe) s.nn_hp[n] |= p_hpe;
          const int count = (int)(wkey >> 32) + 1;
          s.nn_count[n] = count;
          s.nn_tb[n] = -(tick + 1);  // front of the next pod-count block under a stable sort
          H.key(a) = order_key(count, -(tick + 1));
          if (best_slow && (ev.changed || p_itype != KSCHED_NONE)) {
            long long nb1[kHotRes], nb2[kHotRes];
            unsigned short fb;
            bool new_front = true;
            if (coop) {
              commit_reqs(n, fresh_t);
              if (opts_changed) compute_front(s.nn_opts, MAXN, n, nb1, nb2, &fb);
              else new_front = false;  // same option set, same Pareto front
            } else {
              uint64_t meta;
              commit_slow(n, ev, nb1, nb2, &fb, &meta);
            }
            if (new_front) {
#pragma unroll
              for (int r = 0; r < kHotRes; ++r) { H.bound(r, a) = nb1[r]; H.bound2(r, a) = nb2[r]; }
              fl = (unsigned short)((fl & ~(kFlExact | kFlTwo)) | fb);
            }
          }
          H.flags(a) = fl;
          H.rejected(a) = KSCHED_NONE;
          if (simple) H.absorbed(a) = cls;
          long long cb1[kHotRes], cb2[kHotRes];
#pragma unroll
          for (int r = 0; r < kHotRes; ++r) { cb1[r] = H.bound(r, a); cb2[r] = H.bound2(r, a); }
          const bool closed = node_closed(bq, s.min_req, RH, cb1, cb2, fl);
          s.assign[pod] = NE + n;
          s.place_seq[pod] = seq;
          if (closed) {  // the node leaves the active set: its request vector goes back to global memory
            for (int r = 0; r < RH; ++r) s.nn_req[(size_t)r * MAXN + n] = bq[r];
            if (a != n_active - 1) H.move(a, n_active - 1);
          }
          sh.placed_closed = closed ? 1 : 0;
        }
        ++tick;
        ++seq;
        placed = true;
        __syncthreads();
        GK_T(22)
        if (sh.placed_closed) --n_active;
        if (has_topo) topo_record_block(s.nn_vals, s.nn_meta[wn], MAXN, wn, NE + wn);  // Topology.Record, one relation per thread
        GK_T(23)
        break;
      }
    } else if (!placed) {
      nodes_visited += n_new;  // every in-flight node is full; the reference still walks them
    }
    GK_T(3)
    // ------------------------------------------------------------ 3) open a new node, templates in weight order (scheduler.go:194-217)
    if (!placed) {
      GK_C(11)
      const bool f_valid = s.use_F && (first_pass || s.relax_level[pod] == 0);  // K1's row is valid while the pod has its original class
      const uint32_t fpos = first_pass ? (uint32_t)fpos_first : s.pod_pos[pod];
      const bool no_column = f_valid && s.best[fpos] == kNoBest;  // no feasible (template, type) column at all
      if (no_column) nodes_visited += V;
      for (int v = 0; v < V && !placed && !no_column; ++v) {
        const ksched_template& tm = c.templates[v];
        ++nodes_visited;
        if (n_new >= MAXN) { fatal = KSCHED_ERR_OVERFLOW; break; }
        const int n = n_new;  // tentative slot: the hostname placeholder of this attempt (node.go:46)
        const bool limits_active = tm.has_limits && tm.limit_present;
        // Without topology and provisioner limits the outcome of NewNode+Add depends on (class, template) only: memoised.
        const bool memo = !pt_nonempty && !limits_active;
        const size_t fc = ((size_t)cls * V + v);
        __syncthreads();
        if (tid == 0) {
          int path = kPathReject;
          const uint8_t st = memo ? s.fc_state[fc] : 0;
          if (st == 1) path = kPathCached;
          else if (st == 2) path = kPathCachedEmpty;
          else {
            bool ok = (p_tol >> tm.taintset) & 1;
            fresh_t.n = 0;
            if (ok && !plain) ok = requirements_phase(tm.reqs.values, tm.reqs.meta & 0xFFFFFFFFull, 1, 0, NE + n, false, fresh_t);
            if (ok) {
              sh.qp = tm.daemon_res_present | p_res;
              for (int r = 0; r < KSCHED_MAX_RES; ++r) sh.q[r] = r < R ? tm.daemon_requests[r] + (((p_res >> r) & 1) ? row.requests[r] : 0) : 0;
              bool same = f_valid;  // topology left every requirement exactly as K1 saw it
              for (int i = 0; i < fresh_t.n && same; ++i) same = req_equal(fresh_t.fin[i], fresh_t.merged[i]);
              // the new node's requirement set: the template's, overlaid by what this Add touched
              uint64_t meta = tm.reqs.meta & 0xFFFFFFFFull;
              for (int i = 0; i < fresh_t.n; ++i) {
                const int k = fresh_t.key[i];
                const Req& f = fresh_t.fin[i];
                const uint64_t bit = 1ull << k;
                meta &= ~((bit << KSCHED_META_PRESENT_SHIFT) | (bit << KSCHED_META_COMPLEMENT_SHIFT));
                if (f.present) meta |= bit << KSCHED_META_PRESENT_SHIFT;
                if (f.present && f.complement) meta |= bit << KSCHED_META_COMPLEMENT_SHIFT;
              }
              sh.meta = meta;
              sh.fd_slot = -1;
              if (same) path = kPathRow;
              else {
                path = kPathDynamic;
                if (!memo && !limits_active) {  // topology-constrained class: outcome memo keyed by the node's requirement set
                  uint64_t vals[KSCHED_MAX_KEYS];
                  uint64_t hsh = ((uint64_t)fc + 1) * 0x9E3779B97F4A7C15ull ^ meta;
                  for (int k = 0; k < c.n_keys; ++k) {
                    uint64_t val = tm.reqs.values[k];
                    for (int i = 0; i < fresh_t.n; ++i) if (fresh_t.key[i] == k) val = fresh_t.fin[i].values;
                    vals[k] = val;
                    hsh = (hsh ^ val) * 0xBF58476D1CE4E5B9ull;
                    hsh ^= hsh >> 29;
                  }
                  const int slot = (int)((hsh >> 13) & (uint64_t)(s.fd_cap - 1));
                  const uint8_t st = s.fd_state[slot];
                  bool hit = st != 0 && s.fd_fc[slot] == (uint32_t)fc && s.fd_meta[slot] == meta;
                  for (int k = 0; k < c.n_keys && hit; ++k) hit = s.fd_vals[(size_t)slot * KSCHED_MAX_KEYS + k] == vals[k];
                  sh.fd_slot = slot;
                  if (hit) path = st == 1 ? kPathDynCached : kPathDynEmpty;
                  else {
                    s.fd_state[slot] = 0;  // being refilled: tags now, state when the outcome is known
                    s.fd_fc[slot] = (uint32_t)fc;
                    s.fd_meta[slot] = meta;
                    for (int k = 0; k < c.n_keys; ++k) s.fd_vals[(size_t)slot * KSCHED_MAX_KEYS + k] = vals[k];
                  }
                }
                if (path == kPathDynamic)
                  build_type_ctx(fresh_t, sh.q, sh.qp, tm.reqs.values, tm.reqs.meta & 0xFFFFFFFFull, 1, 0, true, alloc_sorted, fresh_x);
              }
            } else if (memo) {
              s.fc_state[fc] = 2;
            }
          }
          sh.path = path;
          sh.any = 0;
        }
        __syncthreads();
        const int path = sh.path;
        GK_C(13 + (path > 4 ? 4 : path))
        GK_T(18)
        if (path == kPathReject || path == kPathCachedEmpty || path == kPathDynEmpty) continue;
        const int fd_slot = (path == kPathDynamic || path == kPathDynCached) ? sh.fd_slot : -1;
        const int a = n_active;
        if (path == kPathCached) {
          for (int w = tid; w < W32; w += blockDim.x) s.nn_opts[(size_t)w * MAXN + n] = s.fc_opts[fc * W32 + w];
          if (tid < c.n_keys) s.nn_vals[(size_t)tid * MAXN + n] = s.fc_vals[fc * KSCHED_MAX_KEYS + tid];
        } else {
          bool local_any = false;
          for (int w = tid; w < W32; w += blockDim.x) {
            uint32_t base = c.member[(size_t)v * W32 + w];
            if (base && limits_active) {  // filterByRemainingResources (scheduler.go:293-309)
              uint32_t m = base;
              while (m) {
                const int b = __ffs(m) - 1;
                m &= m - 1;
                const int t = w * 32 + b;
                for (int r = 0; r < R; ++r)
                  if (((tm.limit_present >> r) & 1) && c.capacity[(size_t)t * KSCHED_MAX_RES + r] > s.remaining[(size_t)v * KSCHED_MAX_RES + r]) base &= ~(1u << b);
              }
            }
            uint32_t sw = 0;
            if (path == kPathDynCached) sw = s.fd_opts[(size_t)fd_slot * W32 + w];
            else if (base) sw = path == kPathRow ? (base & s.F[((size_t)fpos * V + v) * W32 + w]) : type_word(c, s, fresh_x, base, w);
            s.nn_opts[(size_t)w * MAXN + n] = sw;
            if (memo) s.fc_opts[fc * W32 + w] = sw;
            if (path == kPathDynamic && fd_slot >= 0) s.fd_opts[(size_t)fd_slot * W32 + w] = sw;
            local_any = local_any || sw;
          }
          if (local_any) atomicOr(&sh.any, 1u);
          if (tid < c.n_keys) {
            uint64_t val = tm.reqs.values[tid];
            for (int i = 0; i < fresh_t.n; ++i) if (fresh_t.key[i] == tid) val = fresh_t.fin[i].values;
            s.nn_vals[(size_t)tid * MAXN + n] = val;
            if (memo) s.fc_vals[fc * KSCHED_MAX_KEYS + tid] = val;
          }
          __syncthreads();
          if (!sh.any) {
            if (memo && tid == 0) s.fc_state[fc] = 2;
            if (path == kPathDynamic && fd_slot >= 0 && tid == 0) s.fd_state[fd_slot] = 2;
            continue;
          }
        }
        GK_T(19)
        // the Pareto front of a new option set, with every thread (the words were stored before the barrier above)
        const bool front_memo_hit = path == kPathRow && !limits_active && s.fc_front_state[fc];
        const bool front_fresh = path != kPathCached && path != kPathDynCached && !front_memo_hit;
        if (front_fresh) compute_front_block(s.nn_opts, MAXN, n, sh.bound, sh.bound2, &sh.front_bits, red, parity);
        // ---- commit the new node (NewNode + Add, node.go:44-107) — one thread, everything else was written above
        __syncthreads();
        if (tid == 0) {
          uint64_t meta;
          if (path == kPathCached) {
            meta = s.fc_meta[fc];
            for (int r = 0; r < kHotRes; ++r) { sh.bound[r] = s.fc_bound[fc * kHotRes + r]; sh.bound2[r] = s.fc_bound2[fc * kHotRes + r]; }
            sh.front_bits = s.fc_dom[fc];
            sh.qp = s.fc_qp[fc];
            for (int r = 0; r < KSCHED_MAX_RES; ++r) sh.q[r] = s.fc_q[fc * KSCHED_MAX_RES + r];
          } else {
            meta = sh.meta;
            // K1-row path without limits: the option set, hence its Pareto front, depends on (class, template) only
            const bool front_memo = path == kPathRow && !limits_active;
            if (front_memo && s.fc_front_state[fc]) {
              for (int r = 0; r < kHotRes; ++r) { sh.bound[r] = s.fc_bound[fc * kHotRes + r]; sh.bound2[r] = s.fc_bound2[fc * kHotRes + r]; }
              sh.front_bits = s.fc_dom[fc];
            } else if (path == kPathDynCached) {
              for (int r = 0; r < kHotRes; ++r) { sh.bound[r] = s.fd_bound[(size_t)fd_slot * kHotRes + r]; sh.bound2[r] = s.fd_bound2[(size_t)fd_slot * kHotRes + r]; }
              sh.front_bits = s.fd_dom[fd_slot];
            } else {  // (front_fresh: computed by the CTA above)
              if (front_memo) {
                for (int r = 0; r < kHotRes; ++r) { s.fc_bound[fc * kHotRes + r] = sh.bound[r]; s.fc_bound2[fc * kHotRes + r] = sh.bound2[r]; }
                s.fc_dom[fc] = (uint8_t)sh.front_bits;
                s.fc_front_state[fc] = 1;
              }
              if (path == kPathDynamic && fd_slot >= 0) {
                for (int r = 0; r < kHotRes; ++r) { s.fd_bound[(size_t)fd_slot * kHotRes + r] = sh.bound[r]; s.fd_bound2[(size_t)fd_slot * kHotRes + r] = sh.bound2[r]; }
                s.fd_dom[fd_slot] = (uint8_t)sh.front_bits;
                s.fd_state[fd_slot] = 1;
              }
            }
            if (memo) {
              s.fc_meta[fc] = meta;
              for (int r = 0; r < kHotRes; ++r) { s.fc_bound[fc * kHotRes + r] = sh.bound[r]; s.fc_bound2[fc * kHotRes + r] = sh.bound2[r]; }
              s.fc_dom[fc] = (uint8_t)sh.front_bits;
              s.fc_qp[fc] = sh.qp;
              for (int r = 0; r < KSCHED_MAX_RES; ++r) s.fc_q[fc * KSCHED_MAX_RES + r] = sh.q[r];
              s.fc_state[fc] = 1;
            }
          }
          s.nn_meta[n] = meta;
          s.nn_tmpl[n] = (uint8_t)v;
          for (int r = 0; r < KSCHED_MAX_RES; ++r) s.nn_req[(size_t)r * MAXN + n] = sh.q[r];
          s.nn_req_present[n] = sh.qp;
          s.nn_hp[n] = p_hpe;
          s.nn_count[n] = 1;
          s.nn_tb[n] = tick + 1;  // appended: last of the one-pod block
          const bool closed = node_closed(sh.q, s.min_req, RH, sh.bound, sh.bound2, sh.front_bits);
          if (!closed) {
            H.key(a) = order_key(1, tick + 1);
            for (int r = 0; r < kHotRes; ++r) { H.q(r, a) = sh.q[r]; H.bound(r, a) = sh.bound[r]; H.bound2(r, a) = sh.bound2[r]; }
            H.node(a) = n;
            H.flags(a) = (unsigned short)(sh.front_bits | ((sh.qp & 0xF) << 1) | (v << 8));
            H.absorbed(a) = simple ? cls : KSCHED_NONE;
            H.rejected(a) = KSCHED_NONE;
          }
          sh.placed_closed = closed ? 1 : 0;
          s.assign[pod] = NE + n;
          s.place_seq[pod] = seq;
          if (limits_active) {  // subtractMax (scheduler.go:273-290): largest capacity among the surviving options
            for (int r = 0; r < R; ++r) {
              if (!((tm.limit_present >> r) & 1)) continue;
              long long mx = INT64_MIN;
              for (int w = 0; w < W32; ++w) {
                uint32_t m = s.nn_opts[(size_t)w * MAXN + n];
                while (m) {
                  const int b = __ffs(m) - 1;
                  m &= m - 1;
                  const long long cp = c.capacity[(size_t)(w * 32 + b) * KSCHED_MAX_RES + r];
                  mx = cp > mx ? cp : mx;
                }
              }
              if (mx != INT64_MIN) s.remaining[(size_t)v * KSCHED_MAX_RES + r] -= mx;
            }
          }
        }
        ++tick;
        ++seq;
        __syncthreads();
        if (has_topo) topo_record_block(s.nn_vals, s.nn_meta[n], MAXN, n, NE + n);  // Topology.Record, one relation per thread
        ++n_new;
        if (!sh.placed_closed) { L.fresh_valid = 1; L.fresh_a = n_active; L.fresh_cls = cls; ++n_active; }
        placed = true;
        GK_T(20)
      }
      if (fatal) return;
    }
    GK_T(4)
    // ------------------------------------------------------------ failure: relax + requeue (scheduler.go:117-123, queue.go:61-68)
    if (!placed) {
      GK_C(12)
      const uint32_t nx = row.relax_next;
      int tail = head + qlen;
      if (tail >= qcap) tail -= qcap;
      if (tid == 0) {
        s.queue[tail] = pod;
        if (nx != KSCHED_NONE) {
          s.pod_class[pod] = nx;
          s.relax_level[pod] += 1;
          // Topology.Update(pod): groups that only the relaxed spec owns come into existence now
          const ksched_pod_row& nrow = s.classes[nx];
          for (uint32_t e = nrow.topo_begin; e < nrow.topo_end; ++e) {
            const ksched_class_topo ct = s.class_topo[e];
            if ((ct.flags & KSCHED_TOPO_CONSTRAINS) && !s.grp_active[ct.group]) {
              s.grp_active[ct.group] = 1;
              s.grp_min_slot[ct.group] = NE + n_new;
            }
          }
        } else {
          s.last_len[pod] = qlen + 1;
          s.last_epoch[pod] = epoch;
        }
      }
      ++qlen;
      if (nx != KSCHED_NONE) ++epoch;  // a successful relaxation resets the lastLen map
      L.fail_memo = nx == KSCHED_NONE && !has_topo && !pt_nonempty;
      __syncthreads();
    }
  }

// ---- register-resident steady state -----------------------------------------------------------------------------
// When at most 32 in-flight nodes are open, warp 0 keeps one node per lane IN REGISTERS and places consecutive
// "plain" pods (no requirement can change, no host ports) without touching shared or global node state: R compares per
// lane, a 2-REDUX argmin, the winning lane updates its own registers. The other warps wait at a block barrier.
struct WarpIO {
  int qi, head, qlen, tick, seq, n_active;
  long long add_calls;
};

__device__ __forceinline__ bool plain_pod_regs(const PodRegs& r) {
  return ((r.meta >> KSCHED_META_PRESENT_SHIFT) & 0xFFFF) == 0 && r.itype == KSCHED_NONE && r.hostname == KSCHED_NONE && r.topo_begin == r.topo_end;
}
// topology-free, no host ports, resources within the hot vectors: the requirement verdict memo applies
__device__ __forceinline__ bool simple_pod_regs(const PodRegs& r) {
  return r.topo_begin == r.topo_end && r.hpc == 0 && r.hpe == 0 && (r.res >> kHotRes) == 0;
}

__device__ __noinline__ void warp_resident_loop(WarpIO* io) {
  KS_K2
  HotSmem* hs = reinterpret_cast<HotSmem*>(dyn_smem);
  const uint32_t* tmpl_taintset = g_tmpl_taintset;
  const int lane = threadIdx.x & 31;
  const int NE = s.n_existing, MAXN = s.max_new;
  const int RH = c.n_res < kHotRes ? c.n_res : kHotRes;
  const int qcap = s.n_pods + 1;
  int qi = io->qi, head = io->head, qlen = io->qlen, tick = io->tick, seq = io->seq;
  long long add_calls = io->add_calls;
  const int n_active = io->n_active;
  // lane state
  bool live = lane < n_active, dirty = false;
  unsigned long long key = live ? hs->key[lane] : ~0ull;
  long long q[kHotRes], b[kHotRes], b2[kHotRes];
#pragma unroll
  for (int r = 0; r < kHotRes; ++r) { q[r] = live ? hs->q[r][lane] : 0; b[r] = live ? hs->bound[r][lane] : 0; b2[r] = live ? hs->bound2[r][lane] : 0; }
  const int node = live ? hs->node[lane] : 0;
  unsigned short fl = live ? hs->flags[lane] : 0;
  unsigned absorbed = live ? hs->absorbed[lane] : KSCHED_NONE, rejected = live ? hs->rejected[lane] : KSCHED_NONE;
  const ksched_pod_row* ffd_rows = reinterpret_cast<const ksched_pod_row*>(s.rows);
  // Consecutive pods of the queue usually belong to the same class (identical row): only the next pod's id and class are
  // prefetched; the row's words are reloaded on a class change.
  PodRegs cur = load_pod_regs(ffd_rows + qi, s.order[qi]);
  uint32_t npod = 0;
  uint64_t ncls = ~0ull;
  if (qi + 1 < s.n_pods) { npod = s.order[qi + 1]; ncls = ffd_rows[qi + 1].reserved; }
  long long min_req[kHotRes];
#pragma unroll
  for (int r = 0; r < kHotRes; ++r) min_req[r] = r < RH ? s.min_req[r] : 0;

  while (true) {
    if (!simple_pod_regs(cur)) break;  // this pod takes the block-wide path
    const bool plain = plain_pod_regs(cur);
    const unsigned cls = (unsigned)cur.cls64;
    const bool cand = live && rejected != cls && ((cur.tol >> tmpl_taintset[fl >> 8]) & 1);
    const uint32_t qp = ((fl >> 1) & 0xF) | cur.res;
    long long nq[kHotRes];
#pragma unroll
    for (int r = 0; r < kHotRes; ++r) nq[r] = q[r] + cur.req[r];
    const int qf = cand ? quick_fit(nq, qp, RH, b, b2, fl) : 0;
    const bool ok = qf != 0;
    // a candidate whose resource test is not exact, or whose requirement verdict for this class is unknown, needs the full check
    if (__any_sync(0xffffffffu, ok && (qf == 2 || !(plain || absorbed == cls)))) break;
    const unsigned long long wkey = warp_min_u64(ok ? key : ~0ull);
    if (wkey == ~0ull) break;  // nobody accepts: a new node has to be opened
    // ---- level step. The accepting nodes with the FEWEST pods (count L) take the next pods one each, in tie order: a node
    // that accepts moves to the front of block L+1 (scheduler.go:183 re-sort), i.e. behind every node still in block L. With
    // t identical pods ahead, the first t members of the block take them - t iterations of this loop in one.
    const unsigned members = __ballot_sync(0xffffffffu, ok && (key >> 32) == (wkey >> 32));
    if (s.use_level_step && (members & (members - 1)) && ncls == cur.cls64) {
      const bool same = qi + lane < s.n_pods && (lane == 0 || ffd_rows[qi + lane].reserved == cur.cls64);
      const unsigned sm = __ballot_sync(0xffffffffu, same);
      const int run_len = sm == 0xffffffffu ? 32 : __ffs(~sm) - 1;
      const int k = __popc(members);
      const int t = k < run_len ? k : run_len;
      if (t > 1) {
        int rank = 0;
        for (unsigned mm = members; mm; mm &= mm - 1) {
          const unsigned long long k2 = __shfl_sync(0xffffffffu, key, __ffs(mm) - 1);
          rank += k2 < key ? 1 : 0;
        }
        if (((members >> lane) & 1) && rank < t) {
          const uint32_t pod = s.order[qi + rank];
#pragma unroll
          for (int r = 0; r < kHotRes; ++r) q[r] = nq[r];
          const int count = (int)(wkey >> 32) + 1;
          key = order_key(count, -(tick + 1 + rank));
          if ((cur.res & 0xF) & ~((fl >> 1) & 0xF)) {
            s.nn_req_present[node] |= cur.res;
            fl |= (unsigned short)((cur.res & 0xF) << 1);
          }
          dirty = true;
          rejected = KSCHED_NONE;
          s.assign[pod] = NE + node;
          s.place_seq[pod] = seq + rank;
          if (node_closed(q, min_req, RH, b, b2, fl)) {  // the node leaves the active set
            for (int r = 0; r < RH; ++r) s.nn_req[(size_t)r * MAXN + node] = q[r];
            s.nn_count[node] = count;
            s.nn_tb[node] = -(tick + 1 + rank);
            live = false;
            dirty = false;
            key = ~0ull;
          }
        }
        tick += t; seq += t; qi += t; add_calls += t;
        head += t; if (head >= qcap) head -= qcap;
        qlen -= t;
        if (qi >= s.n_pods || qlen == 0) break;
        if (run_len > t) { cur.pod = s.order[qi]; cur.row = ffd_rows + qi; }
        else cur = load_pod_regs(ffd_rows + qi, s.order[qi]);
        if (qi + 1 < s.n_pods) { npod = s.order[qi + 1]; ncls = ffd_rows[qi + 1].reserved; } else ncls = ~0ull;
        if (lane == 0 && qi + 32 < s.n_pods) prefetch_l2(reinterpret_cast<const char*>(ffd_rows + qi + 32) + 128);
        if (lane == 2 && qi + 96 < s.n_pods) prefetch_l2(s.order + qi + 96);
        continue;
      }
    }
    if (ok && key == wkey) {
#pragma unroll
      for (int r = 0; r < kHotRes; ++r) q[r] = nq[r];
      const int count = (int)(wkey >> 32) + 1;
      key = order_key(count, -(tick + 1));
      if ((cur.res & 0xF) & ~((fl >> 1) & 0xF)) {
        s.nn_req_present[node] |= cur.res;
        fl |= (unsigned short)((cur.res & 0xF) << 1);
      }
      dirty = true;
      rejected = KSCHED_NONE;
      s.assign[cur.pod] = NE + node;
      s.place_seq[cur.pod] = seq;
      const bool closed = node_closed(q, min_req, RH, b, b2, fl);
      if (closed) {  // the node leaves the active set
        for (int r = 0; r < RH; ++r) s.nn_req[(size_t)r * MAXN + node] = q[r];
        s.nn_count[node] = count;
        s.nn_tb[node] = -(tick + 1);
        live = false;
        dirty = false;
        key = ~0ull;
      }
    }
    ++tick; ++seq; ++qi; ++add_calls;
    head = head + 1 == qcap ? 0 : head + 1;
    --qlen;
    if (qi >= s.n_pods || qlen == 0) break;
    if (ncls == cur.cls64) { cur.pod = npod; cur.row = ffd_rows + qi; }
    else cur = load_pod_regs(ffd_rows + qi, npod);
    if (qi + 1 < s.n_pods) { npod = s.order[qi + 1]; ncls = ffd_rows[qi + 1].reserved; }
    if (lane == 0 && qi + 32 < s.n_pods) prefetch_l2(reinterpret_cast<const char*>(ffd_rows + qi + 32) + 128);  // the line holding `reserved`
    if (lane == 2 && (qi & 31) == 0 && qi + 96 < s.n_pods) prefetch_l2(s.order + qi + 96);
  }
  // write the lanes back, compacted
  const unsigned livemask = __ballot_sync(0xffffffffu, live);
  const int slot = __popc(livemask & ((1u << lane) - 1));
  __syncwarp();
  if (live) {
    hs->key[slot] = key;
#pragma unroll
    for (int r = 0; r < kHotRes; ++r) { hs->q[r][slot] = q[r]; hs->bound[r][slot] = b[r]; hs->bound2[r][slot] = b2[r]; }
    hs->node[slot] = node;
    hs->flags[slot] = fl;
    hs->absorbed[slot] = absorbed;
    hs->rejected[slot] = rejected;
    if (dirty) {
      s.nn_count[node] = (int)(key >> 32);
      s.nn_tb[node] = (int)((unsigned)key ^ 0x80000000u);
    }
  }
  if (lane == 0) {
    io->qi = qi; io->head = head; io->qlen = qlen; io->tick = tick; io->seq = seq; io->n_active = __popc(livemask);
    io->add_calls = add_calls;
  }
}

// ---- class-run loop ------------------------------------------------------------------------------------------------
// Consecutive pods of the queue usually belong to ONE class (a deployment: identical row, identical topology terms). For
// such a run the whole CTA stays in this loop: ONE block barrier per pod, no global load and (almost) no global store on
// the chain, ~120 instructions per warp and pod.
//  * every open node is owned by thread (slot % blockDim): only its owner ever reads or writes its state, so a commit
//    needs no barrier to become visible; the block argmin carries a payload (slot, domains) from which every warp updates
//    its own copy of the spread counters;
//  * everything the accept test of a run needs from a node collapses into ONE word per node, `rp`:
//      room   = how many more pods of THIS class fit by the exact Pareto-front resource test (computed once per run with
//               integer divisions, decremented by the commits; 0 also covers untolerated taints / a memoised refusal,
//               kRoomSlow = "verdict not exact here"),
//      dead   = a hostname-keyed group of the class (anti-affinity, hostname spread) no longer admits the node - known at
//               the commit that fills it, because only this run's commits change those counts,
//      placed = pods of the run the node took; requests, order statistics and hostname counters are written back from it
//               when the run ends;
//    plus, per spread key of the class, the node's admissible domains (`zv`);
//  * a candidate is accepted here only when the verdict is EXACT and nothing but counters changes: requirements untouched
//    (plain / absorbed classes) or a spread domain that is already pinned on the node - or that can be pinned without
//    touching the option set (DevCatalog::pin_neutral). Any other winner, a pod that fails, or a fresh node of a shape not
//    seen before in the run hands the pod to generic_step (status 1);
//  * a node that becomes full is tombstoned (key = ~0) and the active list is compacted when the run ends; assignments
//    are staged per queue chunk and stored coalesced;
//  * fresh nodes replay a VARIANT: NewNode+Add for (class, template, resulting requirement masks) is a pure function
//    when no provisioner limit is active (same argument as PackState::fd_*), so the node generic_step created last for
//    this class is captured (options, masks, requests, Pareto front) and replayed for every later pod of the run whose
//    spread domains come out the same.
constexpr int kRunHost = 4;      // hostname-keyed relations of a run-eligible class
constexpr int kRunMask = 2;      // spread relations over a mask key
constexpr int kRunDom = 16;      // domains of such a key
constexpr int kTopoCap = 768;    // open nodes whose per-class topology inputs fit in shared memory
constexpr int kRunVariants = 4;
constexpr int kRunW32 = 64;      // option words a variant holds (T <= 2048)
constexpr int kRunWarps = kPackThreads / 32;
constexpr int kRunChunk = 128;   // queue entries staged in shared memory at a time
constexpr unsigned kRoomSlow = 0xFFFFu, kRoomMax = 0x7FFEu, kRpDead = 0x80000000u;
constexpr size_t kRunArrayBytes = (size_t)kTopoCap * (kRunMask * 4 + kRunHost * 2) + (size_t)kActCap * 4;

struct RunVariant {
  uint32_t opts[kRunW32];
  uint64_t vals[KSCHED_MAX_KEYS];
  uint64_t meta;
  long long q[KSCHED_MAX_RES];
  long long b1[kHotRes], b2[kHotRes];
  uint32_t qp;
  uint32_t rp;            // room of the fresh node for further pods of the class (+ dead flag)
  unsigned short fl;      // HotSmem::flags of the fresh node (front bits, request keys, template)
  uint8_t dom[kRunMask];  // domain each spread relation pinned
};
struct RunCtx {
  uint32_t cls;           // class the relation tables and variants belong to (KSCHED_NONE: none)
  int eligible;
  int n_host, n_mask, n_var, var_next;
  int tomb;               // nodes tombstoned by the current run
  int h_row[kRunHost], h_group[kRunHost], h_lim[kRunHost];  // h_lim: largest count of the group on a node that still admits the pod
  int h_inc[kRunHost];    // hostnames that got their first matching pod in this run (grp_host_total)
  uint8_t h_times[kRunHost];
  int m_group[kRunMask], m_skew[kRunMask];
  uint8_t m_key[kRunMask], m_self[kRunMask], m_rec[kRunMask], m_wk[kRunMask];
  uint32_t m_registered[kRunMask], m_neutral[kRunMask], m_tallow[kRunMask];
  int32_t cnt[kRunWarps][kRunMask][kRunDom];  // one copy of the spread counters per warp (updated by its lane 0)
  unsigned long long red_key[2][32];
  unsigned red_pay[2][32];
  uint32_t q_pod[2][kRunChunk], q_cls[2][kRunChunk];  // upcoming queue entries (pod, class), double-buffered
  int32_t q_node[2][kRunChunk];                        // where the entry was placed (ksched_result.assign)
  int q_end[2];           // first staged entry of another class (or the chunk length), per buffer
  int lv_cnt[2];          // level step: members appended to the tie list (double-buffered)
  int lv_fill[2];         // fill step: pods the only eligible node takes
  RunVariant var[kRunVariants];
};
__shared__ RunCtx g_rc;

// ---- mask run: the class-run loop for ONE spread relation over a mask key (zone spread), driven by warp 0 alone ----------
// The accepting nodes are kept in singly linked lists in the reference's order (pod count, then tie-break), one per
// domain they are pinned to plus one for the nodes not pinned yet; they are sorted once per run (buckets by list and count,
// ranks by counting inside the bucket). An accepting node moves to the FRONT of the block of count + 1 of its domain's
// list (its new tie-break is the smallest so far), a fresh node goes to the END of the block of count 1. Each lane keeps
// the head of its list, the node after it and the tail of the head's bucket in registers, so a pod's node is the smallest
// head key over the lists of the admissible domains: a few warp reductions, no block barrier and no shared-memory load on
// the critical path instead of a scan of every open node. Anything the lists cannot represent hands the run back to the
// per-pod loop.
constexpr int kM1Dom = 8;             // domains with ids < kM1Dom; list kM1Dom holds the nodes that admit every registered domain
constexpr int kM1Lists = kM1Dom + 1;
constexpr int kM1Lv = 12;             // pod counts < kM1Lv
constexpr uint16_t kM1None = 0xFFFF;
constexpr int kM1Win = 16;            // lanes kM1Win .. kM1Win + kM1Dom + 1: the first nodes of the unpinned list in a round
static_assert(kM1Win > kM1Dom && kM1Win + kM1Dom + 1 < 32, "the unpinned window needs its own lanes");
struct M1Ctx {
  uint16_t tl[kM1Lv][kM1Lists];       // last node of the bucket (kM1None: empty)
  uint16_t head[kM1Lists];            // first node of the list (between two entries of the warp loop)
  uint16_t ap[kM1Lv][kM1Lists];       // build: the bucket is arr[ap .. ae)
  uint16_t ae[kM1Lv][kM1Lists];
  int bcnt[kM1Lv * kM1Lists];         // build: members per bucket (bucket = list * kM1Lv + count)
  int bad;                            // build: a node the lists cannot represent
  int out_adv, out_reason, out_tick, out_n_new, out_n_active;
  int n_fresh;                        // nodes created by this entry of the warp loop: slot | variant << 16; their global
  uint32_t fr[kRunChunk];             // state (option words, requirement values, requests, ...) is stored by the CTA afterwards
};
__shared__ M1Ctx g_m1;

struct RunIO {
  int qi, head, qlen, tick, seq, n_active, n_new, parity;
  long long add_calls;
  int placed;        // pods this call consumed
  int status;        // 0 the run ended (class change / end of the first pass); 1 the pod at qi needs generic_step; 2 class not eligible
  int fresh_valid, fresh_a;  // in: generic_step has just created node slot fresh_a for fresh_cls (nothing happened since)
  uint32_t fresh_cls;
};
__shared__ RunIO g_rio;

// first domain in (count, id) order among `cand` (non-empty)
__device__ __forceinline__ int run_pick(uint32_t cand, const int32_t* cn) {
  int d = __ffs(cand) - 1;
  cand &= cand - 1;
  int32_t best = cn[d];
  while (cand) {
    const int e = __ffs(cand) - 1;
    cand &= cand - 1;
    if (cn[e] < best) { best = cn[e]; d = e; }
  }
  return d;
}
// How many more pods with request vector `req` (keys `res`) the node at slot a can take: exact by the Pareto front of its
// options (quick_fit for the k-th pod <=> k <= room); kRoomSlow when the front is not exact.
__device__ __noinline__ unsigned run_room(const HotSmem* hs, int a, const long long* req, uint32_t res, int RH) {
  const unsigned short fl = hs->flags[a];
  const uint32_t qp = ((fl >> 1) & 0xF) | res;
  long long best = 0;
  bool inexact_ok = true;
  for (int f = 0; f < 2; ++f) {
    if (f == 1 && !(fl & kFlTwo)) break;
    long long rf = kRoomMax;
    for (int r = 0; r < RH; ++r) {
      if (!((qp >> r) & 1)) continue;
      const long long slack = (f ? hs->bound2[r][a] : hs->bound[r][a]) - hs->q[r][a];
      if (req[r] > 0) {
        const long long k = slack < req[r] ? 0 : slack / req[r];
        rf = k < rf ? k : rf;
      } else if (slack < 0) rf = 0;
    }
    if (f == 0) inexact_ok = rf > 0;
    best = rf > best ? rf : best;
  }
  if (!(fl & kFlExact)) return inexact_ok ? kRoomSlow : 0;  // per-resource maxima only: a necessary test
  return (unsigned)best;
}

__device__ __noinline__ void class_run(const PodRegs& first_in) {
  KS_K2
  RunCtx& rc = g_rc;
  RunIO& io = g_rio;
  HotSmem* hs = reinterpret_cast<HotSmem*>(dyn_smem);
  uint32_t* zv = reinterpret_cast<uint32_t*>(dyn_smem + sizeof(HotSmem) + s.run_off);  // [kRunMask][kTopoCap] bits 0..15 admitted domains, 16 exact (In), 17 present
  uint32_t* rpv = zv + (size_t)kRunMask * kTopoCap;                                      // [kActCap] room | placed << 16 | dead
  uint16_t* hc = reinterpret_cast<uint16_t*>(rpv + kActCap);                             // [kRunHost][kTopoCap]
  const uint32_t* tmpl_taintset = g_tmpl_taintset;
  const int tid = threadIdx.x, T = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = T >> 5;
  const int NE = s.n_existing, MAXN = s.max_new, W32 = c.W32;
  const int RH = c.n_res < kHotRes ? c.n_res : kHotRes;
  const int hstride = s.n_existing + s.max_new;
  // the pod row's words, in registers (identical for every pod of the run)
  const unsigned cls = (unsigned)first_in.cls64;
  const uint32_t p_res = first_in.res;
  const uint64_t p_tol = first_in.tol;
  long long p_req[kHotRes];
#pragma unroll
  for (int r = 0; r < kHotRes; ++r) p_req[r] = first_in.req[r];
  const bool topo = first_in.topo_begin != first_in.topo_end;
  const bool plain = plain_pod_regs(first_in);
  const bool simple = !topo;
  const uint32_t topo_begin = first_in.topo_begin, topo_end = first_in.topo_end;
  const int qi0 = io.qi, seq0 = io.seq;
  int qi = qi0, qlen = io.qlen, tick = io.tick, n_active = io.n_active, n_new = io.n_new, parity = io.parity;
  const int fresh_valid = io.fresh_valid && io.fresh_cls == cls, fresh_a = io.fresh_a;
  const int CH = T < kRunChunk ? T : kRunChunk;  // queue entries staged at a time: one per thread
  if (tid == 0) { rc.q_end[0] = CH; rc.q_end[1] = CH; rc.lv_cnt[0] = 0; rc.lv_cnt[1] = 0; }  // (nobody reads these outside class_run)
  const bool new_cls = rc.cls != cls;  // read BEFORE the barrier: thread 0 rewrites rc.cls right after it (racecheck, round 2)
  __syncthreads();  // everybody has read g_rio; earlier readers of g_rc are done

  // ---- relation tables (once per class)
  if (new_cls) {
    if (tid == 0) {
      rc.cls = cls;
      rc.n_var = 0; rc.var_next = 0; rc.n_host = 0; rc.n_mask = 0;
      int ok = 1;
      if (topo) {
        if (c.n_templates != 1) ok = 0;
        for (uint32_t e = topo_begin; e < topo_end && ok; ++e) {
          const RelX x = s.relx[e];
          const int g = (int)x.group;
          if (!(x.flags & KSCHED_TOPO_CONSTRAINS)) { ok = 0; break; }            // record-only relations: generic step
          if (!s.grp_active[g] || s.grp_min_slot[g] != 0) { ok = 0; break; }      // relaxation-created groups: generic step
          if ((x.flags & KSCHED_TOPO_RECORDS) && x.has_filter) { ok = 0; break; }  // TopologyNodeFilter: generic step
          const int times = ((x.flags & KSCHED_TOPO_RECORDS) ? 1 : 0) + ((x.flags & KSCHED_TOPO_RECORDS_INVERSE) ? 1 : 0);
          const int self = (x.flags & KSCHED_TOPO_SELECTS) ? 1 : 0;
          if (x.key == KSCHED_KEY_HOSTNAME) {
            if (x.type == 1 || rc.n_host == kRunHost) { ok = 0; break; }
            const int j = rc.n_host++;
            rc.h_row[j] = x.host_row; rc.h_group[j] = g; rc.h_times[j] = (uint8_t)times;
            // spread: count + self <= maxSkew (min is 0 for hostnames, topologygroup.go:186-188); anti-affinity: count == 0
            long long lim = x.type == 0 ? (long long)x.max_skew - self : 0;
            rc.h_lim[j] = lim > 0x10000 ? 0x10000 : (lim < -1 ? -1 : (int)lim);
          } else {
            const int k = x.key;
            if (x.type != 0 || rc.n_mask == kRunMask || (x.flags & KSCHED_TOPO_RECORDS_INVERSE) || (c.keys[k].dict_mask >> kRunDom)) { ok = 0; break; }
            for (int i = 0; i < rc.n_mask; ++i) if (rc.m_key[i] == k) ok = 0;
            if (!ok) break;
            const int j = rc.n_mask++;
            rc.m_group[j] = g; rc.m_skew[j] = x.max_skew; rc.m_key[j] = (uint8_t)k;
            rc.m_self[j] = (uint8_t)self; rc.m_rec[j] = (x.flags & KSCHED_TOPO_RECORDS) ? 1 : 0;
            rc.m_wk[j] = c.keys[k].well_known != 0; rc.m_neutral[j] = (uint32_t)c.pin_neutral[k];
            const Req tr = ksched::req_load(c.templates[0].reqs, nullptr, k);
            rc.m_tallow[j] = (uint32_t)(tr.present ? ksched::req_allowed(tr, c.keys[k].dict_mask, key_meta(c, k)) : c.keys[k].dict_mask);
          }
        }
      }
      rc.eligible = ok;
    }
    __syncthreads();
  }
  if (!rc.eligible || (topo && n_active > kTopoCap)) {
    if (tid == 0) { io.status = rc.eligible ? 1 : 2; io.placed = 0; io.parity = parity; }
    __syncthreads();
    return;
  }
  const int n_host = rc.n_host, n_mask = rc.n_mask;

  // ---- queue staging: the next CH (pod, class) entries; the chunk after them is fetched into registers meanwhile
  const ksched_pod_row* ffd_rows = reinterpret_cast<const ksched_pod_row*>(s.rows);
  int cb = qi, buf = 0;
  uint32_t nx_pod = 0, nx_cls = KSCHED_NONE;
  if (tid < CH) {
    const int idx = cb + tid;
    uint32_t pd = 0, pc = KSCHED_NONE;
    if (idx < s.n_pods) { pd = s.order[idx]; pc = (uint32_t)ffd_rows[idx].reserved; }
    rc.q_pod[0][tid] = pd; rc.q_cls[0][tid] = pc;
    const unsigned mm = __ballot_sync(0xffffffffu, pc != cls);  // CH is a multiple of 32: whole warps
    if (lane == 0 && mm) atomicMin(&rc.q_end[0], (tid & ~31) + __ffs(mm) - 1);
    const int idx2 = idx + CH;
    if (idx2 < s.n_pods) { nx_pod = s.order[idx2]; nx_cls = (uint32_t)ffd_rows[idx2].reserved; }
  }
  // ---- per-run state: spread counters (one copy per warp), per-node inputs (each thread fills the slots it owns)
  if (tid == 0) rc.tomb = 0;
  if (tid < kRunHost) rc.h_inc[tid] = 0;
  if (topo) {
    for (int j = 0; j < n_mask; ++j) {
      if (lane < kRunDom) rc.cnt[warp][j][lane] = s.grp_cnt[(size_t)rc.m_group[j] * 64 + lane];
      if (tid == 0) rc.m_registered[j] = (uint32_t)s.grp_registered[rc.m_group[j]];
    }
  }
  for (int a = tid; a < n_active; a += T) {
    const unsigned short fl = hs->flags[a];
    unsigned rm;
    if (!((p_tol >> tmpl_taintset[fl >> 8]) & 1)) rm = 0;                        // Taints.Tolerates
    else if (simple && hs->rejected[a] == cls) rm = 0;                           // memo: refused this class, untouched since
    else if (simple && !plain && hs->absorbed[a] != cls) rm = kRoomSlow;         // requirement verdict unknown for this class
    else rm = run_room(hs, a, p_req, p_res, RH);
    if (topo) {
      const int n = hs->node[a];
      for (int j = 0; j < n_host; ++j) {
        const uint16_t v = s.grp_host[(size_t)rc.h_row[j] * hstride + NE + n];
        hc[j * kTopoCap + a] = v;
        if ((int)v > rc.h_lim[j]) rm |= kRpDead;
      }
      const uint64_t meta = s.nn_meta[n];
      for (int j = 0; j < n_mask; ++j) {
        const int k = rc.m_key[j];
        const Req r = load_soa(s.nn_vals, meta, MAXN, n, k);
        const uint32_t allowed = (uint32_t)(r.present ? ksched::req_allowed(r, c.keys[k].dict_mask, key_meta(c, k)) : c.keys[k].dict_mask);
        zv[j * kTopoCap + a] = allowed | ((r.present && !r.complement) ? 1u << 16 : 0) | (r.present ? 1u << 17 : 0);
      }
    }
    rpv[a] = rm;
  }
  __syncthreads();
  // ---- capture the node generic_step has just created for this class as a fresh-node variant
  if (fresh_valid && !s.any_limits && W32 <= kRunW32 && fresh_a == n_active - 1 && fresh_a >= 0) {
    const int a = fresh_a, n = hs->node[a];
    int dom[kRunMask] = {0, 0};
    bool ok = true;
#pragma unroll
    for (int j = 0; j < kRunMask; ++j) {
      if (j >= n_mask) continue;
      const uint32_t z = zv[j * kTopoCap + a], v = z & 0xFFFF;
      if (!v || (v & (v - 1)) || !(z & (1u << 16))) ok = false;
      else dom[j] = __ffs(v) - 1;
    }
    for (int i = 0; i < rc.n_var && ok; ++i) {
      bool same = (rc.var[i].fl >> 8) == (hs->flags[a] >> 8);
#pragma unroll
      for (int j = 0; j < kRunMask; ++j) same = same && (j >= n_mask || rc.var[i].dom[j] == dom[j]);
      if (same) ok = false;  // already known
    }
    const int slot = rc.var_next;  // read BEFORE the barrier: thread 0 moves it while the others still copy (racecheck warning, round 2)
    __syncthreads();  // rc.n_var / var_next read by everybody before thread 0 moves them
    if (ok) {
      RunVariant& v = rc.var[slot];
      for (int w = tid; w < W32; w += T) v.opts[w] = s.nn_opts[(size_t)w * MAXN + n];
      if (tid < KSCHED_MAX_KEYS) v.vals[tid] = tid < c.n_keys ? s.nn_vals[(size_t)tid * MAXN + n] : 0;
      if (tid == 0) {
        v.meta = s.nn_meta[n];
        for (int r = 0; r < KSCHED_MAX_RES; ++r) v.q[r] = r < kHotRes ? hs->q[r][a] : s.nn_req[(size_t)r * MAXN + n];
        for (int r = 0; r < kHotRes; ++r) { v.b1[r] = hs->bound[r][a]; v.b2[r] = hs->bound2[r][a]; }
        v.qp = s.nn_req_present[n];
        v.fl = hs->flags[a];
        v.rp = rpv[a] & (kRpDead | 0xFFFF);
        for (int j = 0; j < kRunMask; ++j) v.dom[j] = (uint8_t)dom[j];
        rc.var_next = (slot + 1) % kRunVariants;
        if (rc.n_var < kRunVariants) rc.n_var++;
      }
      __syncthreads();
    }
  }

  long long min_req[kHotRes];
#pragma unroll
  for (int r = 0; r < kHotRes; ++r) min_req[r] = r < RH ? s.min_req[r] : 0;
  // relation constants of the commit, in registers
  int h_times_sum = 0;
#pragma unroll
  for (int j = 0; j < kRunHost; ++j) if (j < n_host) h_times_sum += rc.h_times[j];
  const uint32_t m_reg0 = n_mask > 0 ? rc.m_registered[0] : 0, m_reg1 = n_mask > 1 ? rc.m_registered[1] : 0;
  const int m_bias0 = n_mask > 0 ? (int)rc.m_self[0] - rc.m_skew[0] : 0, m_bias1 = n_mask > 1 ? (int)rc.m_self[1] - rc.m_skew[1] : 0;
  const bool m_rec0 = n_mask > 0 && rc.m_rec[0], m_rec1 = n_mask > 1 && rc.m_rec[1];
  int status = 0;
  const bool lvl = s.use_level_run && n_mask == 0;
  // mask run (see M1Ctx): one mask-key spread relation, domains and counts small enough for the lists
  M1Ctx& m1 = g_m1;
  bool m1_ok = s.use_mask_run && n_mask == 1 && (m_reg0 >> kM1Dom) == 0;
  bool m1_built = false;
  uint16_t* m1_arr = reinterpret_cast<uint16_t*>(zv + kTopoCap);  // the second mask relation's plane is unused (n_mask == 1)
  uint16_t* m1_nxt = m1_arr + kTopoCap;
  uint32_t* lvt = zv;  // level step: tie-breaks of the level's members (the zone words are unused when n_mask == 0)
  int lvp = 0;
#ifdef KSCHED_PROFILE_PACK
  const long long cr_t0 = clock64();
  int cr_it[4] = {0, 0, 0, 0};  // iterations: level, fill, fresh, per-pod argmin
#define CR_IT(k) { ++cr_it[k]; }
#else
#define CR_IT(k)
#endif

  while (true) {
    int i = qi - cb;
    if (i == CH) {  // chunk consumed: store its assignments, registers -> the other buffer, fetch the chunk after
      __syncthreads();  // the last commit's q_node entry is visible
      if (tid < CH) {
        const uint32_t pd = rc.q_pod[buf][tid];
        int nd = rc.q_node[buf][tid];
        if (nd < -1) nd = NE + hs->node[-nd - 2];  // the mask run stores the slot
        s.assign[pd] = nd;
        s.place_seq[pd] = seq0 + (cb - qi0) + tid;
      }
      buf ^= 1;
      cb += CH;
      i = 0;
      if (tid < CH) {
        rc.q_pod[buf][tid] = nx_pod; rc.q_cls[buf][tid] = nx_cls;
        const unsigned mm = __ballot_sync(0xffffffffu, nx_cls != cls);
        if (lane == 0 && mm) atomicMin(&rc.q_end[buf], (tid & ~31) + __ffs(mm) - 1);
        const int idx2 = cb + CH + tid;
        nx_cls = KSCHED_NONE;
        if (idx2 < s.n_pods) { nx_pod = s.order[idx2]; nx_cls = (uint32_t)ffd_rows[idx2].reserved; }
      }
      __syncthreads();
      if (tid == 0) rc.q_end[buf ^ 1] = CH;  // the consumed buffer: its next atomicMin comes after the next chunk's first barrier
    }
    if (rc.q_cls[buf][i] != cls) break;  // class change or end of the first pass
#ifdef KSCHED_PROFILE_PACK
    const long long m1_t0 = clock64();
#endif
    if (m1_ok) {
      if (!m1_built) {
        // ---- build the lists (once per call; nothing of this call has been committed yet, so nn_last is free as scratch)
        m1_built = true;
        uint8_t* t_b = reinterpret_cast<uint8_t*>(hs->nn_last);              // bucket of slot a (0xFF: not a member)
        uint16_t* t_pos = reinterpret_cast<uint16_t*>(t_b + kTopoCap);        // its arrival order inside the bucket
        uint16_t* t_slot = t_pos + kTopoCap;                                  // members, bucket by bucket, unsorted
        uint32_t* t_tie = reinterpret_cast<uint32_t*>(t_slot + kTopoCap);     // their tie-breaks
        for (int b = tid; b < kM1Lv * kM1Lists; b += T) m1.bcnt[b] = 0;
        if (tid == 0) m1.bad = 0;
        __syncthreads();
        for (int a = tid; a < n_active; a += T) {
          const uint32_t rp = rpv[a];
          int b = 0xFF;
          if ((rp & 0xFFFF) != 0 && !(rp & kRpDead)) {
            const uint32_t z = zv[a], adm = z & 0xFFFF;
            const unsigned cn = (unsigned)(hs->key[a] >> 32);
            int list = -1;
            if (adm && !(adm & (adm - 1)) && (z & (1u << 16))) {  // pinned to one domain
              if (adm & m_reg0) list = __ffs(adm) - 1;             // (a domain that is not registered never admits a pod)
            } else if ((adm & m_reg0) == m_reg0) list = kM1Dom;     // admits every registered domain
            else if (adm & m_reg0) m1.bad = 1;                      // some of them: per-pod loop
            if (list >= 0) {
              if (cn >= (unsigned)kM1Lv) m1.bad = 1;
              else { b = list * kM1Lv + (int)cn; t_pos[a] = (uint16_t)atomicAdd(&m1.bcnt[b], 1); }
            }
          }
          t_b[a] = (uint8_t)b;
        }
        __syncthreads();
        if (warp == 0) {  // exclusive scan of the bucket sizes -> arr segments
          int run = 0;
          for (int b0 = 0; b0 < kM1Lv * kM1Lists; b0 += 32) {
            const int b = b0 + lane;
            const int v = b < kM1Lv * kM1Lists ? m1.bcnt[b] : 0;
            int inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
            if (b < kM1Lv * kM1Lists) {
              const int list = b / kM1Lv, lv = b - list * kM1Lv;
              m1.ap[lv][list] = (uint16_t)(run + inc - v);
              m1.ae[lv][list] = (uint16_t)(run + inc);
            }
            run += __shfl_sync(0xffffffffu, inc, 31);
          }
        }
        __syncthreads();
        const bool bad = m1.bad != 0;
        if (!bad) {
          for (int a = tid; a < n_active; a += T) {
            const int b = t_b[a];
            if (b == 0xFF) continue;
            const int list = b / kM1Lv, lv = b - list * kM1Lv;
            const int j = m1.ap[lv][list] + t_pos[a];
            t_slot[j] = (uint16_t)a;
            t_tie[j] = (uint32_t)hs->key[a];
          }
        }
        __syncthreads();
        if (!bad) {
          for (int a = tid; a < n_active; a += T) {
            const int b = t_b[a];
            if (b == 0xFF) continue;
            const int list = b / kM1Lv, lv = b - list * kM1Lv;
            const int p0 = m1.ap[lv][list], p1 = m1.ae[lv][list];
            const uint32_t tie = (uint32_t)hs->key[a];
            int rank = 0;
            for (int j = p0; j < p1; ++j) rank += t_tie[j] < tie;
            m1_arr[p0 + rank] = (uint16_t)a;
            t_pos[a] = (uint16_t)(p0 + rank);
          }
        }
        __syncthreads();
        if (!bad) {  // link every list (its buckets are contiguous in arr), tails and heads
          for (int a = tid; a < n_active; a += T) {
            const int b = t_b[a];
            if (b == 0xFF) continue;
            const int list = b / kM1Lv, gp = t_pos[a];
            m1_nxt[a] = gp + 1 < (int)m1.ae[kM1Lv - 1][list] ? m1_arr[gp + 1] : kM1None;
          }
          for (int b = tid; b < kM1Lv * kM1Lists; b += T) {
            const int list = b / kM1Lv, lv = b - list * kM1Lv;
            m1.tl[lv][list] = m1.ae[lv][list] > m1.ap[lv][list] ? m1_arr[m1.ae[lv][list] - 1] : kM1None;
          }
          if (tid < kM1Lists) m1.head[tid] = m1.ae[kM1Lv - 1][tid] > m1.ap[0][tid] ? m1_arr[m1.ap[0][tid]] : kM1None;
        }
        __syncthreads();
        if (bad) m1_ok = false;
#ifdef KSCHED_PROFILE_PACK
        if (tid == 0) { s.counters[38] += clock64() - m1_t0; s.counters[47] += bad ? 1 : 0; }
#endif
      }
    }
#ifdef KSCHED_PROFILE_PACK
    const long long m1_t1 = clock64();
#endif
    if (m1_ok) {
      if (warp == 0) {
        const int L = lane;
        const unsigned FULL = 0xffffffffu;
        int cnt_d = L < kM1Dom ? rc.cnt[0][0][L] : 0;
        const bool valid = L < kM1Dom && ((m_reg0 >> L) & 1);
        // this lane's list: head (slot, key, room word), the node after it, the tail of the head's bucket, the first node
        // behind that bucket and its pod count
        int h = -1, n1 = -1, tcur = -1, bn = -1, bnc = 0;
        unsigned long long hk = ~0ull, nk = ~0ull;
        uint32_t hr = 0, nr = 0;
        auto nxt_of = [&](int sl) -> int { const uint16_t v = m1_nxt[sl]; return v == kM1None ? -1 : (int)v; };
        auto level_state = [&]() {
          if (h < 0) { tcur = -1; bn = -1; bnc = 0; return; }
          tcur = m1.tl[(int)(hk >> 32)][L];
          bn = nxt_of(tcur);
          bnc = bn >= 0 ? (int)(hs->key[bn] >> 32) : 0;
        };
        if (L < kM1Lists) {
          h = m1.head[L] == kM1None ? -1 : (int)m1.head[L];
          if (h >= 0) { hk = hs->key[h]; hr = rpv[h]; n1 = nxt_of(h); }
          if (n1 >= 0) { nk = hs->key[n1]; nr = rpv[n1]; }
          level_state();
        }
        // node a (key ak, room word ar) enters this lane's list at the FRONT of the block of count La
        auto insert_front = [&](int a, int La, unsigned long long ak, uint32_t ar) {
          const int hl = h >= 0 ? (int)(hk >> 32) : 0x7fffffff;
          if (hl >= La) {  // nothing lies below: the new head
            m1_nxt[a] = h >= 0 ? (uint16_t)h : kM1None;
            if (hl > La) { m1.tl[La][L] = (uint16_t)a; tcur = a; bn = h; bnc = hl; }
            n1 = h; nk = hk; nr = hr;
            h = a; hk = ak; hr = ar;
          } else if (bn < 0 || bnc >= La) {  // right behind the head's bucket
            m1_nxt[a] = bn >= 0 ? (uint16_t)bn : kM1None;
            m1_nxt[tcur] = (uint16_t)a;
            if (bn < 0 || bnc > La) m1.tl[La][L] = (uint16_t)a;
            if (tcur == h) { n1 = a; nk = ak; nr = ar; }
            bn = a; bnc = La;
          } else {  // behind the last bucket below La (the head's level is not the one)
            int lv = La - 1;
            while (m1.tl[lv][L] == kM1None) --lv;
            const int pred = m1.tl[lv][L];
            m1_nxt[a] = m1_nxt[pred];
            m1_nxt[pred] = (uint16_t)a;
            if (m1.tl[La][L] == kM1None) m1.tl[La][L] = (uint16_t)a;
            if (pred == h) { n1 = a; nk = ak; nr = ar; }
            if (pred == tcur) { bn = a; bnc = La; }
          }
        };
        // a fresh node (count 1, the largest tie-break so far) enters at the END of the block of count 1
        auto insert_back1 = [&](int a, unsigned long long ak, uint32_t ar) {
          const int hl = h >= 0 ? (int)(hk >> 32) : 0x7fffffff;
          if (hl > 1) {
            m1_nxt[a] = h >= 0 ? (uint16_t)h : kM1None;
            m1.tl[1][L] = (uint16_t)a;
            tcur = a; bn = h; bnc = hl;
            n1 = h; nk = hk; nr = hr;
            h = a; hk = ak; hr = ar;
          } else if (hl == 1) {
            m1_nxt[a] = bn >= 0 ? (uint16_t)bn : kM1None;
            m1_nxt[tcur] = (uint16_t)a;
            m1.tl[1][L] = (uint16_t)a;
            if (tcur == h) { n1 = a; nk = ak; nr = ar; }
            tcur = a;
          } else {  // nodes without pods in front (not produced by the scheduler, kept exact anyway)
            int lv = 1;
            while (m1.tl[lv][L] == kM1None) --lv;
            const int pred = m1.tl[lv][L];
            m1_nxt[a] = m1_nxt[pred];
            m1_nxt[pred] = (uint16_t)a;
            m1.tl[1][L] = (uint16_t)a;
            if (pred == h) { n1 = a; nk = ak; nr = ar; }
            if (pred == tcur) { bn = a; bnc = 1; }
          }
        };
        // the head (pod count c) leaves this lane's list: the node behind it moves up, the one behind that is fetched (it is used
        // at this list's next pop)
        auto pop_head = [&](int c) {
          h = n1; hk = nk; hr = nr;
          n1 = -1; nk = ~0ull; nr = 0;
          if (h >= 0) {
            n1 = nxt_of(h);
            if (n1 >= 0) { nk = hs->key[n1]; nr = rpv[n1]; }
          }
          if (h < 0 || (int)(hk >> 32) != c) {  // the bucket of count c is exhausted
            m1.tl[c][L] = kM1None;
            level_state();
          }
        };
        // skew 1 with a self-matching selector: only the domains with the fewest pods admit a pod, so once every one of them has
        // a pinned node at hand and the unpinned nodes come later in the order, the next pods go one to each of these domains,
        // smallest head key first - a whole round is committed at once, every lane its own domain
        const bool rounds = m_rec0 && m_bias0 == 0;
        int li = i, ltick = tick, lnew = n_new, lact = n_active, nfr = 0;
        int i_end = rc.q_end[buf];
        if (i + qlen < i_end) i_end = i + qlen;
        int reason = 0;  // 0: the staged entries of the class are consumed; 1: the pod at li needs generic_step; 2: per-pod loop from li on
        // count + self - min <= maxSkew as count - min <= slack in 32 bits: counts are pod counts (< 2^30), so a slack of 2^30
        // or more admits every domain exactly like the 64-bit form of the per-pod loop
        const int slack = m_bias0 < -(1 << 30) ? (1 << 30) : -m_bias0;
#ifdef KSCHED_PROFILE_PACK
        // iterations by kind (k: 0 round of pinned heads, 1 round with fresh nodes, 2 round that pins unpinned nodes, 3 single
        // step on a pinned head, 4 single step that pins an unpinned node, 5 single fresh node): count, pods, cycles
#define M1_KIND(k, pods) { if (L == 0) { s.counters[48 + 3 * (k)] += 1; s.counters[49 + 3 * (k)] += (pods); s.counters[50 + 3 * (k)] += clock64() - it_t0; } }
        // declined rounds (r: 0 na <= 1, 1 too few staged entries, 2 unpinned head first, 3 room kRoomSlow, 4 count + 1 >= kM1Lv,
        // 5 no fresh node possible, 6 unpinned round: too few candidates, 7 unpinned round: a pin precondition fails)
#define M1_DECLINE(r) { if (L == 0) s.counters[66 + (r)] += 1; }
#else
#define M1_KIND(k, pods) {}
#define M1_DECLINE(r) {}
#endif
        while (li < i_end) {
#ifdef KSCHED_PROFILE_PACK
          const long long it_t0 = clock64();
#endif
          const int mn = __reduce_min_sync(FULL, valid ? cnt_d : INT32_MAX);
          const bool allowed = valid && cnt_d - mn <= slack;
          const unsigned okm = __ballot_sync(FULL, allowed);
          const bool cand_ok = L < kM1Dom ? allowed : (L == kM1Dom && okm != 0);  // an empty list keeps hk = ~0
          const unsigned long long key = cand_ok ? hk : ~0ull;
          const unsigned long long wkey = warp_min_u64(key);
#ifdef KSCHED_PROFILE_PACK
          {  // how often a whole round (one pod per admissible domain, all from pinned lists) could be placed at once
            const unsigned have = __ballot_sync(FULL, L < kM1Dom && allowed && h >= 0);
            const unsigned long long ukey = __shfl_sync(FULL, hk, kM1Dom);
            unsigned long long mx = (L < kM1Dom && allowed && h >= 0) ? hk : 0ull;
            for (int o = 16; o; o >>= 1) { const unsigned long long t = __shfl_xor_sync(FULL, mx, o); mx = t > mx ? t : mx; }
            const int na = __popc(okm);
            if (L == 0 && na > 1 && have == okm && ukey > mx && i_end - li >= na) s.counters[17] += 1;
            if (L == 0) s.counters[18] += 1;
            if (L == 0 && na > 1) s.counters[19] += 1;
          }
#endif
          if (rounds) {
            const int na = __popc(okm);
            if (na > 1 && i_end - li >= na) {
              const bool act = L < kM1Dom && allowed;
              const bool hd = act && h >= 0;                       // this domain's pod goes to the head of its list
              const unsigned hv = __ballot_sync(FULL, hd), fv = okm & ~hv;  // fv: domains that get a fresh node (no pinned node at hand)
              const bool bad_l = hd && ((hr & 0xFFFF) == kRoomSlow || (int)(hk >> 32) + 1 >= kM1Lv);
              const unsigned long long ukey = __shfl_sync(FULL, hk, kM1Dom);
              const unsigned hi = hd ? (unsigned)(hk >> 32) : 0u;
              const unsigned mhi = __reduce_max_sync(FULL, hi);
              const unsigned mlo = __reduce_max_sync(FULL, (hd && hi == mhi) ? (unsigned)hk : 0u);
              const unsigned long long mx = ((unsigned long long)mhi << 32) | mlo;  // largest head key of the round
              // fresh nodes come last in a round, lowest domain id first (every admissible domain has the same count: run_pick
              // takes the lowest id), and only when no unpinned node is left (it would be taken first)
              int vi_l = -1;
              const int nf = __popc(fv);
              bool fresh_ok = true;
              if (fv) {
                const bool fl = act && h < 0;
                if (fl) for (int v2 = 0; v2 < rc.n_var && vi_l < 0; ++v2) if (rc.var[v2].dom[0] == L) vi_l = v2;
                fresh_ok = ukey == ~0ull && (fv & ~rc.m_tallow[0]) == 0 && !__any_sync(FULL, fl && vi_l < 0) && lnew + nf <= MAXN &&
                           lact + nf <= kActCap && lact + nf <= kTopoCap;
                for (int j = 0; j < n_host; ++j) fresh_ok = fresh_ok && rc.h_lim[j] >= 0;
              }
              if (fresh_ok && !__any_sync(FULL, bad_l) && (hv == 0 || ukey > mx)) {
                int rank = 0;  // position of this lane's node in the round
                for (unsigned m = hv; m; m &= m - 1) {
                  const unsigned long long k2 = __shfl_sync(FULL, hk, __ffs(m) - 1);
                  rank += k2 < hk;
                }
                bool closed_l = false;
                if (hd) {
                  const int a = h;
                  const uint32_t rp = hr;
                  const int c = (int)(hk >> 32);
                  const int mytick = ltick + rank;
                  pop_head(c);
                  uint32_t rp2 = rp - 1 + (1u << 16);
                  for (int j = 0; j < n_host; ++j) {  // Topology.Record, hostname groups
                    const int times = rc.h_times[j];
                    const int old = hc[j * kTopoCap + a];
                    const int now = old + times > 0xFFFF ? 0xFFFF : old + times;
                    if (times) hc[j * kTopoCap + a] = (uint16_t)now;
                    if (now > rc.h_lim[j]) rp2 |= kRpDead;
                  }
                  const unsigned long long nkey = order_key(c + 1, -(mytick + 1));
                  unsigned long long skey = nkey;
                  rc.q_node[buf][li + rank] = -(a + 2);
                  if ((rp2 & 0xFFFF) == 0) {  // the class no longer fits by resources: does anything? (node_closed)
                    const int placed = (rp2 >> 16) & 0x7FFF;
                    long long nq[kHotRes], cb1[kHotRes], cb2[kHotRes];
#pragma unroll
                    for (int r = 0; r < kHotRes; ++r) { nq[r] = hs->q[r][a] + placed * p_req[r]; cb1[r] = hs->bound[r][a]; cb2[r] = hs->bound2[r][a]; }
                    const unsigned short fl = (unsigned short)(hs->flags[a] | ((p_res & 0xF) << 1));
                    if (node_closed(nq, min_req, RH, cb1, cb2, fl)) {
                      skey = ~0ull;
                      hs->nn_last[a] = ((unsigned long long)(unsigned)(c + 1) << 32) | (unsigned)(-(mytick + 1));
                      closed_l = true;
                    }
                  }
                  hs->key[a] = skey;
                  rpv[a] = rp2;
                  if ((rp2 & 0xFFFF) != 0 && !(rp2 & kRpDead)) insert_front(a, c + 1, nkey, rp2);
                  ++cnt_d;
                } else if (act) {  // NewNode + Add replayed from the variant of this lane's domain
                  const RunVariant& v = rc.var[vi_l];
                  const int idx = __popc(fv & ((1u << L) - 1u));
                  const int n = lnew + idx, a = lact + idx;
                  const int mytick = ltick + __popc(hv) + idx;
                  for (int j = 0; j < n_host; ++j) {
                    const int times = rc.h_times[j];
                    hc[j * kTopoCap + a] = (uint16_t)times;
                    if (times) s.grp_host[(size_t)rc.h_row[j] * hstride + NE + n] = (uint16_t)times;
                  }
                  const unsigned long long fkey = order_key(1, mytick + 1);
                  hs->key[a] = fkey;
#pragma unroll
                  for (int r = 0; r < kHotRes; ++r) { hs->q[r][a] = v.q[r]; hs->bound[r][a] = v.b1[r]; hs->bound2[r][a] = v.b2[r]; }
                  hs->node[a] = n;
                  hs->flags[a] = v.fl;
                  hs->absorbed[a] = simple ? cls : KSCHED_NONE;
                  hs->rejected[a] = KSCHED_NONE;
                  rpv[a] = v.rp;
                  rc.q_node[buf][li + __popc(hv) + idx] = NE + n;
                  zv[a] = (1u << L) | (3u << 16);
                  m1.fr[nfr + idx] = (uint32_t)a | ((uint32_t)vi_l << 16);
                  if ((v.rp & 0xFFFF) != 0 && !(v.rp & kRpDead)) insert_back1(a, fkey, v.rp);
                  ++cnt_d;
                }
                if (nf && L < n_host && rc.h_times[L]) rc.h_inc[L] = rc.h_inc[L] + nf;
                const unsigned tb = __ballot_sync(FULL, closed_l);
                if (L == 0 && tb) rc.tomb = rc.tomb + __popc(tb);
                lnew += nf;
                lact += nf;
                nfr += nf;
                ltick += na;
                li += na;
                __syncwarp();
                M1_KIND(nf ? 1 : 0, na)
                continue;
              }
              if (ukey != ~0ull && !(hv == okm && ukey > mx)) {
                // an unpinned node comes before some head (or a domain has no head): the one-pod steps of the round, replayed
                // in key order over the candidates - the heads of the admissible lists and the first na unpinned nodes. A
                // head takes a pod while its domain is still open in the round; an unpinned node takes one and is pinned to
                // the lowest open domain id (run_pick). The window walks one node further than the round can take, so the
                // unpinned list's next head and the node behind it are known without another load.
                const int u0 = __shfl_sync(FULL, h, kM1Dom), u1 = __shfl_sync(FULL, n1, kM1Dom);
                int us = L == kM1Win ? u0 : (L == kM1Win + 1 ? u1 : -1);  // lane kM1Win + j: the j-th node of the unpinned list
                int cur = u1;
                for (int j = 2; j <= na + 1; ++j) {
                  cur = cur >= 0 ? nxt_of(cur) : -1;
                  if (L == kM1Win + j) us = cur;
                }
                unsigned long long uk = ~0ull;
                uint32_t ur = 0;
                if (us >= 0) { uk = hs->key[us]; ur = rpv[us]; }
                const bool un = L >= kM1Win && L < kM1Win + na && us >= 0;
                const bool cnd = hd || un;
                const unsigned long long ck = hd ? hk : uk;
                const unsigned cm = __ballot_sync(FULL, cnd);
                int pos = 0;  // position among the candidates
                for (unsigned m = cm; m; m &= m - 1) pos += __shfl_sync(FULL, ck, __ffs(m) - 1) < ck;
                // 4 bits per position: the head's domain, or 8 for an unpinned node (those come in list order)
                const unsigned long long code = cnd ? (unsigned long long)(un ? 8 : L) << (4 * pos) : 0ull;
                const unsigned long long desc = ((unsigned long long)__reduce_or_sync(FULL, (unsigned)(code >> 32)) << 32) |
                                                __reduce_or_sync(FULL, (unsigned)code);
                unsigned open = okm;
                unsigned long long asg = 0;  // one byte per domain: 0x80 gets a pod | 0x40 from unpinned node j << 3 | position
                int ju = 0;                  // unpinned nodes the round takes
                for (int p = 0, nc = __popc(cm); p < nc && open; ++p) {
                  const int cd = (int)(desc >> (4 * p)) & 15;
                  const int d = cd == 8 ? __ffs(open) - 1 : cd;
                  if ((open >> d) & 1) {
                    asg |= (unsigned long long)(0x80 | (cd == 8 ? 0x40 | ju << 3 : 0) | (na - __popc(open))) << (8 * d);
                    open &= ~(1u << d);
                  }
                  ju += cd == 8;
                }
                const unsigned b = L < kM1Dom ? (unsigned)(asg >> (8 * L)) & 0xFF : 0u;
                const int src = (b & 0x40) ? kM1Win + ((b >> 3) & 7) : L;
                const int ua = __shfl_sync(FULL, us, src);
                const unsigned long long uka = __shfl_sync(FULL, uk, src);
                const uint32_t ura = __shfl_sync(FULL, ur, src);
                // this lane's pod goes to node a (room word rp2's source, count c) at position rank of the round: its own
                // head, or with `pin` the unpinned node the commit pins to this domain
                const bool mine = (b & 0x80) != 0, pin = (b & 0x40) != 0;
                const int rank = b & 7, a = pin ? ua : h;
                const uint32_t rp = pin ? ura : hr;
                const int c = (int)((pin ? uka : hk) >> 32);
                bool bad_m = mine && ((rp & 0xFFFF) == kRoomSlow || c + 1 >= kM1Lv);
                if (pin) bad_m = bad_m || !((rc.m_neutral[0] >> L) & 1) || !((zv[a] & (1u << 17)) || rc.m_wk[0]);
#ifdef KSCHED_PROFILE_PACK
                if (open) M1_DECLINE(6)
                else if (__any_sync(FULL, bad_m)) M1_DECLINE(7)
#endif
                // a domain left open needs a fresh node, and these are only replayed when no unpinned node is left
                if (open == 0 && !__any_sync(FULL, bad_m)) {
                  bool closed_l = false;
                  if (mine) {
                    const int mytick = ltick + rank;
                    if (!pin) pop_head(c);
                    uint32_t rp2 = rp - 1 + (1u << 16);
                    for (int j = 0; j < n_host; ++j) {  // Topology.Record, hostname groups
                      const int times = rc.h_times[j];
                      const int old = hc[j * kTopoCap + a];
                      const int now = old + times > 0xFFFF ? 0xFFFF : old + times;
                      if (times) hc[j * kTopoCap + a] = (uint16_t)now;
                      if (now > rc.h_lim[j]) rp2 |= kRpDead;
                    }
                    const unsigned long long nkey = order_key(c + 1, -(mytick + 1));
                    unsigned long long skey = nkey;
                    rc.q_node[buf][li + rank] = -(a + 2);
                    if (pin) {  // requirements.Add(In{L}) on the node, as the one-pod step does it
                      const int n = hs->node[a], k = rc.m_key[0];
                      zv[a] = (1u << L) | (3u << 16);
                      s.nn_vals[(size_t)k * MAXN + n] = 1ull << L;
                      atomicOr(reinterpret_cast<unsigned long long*>(&s.nn_meta[n]), 1ull << (KSCHED_META_PRESENT_SHIFT + k));
                      atomicAnd(reinterpret_cast<unsigned long long*>(&s.nn_meta[n]), ~(1ull << (KSCHED_META_COMPLEMENT_SHIFT + k)));
                    }
                    if ((rp2 & 0xFFFF) == 0) {  // the class no longer fits by resources: does anything? (node_closed)
                      const int placed = (rp2 >> 16) & 0x7FFF;
                      long long nq[kHotRes], cb1[kHotRes], cb2[kHotRes];
#pragma unroll
                      for (int r = 0; r < kHotRes; ++r) { nq[r] = hs->q[r][a] + placed * p_req[r]; cb1[r] = hs->bound[r][a]; cb2[r] = hs->bound2[r][a]; }
                      const unsigned short fl = (unsigned short)(hs->flags[a] | ((p_res & 0xF) << 1));
                      if (node_closed(nq, min_req, RH, cb1, cb2, fl)) {
                        skey = ~0ull;
                        hs->nn_last[a] = ((unsigned long long)(unsigned)(c + 1) << 32) | (unsigned)(-(mytick + 1));
                        closed_l = true;
                      }
                    }
                    hs->key[a] = skey;
                    rpv[a] = rp2;
                    // (a pinned node enters a list whose own head is not placed in this round: lane L stays its only writer)
                    if ((rp2 & 0xFFFF) != 0 && !(rp2 & kRpDead)) insert_front(a, c + 1, nkey, rp2);
                    ++cnt_d;
                  }
                  // the unpinned list loses its first ju nodes; a bucket they emptied has no tail any more
                  const int nh = __shfl_sync(FULL, us, kM1Win + ju), nn = __shfl_sync(FULL, us, kM1Win + ju + 1);
                  const unsigned long long nhk = __shfl_sync(FULL, uk, kM1Win + ju), nnk = __shfl_sync(FULL, uk, kM1Win + ju + 1);
                  const uint32_t nhr = __shfl_sync(FULL, ur, kM1Win + ju), nnr = __shfl_sync(FULL, ur, kM1Win + ju + 1);
                  const unsigned long long uk_nx = __shfl_down_sync(FULL, uk, 1);
                  const bool emptied = L >= kM1Win && L < kM1Win + ju && (uk_nx >> 32) != (uk >> 32);
                  if (emptied) m1.tl[(int)(uk >> 32)][kM1Dom] = kM1None;
                  const bool any_emptied = __any_sync(FULL, emptied);
                  if (L == kM1Dom) { h = nh; hk = nhk; hr = nhr; n1 = nn; nk = nnk; nr = nnr; }
                  if (any_emptied) {
                    __syncwarp();
                    if (L == kM1Dom) level_state();
                  }
                  const unsigned tb = __ballot_sync(FULL, closed_l);
                  if (L == 0 && tb) rc.tomb = rc.tomb + __popc(tb);
                  ltick += na;
                  li += na;
                  __syncwarp();
                  M1_KIND(2, na)
                  continue;
                }
              }
#ifdef KSCHED_PROFILE_PACK
              else if (ukey != ~0ull && hv != 0 && ukey <= mx) M1_DECLINE(2)
              else if (__any_sync(FULL, bad_l && (hr & 0xFFFF) == kRoomSlow)) M1_DECLINE(3)
              else if (__any_sync(FULL, bad_l)) M1_DECLINE(4)
              else M1_DECLINE(5)
#endif
            } else if (na <= 1) M1_DECLINE(0)
            else M1_DECLINE(1)
          }
          if (wkey != ~0ull) {
            const int wl = __ffs(__ballot_sync(FULL, key == wkey)) - 1;
            const int a = __shfl_sync(FULL, h, wl);
            const uint32_t rp = __shfl_sync(FULL, hr, wl);
            if ((rp & 0xFFFF) == kRoomSlow) { reason = 1; break; }  // the winner needs the full evaluation
            int d = wl;
            const bool pin = wl == kM1Dom;
            if (pin) {  // the placement pins the node's domain: fewest pods, lowest id among the admissible ones (run_pick)
              const int mc = __reduce_min_sync(FULL, allowed ? cnt_d : INT32_MAX);
              d = __ffs(__ballot_sync(FULL, allowed && cnt_d == mc)) - 1;
              if (!((rc.m_neutral[0] >> d) & 1) || !((zv[a] & (1u << 17)) || rc.m_wk[0])) { reason = 1; break; }
            }
            const int c = (int)(wkey >> 32);
            if (L == wl) pop_head(c);
            // ---- commit (the per-pod loop's commit, relation by relation on the first lanes)
            uint32_t rp2 = rp - 1 + (1u << 16);
            bool dead_l = false;
            if (L < n_host) {  // Topology.Record, hostname groups
              const int times = rc.h_times[L];
              const int old = hc[L * kTopoCap + a];
              const int now = old + times > 0xFFFF ? 0xFFFF : old + times;
              if (times) hc[L * kTopoCap + a] = (uint16_t)now;
              dead_l = now > rc.h_lim[L];
            }
            if (n_host > 0 && __any_sync(FULL, dead_l)) rp2 |= kRpDead;
            const unsigned long long nkey = order_key(c + 1, -(ltick + 1));
            if (L == 0) {
              unsigned long long skey = nkey;
              if (pin) {  // requirements.Add(In{d}) on the node
                const int n = hs->node[a], k = rc.m_key[0];
                zv[a] = (1u << d) | (3u << 16);
                s.nn_vals[(size_t)k * MAXN + n] = 1ull << d;
                // two reductions instead of a read-modify-write: the load would stall the whole chain for an L2 round trip
                atomicOr(reinterpret_cast<unsigned long long*>(&s.nn_meta[n]), 1ull << (KSCHED_META_PRESENT_SHIFT + k));
                atomicAnd(reinterpret_cast<unsigned long long*>(&s.nn_meta[n]), ~(1ull << (KSCHED_META_COMPLEMENT_SHIFT + k)));
              }
              rc.q_node[buf][li] = -(a + 2);  // the slot: translated to the node when the chunk is stored
              if ((rp2 & 0xFFFF) == 0) {  // the class no longer fits by resources: does anything? (node_closed)
                const int placed = (rp2 >> 16) & 0x7FFF;
                long long nq[kHotRes], cb1[kHotRes], cb2[kHotRes];
#pragma unroll
                for (int r = 0; r < kHotRes; ++r) { nq[r] = hs->q[r][a] + placed * p_req[r]; cb1[r] = hs->bound[r][a]; cb2[r] = hs->bound2[r][a]; }
                const unsigned short fl = (unsigned short)(hs->flags[a] | ((p_res & 0xF) << 1));
                if (node_closed(nq, min_req, RH, cb1, cb2, fl)) {
                  skey = ~0ull;
                  hs->nn_last[a] = ((unsigned long long)(unsigned)(c + 1) << 32) | (unsigned)(-(ltick + 1));
                  rc.tomb = rc.tomb + 1;
                }
              }
              hs->key[a] = skey;
              rpv[a] = rp2;
            }
            if ((rp2 & 0xFFFF) != 0 && !(rp2 & kRpDead)) {  // still accepts the class: front of the block of count + 1
              if (c + 1 >= kM1Lv) reason = 2;
              else if (L == d) insert_front(a, c + 1, nkey, rp2);
            }
            if (m_rec0 && L == d) ++cnt_d;
            ++ltick;
            ++li;
            __syncwarp();  // lane 0's key / room words before a later pop fetches them
            M1_KIND(pin ? 4 : 3, 1)
            if (reason == 2) break;
          } else {
            // ---- nobody accepts: NewNode + Add replayed from the variant of the domain a fresh node gets
            if (lnew >= MAXN || lact >= kActCap || lact >= kTopoCap || rc.n_var == 0) { reason = 1; break; }
            bool ok = true;
            for (int j = 0; j < n_host; ++j) ok = ok && rc.h_lim[j] >= 0;
            const unsigned cand = rc.m_tallow[0] & okm;
            if (!ok || !cand) { reason = 1; break; }
            const bool in_c = (cand >> L) & 1;  // (cand is a subset of okm: lanes below kM1Dom)
            const int mc = __reduce_min_sync(FULL, in_c ? cnt_d : INT32_MAX);
            const int fd = __ffs(__ballot_sync(FULL, in_c && cnt_d == mc)) - 1;
            int vi = -1;
            for (int v2 = 0; v2 < rc.n_var && vi < 0; ++v2) if (rc.var[v2].dom[0] == fd) vi = v2;
            if (vi < 0) { reason = 1; break; }
            const RunVariant& v = rc.var[vi];
            const int n = lnew, a = lact;
            if (L < n_host) {
              const int times = rc.h_times[L];
              hc[L * kTopoCap + a] = (uint16_t)times;
              if (times) {
                s.grp_host[(size_t)rc.h_row[L] * hstride + NE + n] = (uint16_t)times;
                rc.h_inc[L] = rc.h_inc[L] + 1;
              }
            }
            const unsigned long long fkey = order_key(1, ltick + 1);
            if (L == 0) {
              hs->key[a] = fkey;
#pragma unroll
              for (int r = 0; r < kHotRes; ++r) { hs->q[r][a] = v.q[r]; hs->bound[r][a] = v.b1[r]; hs->bound2[r][a] = v.b2[r]; }
              hs->node[a] = n;
              hs->flags[a] = v.fl;
              hs->absorbed[a] = simple ? cls : KSCHED_NONE;
              hs->rejected[a] = KSCHED_NONE;
              rpv[a] = v.rp;
              rc.q_node[buf][li] = NE + n;
              zv[a] = (1u << fd) | (3u << 16);
              m1.fr[nfr] = (uint32_t)a | ((uint32_t)vi << 16);  // nothing in this loop reads the node's global state
            }
            ++nfr;
            if (L == fd) {
              if ((v.rp & 0xFFFF) != 0 && !(v.rp & kRpDead)) insert_back1(a, fkey, v.rp);  // accepts further pods of the class
              if (m_rec0) ++cnt_d;
            }
            ++ltick; ++lnew; ++lact; ++li;
            __syncwarp();
            M1_KIND(5, 1)
          }
        }
#undef M1_KIND
#undef M1_DECLINE
        __syncwarp();
        // every warp's copy of the spread counters follows (the per-pod loop and the write-back read them)
        if (L < kM1Dom) for (int w = 0; w < nwarps; ++w) rc.cnt[w][0][L] = cnt_d;
        if (L < kM1Lists) m1.head[L] = h >= 0 ? (uint16_t)h : kM1None;
        if (L == 0) { m1.out_adv = li - i; m1.out_reason = reason; m1.out_tick = ltick; m1.out_n_new = lnew; m1.out_n_active = lact; m1.n_fresh = nfr; }
      }
      __syncthreads();
      {  // the global state of the nodes the warp loop created, 64 words per node across the CTA
        const int nfr = m1.n_fresh;
        for (int e = tid; e < nfr * 64; e += T) {
          const uint32_t rec = m1.fr[e >> 6];
          const int a = (int)(rec & 0xFFFF), w = e & 63;
          const RunVariant& v = rc.var[rec >> 16];
          const int n = hs->node[a];
          if (w < W32) s.nn_opts[(size_t)w * MAXN + n] = v.opts[w];
          if (w < c.n_keys) s.nn_vals[(size_t)w * MAXN + n] = v.vals[w];
          if (w < KSCHED_MAX_RES) s.nn_req[(size_t)w * MAXN + n] = v.q[w];
          if (w == 0) {
            s.nn_meta[n] = v.meta;
            s.nn_tmpl[n] = (uint8_t)(v.fl >> 8);
            s.nn_req_present[n] = v.qp;
            s.nn_hp[n] = 0;
            if (((rpv[a] >> 16) & 0x7FFF) == 0) {  // no further pod so far: (1, creation tick); otherwise the run's write-back stores them
              s.nn_count[n] = 1;
              s.nn_tb[n] = (int)((unsigned)hs->key[a] ^ 0x80000000u);
            }
          }
        }
      }
      const int m_adv = m1.out_adv, m_reason = m1.out_reason;
      tick = m1.out_tick; n_new = m1.out_n_new; n_active = m1.out_n_active;
      qi += m_adv;
      qlen -= m_adv;
      __syncthreads();  // out_* are rewritten by the next entry
#ifdef KSCHED_PROFILE_PACK
      if (tid == 0) { s.counters[6] += clock64() - m1_t1; s.counters[7] += m_adv; s.counters[16] += 1; }
#endif
      if (m_reason == 1) { status = 1; break; }
      if (qlen == 0) break;
      if (m_reason == 2) m1_ok = false;
      continue;
    }
    if (lvl && n_active > 0 && n_active <= 32 && s.use_level_warp) {
      // ---- at most 32 open nodes: the level / fill steps of the block below with ONE node per lane of warp 0 and no block
      // barrier (slot a belongs to thread a, as in the block-wide form). Fresh nodes and winners that need the full evaluation
      // go to the block-wide iteration below.
      if (warp == 0) {
        const unsigned FULL = 0xffffffffu;
        const int a = lane;
        const bool mine = a < n_active;
        int li = i, ltick = tick, reason = 0;
        int i_end = rc.q_end[buf];
        if (i + qlen < i_end) i_end = i + qlen;
        while (li < i_end) {
          const uint32_t rp = mine ? rpv[a] : 0u;
          const unsigned long long key = mine ? hs->key[a] : ~0ull;
          const bool el = mine && (rp & 0xFFFF) != 0 && !(rp & kRpDead);
          const unsigned elm = __ballot_sync(FULL, el);
          if (!elm || __any_sync(FULL, el && (rp & 0xFFFF) == kRoomSlow)) { reason = 1; break; }
          const unsigned cn = el ? (unsigned)(key >> 32) : 0xFFFFFFFFu;
          const unsigned c_min = __reduce_min_sync(FULL, cn);
          const bool mem = el && cn == c_min;
          const unsigned memm = __ballot_sync(FULL, mem);
          const int k_av = i_end - li;
          int t = 1, rank = 0, adv_w;
          if (!(elm & (elm - 1))) {  // fill: the only accepting node takes pods until it refuses
            int cap = (int)(rp & 0xFFFF);
            if (mem) {
              for (int j = 0; j < n_host; ++j) {
                const int times = rc.h_times[j], lim = rc.h_lim[j];
                if (!times || lim >= 0x10000) continue;
                if (lim >= 0xFFF0) { cap = 1; continue; }
                const int td = (lim - (int)hc[j * kTopoCap + a]) / times + 1;
                cap = td < cap ? td : cap;
              }
            }
            t = __shfl_sync(FULL, cap, __ffs(memm) - 1);
            t = t < k_av ? t : k_av;
            adv_w = t;
          } else {  // level: the accepting nodes with the fewest pods, one pod each in tie order
            const unsigned tie = (unsigned)key;
            for (unsigned m = memm; m; m &= m - 1) {
              const unsigned tm = __shfl_sync(FULL, tie, __ffs(m) - 1);
              rank += tm < tie;
            }
            const int n_s = __popc(memm);
            adv_w = n_s < k_av ? n_s : k_av;
          }
          if (mem && rank < adv_w) {  // (fill: rank 0 < t)
            uint32_t rp2 = rp - (uint32_t)t + ((uint32_t)t << 16);
            for (int j = 0; j < n_host; ++j) {  // Topology.Record, hostname groups
              const int times = rc.h_times[j];
              const int old = hc[j * kTopoCap + a];
              const int now = old + t * times > 0xFFFF ? 0xFFFF : old + t * times;
              if (times) hc[j * kTopoCap + a] = (uint16_t)now;
              if (now > rc.h_lim[j]) rp2 |= kRpDead;
            }
            const int count = (int)c_min + t;
            const int tb = -(ltick + rank + t);
            unsigned long long nkey = order_key(count, tb);
            const int nd = NE + hs->node[a];
            for (int e = 0; e < t; ++e) rc.q_node[buf][li + rank + e] = nd;
            if ((rp2 & 0xFFFF) == 0) {  // the class no longer fits by resources: does anything? (node_closed)
              const int placed = (rp2 >> 16) & 0x7FFF;
              long long nq[kHotRes], cb1[kHotRes], cb2[kHotRes];
#pragma unroll
              for (int r = 0; r < kHotRes; ++r) { nq[r] = hs->q[r][a] + placed * p_req[r]; cb1[r] = hs->bound[r][a]; cb2[r] = hs->bound2[r][a]; }
              const unsigned short fl = (unsigned short)(hs->flags[a] | ((p_res & 0xF) << 1));
              if (node_closed(nq, min_req, RH, cb1, cb2, fl)) {
                nkey = ~0ull;
                hs->nn_last[a] = ((unsigned long long)(unsigned)count << 32) | (unsigned)tb;
                atomicAdd(&rc.tomb, 1);
              }
            }
            hs->key[a] = nkey;
            rpv[a] = rp2;
          }
          ltick += adv_w;
          li += adv_w;
        }
        if (lane == 0) { g_m1.out_adv = li - i; g_m1.out_reason = reason; g_m1.out_tick = ltick; }
      }
      __syncthreads();
      const int w_adv = g_m1.out_adv, w_reason = g_m1.out_reason;
      tick = g_m1.out_tick;
      qi += w_adv;
      qlen -= w_adv;
      i += w_adv;
      __syncthreads();  // out_* are rewritten by the next entry
      if (qlen == 0) break;
      if (w_reason == 0) continue;  // the staged entries of the class are consumed
      // w_reason == 1: the pod at i takes the block-wide iteration (fresh nodes / full evaluation)
    }
    int adv = 1;       // pods this iteration consumes
    int mode = 0;      // 0: per-pod argmin below; 1: placed by a level / fill step; 2: nobody accepts (fresh node)
    int k_avail = 1;   // pods of the class that may be consumed now: staged, same class, still queued
    if (lvl) {
      // ---- classes without mask-key spread: a node's verdict depends on the node alone, so
      //  * level step: the n accepting nodes with the fewest pods take the next n pods one each, in tie order (each leaves
      //    for the block of count + 1, behind every node of the level);
      //  * fill step: the only accepting node takes pods until it refuses (resources / hostname limits);
      //  * a fresh node is filled the same way in the iteration that creates it.
      k_avail = rc.q_end[buf] - i;
      k_avail = k_avail < qlen ? k_avail : qlen;
      unsigned cmin = 0xFFFFFFFFu;
      int ne = 0;
      bool slow = false;
      for (int a = tid; a < n_active; a += T) {
        const uint32_t rp = rpv[a];
        if ((rp & 0xFFFF) != 0 && !(rp & kRpDead)) {  // tombstones have no room
          const unsigned cn = (unsigned)(hs->key[a] >> 32);
          cmin = cn < cmin ? cn : cmin;
          ++ne;
          slow = slow || (rp & 0xFFFF) == kRoomSlow;
        }
      }
      const unsigned wc = __reduce_min_sync(0xffffffffu, cmin);
      const unsigned wn = __reduce_add_sync(0xffffffffu, (unsigned)ne) | (__any_sync(0xffffffffu, slow) ? 0x80000000u : 0u);
      if (lane == 0) rc.red_key[parity][warp] = ((unsigned long long)wc << 32) | wn;
      __syncthreads();
      const unsigned long long rr = lane < nwarps ? rc.red_key[parity][lane] : 0xFFFFFFFF00000000ull;
      parity ^= 1;
      const unsigned c_min = __reduce_min_sync(0xffffffffu, (unsigned)(rr >> 32));
      const int n_el = (int)__reduce_add_sync(0xffffffffu, (unsigned)rr & 0x7FFFFFFFu);
      const bool any_slow = __any_sync(0xffffffffu, ((unsigned)rr >> 31) != 0);
      if (!any_slow) {
        if (n_el == 0) mode = 2;
        else {
          mode = 1;
          const int lp = lvp;
          lvp ^= 1;
          if (tid == 0) rc.lv_cnt[lp ^ 1] = 0;  // last read before this iteration's first barrier
          // the level's members append their tie-breaks to the list (any order)
          for (int base = 0; base < n_active; base += T) {
            const int a = base + tid;
            bool mem = false;
            unsigned tie = 0;
            if (a < n_active) {
              const uint32_t rp = rpv[a];
              const unsigned long long key = hs->key[a];
              mem = (rp & 0xFFFF) != 0 && !(rp & kRpDead) && (unsigned)(key >> 32) == c_min;
              tie = (unsigned)key;
              if (mem && n_el == 1) {  // fill: how many pods this node takes before it refuses
                int cap = (int)(rp & 0xFFFF);
                for (int j = 0; j < n_host; ++j) {
                  const int times = rc.h_times[j], lim = rc.h_lim[j];
                  if (!times || lim >= 0x10000) continue;
                  if (lim >= 0xFFF0) { cap = 1; continue; }  // saturating counters nearby: one pod at a time
                  const int td = (lim - (int)hc[j * kTopoCap + a]) / times + 1;
                  cap = td < cap ? td : cap;
                }
                rc.lv_fill[lp] = cap < k_avail ? cap : k_avail;
              }
            }
            const unsigned bal = __ballot_sync(0xffffffffu, mem);
            if (bal) {
              const int src = __ffs(bal) - 1;
              int pos0 = 0;
              if (lane == src) pos0 = atomicAdd(&rc.lv_cnt[lp], __popc(bal));
              pos0 = __shfl_sync(0xffffffffu, pos0, src);
              if (mem) lvt[pos0 + __popc(bal & ((1u << lane) - 1u))] = tie;
            }
          }
          __syncthreads();
          const int n_s = rc.lv_cnt[lp];
          const int t_fill = n_el == 1 ? rc.lv_fill[lp] : 1;
          const int k_lvl = n_el == 1 ? 1 : (n_s < k_avail ? n_s : k_avail);
          adv = n_el == 1 ? t_fill : k_lvl;
          CR_IT(n_el == 1 ? 1 : 0)
          for (int a = tid; a < n_active; a += T) {
            const uint32_t rp = rpv[a];
            const unsigned long long key = hs->key[a];
            if (!((rp & 0xFFFF) != 0 && !(rp & kRpDead) && (unsigned)(key >> 32) == c_min)) continue;
            const unsigned tie = (unsigned)key;
            int rank = 0;
            if (n_el != 1) {
              int j = 0;
              for (; j + 4 <= n_s; j += 4) {
                const uint4 v = *reinterpret_cast<const uint4*>(lvt + j);
                rank += (v.x < tie) + (v.y < tie) + (v.z < tie) + (v.w < tie);
              }
              for (; j < n_s; ++j) rank += lvt[j] < tie;
              if (rank >= k_lvl) continue;
            }
            // the owner commits: pods i + rank .. i + rank + t - 1 of the chunk
            const int t = t_fill;
            uint32_t rp2 = rp - (uint32_t)t + ((uint32_t)t << 16);
            for (int j = 0; j < n_host; ++j) {  // Topology.Record, hostname groups
              const int times = rc.h_times[j];
              const int old = hc[j * kTopoCap + a];
              const int now = old + t * times > 0xFFFF ? 0xFFFF : old + t * times;
              if (times) hc[j * kTopoCap + a] = (uint16_t)now;
              if (now > rc.h_lim[j]) rp2 |= kRpDead;
            }
            const int count = (int)c_min + t;
            const int tb = -(tick + rank + t);
            unsigned long long nkey = order_key(count, tb);
            const int nd = NE + hs->node[a];
            for (int e = 0; e < t; ++e) rc.q_node[buf][i + rank + e] = nd;
            if ((rp2 & 0xFFFF) == 0) {  // the class no longer fits by resources: does anything? (node_closed)
              const int placed = (rp2 >> 16) & 0x7FFF;
              long long nq[kHotRes], cb1[kHotRes], cb2[kHotRes];
#pragma unroll
              for (int r = 0; r < kHotRes; ++r) { nq[r] = hs->q[r][a] + placed * p_req[r]; cb1[r] = hs->bound[r][a]; cb2[r] = hs->bound2[r][a]; }
              const unsigned short fl = (unsigned short)(hs->flags[a] | ((p_res & 0xF) << 1));
              if (node_closed(nq, min_req, RH, cb1, cb2, fl)) {
                nkey = ~0ull;
                hs->nn_last[a] = ((unsigned long long)(unsigned)count << 32) | (unsigned)tb;
                atomicAdd(&rc.tomb, 1);
              }
            }
            hs->key[a] = nkey;
            rpv[a] = rp2;
          }
          tick += adv;
        }
      }
    }
    // node-independent half of nextDomainTopologySpread, one domain per lane: min count over the pod's domains, the
    // domains within max-skew (count + self - min <= maxSkew)
    uint32_t okm0 = 0, okm1 = 0;
    int fd0 = 0, fd1 = 0;
    if (mode == 0) {
    CR_IT(3)
    if (n_mask > 0) {
      const bool valid = (m_reg0 >> lane) & 1;  // registered domains have ids < kRunDom
      const int cn = rc.cnt[warp][0][lane & (kRunDom - 1)];
      const int mn = __reduce_min_sync(0xffffffffu, valid ? cn : INT32_MAX);
      okm0 = __ballot_sync(0xffffffffu, valid && (long long)cn + m_bias0 <= (long long)mn);
      if (n_mask > 1) {
        const bool valid1 = (m_reg1 >> lane) & 1;
        const int cn1 = rc.cnt[warp][1][lane & (kRunDom - 1)];
        const int mn1 = __reduce_min_sync(0xffffffffu, valid1 ? cn1 : INT32_MAX);
        okm1 = __ballot_sync(0xffffffffu, valid1 && (long long)cn1 + m_bias1 <= (long long)mn1);
      }
    }
    // ---- scan the slots this thread owns: key, rp and (topology classes) the admissible domains
    unsigned long long mine = ~0ull;
    int best_a = 0;
    uint32_t best_rp = 0, best_z0 = 0, best_z1 = 0;
    for (int a = tid; a < n_active; a += T) {
      const unsigned long long key = hs->key[a];
      const uint32_t rp = rpv[a];
      uint32_t z0 = 0, z1 = 0;
      bool ok = key < mine && (rp & 0xFFFF) != 0 && !(rp & kRpDead);  // tombstones carry key = ~0
      if (n_mask > 0) { z0 = zv[a]; ok = ok && (z0 & okm0) != 0; }
      if (n_mask > 1) { z1 = zv[kTopoCap + a]; ok = ok && (z1 & okm1) != 0; }
      if (ok) { mine = key; best_a = a; best_rp = rp; best_z0 = z0; best_z1 = z1; }
    }
    // payload of this thread's candidate: slot | slow << 11 | pin bits << 13 | domains << 15 / 19
    unsigned pay = (unsigned)best_a;
    if (mine != ~0ull) {
      if ((best_rp & 0xFFFF) == kRoomSlow) pay |= 1u << 11;
      if (n_mask > 0) {
        const uint32_t cand = best_z0 & okm0;
        int d;
        if (!(best_z0 & 0xFFFF & ((best_z0 & 0xFFFF) - 1)) && (best_z0 & (1u << 16))) d = __ffs(cand) - 1;  // pinned already
        else {  // the placement pins the node's domain
          d = run_pick(cand, rc.cnt[warp][0]);
          pay |= 1u << 13;
          if (!((rc.m_neutral[0] >> d) & 1) || !((best_z0 & (1u << 17)) || rc.m_wk[0])) pay |= 1u << 11;
        }
        pay |= (unsigned)d << 15;
      }
      if (n_mask > 1) {
        const uint32_t cand = best_z1 & okm1;
        int d;
        if (!(best_z1 & 0xFFFF & ((best_z1 & 0xFFFF) - 1)) && (best_z1 & (1u << 16))) d = __ffs(cand) - 1;
        else {
          d = run_pick(cand, rc.cnt[warp][1]);
          pay |= 1u << 14;
          if (!((rc.m_neutral[1] >> d) & 1) || !((best_z1 & (1u << 17)) || rc.m_wk[1])) pay |= 1u << 11;
        }
        pay |= (unsigned)d << 19;
      }
    }
    // ---- block argmin with payload: ONE barrier (double-buffered scratch)
    const unsigned long long wmin = warp_min_u64(mine);
    if (mine == wmin && mine != ~0ull) { rc.red_key[parity][warp] = wmin; rc.red_pay[parity][warp] = pay; }
    else if (lane == 0 && wmin == ~0ull) rc.red_key[parity][warp] = ~0ull;
    __syncthreads();
    const unsigned long long rk = lane < nwarps ? rc.red_key[parity][lane] : ~0ull;
    const unsigned rp_l = lane < nwarps ? rc.red_pay[parity][lane] : 0;
    parity ^= 1;
    const unsigned long long wkey = warp_min_u64(rk);
    if (wkey != ~0ull) {
      const unsigned src = __ballot_sync(0xffffffffu, rk == wkey);
      const unsigned wp = __shfl_sync(0xffffffffu, rp_l, __ffs(src) - 1);
      if (wp & (1u << 11)) { status = 1; break; }  // the winner needs the full evaluation
      fd0 = (wp >> 15) & 0xF;
      fd1 = (wp >> 19) & 0xF;
      if (mine == wkey) {  // the owner commits its node: a handful of shared-memory stores
        const int a = best_a;
        uint32_t rp = best_rp - 1 + (1u << 16);
        bool host_first = false;
#pragma unroll
        for (int j = 0; j < kRunHost; ++j) {  // Topology.Record, hostname groups
          if (j >= n_host) continue;
          const int times = rc.h_times[j];
          const int old = hc[j * kTopoCap + a];
          const int now = old + times > 0xFFFF ? 0xFFFF : old + times;
          if (times) hc[j * kTopoCap + a] = (uint16_t)now;
          if (now > rc.h_lim[j]) rp |= kRpDead;  // no further pod of the class here
          host_first = host_first || (times && old == 0);
        }
        if (pay & (3u << 13)) {  // requirements.Add(In{d}) on the node: once per node and key
          const int n = hs->node[a];
          for (int j = 0; j < n_mask; ++j) {
            if (!((pay >> (13 + j)) & 1)) continue;
            const int d = j ? fd1 : fd0, k = rc.m_key[j];
            zv[j * kTopoCap + a] = (1u << d) | (3u << 16);
            s.nn_vals[(size_t)k * MAXN + n] = 1ull << d;
            s.nn_meta[n] = (s.nn_meta[n] | (1ull << (KSCHED_META_PRESENT_SHIFT + k))) & ~(1ull << (KSCHED_META_COMPLEMENT_SHIFT + k));
          }
        }
        const int count = (int)(wkey >> 32) + 1;
        unsigned long long nkey = order_key(count, -(tick + 1));
        rc.q_node[buf][i] = NE + hs->node[a];
        if ((rp & 0xFFFF) == 0) {  // the class no longer fits by resources: does anything? (node_closed)
          const int placed = (rp >> 16) & 0x7FFF;
          long long nq[kHotRes], cb1[kHotRes], cb2[kHotRes];
#pragma unroll
          for (int r = 0; r < kHotRes; ++r) { nq[r] = hs->q[r][a] + placed * p_req[r]; cb1[r] = hs->bound[r][a]; cb2[r] = hs->bound2[r][a]; }
          const unsigned short fl = (unsigned short)(hs->flags[a] | ((p_res & 0xF) << 1));
          if (node_closed(nq, min_req, RH, cb1, cb2, fl)) {  // leaves the active set: tombstone, compacted when the run ends
            nkey = ~0ull;
            hs->nn_last[a] = ((unsigned long long)(unsigned)count << 32) | (unsigned)(-(tick + 1));
            rc.tomb = rc.tomb + 1;
          }
        }
        hs->key[a] = nkey;
        rpv[a] = rp;
        (void)host_first;
      }
      if (n_mask > 0) {  // every warp keeps its copy of the spread counters in step (the node's domain is the single value d)
        if (lane == 0) {
          if (m_rec0) rc.cnt[warp][0][fd0]++;
          if (m_rec1) rc.cnt[warp][1][fd1]++;
        }
        __syncwarp();
      }
      ++tick;
    } else mode = 2;
    }
    if (mode == 2) {
      // ---- nobody accepts: NewNode + Add replayed from a variant (templates: the one the variant was created from)
      if (n_new >= MAXN || n_active >= kActCap || (topo && n_active >= kTopoCap) || rc.n_var == 0) { status = 1; break; }
      bool ok = true;
#pragma unroll
      for (int j = 0; j < kRunHost; ++j) ok = ok && (j >= n_host || rc.h_lim[j] >= 0);  // a fresh hostname has count 0
      if (n_mask > 0 && ok) {
        const uint32_t cand = rc.m_tallow[0] & okm0;
        if (!cand) ok = false; else fd0 = run_pick(cand, rc.cnt[warp][0]);
      }
      if (n_mask > 1 && ok) {
        const uint32_t cand = rc.m_tallow[1] & okm1;
        if (!cand) ok = false; else fd1 = run_pick(cand, rc.cnt[warp][1]);
      }
      int vi = -1;
      for (int v2 = 0; v2 < rc.n_var && ok && vi < 0; ++v2)
        if ((n_mask < 1 || rc.var[v2].dom[0] == fd0) && (n_mask < 2 || rc.var[v2].dom[1] == fd1)) vi = v2;
      if (vi < 0) { status = 1; break; }
      const RunVariant& v = rc.var[vi];
      CR_IT(2)
      // Fill step on the fresh node: it takes `cap` further pods of the class while it is the only accepting node and then
      // refuses (room 0 or a hostname limit reached). With an exact cap the run needs F such nodes in a row, m = 1 + cap pods
      // each: all of them are created in this iteration, one per thread (slot a belongs to thread a % T as everywhere).
      int cap = 0, F = 1;
      bool cap_exact = false;
      if (lvl && (v.rp & 0xFFFF) != kRoomSlow) {
        cap_exact = true;
        if (!(v.rp & kRpDead)) {
          cap = (int)(v.rp & 0xFFFF);
          for (int j = 0; j < n_host; ++j) {
            const int times = rc.h_times[j], lim = rc.h_lim[j];
            if (!times || lim >= 0x10000) continue;
            if (lim >= 0xFFF0) { cap = 0; cap_exact = false; continue; }  // saturating counters nearby: one pod at a time
            const int td = (lim - times) / times + 1;  // the count is `times` after the first pod
            cap = td < cap ? td : cap;
          }
        }
      }
      const int m = 1 + cap;
      if (cap_exact) {
        F = (k_avail + m - 1) / m;
        if (F > MAXN - n_new) F = MAXN - n_new;
        if (F > kActCap - n_active) F = kActCap - n_active;
        if (topo && F > kTopoCap - n_active) F = kTopoCap - n_active;
      }
      const int K = k_avail < F * m ? k_avail : F * m;  // pods consumed (k_avail is 1 outside level mode: F = m = K = 1)
      for (int idx = tid; idx < W32 * F; idx += T) { const int w = idx / F, j = idx - w * F; s.nn_opts[(size_t)w * MAXN + n_new + j] = v.opts[w]; }
      for (int idx = tid; idx < c.n_keys * F; idx += T) { const int k = idx / F, j = idx - k * F; s.nn_vals[(size_t)k * MAXN + n_new + j] = v.vals[k]; }
      for (int idx = tid; idx < KSCHED_MAX_RES * F; idx += T) { const int r = idx / F, j = idx - r * F; s.nn_req[(size_t)r * MAXN + n_new + j] = v.q[r]; }
      for (int e = tid; e < K; e += T) rc.q_node[buf][i + e] = NE + n_new + e / m;
      if (tid == 0)
        for (int j = 0; j < n_host; ++j) if (rc.h_times[j]) rc.h_inc[j] = rc.h_inc[j] + F;
      for (int j = (tid + T - n_active % T) % T; j < F; j += T) {  // the new slots this thread owns
        const int a = n_active + j, n = n_new + j;
        const int t = (K - j * m < m ? K - j * m : m) - 1;  // further pods on this node (the last one may get fewer)
        const int tk = tick + j * m;                          // tick of its first pod
#pragma unroll
        for (int r = 0; r < kHotRes; ++r) { hs->q[r][a] = v.q[r]; hs->bound[r][a] = v.b1[r]; hs->bound2[r][a] = v.b2[r]; }
        hs->node[a] = n;
        hs->flags[a] = v.fl;
        hs->absorbed[a] = simple ? cls : KSCHED_NONE;
        hs->rejected[a] = KSCHED_NONE;
        s.nn_meta[n] = v.meta;
        s.nn_tmpl[n] = (uint8_t)(v.fl >> 8);
        s.nn_req_present[n] = v.qp;
        s.nn_hp[n] = 0;
        s.nn_count[n] = 1;
        s.nn_tb[n] = tk + 1;
        if (n_mask > 0) zv[a] = (1u << fd0) | (3u << 16);
        if (n_mask > 1) zv[kTopoCap + a] = (1u << fd1) | (3u << 16);
        uint32_t rp2 = t > 0 ? v.rp - (uint32_t)t + ((uint32_t)t << 16) : v.rp;
        for (int jj = 0; jj < n_host; ++jj) {
          const int times = rc.h_times[jj];
          const int now = times + t * times > 0xFFFF ? 0xFFFF : times + t * times;
          hc[jj * kTopoCap + a] = (uint16_t)now;
          if (times) s.grp_host[(size_t)rc.h_row[jj] * hstride + NE + n] = (uint16_t)times;  // (the run's write-back stores the final count)
          if (t > 0 && now > rc.h_lim[jj]) rp2 |= kRpDead;
        }
        unsigned long long nkey = t > 0 ? order_key(1 + t, -(tk + 1 + t)) : order_key(1, tk + 1);
        if (t > 0 && (rp2 & 0xFFFF) == 0) {  // full for the class: closed for every class? (same test as the accept that fills a node)
          long long nq[kHotRes], cb1[kHotRes], cb2[kHotRes];
#pragma unroll
          for (int r = 0; r < kHotRes; ++r) { nq[r] = v.q[r] + t * p_req[r]; cb1[r] = v.b1[r]; cb2[r] = v.b2[r]; }
          const unsigned short fl = (unsigned short)(v.fl | ((p_res & 0xF) << 1));
          if (node_closed(nq, min_req, RH, cb1, cb2, fl)) {
            nkey = ~0ull;
            hs->nn_last[a] = ((unsigned long long)(unsigned)(1 + t) << 32) | (unsigned)(-(tk + 1 + t));
            atomicAdd(&rc.tomb, 1);
          }
        }
        hs->key[a] = nkey;
        rpv[a] = rp2;
      }
      if (n_mask > 0) {
        if (lane == 0) {
          if (m_rec0) rc.cnt[warp][0][fd0]++;
          if (m_rec1) rc.cnt[warp][1][fd1]++;
        }
        __syncwarp();
      }
      adv = K;
      tick += K;
      n_new += F;
      n_active += F;
    }
    // ---- the pods are placed: pop them
    qi += adv;
    qlen -= adv;
    if (qlen == 0) break;
  }
  __syncthreads();
  // ---- the run is over: write back what the commits deferred
  const int placed_total = qi - qi0;
  if (tid < CH && tid < qi - cb) {  // assignments of the partly consumed chunk
    const uint32_t pd = rc.q_pod[buf][tid];
    int nd = rc.q_node[buf][tid];
    if (nd < -1) nd = NE + hs->node[-nd - 2];  // the mask run stores the slot
    s.assign[pd] = nd;
    s.place_seq[pd] = seq0 + (cb - qi0) + tid;
  }
  for (int a = tid; a < n_active; a += T) {  // requests, order statistics, hostname counters of the nodes that took pods
    const uint32_t rp = rpv[a];
    const int placed = (rp >> 16) & 0x7FFF;
    if (!placed) continue;
    const int n = hs->node[a];
    unsigned long long key = hs->key[a];
    const bool tomb = key == ~0ull;
    if (tomb) key = hs->nn_last[a];
#pragma unroll
    for (int r = 0; r < kHotRes; ++r) {
      const long long nq = hs->q[r][a] + placed * p_req[r];
      hs->q[r][a] = nq;
      if (tomb && r < RH) s.nn_req[(size_t)r * MAXN + n] = nq;
    }
    hs->rejected[a] = KSCHED_NONE;
    const unsigned short fl = hs->flags[a];
    if ((p_res & 0xF) & ~((fl >> 1) & 0xF)) {  // a request key new to the node
      s.nn_req_present[n] |= p_res;
      hs->flags[a] = fl | (unsigned short)((p_res & 0xF) << 1);
    }
    s.nn_count[n] = (int)(key >> 32);
    s.nn_tb[n] = (int)((unsigned)key ^ 0x80000000u);
    for (int j = 0; j < n_host; ++j) {
      const int times = rc.h_times[j];
      if (!times) continue;
      const int now = hc[j * kTopoCap + a];
      s.grp_host[(size_t)rc.h_row[j] * hstride + NE + n] = (uint16_t)now;
      if (now - placed * times == 0) atomicAdd(&rc.h_inc[j], 1);  // the hostname's first matching pod (not saturated: counts <= pods per node)
    }
  }
  for (int j = 0; j < n_mask; ++j)
    if (rc.m_rec[j] && warp == 0 && lane < kRunDom && ((rc.m_registered[j] >> lane) & 1)) s.grp_cnt[(size_t)rc.m_group[j] * 64 + lane] = rc.cnt[0][j][lane];
  __syncthreads();
  if (tid < n_host && rc.h_inc[tid]) s.grp_host_total[rc.h_group[tid]] += rc.h_inc[tid];
  // ---- compact the active list (tombstones out); slot order is irrelevant, ownership ends with the run
  if (rc.tomb > 0) {
    if (tid == 0) {
      int i = 0, j = n_active - 1;
      while (true) {
        while (j >= 0 && hs->key[j] == ~0ull) --j;
        while (i < j && hs->key[i] != ~0ull) ++i;
        if (i >= j) break;
        hs->key[i] = hs->key[j];
        for (int r = 0; r < kHotRes; ++r) { hs->q[r][i] = hs->q[r][j]; hs->bound[r][i] = hs->bound[r][j]; hs->bound2[r][i] = hs->bound2[r][j]; }
        hs->node[i] = hs->node[j]; hs->flags[i] = hs->flags[j]; hs->absorbed[i] = hs->absorbed[j]; hs->rejected[i] = hs->rejected[j];
        hs->key[j] = ~0ull;
      }
    }
    n_active -= rc.tomb;
  }
#ifdef KSCHED_PROFILE_PACK
  if (tid == 0) {
    const int b = lvl ? 32 : 36;  // [cycles, pods, level+fill iterations, fresh iterations] ; per-pod iterations go to 44 / 45
    s.counters[b] += clock64() - cr_t0; s.counters[b + 1] += placed_total; s.counters[b + 2] += cr_it[0] + cr_it[1]; s.counters[b + 3] += cr_it[2];
    s.counters[lvl ? 44 : 45] += cr_it[3];
    s.counters[46] += cr_it[1];
  }
#endif
  if (tid == 0) {
    const int qcap = s.n_pods + 1;
    io.qi = qi; io.head = (io.head + placed_total) % qcap; io.qlen = qlen; io.tick = tick; io.seq = seq0 + placed_total; io.n_active = n_active; io.n_new = n_new; io.parity = parity;
    io.add_calls += placed_total; io.placed = placed_total; io.status = status;
  }
  __syncthreads();
}


#ifdef KSCHED_PROFILE_PACK
#define PK_T(i) { long long _now = clock64(); pk_acc[i] += _now - pk_last; pk_last = _now; }
#else
#define PK_T(i)
#endif

__global__ void __launch_bounds__(kPackThreads, 1) pack_kernel() {
#ifdef KSCHED_PROFILE_PACK
  long long pk_acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  long long pk_last = clock64();
#endif
  KS_K2
  const int tid = threadIdx.x;
  const int NE = s.n_existing, MAXN = s.max_new;
  const int R = c.n_res, RH = R < kHotRes ? R : kHotRes;

  int64_t* sm_alloc = reinterpret_cast<int64_t*>(dyn_smem + sizeof(HotSmem));
  const Hot H = make_hot(s);
  if (s.alloc_in_smem)
    for (int i = tid; i < R * c.n_types; i += blockDim.x) sm_alloc[i] = c.alloc_sorted[i];

  PodTopo& pt = g_pt;
  uint32_t* tmpl_taintset = g_tmpl_taintset;
  __shared__ WarpIO wio;
  if (tid < c.n_templates) tmpl_taintset[tid] = c.templates[tid].taintset;
  if (tid == 0) { pt.n = 0; g_rc.cls = KSCHED_NONE; g_rc.eligible = 0; }

  int head = 0, qlen = s.n_pods;
  const int qcap = s.n_pods + 1;
  int n_new = 0, n_active = 0, tick = 0, seq = 0, parity = 0;
  uint32_t epoch = 1;
  long long nodes_visited = 0, add_calls = 0;
  int fatal = 0;
  bool pt_nonempty = false;
  uint32_t pt_class = KSCHED_NONE, row_class = KSCHED_NONE;
  int fresh_valid = 0, fresh_a = 0;
  uint32_t fresh_cls = KSCHED_NONE;
  // class-run bookkeeping: classes found ineligible are not tried again; a run that places nothing backs off
  uint32_t run_block_cls = KSCHED_NONE;
  int run_skip = 0, run_fail = 0;
  uint32_t xrun_block_cls = KSCHED_NONE;  // existing-node run: class the existing nodes have no room left for
  // failure memo: the class whose Scheduler.add has just failed, valid while nothing is placed (seq) or relaxed (epoch)
  uint32_t fail_cls = KSCHED_NONE, fail_epoch = 0;
  int fail_seq = 0;

  for (int i = tid; i < s.n_pods; i += blockDim.x) {
    s.queue[i] = s.order[i];
    s.pod_pos[s.order[i]] = (uint32_t)i;
    s.assign[i] = -1;
    s.place_seq[i] = -1;
    s.last_epoch[i] = 0;
  }
  __syncthreads();

  // First pass over the queue = FFD order: row qi of the dense pod-row matrix (K0) belongs to pod order[qi], so the
  // next pod's words are fetched one iteration ahead with addresses that depend on no earlier load.
  int qi = 0;
  const ksched_pod_row* ffd_rows = reinterpret_cast<const ksched_pod_row*>(s.rows);
  PodRegs nxt{};
  if (s.n_pods > 0) nxt = load_pod_regs(ffd_rows, s.order[0]);
  const bool fast_allowed = NE == 0 && !s.count_visited;

  while (qlen > 0) {
    // ---- failure memo: pods at the head of the queue of the class that has just failed fail again (same class, same state:
    // scheduler.go:117-123 pushes them back unchanged, queue.go:61-68) - requeued in one step, up to one per thread
    if (fast_allowed && fail_cls != KSCHED_NONE && seq == fail_seq && epoch == fail_epoch) {
      const int T = blockDim.x;
      int lim = qlen < T ? qlen : T;
      if (qi < s.n_pods && s.n_pods - qi < lim) lim = s.n_pods - qi;  // the first pass ends with its last pod
      uint32_t pj = 0;
      bool stop = true;
      if (tid < lim) {
        int pos = head + tid;
        if (pos >= qcap) pos -= qcap;
        pj = s.queue[pos];
        stop = s.pod_class[pj] != fail_cls || (s.last_epoch[pj] == epoch && s.last_len[pj] == qlen);  // Pop() would stop here
      }
      unsigned first, unused;
      block_min2_u32_db(stop ? (unsigned)tid : 0xFFFFFFFFu, 0u, g_red, parity, &first, &unused);
      const int k = first < (unsigned)lim ? (int)first : lim;
      if (k > 0) {
        if (tid < k) {
          s.queue[(head + qlen + tid) % qcap] = pj;  // (every read of the old entries happened before the barrier above)
          s.last_len[pj] = qlen;
          s.last_epoch[pj] = epoch;
        }
        if (qi < s.n_pods) qi += k;
        head = (head + k) % qcap;
        add_calls += k;
        __syncthreads();
        if (qi < s.n_pods) nxt = load_pod_regs(ffd_rows + qi, s.order[qi]);
        continue;
      }
    }
    // ---- register-resident mode (see warp_resident_loop): entered when the next pod is plain and <= 32 nodes are open
    if (fast_allowed && s.use_warp_loop && !fresh_valid && qi < s.n_pods && n_active > 0 && n_active <= 32 && simple_pod_regs(nxt)) {
      __syncthreads();
      if (tid == 0) { wio.qi = qi; wio.head = head; wio.qlen = qlen; wio.tick = tick; wio.seq = seq; wio.n_active = n_active; wio.add_calls = add_calls; }
      __syncthreads();
      if (tid < 32) warp_resident_loop(&wio);
      __syncthreads();
      qi = wio.qi; head = wio.head; qlen = wio.qlen; tick = wio.tick; seq = wio.seq; n_active = wio.n_active; add_calls = wio.add_calls;
      if (qlen == 0) break;
      if (qi < s.n_pods) nxt = load_pod_regs(ffd_rows + qi, s.order[qi]);
      // the pod the warp loop stopped at (new node needed, non-plain pod, end of the first pass) takes the block-wide path
    }
    PK_T(0)
    // ---- class-run mode (see class_run): first-pass pods of a class whose accept test is exact from shared memory
    bool skip_run = true;
    if (fast_allowed && s.use_class_run && qi < s.n_pods && n_active <= kActCap) {
      const bool topo_cls = nxt.topo_begin != nxt.topo_end;
      const bool shape_ok = nxt.hpc == 0 && nxt.hpe == 0 && (nxt.res >> kHotRes) == 0 &&
                            (!topo_cls || (((nxt.meta >> KSCHED_META_PRESENT_SHIFT) & 0xFFFF) == 0 && nxt.itype == KSCHED_NONE && nxt.hostname == KSCHED_NONE));
      if (shape_ok && (unsigned)nxt.cls64 != run_block_cls) {
        if (fresh_valid && fresh_cls == (unsigned)nxt.cls64) skip_run = false;  // a fresh node of this class to capture
        else if (run_skip > 0) --run_skip;
        else skip_run = false;
      }
    }
    if (!skip_run) {
      __syncthreads();
      if (tid == 0) {
        RunIO& io = g_rio;
        io.qi = qi; io.head = head; io.qlen = qlen; io.tick = tick; io.seq = seq; io.n_active = n_active; io.n_new = n_new; io.parity = parity;
        io.add_calls = add_calls; io.placed = 0; io.status = 0;
        io.fresh_valid = fresh_valid; io.fresh_a = fresh_a; io.fresh_cls = fresh_cls;
      }
      __syncthreads();
      class_run(nxt);
      const RunIO& io = g_rio;
      const int placed = io.placed, status = io.status;
      qi = io.qi; head = io.head; qlen = io.qlen; tick = io.tick; seq = io.seq; n_active = io.n_active; n_new = io.n_new; parity = io.parity;
      add_calls = io.add_calls;
      fresh_valid = 0;
#ifdef KSCHED_PROFILE_PACK
      if (tid == 0) { s.counters[40] += 1; s.counters[41] += placed; s.counters[42] += status == 1; s.counters[43] += status == 2; }
#endif
      if (status == 2) run_block_cls = (unsigned)nxt.cls64;
      if (placed == 0 && status == 1) { run_fail = run_fail < 6 ? run_fail + 1 : 6; run_skip = (1 << run_fail) - 1; }
      else if (placed > 0) run_fail = 0;
      PK_T(1)
      if (qlen == 0) break;
      if (placed > 0) {
        if (qi < s.n_pods) nxt = load_pod_regs(ffd_rows + qi, s.order[qi]);
        if (status == 0) continue;  // class change / end of the first pass: pick the mode for the next pod
      }
      // status 1 / 2: the pod at qi takes the generic step
    }
    // ---- existing-node run (see existing_run): identical plain pods take the existing nodes in one prefix-sum pass
    if (NE > 0 && !s.count_visited && qi < s.n_pods && (unsigned)nxt.cls64 != xrun_block_cls &&
        ((nxt.meta >> KSCHED_META_PRESENT_SHIFT) & 0xFFFF) == 0 && nxt.topo_begin == nxt.topo_end && nxt.itype == KSCHED_NONE &&
        nxt.hostname == KSCHED_NONE && nxt.hpc == 0 && nxt.hpe == 0 && (nxt.res >> kHotRes) == 0 && !class_has_volumes(s, (unsigned)nxt.cls64)) {
      __syncthreads();
      if (tid == 0) { ExRunIO& io = g_xio; io.qi = qi; io.head = head; io.qlen = qlen; io.seq = seq; io.parity = parity; io.add_calls = add_calls; io.placed = 0; }
      __syncthreads();
      existing_run(nxt);
      const ExRunIO& io = g_xio;
      const int placed = io.placed;
      qi = io.qi; head = io.head; qlen = io.qlen; seq = io.seq; parity = io.parity; add_calls = io.add_calls;
      __syncthreads();  // g_xio is rewritten by the next run
      if (placed == 0) xrun_block_cls = (unsigned)nxt.cls64;  // no existing node takes this class: the generic step does the rest of it
      if (placed > 0) {
        fresh_valid = 0;
        if (qlen == 0) break;
        if (qi < s.n_pods) nxt = load_pod_regs(ffd_rows + qi, s.order[qi]);
        if ((unsigned)nxt.cls64 == (unsigned)ffd_rows[qi - 1].reserved) xrun_block_cls = (unsigned)nxt.cls64;  // the existing nodes are full for this class
        continue;
      }
    }
    if (s.stop_new_nodes > 0 && n_new >= s.stop_new_nodes) break;  // simulation: the verdict no longer depends on the rest (cluster.cuh)
    PodRegs cur;
    const bool first_pass = qi < s.n_pods;
    if (first_pass) {
      cur = nxt;
      if (qi + 1 < s.n_pods) nxt = load_pod_regs(ffd_rows + qi + 1, s.order[qi + 1]);
      if (tid < 2 && qi + 24 < s.n_pods) prefetch_l2(reinterpret_cast<const char*>(ffd_rows + qi + 24) + tid * 128);
      if (tid == 2 && (qi & 31) == 0 && qi + 96 < s.n_pods) prefetch_l2(s.order + qi + 96);
    } else {
      const uint32_t qpod = s.queue[head];
      if (s.last_epoch[qpod] == epoch && s.last_len[qpod] == qlen) break;  // Pop(): no progress in a whole cycle (queue.go:52)
      cur = load_pod_regs(s.classes + s.pod_class[qpod], qpod);
    }
    const int fpos_first = qi;
    ++qi;
    head = head + 1 == qcap ? 0 : head + 1;
    --qlen;
    ++add_calls;
#ifdef KSCHED_PROFILE_PACK
    if (tid == 0) s.counters[8 + 9] += 1;
#endif
    LoopVars L{head, qlen, n_new, n_active, tick, seq, parity, fatal, epoch, pt_nonempty, nodes_visited, pt_class, row_class, 0, 0, KSCHED_NONE, 0};
    generic_step(cur, first_pass, fpos_first, L);
    if (L.fail_memo) { fail_cls = (unsigned)cur.cls64; fail_seq = L.seq; fail_epoch = L.epoch; } else fail_cls = KSCHED_NONE;
    head = L.head; qlen = L.qlen; n_new = L.n_new; n_active = L.n_active; tick = L.tick; seq = L.seq; parity = L.parity; fatal = L.fatal;
    epoch = L.epoch; pt_nonempty = L.pt_nonempty; nodes_visited = L.nodes_visited; pt_class = L.pt_class; row_class = L.row_class;
    fresh_valid = L.fresh_valid; fresh_a = L.fresh_a; fresh_cls = L.fresh_cls;
    if (fatal) break;
    PK_T(5)
  }
  __syncthreads();
  for (int a = tid; a < n_active; a += blockDim.x) {
    const int n = H.node(a);
    for (int r = 0; r < RH; ++r) s.nn_req[(size_t)r * MAXN + n] = H.q(r, a);
  }
  if (tid == 0) {
    s.counters[0] = n_new;
    s.counters[1] = qlen;
    s.counters[2] = nodes_visited;
    s.counters[3] = add_calls;
    s.counters[4] = fatal;
    s.counters[5] = add_calls;
#ifdef KSCHED_PROFILE_PACK
    s.counters[8 + 6] = pk_acc[1];  // cycles inside class_run calls
    s.counters[8 + 7] = pk_acc[5];  // cycles inside generic calls (incl. call)
#endif
  }
}

// options_true = options_stored AND Fits(requests): one warp per new node (resources.Fits, utils/resources/resources.go:138).
__global__ void finalize_options_kernel(DevCatalog c, const long long* counters, const int64_t* nn_req, const uint32_t* nn_req_present,
                                        uint32_t* nn_opts, int max_new) {
  const int n_new = (int)counters[0];
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int n = warp; n < n_new; n += nwarps) {
    const uint32_t qp = nn_req_present[n];
    int rank = 0;
    if (lane < c.n_res && ((qp >> lane) & 1)) rank = fit_rank(c.alloc_sorted, c.n_types, lane, nn_req[(size_t)lane * max_new + n]);
    int ranks[KSCHED_MAX_RES];
#pragma unroll
    for (int r = 0; r < KSCHED_MAX_RES; ++r) ranks[r] = __shfl_sync(0xffffffffu, rank, r);  // every lane takes part
    for (int w = lane; w < c.W32; w += 32) {
      uint32_t sw = nn_opts[(size_t)w * max_new + n];
#pragma unroll
      for (int r = 0; r < KSCHED_MAX_RES; ++r)
        if (r < c.n_res && ((qp >> r) & 1)) sw &= c.fitset[((size_t)r * (c.n_types + 1) + ranks[r]) * c.W32 + w];
      nn_opts[(size_t)w * max_new + n] = sw;
    }
  }
}

}  // namespace
