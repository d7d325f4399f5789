// Host orchestration + C ABI (include/rootba_b200.h) of the B200-native square-root BA inner loop.
// One rba_handle = one landmark shard on one GPU; everything is enqueued on one CUDA stream.
// "ref:" citations are relative to /root/reference/src/rootba/.
#include <cuda_runtime.h>
#include <dlfcn.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <limits>
#include <memory>
#include <string>
#include <vector>

#include "../../include/rootba_b200.h"
#include "../host/bal_io_fast.hpp"
#include "kernels.cuh"
#include "nccl_dyn.hpp"

namespace rba {

thread_local std::string g_err;

#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess) {                                                                      \
      g_err = std::string(#call) + ": " + cudaGetErrorString(e__) + " (" __FILE__ ":" + std::to_string(__LINE__) + ")"; \
      return RBA_ERR_CUDA;                                                                         \
    }                                                                                              \
  } while (0)

struct EventPair {
  cudaEvent_t a = nullptr, b = nullptr;
  bool used = false;
};

}  // namespace rba

using namespace rba;

// type-erased base so the C ABI can hold either scalar type
struct rba_handle {
  int scalar_size = 0;
  virtual ~rba_handle() {}
  virtual int set_state(const void* cams, const void* lms) = 0;
  virtual int get_state(void* cams, void* lms) = 0;
  virtual int backup() = 0;
  virtual int restore() = 0;
  virtual int compute_error(rba_residual_info* out) = 0;
  virtual int linearize() = 0;
  virtual int solve(double lambda, void* inc_out, rba_cg_summary* cg) = 0;
  virtual int apply(const void* inc, void* l_diff_out, bool update_cameras) = 0;
  virtual int lm_step(bool linearize_first, double lambda, rba_lm_step_result* out) = 0;
  virtual int lm_run(const rba_lm_opts* o, int max_steps, rba_lm_iteration* log, int* steps_done, int* terminated, rba_stage_timings* totals) = 0;
  virtual int get_timings(rba_stage_timings* out) const = 0;
  virtual int get_stats(rba_workload_stats* out) const = 0;
  virtual int get_scaling(void* scaling, void* diag2) = 0;
  virtual int get_rhs(void* b) = 0;
  virtual int get_precond(void* inv, void* blocks) = 0;
  virtual int right_multiply(const void* x, void* y) = 0;
  virtual int debug_get_block(int lm, void* out, int rows, int cols, void* jls) = 0;
  virtual int time_matvec(int reps, double* sec) = 0;
  virtual int timer_start() = 0;
  virtual int timer_stop(double* sec) = 0;
  virtual void* stream_ptr() = 0;
  virtual int synchronize() = 0;
  virtual int comm_init(const void* uid) = 0;
  virtual int ipc_export(void* out128) = 0;
  virtual int ipc_import(const void* all) = 0;
};

#ifndef RBA_IMP_NS
#define RBA_IMP_NS 1
#endif

namespace rba {

template <class S>
struct Solver : rba_handle {
  rba_solver_opts opt{};
  KOpts ko{};
  Layout L;
  int nc = 0, nl_total = 0;
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  std::vector<void*> allocs;
  size_t device_bytes = 0;
  DevPtrs<S> D{};
  // device-only helpers
  S* cams_bk = nullptr; S* lms_bk = nullptr;
  MatvecItem* d_items = nullptr;
  std::vector<MatvecItem> dealt_items;  // L.items, the small-KP part dealt to the persistent warps (see init)
  int n_dealt = 0, dealt_grid = 0, dealt_bps = 0;
  long long state_version = 0;     // bumped whenever cameras / landmarks change (set_state, apply, restore)
  rba_residual_info error_cache{}; long long error_cache_version = -1, error_enqueue_version = -1; bool error_cache_valid = false;
  int* d_csr_obs_slots = nullptr; ReduceItem* d_csr_obs_items = nullptr; int* d_csr_obs_item_ptr = nullptr;
  int* d_csr_y_slots = nullptr; ReduceItem* d_csr_y_items = nullptr; int* d_csr_y_item_ptr = nullptr;
  int n_obs_items = 0, n_y_items = 0;
  // camera-major CSR the operator's per-slot output is reduced over: the y-slot CSR of the dense form (one slot per
  // observation and row chunk) or the observation CSR of the implicit form
  const int* op_slots = nullptr; const ReduceItem* op_items = nullptr; const int* op_item_ptr = nullptr; int n_op_items = 0;
  bool implicit_op = false;
  int e0_only_flag = 0;          // Power-SC: the implicit operator kernels return E_0 x = Q1d^T Q1d x alone
  bool panel_form = true;        // gradient and SCHUR_JACOBI blocks from the Q2 panels (reference form) instead of the identities
  int imp_tile_split = 0;        // tiles [0, split) have <= IMP_MAXSLOTS slots and take the streamed kernel
  size_t imp_smem = 0; int imp_grid = 1;
  ReduceItem* d_pb_items = nullptr; int* d_pb_item_ptr = nullptr; int n_pb_items = 0;
  int pcg_cluster = 16;
  bool use_pdl = true;
  int* h_prog = nullptr; int* d_prog = nullptr;  // PCG progress in host-mapped pinned memory: [0] last completed iteration, [1] solve ended
  int pcg_solve_id = 0;
  bool pcg_partials = true;      // one GPU: k_pcg_vec consumes the per-segment sums of k_cam_reduce (RBA_PCG_PARTIALS=0: k_cam_reduce_final)
  double* d_epart = nullptr;     // [EBLOCKS][6]
  double* d_red = nullptr;       // [8] reduced doubles (error / l_diff)
  int* d_flags = nullptr;        // [4] bad flags
  int* d_cam_cnt = nullptr;      // per-camera arrival counters of k_cam_reduce_final (zero between launches)
  PcgState* d_state = nullptr;
  PcgState* h_state = nullptr;   // pinned [2]
  double* h_red = nullptr;       // pinned [8]
  int* h_flags = nullptr;        // pinned [4]
  cudaEvent_t poll_ev[2] = {nullptr, nullptr};
  // status
  bool linearized = false;
  bool new_linearization_point = false;
  bool have_inc = false;
  S last_lambda = 0;
  bool damping_valid = false;
  rba_stage_timings tm{};
  EventPair ev_stage1, ev_stage2, ev_precond, ev_pcg, ev_backsub, ev_update, ev_error, ev_mv, ev_user;
  long long launches = 0;
  // NCCL
  NcclApi* nccl = nullptr;
  ncclComm_t comm = nullptr;
  // peer-memory all-reduce fused into the PCG vector kernel
  char* peer_mem = nullptr;      // this rank's exchange region (flags + staging areas, see PeerComm), IPC-exported
  size_t peer_bytes = 0;
  PeerComm pc{};
  bool peer_ok = false;
  int ar_seq = 0, c_seq = 0, s_seq = 0;  // sequence numbers of the three flag families (operator output / vectors / scalars)
  std::vector<void*> ipc_opened;
  static constexpr int EBLOCKS = 592;
  static constexpr int KPMAX = sizeof(S) == 4 ? 16 : 10;

  ~Solver() override {
    if (comm && nccl) nccl->CommDestroy(comm);
    for (void* p : ipc_opened) cudaIpcCloseMemHandle(p);
    for (void* p : allocs) cudaFree(p);
    if (h_prog) cudaFreeHost(h_prog);
    if (h_state) cudaFreeHost(h_state);
    if (h_red) cudaFreeHost(h_red);
    if (h_flags) cudaFreeHost(h_flags);
    for (EventPair* e : {&ev_stage1, &ev_stage2, &ev_precond, &ev_pcg, &ev_backsub, &ev_update, &ev_error, &ev_mv, &ev_user}) {
      if (e->a) cudaEventDestroy(e->a);
      if (e->b) cudaEventDestroy(e->b);
    }
    for (auto& e : poll_ev) if (e) cudaEventDestroy(e);
    if (stream) cudaStreamDestroy(stream);
  }

  template <class T>
  int dalloc(T** p, size_t count, bool zero = true) {
    const size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
    void* q = nullptr;
    CU(cudaMalloc(&q, bytes));
    allocs.push_back(q);
    device_bytes += bytes;
    if (zero) CU(cudaMemsetAsync(q, 0, bytes, stream));
    *p = (T*)q;
    return RBA_OK;
  }
  template <class T>
  int upload(T** p, const std::vector<T>& v) {
    int rc = dalloc(p, v.size(), false);
    if (rc) return rc;
    if (!v.empty()) CU(cudaMemcpyAsync(*p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, stream));
    return RBA_OK;
  }

  int start(EventPair& e) { e.used = true; CU(cudaEventRecord(e.a, stream)); return RBA_OK; }
  int stop(EventPair& e) { CU(cudaEventRecord(e.b, stream)); return RBA_OK; }
  static double elapsed(EventPair& e) {
    if (!e.used) return 0.0;
    float ms = 0;
    if (cudaEventElapsedTime(&ms, e.a, e.b) != cudaSuccess) return 0.0;
    return 1e-3 * ms;
  }

  // ------------------------------------------------------------------------------------------
  int init(const rba_problem_view* pv, const rba_solver_opts* o) {
    opt = *o;
    if (opt.nranks < 1 || opt.rank < 0 || opt.rank >= opt.nranks) { g_err = "bad rank/nranks"; return RBA_ERR_INVALID_ARGUMENT; }
    if (opt.pcg_check_period <= 0) opt.pcg_check_period = 4;
    if (opt.residual_reset_period <= 0) opt.residual_reset_period = 10;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
      g_err = "no CUDA device: rootba_b200 has no CPU fallback";
      return RBA_ERR_NO_DEVICE;
    }
    if (opt.device >= 0) CU(cudaSetDevice(opt.device));
    CU(cudaGetDevice(&device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    for (EventPair* e : {&ev_stage1, &ev_stage2, &ev_precond, &ev_pcg, &ev_backsub, &ev_update, &ev_error, &ev_mv, &ev_user}) {
      CU(cudaEventCreate(&e->a));
      CU(cudaEventCreate(&e->b));
    }
    for (auto& e : poll_ev) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    nc = pv->num_cameras;
    nl_total = pv->num_landmarks;
    ko.use_valid_projections_only = opt.use_valid_projections_only;
    ko.robust_norm = opt.robust_norm;
    ko.write_panel = (opt.operator_form == 1 || opt.solver_type != 0) ? 0 : 1;
    ko.huber = opt.huber_parameter;
    ko.jacobi_eps = opt.jacobi_scaling_epsilon > 0 ? opt.jacobi_scaling_epsilon : (double)ST<S>::eps_sqrt();  // ref: linearizor_base.cpp:72-79
    std::string msg = build_layout(nc, nl_total, pv->lm_obs_offset, pv->obs_cam_idx, opt.rank, opt.nranks, KPMAX, L);
    if (!msg.empty()) { g_err = msg; return RBA_ERR_INVALID_ARGUMENT; }
    // observation coordinates in slot order
    std::vector<S> xy((size_t)2 * L.nslots, S(0));
    const S* src = (const S*)pv->obs_xy;
    for (int s = 0; s < L.nslots; ++s)
      if (L.slot_obs[s] >= 0) { xy[2 * (size_t)s] = src[2 * L.slot_obs[s]]; xy[2 * (size_t)s + 1] = src[2 * L.slot_obs[s] + 1]; }
    int rc;
    TileInfo* d_tiles; int* d_sorted; int* d_slot_cam; int* d_slot_lm; S* d_xy;
#define TRY(x) do { rc = (x); if (rc) return rc; } while (0)
    TRY(upload(&d_tiles, L.tiles));
    TRY(upload(&d_sorted, L.sorted_lm));
    TRY(upload(&d_slot_cam, L.slot_cam));
    TRY(upload(&d_slot_lm, L.slot_lm));
    TRY(upload(&d_xy, xy));
    // The persistent warps of the TMA matvec take the items q = first + k * (number of warps).  Dealing the items sorted by size
    // round-robin leaves a warp with up to 1.6x the mean work on Ladybug-1723 (13 045 items for 2 960 warps: some get 5, some
    // 4, and warp 0 the largest of every round); instead the small-KP items are dealt longest-processing-time-first on the host
    // (greedy on bytes + a per-item constant) and laid out so that position k * W + w holds the k-th item of warp w, padded
    // with empty items (nrows = 0 = end of a warp's list).  RBA_MATVEC_DEAL=rr keeps the round-robin order.
    dealt_items = L.items;
    n_dealt = (int)L.items.size();
    {
      const char* e = getenv("RBA_MATVEC_DEAL");
      long long deal_ovh = 48;  // per-item constant (~12 KB-equivalent); 0 / 16 / 48 / 128 measured within 1 % of each other
      if (const char* o2 = getenv("RBA_MATVEC_DEAL_OVH")) deal_ovh = atoll(o2);
      const int nsmall = (int)L.items.size() - L.n_items_large;
      // resident CTAs per SM of the TMA matvec (shared memory: 5; the float64 instance is register-limited to 2): the grid
      // must be exactly the co-resident CTAs, or the longest-first lists of a later wave would start when the first is done
      int tma_bps = std::max(1, (int)((220 * 1024) / ((size_t)K4_WARPS * K4_NS * K4_STAGE + 1024)));
      {
        const size_t smem = (size_t)K4_WARPS * K4_NS * K4_STAGE;
        int occ = 0;
        if (cudaFuncSetAttribute((k_matvec_small_tma<S, K4_WARPS, K4_NS, K4_STAGE>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) == cudaSuccess &&
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, (k_matvec_small_tma<S, K4_WARPS, K4_NS, K4_STAGE>), K4_WARPS * 32, smem) == cudaSuccess && occ > 0)
          tma_bps = std::min(tma_bps, occ);
        else
          cudaGetLastError();
      }
      dealt_bps = tma_bps;
      const int W = grid_for(nsmall, K4_WARPS, tma_bps) * K4_WARPS;
      if (!(e && std::string(e) == "rr") && nsmall > W && !implicit_op) {
        std::vector<std::vector<int>> lists(W);
        std::vector<std::pair<long long, int>> heap(W);  // (load, warp), min-heap on the load
        for (int w = 0; w < W; ++w) heap[w] = {0, w};
        auto cmp = [](const std::pair<long long, int>& a, const std::pair<long long, int>& b) { return a > b; };
        std::make_heap(heap.begin(), heap.end(), cmp);
        for (int q = L.n_items_large; q < (int)L.items.size(); ++q) {  // already sorted by decreasing work
          std::pop_heap(heap.begin(), heap.end(), cmp);
          auto& top = heap.back();
          lists[top.second].push_back(q);
          top.first += (long long)L.items[q].nrows * L.tiles[L.items[q].tile].KP + deal_ovh;  // rows x KP x 256 B, + a per-item constant
          std::push_heap(heap.begin(), heap.end(), cmp);
        }
        size_t maxlen = 0;
        for (auto& l : lists) maxlen = std::max(maxlen, l.size());
        MatvecItem empty{}; empty.tile = 0; empty.row0 = 0; empty.nrows = 0; empty.yslot_base = 0; empty.pad = 0;
        dealt_items.assign(L.items.begin(), L.items.begin() + L.n_items_large);
        dealt_items.resize(L.n_items_large + maxlen * W, empty);
        for (int w = 0; w < W; ++w)
          for (size_t k = 0; k < lists[w].size(); ++k) dealt_items[L.n_items_large + k * W + w] = L.items[lists[w][k]];
        n_dealt = (int)dealt_items.size();
        dealt_grid = W / K4_WARPS;
      }
    }
    TRY(upload(&d_items, dealt_items));

    TRY(upload(&d_csr_obs_slots, L.csr_obs.slots));
    TRY(upload(&d_csr_obs_items, L.csr_obs.items));
    TRY(upload(&d_csr_obs_item_ptr, L.csr_obs.cam_item_ptr));
    n_obs_items = (int)L.csr_obs.items.size();
    if (L.csr_y_is_obs) {
      d_csr_y_slots = d_csr_obs_slots; d_csr_y_items = d_csr_obs_items; d_csr_y_item_ptr = d_csr_obs_item_ptr;
      n_y_items = n_obs_items;
    } else {
      TRY(upload(&d_csr_y_slots, L.csr_y.slots));
      TRY(upload(&d_csr_y_items, L.csr_y.items));
      TRY(upload(&d_csr_y_item_ptr, L.csr_y.cam_item_ptr));
      n_y_items = (int)L.csr_y.items.size();
    }
    implicit_op = opt.operator_form == 1 || opt.solver_type != 0;
    if (opt.operator_form != 0 && opt.operator_form != 1) { g_err = "operator_form must be 0 (dense) or 1 (implicit)"; return RBA_ERR_INVALID_ARGUMENT; }
    if (opt.solver_type < 0 || opt.solver_type > 2) { g_err = "solver_type must be 0 (SQUARE_ROOT), 1 (SCHUR_COMPLEMENT) or 2 (POWER_SCHUR_COMPLEMENT)"; return RBA_ERR_INVALID_ARGUMENT; }
    if (opt.solver_type == 2 && opt.nranks > 1) { g_err = "POWER_SCHUR_COMPLEMENT runs on one GPU (the power-series vector kernel has no peer exchange yet)"; return RBA_ERR_UNSUPPORTED; }
    if (opt.power_order <= 0) opt.power_order = 20;  // solver_options.hpp:270
    // the Schur-complement solvers share the per-observation records and the implicit operator kernels (k_sc_stage2)
    if (opt.solver_type != 0) implicit_op = true;
    if (opt.stage2_form != 0 && opt.stage2_form != 1) { g_err = "stage2_form must be 0 (Q2 panel, reference) or 1 (orthogonality identity)"; return RBA_ERR_INVALID_ARGUMENT; }
    // gradient / SCHUR_JACOBI blocks from the stored Q2 panels like the reference, unless there are no panels (implicit operator)
    panel_form = !implicit_op && opt.stage2_form == 0;
    if (implicit_op) {
      while (imp_tile_split < (int)L.tiles.size() && (32 / L.tiles[imp_tile_split].G) * L.tiles[imp_tile_split].n <= IMP_MAXSLOTS) ++imp_tile_split;
      imp_smem = (size_t)IMP_WARPS * IMP_NS * (size_t)IMP_MAXSLOTS * 48 * sizeof(S);
      CU(cudaFuncSetAttribute((k_matvec_implicit_tma<S, IMP_WARPS, IMP_MAXSLOTS, IMP_NS>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)imp_smem));
      int bps = 0;
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, (k_matvec_implicit_tma<S, IMP_WARPS, IMP_MAXSLOTS, IMP_NS>), IMP_WARPS * 32, imp_smem));
      imp_grid = std::max(1, std::min((imp_tile_split + IMP_WARPS - 1) / IMP_WARPS, sm_count * std::max(1, bps)));
    }
    if (implicit_op) { op_slots = d_csr_obs_slots; op_items = d_csr_obs_items; op_item_ptr = d_csr_obs_item_ptr; n_op_items = n_obs_items; }
    else { op_slots = d_csr_y_slots; op_items = d_csr_y_items; op_item_ptr = d_csr_y_item_ptr; n_op_items = n_y_items; }
    TRY(upload(&d_pb_items, L.pb_items));
    TRY(upload(&d_pb_item_ptr, L.pb_cam_item_ptr));
    n_pb_items = (int)L.pb_items.size();
    D.tiles = d_tiles; D.ntiles = (int)L.tiles.size(); D.sorted_lm = d_sorted;
    D.slot_cam = d_slot_cam; D.slot_lm = d_slot_lm; D.slot_xy = d_xy; D.nslots = L.nslots; D.nc = nc;
    TRY(dalloc(&D.cams, (size_t)10 * nc)); TRY(dalloc(&cams_bk, (size_t)10 * nc));
    TRY(dalloc(&D.lms, (size_t)3 * L.nl_local)); TRY(dalloc(&lms_bk, (size_t)3 * L.nl_local));
    if (ko.write_panel) TRY(dalloc(&D.panel, (size_t)L.panel_scalars));  // the implicit operator never touches the panels
    TRY(dalloc(&D.jp, (size_t)20 * L.nslots));
    TRY(dalloc(&D.q1u, (size_t)28 * L.nslots));
    TRY(dalloc(&D.q1d, (size_t)28 * L.nslots));
    TRY(dalloc(&D.jl, (size_t)6 * L.nslots));
    TRY(dalloc(&D.res, (size_t)2 * L.nslots));
    TRY(dalloc(&D.lmk, (size_t)24 * L.sorted_lm.size()));
    TRY(dalloc(&D.qtr, (size_t)2 * L.nslots));
    if (panel_form) {
      TRY(dalloc(&D.dmp, (size_t)28 * L.nslots));
      if (opt.preconditioner_type == 1) TRY(dalloc(&D.blk0, (size_t)48 * L.nslots));
      TRY(dalloc(&D.blocks0, (size_t)81 * nc));
      TRY(dalloc(&D.b0, (size_t)9 * nc));
    }
    for (S** v : {&D.diag2, &D.scaling, &D.b, &D.x, &D.r, &D.z, &D.p, &D.q, &D.y, &D.inc}) TRY(dalloc(v, (size_t)9 * nc));
    TRY(dalloc(&D.blocks, (size_t)81 * nc)); TRY(dalloc(&D.jblocks, (size_t)81 * nc)); TRY(dalloc(&D.inv, (size_t)81 * nc));
    TRY(dalloc(&D.yobs, (size_t)9 * L.nyslots));
    TRY(dalloc(&D.partial, (size_t)9 * std::max(n_obs_items, n_y_items)));
    TRY(dalloc(&D.pblk, (size_t)48 * n_pb_items));

    pc.nranks = 1; pc.rank = opt.rank;
    if (opt.nranks > 1 && opt.nranks <= MAX_PEERS) {
      pc.off_y = 4096;
      pc.off_c = pc.off_y + (((long long)2 * opt.nranks * 9 * nc * (long long)sizeof(S) + 255) & ~255LL);
      pc.cmax = (long long)81 * nc;
      peer_bytes = (size_t)(pc.off_c + (long long)2 * opt.nranks * pc.cmax * (long long)sizeof(S));
      TRY(dalloc(&peer_mem, peer_bytes));
      pc.base[opt.rank] = peer_mem;
      TRY(dalloc(&pc.dead, 1));
    }
    TRY(dalloc(&d_epart, (size_t)EBLOCKS * 6)); TRY(dalloc(&d_red, 8)); TRY(dalloc(&d_flags, 4));
    TRY(dalloc(&d_cam_cnt, (size_t)nc));
    TRY(dalloc(&d_state, 1));
    CU(cudaHostAlloc((void**)&h_prog, 64, cudaHostAllocMapped));
    CU(cudaHostGetDevicePointer((void**)&d_prog, h_prog, 0));
    h_prog[0] = 0; h_prog[1] = 0;
    CU(cudaMallocHost((void**)&h_state, 2 * sizeof(PcgState)));
    CU(cudaMallocHost((void**)&h_red, 24 * sizeof(double)));
    CU(cudaMallocHost((void**)&h_flags, 12 * sizeof(int)));
    // tile kernels (linearize+QR, stage 2): scratch in shared memory when the tile fits in the kernel's cap (scalars per
    // warp), else in a per-warp slice of a global buffer (very long tracks; slow but general)
    {
      long long need1 = 0, need2 = 0;
      for (const TileInfo& T : L.tiles) {
        const int Wn = (32 / T.G) * T.n;
        need1 = std::max<long long>(need1, (long long)Wn * 60 + 64);
        need2 = std::max<long long>(need2, (long long)stage2_need(T.n, T.G, T.KP));
      }
      auto setup = [&](Scratch<S>& sc, int cap, long long need, size_t& smem, int& blocks_per_sm, int& max_blocks) -> int {
        sc.smem_cap = cap; sc.gbase = nullptr; sc.gstride = 0;
        smem = (size_t)TILE_WARPS * cap * sizeof(S);
        blocks_per_sm = std::max(1, (int)((220 * 1024) / (smem + 1024)));
        max_blocks = sm_count * blocks_per_sm;
        if (need > cap) {
          long long warps = (long long)max_blocks * TILE_WARPS;
          while (warps > TILE_WARPS && warps * need * (long long)sizeof(S) > (1LL << 30)) warps /= 2;
          max_blocks = (int)std::max<long long>(1, warps / TILE_WARPS);
          sc.gstride = (need + 3) & ~3LL;
          int rc2 = dalloc(&sc.gbase, (size_t)(max_blocks * TILE_WARPS) * sc.gstride, false);
          if (rc2) return rc2;
        }
        return RBA_OK;
      };
      TRY(setup(k1_sc, K1_CAP, need1, k1_smem, k1_bps, k1_max_blocks));
      TRY(setup(k2_sc, K2_CAP, need2, k2_smem, k2_bps, k2_max_blocks));
      // tiles dealt to the persistent warps longest-first (the kernels' work per tile grows like n^2: panel rows x columns)
      if (!(getenv("RBA_TILE_DEAL") && std::string(getenv("RBA_TILE_DEAL")) == "rr")) {
        TRY(deal_tiles(tile_grid(k1_max_blocks) * TILE_WARPS, order_k1));
        TRY(deal_tiles(tile_grid(sm_count * 8) * TILE_WARPS, order_kp));
      }
      CU(cudaFuncSetAttribute((k_linearize_qr<S, false>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1_smem));
      CU(cudaFuncSetAttribute((k_linearize_qr<S, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k1_smem));
      CU(cudaFuncSetAttribute((k_stage2<S, true>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k2_smem));
      CU(cudaFuncSetAttribute((k_stage2<S, false>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k2_smem));
    }
    k4_smem_small = (size_t)K4_WARPS * L.k4_scratch_per_warp * sizeof(S);
    if (k4_smem_small > 200 * 1024) { g_err = "matvec scratch exceeds shared memory"; return RBA_ERR_UNSUPPORTED; }
    CU(cudaFuncSetAttribute(k_matvec_small<S, K4_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(k4_smem_small, 1024)));
    CU(cudaFuncSetAttribute((k_matvec_large<S, K4_WARPS, KPMAX>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(k4_smem_small, 1024)));
    {
      // the PCG vector step runs on one thread-block cluster (16 CTAs if the device grants it, else 8)
      CU(cudaFuncSetAttribute(k_pcg_vec<S>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
      CU(cudaFuncSetAttribute(k_power_vec<S>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
      pcg_cluster = 16;
      if (const char* e = getenv("RBA_PDL")) use_pdl = atoi(e) != 0;
      if (const char* e = getenv("RBA_PCG_PARTIALS")) pcg_partials = atoi(e) != 0;
      if (const char* e = getenv("RBA_PCG_CLUSTER")) pcg_cluster = std::max(1, std::min(atoi(e), 16));
      for (; pcg_cluster > 1; pcg_cluster >>= 1) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(pcg_cluster); cfg.blockDim = dim3(VEC_THREADS);
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = pcg_cluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        int ncl = 0;
        if (cudaOccupancyMaxActiveClusters(&ncl, k_pcg_vec<S>, &cfg) == cudaSuccess && ncl >= 1) break;
        cudaGetLastError();
      }
    }
    {
      const char* e = getenv("RBA_MATVEC");
      use_tma = !(e && std::string(e) == "ldg");
      k4_smem_tma = (size_t)K4_WARPS * K4_NS * K4_STAGE;
      if (k4_smem_tma > 220 * 1024) use_tma = false;
      if (use_tma) {
        CU(cudaFuncSetAttribute((k_matvec_small_tma<S, K4_WARPS, K4_NS, K4_STAGE>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)k4_smem_tma));
        k4_tma_blocks_per_sm = std::max(1, (int)((220 * 1024) / (k4_smem_tma + 1024)));
        if (dealt_bps > 0) k4_tma_blocks_per_sm = dealt_bps;
        if (const char* b = getenv("RBA_MATVEC_BLOCKS_PER_SM")) k4_tma_blocks_per_sm = std::max(1, atoi(b));
      }
    }
#undef TRY
    CU(cudaStreamSynchronize(stream));
    return RBA_OK;
  }
  static constexpr int K4_WARPS = 4;
  static constexpr int IMP_WARPS = 2, IMP_MAXSLOTS = 64, IMP_NS = RBA_IMP_NS;  // streamed implicit operator: warps per block, slots per stage, stages per warp
#ifndef RBA_K4_NS
#define RBA_K4_NS 2
#endif
#ifndef RBA_K4_STAGE
#define RBA_K4_STAGE 4608
#endif
  static constexpr int K4_NS = RBA_K4_NS;        // TMA ring stages per warp
  static constexpr int K4_STAGE = RBA_K4_STAGE;  // bytes per stage (2 rows of an f32 KP=9 tile)
  static constexpr int TILE_WARPS = 4;
  static constexpr int K1_CAP = 3904;   // scalars of shared memory per warp: linearize+QR needs 60 * W * n + 64 (= 3904 for the standard tiles)
  static constexpr int K2_CAP = 3072;   // stage 2 needs 3 * W * CS + 9 * W * n + 20 W + 8 (<= 3048 for the standard tiles)
  Scratch<S> k1_sc{}, k2_sc{};
  size_t k1_smem = 0, k2_smem = 0;
  int k1_bps = 2, k2_bps = 2, k1_max_blocks = 296, k2_max_blocks = 296;
  size_t k4_smem_small = 0, k4_smem_tma = 0;
  bool use_tma = true;
  int k4_tma_blocks_per_sm = 2;

  // ------------------------------------------------------------------------------------------
  // sum over the shards, in place, on the solver stream: peer-memory push exchange when the ranks have mapped each other's
  // regions (rba_ipc_import), else NCCL
  int allreduce(S* buf, size_t count) {
    if (opt.nranks == 1) return RBA_OK;
    if (peer_ok && (long long)count <= pc.cmax) {
      ++c_seq;
      const int g = (int)std::max<size_t>(1, std::min<size_t>((size_t)sm_count, (count + 255) / 256));
      k_peer_push<S><<<g, 256, 0, stream>>>(pc, buf, (long long)count, c_seq & 1);
      k_peer_sum<S><<<g, 256, 0, stream>>>(pc, buf, (long long)count, c_seq & 1, c_seq, d_flags + 1);
      launches += 2;
      return RBA_OK;
    }
    if (!comm) { g_err = "rba_comm_init has not been called on a sharded handle"; return RBA_ERR_STATE; }
    ncclResult_t r = nccl->AllReduce(buf, buf, count, sizeof(S) == 4 ? ncclFloat : ncclDouble, ncclSum, comm, stream);
    if (r != ncclSuccess) { g_err = std::string("ncclAllReduce: ") + nccl->GetErrorString(r); return RBA_ERR_NCCL; }
    return RBA_OK;
  }
  // nd doubles (d_red) and the bad flags (d_flags, summed = OR) in one exchange
  int allreduce_scalars(int nd) {
    if (opt.nranks == 1) return RBA_OK;
    if (peer_ok) {
      ++s_seq;
      k_peer_small<<<1, 64, 0, stream>>>(pc, d_red, nd, d_flags, 4, s_seq & 1, s_seq, d_flags + 1);
      ++launches;
      return RBA_OK;
    }
    if (!comm) { g_err = "rba_comm_init has not been called on a sharded handle"; return RBA_ERR_STATE; }
    ncclResult_t r = ncclSuccess;
    if (nd > 0) r = nccl->AllReduce(d_red, d_red, nd, ncclDouble, ncclSum, comm, stream);
    if (r == ncclSuccess) r = nccl->AllReduce(d_flags, d_flags, 4, ncclInt, ncclSum, comm, stream);
    if (r != ncclSuccess) { g_err = std::string("ncclAllReduce: ") + nccl->GetErrorString(r); return RBA_ERR_NCCL; }
    return RBA_OK;
  }

  int comm_init(const void* uid) override {
    if (opt.nranks == 1) return RBA_OK;
    nccl = nccl_api();
    if (!nccl) { g_err = "libnccl.so.2 could not be loaded"; return RBA_ERR_NCCL; }
    ncclUniqueId id;
    std::memcpy(&id, uid, sizeof(id));
    CU(cudaSetDevice(device));
    ncclResult_t r = nccl->CommInitRank(&comm, opt.nranks, id, opt.rank);
    if (r != ncclSuccess) { g_err = std::string("ncclCommInitRank: ") + nccl->GetErrorString(r); return RBA_ERR_NCCL; }
    return RBA_OK;
  }

  int ipc_export(void* out128) override {
    std::memset(out128, 0, 128);
    if (!peer_mem) return RBA_OK;  // single rank
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, peer_mem));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    std::memcpy(out128, &h, 64);
    return RBA_OK;
  }
  int ipc_import(const void* all) override {
    if (opt.nranks == 1) return RBA_OK;
    if (opt.nranks > MAX_PEERS) { g_err = "the peer-memory exchange supports at most 8 ranks"; return RBA_ERR_UNSUPPORTED; }
    if (const char* e = getenv("RBA_PEER_AR")) if (atoi(e) == 0) return RBA_OK;
    CU(cudaSetDevice(device));
    for (int r = 0; r < opt.nranks; ++r) {
      if (r == opt.rank) continue;
      cudaIpcMemHandle_t h;
      std::memcpy(&h, (const char*)all + (size_t)128 * r, 64);
      void* p = nullptr;
      if (cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
        cudaGetLastError();
        g_err = "cudaIpcOpenMemHandle failed; using NCCL for the reductions across shards";
        return RBA_OK;  // peer_ok stays false: NCCL
      }
      ipc_opened.push_back(p);
      pc.base[r] = (char*)p;
    }
    pc.nranks = opt.nranks; pc.rank = opt.rank;
    peer_ok = true;
    return RBA_OK;
  }

  // ------------------------------------------------------------------------------------------
  int set_state(const void* cams, const void* lms) override {
    ++state_version;
    CU(cudaMemcpyAsync(D.cams, cams, (size_t)10 * nc * sizeof(S), cudaMemcpyHostToDevice, stream));
    CU(cudaMemcpyAsync(D.lms, (const S*)lms + (size_t)3 * L.lm_begin, (size_t)3 * L.nl_local * sizeof(S), cudaMemcpyHostToDevice, stream));
    CU(cudaStreamSynchronize(stream));
    return RBA_OK;
  }
  int get_state(void* cams, void* lms) override {
    CU(cudaMemcpyAsync(cams, D.cams, (size_t)10 * nc * sizeof(S), cudaMemcpyDeviceToHost, stream));
    CU(cudaMemcpyAsync((S*)lms + (size_t)3 * L.lm_begin, D.lms, (size_t)3 * L.nl_local * sizeof(S), cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    return RBA_OK;
  }
  int backup() override {  // ref: bal/bal_problem.cpp:590-598
    CU(cudaMemcpyAsync(cams_bk, D.cams, (size_t)10 * nc * sizeof(S), cudaMemcpyDeviceToDevice, stream));
    CU(cudaMemcpyAsync(lms_bk, D.lms, (size_t)3 * L.nl_local * sizeof(S), cudaMemcpyDeviceToDevice, stream));
    return RBA_OK;
  }
  int restore() override {  // ref: bal/bal_problem.cpp:600-608
    ++state_version;
    CU(cudaMemcpyAsync(D.cams, cams_bk, (size_t)10 * nc * sizeof(S), cudaMemcpyDeviceToDevice, stream));
    CU(cudaMemcpyAsync(D.lms, lms_bk, (size_t)3 * L.nl_local * sizeof(S), cudaMemcpyDeviceToDevice, stream));
    return RBA_OK;
  }

  // launch with optional programmatic dependent launch (the kernel may start before its predecessor in the stream has
  // finished and orders itself with griddepcontrol.wait) and optional thread-block-cluster dimension
  template <class... KArgs, class... Args>
  int launch_ex(void (*kern)(KArgs...), int grid, int block, size_t smem, bool pdl, int cluster, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute at[2];
    int na = 0;
    if (pdl) { at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[na].val.programmaticStreamSerializationAllowed = 1; ++na; }
    if (cluster > 1) { at[na].id = cudaLaunchAttributeClusterDimension; at[na].val.clusterDim.x = cluster; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1; ++na; }
    cfg.attrs = at; cfg.numAttrs = na;
    CU(cudaLaunchKernelEx(&cfg, kern, KArgs(args)...));
    ++launches;
    return RBA_OK;
  }
  TileOrder order_k1{nullptr, 0}, order_kp{nullptr, 0};
  // longest-processing-time-first lists of tiles for nw persistent warps, laid out so that position k * nw + w is the k-th
  // tile of warp w (-1 = end of the warp's list)
  int deal_tiles(int nw, TileOrder& out) {
    const int nt = (int)L.tiles.size();
    if (nt <= nw) return RBA_OK;  // at most one tile per warp: nothing to balance
    std::vector<int> idx(nt);
    std::vector<long long> cost(nt);
    for (int t = 0; t < nt; ++t) {
      idx[t] = t;
      const TileInfo& T = L.tiles[t];
      cost[t] = (long long)2 * T.n * T.KP + (long long)(32 / T.G) * T.n / 2 + 8;  // panel rows x column steps + per-observation work + constant
    }
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return cost[a] > cost[b]; });
    std::vector<std::vector<int>> lists(nw);
    std::vector<std::pair<long long, int>> heap(nw);
    for (int w = 0; w < nw; ++w) heap[w] = {0, w};
    auto cmp = [](const std::pair<long long, int>& a, const std::pair<long long, int>& b) { return a > b; };
    std::make_heap(heap.begin(), heap.end(), cmp);
    for (int t : idx) {
      std::pop_heap(heap.begin(), heap.end(), cmp);
      heap.back().first += cost[t];
      lists[heap.back().second].push_back(t);
      std::push_heap(heap.begin(), heap.end(), cmp);
    }
    size_t maxlen = 0;
    for (auto& l : lists) maxlen = std::max(maxlen, l.size());
    std::vector<int> order(maxlen * nw, -1);
    for (int w = 0; w < nw; ++w)
      for (size_t k = 0; k < lists[w].size(); ++k) order[k * nw + w] = lists[w][k];
    int* d = nullptr;
    int rc = upload(&d, order); if (rc) return rc;
    out.order = d; out.count = (int)order.size();
    return RBA_OK;
  }
  int tile_grid(int max_blocks) const { return std::max(1, std::min(max_blocks, (D.ntiles + TILE_WARPS - 1) / TILE_WARPS)); }
  int grid_for(long long work_items, int per_block, int blocks_per_sm) const {
    long long g = (work_items + per_block - 1) / per_block;
    g = std::min<long long>(g, (long long)sm_count * blocks_per_sm);
    return (int)std::max<long long>(g, 1);
  }

  // deterministic per-camera sum of yobs[slot][9] over a CSR -> dst[9 nc] (+ all-reduce across shards)
  int camera_reduce(const int* slots, const ReduceItem* items, int nitems, const int* item_ptr, S* dst, const int* done,
                    const S* addend = nullptr, bool reduce_ranks = true) {
    k_cam_reduce<S><<<grid_for(nitems, 8, 8), 256, 0, stream>>>(D.yobs, slots, items, nitems, D.partial, done, 0);
    k_cam_final9<S><<<(9 * nc + 255) / 256, 256, 0, stream>>>(D.partial, item_ptr, nc, dst, done, addend);
    launches += 2;
    return reduce_ranks ? allreduce(dst, (size_t)9 * nc) : RBA_OK;
  }

  // ------------------------------------------------------------------------------------------
  // ref: solver/linearizor_base.cpp:59-67
  // Every entry point is split into an enqueue half (kernels + asynchronous copies into its OWN pinned slot) and a finish
  // half (after a stream synchronisation): the public calls are enqueue + synchronise + finish, rba_lm_step strings the
  // enqueue halves of a whole LM inner iteration together and synchronises once.
  // pinned slots: h_red + 8 * slot, h_flags + 4 * slot;  slot 0 compute_error, 1 linearize, 2 apply
  bool error_enqueued = false;
  int compute_error_enqueue() {
    error_enqueued = false;
    if (error_cache_valid && error_cache_version == state_version) return RBA_OK;  // answered from the cache in finish
    int rc = start(ev_error); if (rc) return rc;
    CU(cudaMemsetAsync(d_flags, 0, 4 * sizeof(int), stream));
    k_error<S><<<EBLOCKS, 256, 0, stream>>>(D, ko, d_epart, d_flags);
    k_sum_partials<6><<<1, 256, 0, stream>>>(d_epart, EBLOCKS, d_red);
    launches += 2;
    rc = allreduce_scalars(6); if (rc) return rc;
    CU(cudaMemcpyAsync(h_red, d_red, 6 * sizeof(double), cudaMemcpyDeviceToHost, stream));
    CU(cudaMemcpyAsync(h_flags, d_flags, 4 * sizeof(int), cudaMemcpyDeviceToHost, stream));
    rc = stop(ev_error); if (rc) return rc;
    error_enqueued = true;
    error_enqueue_version = state_version;
    return RBA_OK;
  }
  int compute_error_finish(rba_residual_info* out) {
    // The LM loop evaluates the cost at the end of an accepted step and again, unchanged state, before the next
    // linearisation (the reference's own TODO, bal_bundle_adjustment.cpp:298-301): the evaluation is deterministic, so
    // the second call returns the cached ResidualInfo without touching the GPU.
    if (!error_enqueued) {
      *out = error_cache;
      tm.residual_evaluation_time = 0.0;
      return RBA_OK;
    }
    out->all_num_obs = (int64_t)llround(h_red[0]); out->all_error = h_red[1]; out->all_residual_sum = h_red[2];
    out->valid_num_obs = (int64_t)llround(h_red[3]); out->valid_error = h_red[4]; out->valid_residual_sum = h_red[5];
    if (h_flags[1]) { g_err = "a peer rank did not take part in a cross-shard reduction in time (peer-memory exchange timed out)"; return RBA_ERR_NCCL; }
    out->is_numerically_valid = h_flags[0] ? 0 : 1;
    out->pad_ = 0;
    tm.residual_evaluation_time = elapsed(ev_error);
    error_cache = *out; error_cache_version = error_enqueue_version; error_cache_valid = true;
    return RBA_OK;
  }
  int compute_error(rba_residual_info* out) override {
    int rc = compute_error_enqueue(); if (rc) return rc;
    if (error_enqueued) CU(cudaStreamSynchronize(stream));
    return compute_error_finish(out);
  }

  // ref: solver/linearizor_qr.cpp:78-138 (staged: LinearizationQR::get_stage1, linearization_qr.hpp:634-712)
  long long lin_l0 = 0;
  int linearize_enqueue() {
    lin_l0 = launches;
    int rc = start(ev_stage1); if (rc) return rc;
    CU(cudaMemsetAsync(d_flags, 0, 4 * sizeof(int), stream));
    // pass A: squared column norms of the weighted pose Jacobians -> pose_jacobian_scaling_
    k_jp_norms<S><<<grid_for(L.nslots, 256, 8), 256, 0, stream>>>(D, ko, d_flags);
    ++launches;
    rc = camera_reduce(d_csr_obs_slots, d_csr_obs_items, n_obs_items, d_csr_obs_item_ptr, D.diag2, nullptr); if (rc) return rc;
    k_scaling<S><<<(9 * nc + 255) / 256, 256, 0, stream>>>(D.diag2, D.scaling, 9 * nc, (S)ko.jacobi_eps);
    // pass B: linearize (scaled) + Jl scaling + Householder QR + panel write
    if (opt.use_householder_marginalization)
      k_linearize_qr<S, false><<<tile_grid(k1_max_blocks), TILE_WARPS * 32, k1_smem, stream>>>(D, ko, k1_sc, d_flags, order_k1);
    else  // ref: ipp:149-163 selects perform_qr_givens
      k_linearize_qr<S, true><<<tile_grid(k1_max_blocks), TILE_WARPS * 32, k1_smem, stream>>>(D, ko, k1_sc, d_flags, order_k1);
    launches += 2;
    if (opt.preconditioner_type == 0 || opt.solver_type == 2) {
      // JACOBI: D (sum Jp^T Jp) D from the stored scaled Jacobians (Power-SC: these blocks are Hpp, sc/linearization_power_sc.hpp:92-128) (ref: ipp:554-569, block_sparse_matrix.hpp:89-100)
      rc = precond_blocks(0, D.jblocks, nullptr, true); if (rc) return rc;
    }
    if (panel_form) {
      // rows 3..2n-1 of the Q2 panels do not change with lambda: their part of the gradient (ipp:443-466) and of the
      // SCHUR_JACOBI blocks (ipp:520-552) is accumulated once per linearisation (this shard only; the sum over the
      // shards happens in solve() together with the damping-row part)
      const int want_blocks = opt.preconditioner_type == 1 ? 1 : 0;
      k_panel_grad_blocks<S><<<tile_grid(sm_count * 8), TILE_WARPS * 32, 0, stream>>>(D, want_blocks, order_kp);
      ++launches;
      rc = camera_reduce(d_csr_obs_slots, d_csr_obs_items, n_obs_items, d_csr_obs_item_ptr, D.b0, nullptr, nullptr, false); if (rc) return rc;
      if (want_blocks) { rc = precond_blocks(3, D.blocks0, nullptr, false); if (rc) return rc; }
    }
    rc = allreduce_scalars(0); if (rc) return rc;
    CU(cudaMemcpyAsync(h_flags + 4, d_flags, 4 * sizeof(int), cudaMemcpyDeviceToHost, stream));
    rc = stop(ev_stage1); if (rc) return rc;
    linearized = true;  // provisional: linearize_finish withdraws it on a numerical failure
    new_linearization_point = true;
    damping_valid = false;
    have_inc = false;
    return RBA_OK;
  }
  int linearize_finish() {
    CU(cudaGetLastError());
    tm.stage1_time = elapsed(ev_stage1);
    tm.kernel_launches = launches - lin_l0;
    if (h_flags[4 + 1]) { linearized = false; g_err = "a peer rank did not take part in a cross-shard reduction in time (peer-memory exchange timed out)"; return RBA_ERR_NCCL; }
    if (h_flags[4 + 0]) { linearized = false; return RBA_NUMERICAL_FAILURE; }  // reference: CHECK abort (linearizor_qr.cpp:121-122)
    return RBA_OK;
  }
  int linearize() override {
    int rc = linearize_enqueue(); if (rc) return rc;
    CU(cudaStreamSynchronize(stream));
    return linearize_finish();
  }

  // per-camera 9x9 blocks: deterministic two-phase sum over the camera-major observation CSR (modes: see k_precond_partial)
  int precond_blocks(int mode, S* dst, const S* addend, bool reduce_ranks) {
    const int g = (n_pb_items + 127) / 128;
    switch (mode) {
      case 0: k_precond_partial<S, 0><<<g, 128, 0, stream>>>(D.jp, (const S*)nullptr, d_csr_obs_slots, d_pb_items, n_pb_items, D.pblk); break;
      case 1: k_precond_partial<S, 1><<<g, 128, 0, stream>>>(D.jp, D.q1d, d_csr_obs_slots, d_pb_items, n_pb_items, D.pblk); break;
      case 2: k_precond_partial<S, 2><<<g, 128, 0, stream>>>(D.dmp, (const S*)nullptr, d_csr_obs_slots, d_pb_items, n_pb_items, D.pblk); break;
      default: k_precond_partial<S, 3><<<g, 128, 0, stream>>>(D.blk0, (const S*)nullptr, d_csr_obs_slots, d_pb_items, n_pb_items, D.pblk); break;
    }
    k_precond_final<S><<<(45 * nc + 255) / 256, 256, 0, stream>>>(D.pblk, d_pb_item_ptr, nc, addend, dst);
    launches += 2;
    return reduce_ranks ? allreduce(dst, (size_t)81 * nc) : RBA_OK;
  }

  // operator part of one matvec: yobs = P^T P x_red for every landmark, then per-camera sums -> D.partial
  // one complete operator application outside PCG: y = sum over the landmarks of P^T P x_red (this shard), per camera in D.y
  void matvec_launch(const S* xvec, const int* done) {
    matvec_kernels(xvec, done);
    k_cam_reduce_final<S, false><<<grid_for(n_op_items, 8, 8), 256, 0, stream>>>((const S*)D.yobs, op_slots, op_items, n_op_items, op_item_ptr, D.partial,
                                                                               d_cam_cnt, D.y, done, 0, pc, 0, nc);
    ++launches;
  }
  void matvec_kernels(const S* xvec, const int* done, bool pdl = false) {
    if (implicit_op) {
      const int ntl = (int)L.tiles.size();
      const bool p = pdl && use_pdl && imp_tile_split == ntl;  // a single kernel between the PCG vector step and the reduction
      if (imp_tile_split > 0 && use_tma)
        launch_ex((k_matvec_implicit_tma<S, IMP_WARPS, IMP_MAXSLOTS, IMP_NS>), imp_grid, IMP_WARPS * 32, imp_smem, p, 1, D, imp_tile_split, xvec, done, (int)p, e0_only_flag);
      const int tb = use_tma ? imp_tile_split : 0;
      if (tb < ntl)
        launch_ex(k_matvec_implicit<S>, (ntl - tb + TILE_WARPS - 1) / TILE_WARPS, TILE_WARPS * 32, 0, false, 1, D, tb, xvec, done, 0, e0_only_flag);
      ++tm.matvec_launches;
      return;
    }
    const int nitems = n_dealt;
    if (L.n_items_large > 0) {
      k_matvec_large<S, K4_WARPS, KPMAX><<<grid_for(L.n_items_large, K4_WARPS, 4), K4_WARPS * 32, k4_smem_small, stream>>>(
          D, d_items, 0, L.n_items_large, L.k4_scratch_per_warp, xvec, done);
      ++launches;
    }
    if (nitems > L.n_items_large) {
      if (use_tma) {
        launch_ex(k_matvec_small_tma<S, K4_WARPS, K4_NS, K4_STAGE>, dealt_grid > 0 ? dealt_grid : grid_for(nitems - L.n_items_large, K4_WARPS, k4_tma_blocks_per_sm), K4_WARPS * 32,
                  k4_smem_tma, pdl && use_pdl && L.n_items_large == 0, 1, D, (const MatvecItem*)d_items, L.n_items_large, nitems, L.k4_scratch_per_warp, xvec, done,
                  (int)(pdl && use_pdl && L.n_items_large == 0));
        --launches;
      } else
        k_matvec_small<S, K4_WARPS><<<grid_for(nitems - L.n_items_large, K4_WARPS, 5), K4_WARPS * 32, k4_smem_small, stream>>>(
            D, d_items, L.n_items_large, nitems, L.k4_scratch_per_warp, xvec, done);
      ++launches;
    }
    ++tm.matvec_launches;
  }
  int pcg_vec(int i, int mode, bool pdl, int is_last, S lambda, bool fused_ar = false, bool from_partials = false) {
    PeerComm c = pc;
    if (!fused_ar) c.nranks = 1;
    return launch_ex(k_pcg_vec<S>, pcg_cluster, VEC_THREADS, 0, pdl && use_pdl, pcg_cluster, D, d_state, lambda, i, mode, (double)opt.eta,
                     (int)opt.min_linear_solver_iterations, is_last, (int)(pdl && use_pdl), c, ar_seq, from_partials ? op_item_ptr : (const int*)nullptr, d_prog);
  }
  // The hand-over through per-segment sums is taken when a cluster CTA's share of the cameras fits the vector kernel's
  // register-resident layout: 9 * ceil(nc / cluster) <= VEC_THREADS * VEC_EPT = 1024, i.e. <= 1808 cameras with a 16-CTA
  // cluster.  Larger camera counts on one GPU (Final-13682) keep the arrival-counter reduction into D.y (pcg_apply), the
  // combination that was measured at that size.
  bool pcg_from_partials() const {
    return opt.nranks == 1 && pcg_partials && 9 * ((nc + pcg_cluster - 1) / pcg_cluster) <= VEC_THREADS * VEC_EPT;
  }
  // finish one operator application inside PCG (H v for v = p in mode 0/1, x in mode 2) and do the vector step
  int pcg_apply(int i, int mode, int is_last, S lambda) {
    if (pcg_from_partials()) {
      // one GPU: the vector kernel adds the per-segment sums itself (same order as k_cam_reduce_final's last arriver:
      // bit-identical) -- no arrival counters, fences or second pass in the reduction
      int rc = launch_ex(k_cam_reduce<S>, grid_for(n_op_items, 8, 8), 256, 0, use_pdl, 1, (const S*)D.yobs, op_slots, op_items, n_op_items, D.partial,
                         (const int*)&d_state->done, (int)use_pdl);
      if (rc) return rc;
      return pcg_vec(i, mode, true, is_last, lambda, false, true);
    }
    const bool fused = opt.nranks > 1 && peer_ok;
    if (fused) ++ar_seq;
    // NCCL path: k_cam_reduce_final writes y only for cameras that have observations in this shard; D.y is all-reduced IN
    // PLACE, so without this the other cameras would carry the previous iteration's global sum into the next all-reduce
    if (opt.nranks > 1 && !fused) CU(cudaMemsetAsync(D.y, 0, (size_t)9 * nc * sizeof(S), stream));
    int rc = fused ? launch_ex((k_cam_reduce_final<S, true>), grid_for(n_op_items, 8, 8), 256, 0, use_pdl, 1, (const S*)D.yobs, op_slots,
                               op_items, n_op_items, op_item_ptr, D.partial, d_cam_cnt, D.y, (const int*)&d_state->done, (int)use_pdl, pc, ar_seq, nc)
                   : launch_ex((k_cam_reduce_final<S, false>), grid_for(n_op_items, 8, 8), 256, 0, use_pdl, 1, (const S*)D.yobs, op_slots,
                               op_items, n_op_items, op_item_ptr, D.partial, d_cam_cnt, D.y, (const int*)&d_state->done, (int)use_pdl, pc, ar_seq, nc);
    if (rc) return rc;
    if (opt.nranks == 1) return pcg_vec(i, mode, true, is_last, lambda);
    if (fused) return pcg_vec(i, mode, true, is_last, lambda, true);
    rc = allreduce(D.y, (size_t)9 * nc); if (rc) return rc;
    return pcg_vec(i, mode, false, is_last, lambda);
  }
  // q_out = H vec = sum + lambda vec ; optional partial p.q
  int matvec_finish(const S* vec, S* out, S lambda, PcgState* st, double* part) {
    int rc = allreduce(D.y, (size_t)9 * nc); if (rc) return rc;  // no-op on one GPU
    k_pcg_q<S><<<NPART, 128, 0, stream>>>(D, st, nullptr, nullptr, D.y, vec, out, lambda, part);
    ++launches;
    return RBA_OK;
  }

  // ref: solver/linearizor_qr.cpp:140-265
  // Power-series solve of the reduced camera system (ref: sc/linearization_power_sc.hpp:130-160, driven by
  // solver/linearizor_power_sc.cpp:140-160 with q_tolerance = eta): per term one E_0 application (the implicit operator
  // kernels with e0_only), the per-camera reduction and k_power_vec; the device convergence flag is polled like in PCG.
  int power_enqueue(void* inc_out) {
    int rc = start(ev_pcg); if (rc) return rc;
    CU(cudaMemsetAsync(d_state, 0, sizeof(PcgState), stream));
    const int order = opt.power_order, chk = opt.pcg_check_period;
    rc = launch_ex(k_power_vec<S>, pcg_cluster, VEC_THREADS, 0, false, pcg_cluster, D, d_state, 0, (double)opt.eta, 0, 0); if (rc) return rc;
    e0_only_flag = 1;
    int i = 1, pending[2] = {0, 0}, slot = 0;
    bool finished = false;
    while (i <= order && !finished) {
      const int chunk_end = std::min(i + chk - 1, order);
      for (; i <= chunk_end; ++i) {
        matvec_kernels(D.p, &d_state->done, true);
        rc = launch_ex((k_cam_reduce_final<S, false>), grid_for(n_op_items, 8, 8), 256, 0, use_pdl, 1, (const S*)D.yobs, op_slots, op_items,
                       n_op_items, op_item_ptr, D.partial, d_cam_cnt, D.y, (const int*)&d_state->done, (int)use_pdl, pc, 0, nc);
        if (rc) { e0_only_flag = 0; return rc; }
        rc = launch_ex(k_power_vec<S>, pcg_cluster, VEC_THREADS, 0, use_pdl, pcg_cluster, D, d_state, i, (double)opt.eta, (int)(i == order), (int)use_pdl);
        if (rc) { e0_only_flag = 0; return rc; }
      }
      CU(cudaMemcpyAsync(&h_state[slot], d_state, sizeof(PcgState), cudaMemcpyDeviceToHost, stream));
      CU(cudaEventRecord(poll_ev[slot], stream));
      pending[slot] = 1;
      const int other = slot ^ 1;
      if (pending[other]) {
        CU(cudaEventSynchronize(poll_ev[other]));
        pending[other] = 0;
        if (h_state[other].done) finished = true;
      }
      slot = other;
    }
    e0_only_flag = 0;
    CU(cudaMemcpyAsync(&h_state[0], d_state, sizeof(PcgState), cudaMemcpyDeviceToHost, stream));
    if (inc_out) CU(cudaMemcpyAsync(inc_out, D.inc, (size_t)9 * nc * sizeof(S), cudaMemcpyDeviceToHost, stream));
    rc = stop(ev_pcg); if (rc) return rc;
    have_inc = true;
    new_linearization_point = false;
    return RBA_OK;
  }

  long long solve_l0 = 0;
  int solve_enqueue(double lambda_d, void* inc_out) {
    if (!linearized) { g_err = "rba_solve called before a successful rba_linearize"; return RBA_ERR_STATE; }
    const S lambda = (S)lambda_d;
    solve_l0 = launches;
    tm.matvec_launches = 0;
    int rc = start(ev_stage2); if (rc) return rc;
    // stage 2: landmark damping + gradient (+ SCHUR_JACOBI blocks)
    if (opt.solver_type != 0) {
      // Schur-complement solvers: landmark eliminated through the normal equations (Cholesky of Jl^T Jl + lambda I)
      CU(cudaMemsetAsync(d_flags, 0, 4 * sizeof(int), stream));
      k_sc_stage2<S><<<tile_grid(sm_count * 8), TILE_WARPS * 32, 0, stream>>>(D, lambda, d_flags);
    } else if (panel_form) k_stage2<S, true><<<tile_grid(k2_max_blocks), TILE_WARPS * 32, k2_smem, stream>>>(D, lambda, k2_sc, ko.write_panel);
    else k_stage2<S, false><<<tile_grid(k2_max_blocks), TILE_WARPS * 32, k2_smem, stream>>>(D, lambda, k2_sc, ko.write_panel);
    ++launches;
    rc = camera_reduce(d_csr_obs_slots, d_csr_obs_items, n_obs_items, d_csr_obs_item_ptr, D.b, nullptr, panel_form ? D.b0 : nullptr); if (rc) return rc;
    const bool power = opt.solver_type == 2;
    const bool schur = opt.preconditioner_type == 1 && !power;  // Power-SC inverts Hpp = sum Jp^T Jp + lambda I instead
    if (schur) { rc = panel_form ? precond_blocks(2, D.blocks, D.blocks0, true) : precond_blocks(1, D.blocks, nullptr, true); if (rc) return rc; }
    rc = stop(ev_stage2); if (rc) return rc;
    rc = start(ev_precond); if (rc) return rc;
    // pose damping lambda*I added to the blocks, then explicit inverse (ref: linearization_qr.hpp:796-802, linearizor_qr.cpp:228-237)
    k_precond_invert<S><<<(nc + 63) / 64, 64, 0, stream>>>(schur ? D.blocks : D.jblocks, lambda, nc, schur ? D.blocks : nullptr, D.inv);
    ++launches;
    rc = stop(ev_precond); if (rc) return rc;
    last_lambda = lambda;
    damping_valid = true;
    // One GPU, operator sums through D.y (Power-SC, or PCG without the per-segment hand-over): k_cam_reduce_final writes y only
    // for cameras that have observations, so the others must start at 0 -- not at what rba_right_multiply left there
    // (H x + lambda x).  Every iteration of the solve then leaves them 0.
    if (opt.nranks == 1 && (power || !pcg_from_partials())) CU(cudaMemsetAsync(D.y, 0, (size_t)9 * nc * sizeof(S), stream));
    if (power) return power_enqueue(inc_out);
    // PCG (ref: cg/conjugate_gradient.hpp:113-298 ; linearizor_base.cpp:81-103)
    rc = start(ev_pcg); if (rc) return rc;
    CU(cudaMemsetAsync(d_state, 0, sizeof(PcgState), stream));
    const int max_it = std::max(opt.max_linear_solver_iterations, 1);
    const int period = opt.residual_reset_period;
    // The vector kernel publishes the number of the last completed iteration and the end of the solve in host-mapped pinned
    // memory (h_prog); the host enqueues at most pcg_check_period iterations beyond that and stops as soon as it sees the
    // end: no copy or event between the kernels of the loop, and at most pcg_check_period no-op iterations after the end
    // (one GPU, and the peer-memory exchange, whose no-op kernels leave before they communicate).
    const int depth = opt.pcg_check_period;
    h_prog[0] = 0; h_prog[1] = 0;  // nothing in flight writes them: the stream has been synchronised since the previous solve
    // The ranks stop enqueueing at slightly different iterations (whenever each sees the end), so the sequence numbers of the
    // operator exchange restart from a per-solve base that every rank computes alike
    ar_seq = (++pcg_solve_id) * (2 * max_it + 4);
    rc = pcg_vec(0, 3, false, 0, lambda); if (rc) return rc;  // x = 0, r = b, z = M^-1 r, rho, p = z
    auto enqueue_iteration = [&](int i) -> int {
      const int is_last = (i == max_it) ? 1 : 0;
      matvec_kernels(D.p, &d_state->done, true);
      if (i % period == 0) {
        int r2 = pcg_apply(i, 1, 0, lambda); if (r2) return r2;
        matvec_kernels(D.x, &d_state->done, true);
        return pcg_apply(i, 2, is_last, lambda);
      }
      return pcg_apply(i, 0, is_last, lambda);
    };
    if (opt.nranks > 1 && !peer_ok) {
      // NCCL exchange: every rank must enqueue the SAME number of all-reduces, so the decision to stop may depend only on
      // the iteration count -- the flag is polled once per chunk of `depth` iterations, one chunk behind
      int i = 1, pending[2] = {0, 0}, slot = 0;
      bool finished = false;
      while (i <= max_it && !finished) {
        const int chunk_end = std::min(i + depth - 1, max_it);
        for (; i <= chunk_end; ++i) { rc = enqueue_iteration(i); if (rc) return rc; }
        CU(cudaMemcpyAsync(&h_state[slot], d_state, sizeof(PcgState), cudaMemcpyDeviceToHost, stream));
        CU(cudaEventRecord(poll_ev[slot], stream));
        pending[slot] = 1;
        const int other = slot ^ 1;
        if (pending[other]) {
          CU(cudaEventSynchronize(poll_ev[other]));
          pending[other] = 0;
          if (h_state[other].done) finished = true;
        }
        slot = other;
      }
    } else {
      volatile int* prog = h_prog;
      for (int i = 1; i <= max_it; ++i) {
        unsigned spins = 0;
        while (!prog[1] && i - prog[0] > depth) {
          // every 64k polls: has the stream run dry (a launch failed, or the kernels ended without publishing)?  Then do not wait.
          if ((++spins & 0xffffu) == 0 && cudaStreamQuery(stream) != cudaErrorNotReady) break;
        }
        if (prog[1]) break;
        rc = enqueue_iteration(i); if (rc) return rc;
      }
    }
    CU(cudaMemcpyAsync(&h_state[0], d_state, sizeof(PcgState), cudaMemcpyDeviceToHost, stream));
    if (inc_out) CU(cudaMemcpyAsync(inc_out, D.inc, (size_t)9 * nc * sizeof(S), cudaMemcpyDeviceToHost, stream));
    rc = stop(ev_pcg); if (rc) return rc;
    have_inc = true;
    new_linearization_point = false;
    return RBA_OK;
  }
  int solve_finish(rba_cg_summary* cg) {
    CU(cudaGetLastError());
    tm.stage2_time = elapsed(ev_stage2);
    tm.compute_preconditioner_time = elapsed(ev_precond);
    tm.solve_reduced_system_time = elapsed(ev_pcg);
    tm.kernel_launches = launches - solve_l0;
    if (cg) {
      cg->termination_type = h_state[0].term;
      cg->num_iterations = h_state[0].iter;
      cg->reason = h_state[0].reason;
      cg->num_matvecs = h_state[0].iter + h_state[0].iter / opt.residual_reset_period;
    }
    if (h_state[0].reason == 99) {
      g_err = "PCG: a peer rank did not publish its operator output in time (peer-memory exchange timed out)";
      return RBA_ERR_NCCL;
    }
    return RBA_OK;
  }
  int solve(double lambda_d, void* inc_out, rba_cg_summary* cg) override {
    int rc = solve_enqueue(lambda_d, inc_out); if (rc) return rc;
    CU(cudaStreamSynchronize(stream));
    return solve_finish(cg);
  }

  // ref: solver/linearizor_qr.cpp:267-291
  long long apply_l0 = 0;
  int apply_enqueue(const void* inc_host, bool update_cameras) {
    if (!linearized || !damping_valid) { g_err = "rba_apply / rba_back_substitute need rba_linearize + rba_solve first"; return RBA_ERR_STATE; }
    apply_l0 = launches;
    ++state_version;
    if (inc_host) CU(cudaMemcpyAsync(D.inc, inc_host, (size_t)9 * nc * sizeof(S), cudaMemcpyHostToDevice, stream));
    else if (!have_inc) { g_err = "no device-resident increment"; return RBA_ERR_STATE; }
    int rc = start(ev_backsub); if (rc) return rc;
    CU(cudaMemsetAsync(d_flags, 0, 4 * sizeof(int), stream));
    const int grid = std::min(tile_grid(sm_count * 4), EBLOCKS);
    k_back_substitute<S><<<grid, TILE_WARPS * 32, 0, stream>>>(D, D.inc, d_epart, d_flags);
    k_sum_partials<1><<<1, 256, 0, stream>>>(d_epart, grid, d_red);
    launches += 2;
    rc = allreduce_scalars(1); if (rc) return rc;
    rc = stop(ev_backsub); if (rc) return rc;
    rc = start(ev_update); if (rc) return rc;
    if (update_cameras) {
      // NOTE: the reference skips the camera update when l_diff is not finite (linearizor_qr.cpp:275-277); the LM loop
      // then rejects the step and restores the backup, so updating unconditionally is equivalent for the caller.
      k_camera_update<S><<<(nc + 127) / 128, 128, 0, stream>>>(D, D.inc);
      ++launches;
    }
    rc = stop(ev_update); if (rc) return rc;
    CU(cudaMemcpyAsync(h_red + 16, d_red, sizeof(double), cudaMemcpyDeviceToHost, stream));
    CU(cudaMemcpyAsync(h_flags + 8, d_flags, 4 * sizeof(int), cudaMemcpyDeviceToHost, stream));
    return RBA_OK;
  }
  int apply_finish(void* l_diff_out) {
    CU(cudaGetLastError());
    tm.back_substitution_time = elapsed(ev_backsub);
    tm.update_cameras_time = elapsed(ev_update);
    tm.kernel_launches = launches - apply_l0;
    if (h_flags[8 + 1]) { g_err = "a peer rank did not take part in a cross-shard reduction in time (peer-memory exchange timed out)"; return RBA_ERR_NCCL; }
    S l = (S)h_red[16];
    int ret = RBA_OK;
    if (h_flags[8 + 0] || !std::isfinite((double)l)) { l = std::numeric_limits<S>::quiet_NaN(); ret = RBA_NUMERICAL_FAILURE; }
    *(S*)l_diff_out = l;
    return ret;
  }
  int apply(const void* inc_host, void* l_diff_out, bool update_cameras) override {
    int rc = apply_enqueue(inc_host, update_cameras); if (rc) return rc;
    CU(cudaStreamSynchronize(stream));
    return apply_finish(l_diff_out);
  }

  // One LM inner iteration with ONE host synchronisation (SURVEY 8f row 2): [linearize] + solve(lambda) + backup + apply with
  // the device-resident increment + compute_error, the enqueue halves back to back.  Same kernels in the same order as the
  // separate calls, hence bit-identical results.  The reference skips apply when the increment is not finite
  // (bal_bundle_adjustment.cpp:360-399); here the step is applied on the device regardless and the caller restores the
  // backup when `solve_failed` is set (the backup is taken inside).
  int lm_step(bool linearize_first, double lambda, rba_lm_step_result* out) override {
    std::memset(out, 0, sizeof(*out));
    int rc;
    if (linearize_first) { rc = linearize_enqueue(); if (rc) return rc; }
    rc = solve_enqueue(lambda, nullptr); if (rc) return rc;
    rc = backup(); if (rc) return rc;
    rc = apply_enqueue(nullptr, true); if (rc) return rc;
    rc = compute_error_enqueue(); if (rc) return rc;
    CU(cudaStreamSynchronize(stream));
    if (linearize_first) { rc = linearize_finish(); if (rc) return rc; }  // numerical failure of the linearisation: as rba_linearize
    rc = solve_finish(&out->cg); if (rc) return rc;
    out->solve_failed = out->cg.termination_type == 2 ? 1 : 0;  // FAILURE: the increment is not usable (reference: non-finite inc)
    S l = 0;
    rc = apply_finish(&l);
    if (rc < 0) return rc;
    out->l_diff = (double)l;
    int rc2 = compute_error_finish(&out->cost); if (rc2) return rc2;
    return rc;  // RBA_NUMERICAL_FAILURE when l_diff is not finite (as rba_apply)
  }

  // optimize_lm_ours (solver/bal_bundle_adjustment.cpp:291-521) on top of lm_step; see rba_lm_run in the header
  static double cost_of(const rba_residual_info& r, int optimized_cost) {
    if (optimized_cost == 0) return r.all_error;
    if (optimized_cost == 1) return r.valid_error;
    return r.valid_num_obs > 0 ? r.valid_error / (double)r.valid_num_obs : 0.0;
  }
  int lm_run(const rba_lm_opts* o, int max_steps, rba_lm_iteration* log, int* steps_done, int* terminated_out, rba_stage_timings* totals) override {
    const S min_lambda = (S)(1.0 / o->max_trust_region_radius), max_lambda = (S)(1.0 / o->min_trust_region_radius);
    const S vee_factor = (S)o->vee_factor, initial_vee = (S)o->initial_vee;
    S lam = (S)(1.0 / o->initial_trust_region_radius), vee = initial_vee;
    bool new_outer = true, terminated = false;
    rba_residual_info ri{};
    // cost of the previous log entry in the ERROR / ERROR_VALID sense, which the function tolerance compares against
    // (:69-72, :174-201): the initial cost, then every logged step's cost -- a rejected step's too -- and 0 after a failed solve
    const int prev_kind = o->optimized_cost == 0 ? 0 : 1;
    double prev_logged = 0;
    if (totals) std::memset(totals, 0, sizeof(*totals));
    int it = 0;
    for (; it < max_steps && !terminated; ++it) {
      rba_lm_iteration& L2 = log[it];
      std::memset(&L2, 0, sizeof(L2));
      L2.lambda = (double)lam;
      const bool lin_first = new_outer;
      double dev = 0;
      if (new_outer) {
        int rc = compute_error(&ri); if (rc) return rc;   // answered from the cache after an accepted step
        if (!ri.is_numerically_valid) { g_err = "did not expect numerical failure during linearization"; return RBA_NUMERICAL_FAILURE; }  // :307-308
        if (it == 0) prev_logged = cost_of(ri, prev_kind);
        dev += tm.residual_evaluation_time;
        if (totals) totals->residual_evaluation_time += tm.residual_evaluation_time;
        new_outer = false;
      }
      rba_lm_step_result r;
      int rc = lm_step(lin_first, (double)lam, &r);
      if (rc < 0) return rc;
      if (lin_first && rc == RBA_NUMERICAL_FAILURE && !linearized) return rc;  // the linearisation itself failed (reference: CHECK abort)
      const double t_step = (lin_first ? tm.stage1_time : 0.0) + tm.stage2_time + tm.compute_preconditioner_time + tm.solve_reduced_system_time +
                            tm.back_substitution_time + tm.update_cameras_time + tm.residual_evaluation_time;
      dev += t_step;
      if (totals) {
        if (lin_first) totals->stage1_time += tm.stage1_time;
        totals->stage2_time += tm.stage2_time; totals->compute_preconditioner_time += tm.compute_preconditioner_time;
        totals->solve_reduced_system_time += tm.solve_reduced_system_time; totals->back_substitution_time += tm.back_substitution_time;
        totals->update_cameras_time += tm.update_cameras_time; totals->residual_evaluation_time += tm.residual_evaluation_time;
        totals->matvec_launches += tm.matvec_launches;
      }
      L2.device_seconds = dev;
      L2.cg_iterations = r.cg.num_iterations; L2.cg_termination = r.cg.termination_type;
      L2.l_diff = r.l_diff;
      L2.cost = std::numeric_limits<double>::quiet_NaN();
      bool success = false;
      const double prev = prev_logged;
      if (r.solve_failed) {
        // non-finite increment (:360-399): not applied by the reference; here undone
        rc = restore(); if (rc) return rc;
        prev_logged = 0;
      } else {
        const double cur = cost_of(r.cost, prev_kind);
        prev_logged = cur;
        const S l_diff = (S)r.l_diff;
        const bool ok = std::isfinite((double)l_diff) && r.cost.is_numerically_valid;
        L2.cost = cost_of(r.cost, o->optimized_cost);
        if (ok) {
          const S f_diff = (S)(cost_of(ri, o->optimized_cost) - cost_of(r.cost, o->optimized_cost));
          S ld = l_diff;
          if (o->optimized_cost == 2) ld = (S)(l_diff / (S)ri.valid_num_obs);  // :436-438
          const S q = (S)(f_diff / ld);
          L2.relative_decrease = (double)q;
          success = ld > S(0) && (double)q > o->min_relative_decrease;     // :443-446
          if (success) {
            const double fac = std::max(1.0 / 3.0, 1.0 - std::pow(2.0 * (double)q - 1.0, 3));
            lam = (S)(lam * (S)fac);                                         // :462-466
            lam = std::max(min_lambda, lam);
            vee = initial_vee;
            new_outer = true;
            terminated = std::fabs(prev - cur) <= o->function_tolerance * cur;  // function_tolerance_reached (:174-201)
          }
        }
        if (!success) { rc = restore(); if (rc) return rc; }
      }
      if (!success) {
        lam = (S)(vee * lam); vee = (S)(vee * vee_factor);                   // :378-379, :499-500
        if (lam > max_lambda) terminated = true;
      }
      L2.accepted = success ? 1 : 0;
      if (it + 1 >= o->max_num_iterations) terminated = true;
      L2.terminated = terminated ? 1 : 0;
    }
    *steps_done = it;
    *terminated_out = terminated ? 1 : 0;
    return RBA_OK;
  }

  int get_timings(rba_stage_timings* out) const override { *out = tm; out->kernel_launches = launches; return RBA_OK; }
  int get_stats(rba_workload_stats* out) const override {
    std::memset(out, 0, sizeof(*out));
    out->num_landmarks_local = L.nl_local;
    out->num_observations_local = L.nobs_local;
    out->sum_n2 = L.sum_n2;
    out->max_n = L.max_n;
    out->num_tiles = (int)L.tiles.size();
    out->panel_scalars = L.panel_scalars;
    out->panel_scalars_algorithmic = 18 * L.sum_n2;
    out->device_bytes = (int64_t)device_bytes;
    out->matvec_algorithmic_bytes = (18 * L.sum_n2 + 18 * L.nobs_local) * (int64_t)sizeof(S) + 4 * L.nobs_local;
    out->landmark_begin = L.lm_begin;
    out->landmark_end = L.lm_end;
    out->num_matvec_items = (int)L.items.size();
    return RBA_OK;
  }

  int get_scaling(void* scaling, void* diag2) override {
    if (scaling) CU(cudaMemcpyAsync(scaling, D.scaling, (size_t)9 * nc * sizeof(S), cudaMemcpyDeviceToHost, stream));
    if (diag2) CU(cudaMemcpyAsync(diag2, D.diag2, (size_t)9 * nc * sizeof(S), cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    return RBA_OK;
  }
  int get_rhs(void* b) override {
    CU(cudaMemcpyAsync(b, D.b, (size_t)9 * nc * sizeof(S), cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    return RBA_OK;
  }
  int get_precond(void* inv, void* blocks) override {
    if (inv) CU(cudaMemcpyAsync(inv, D.inv, (size_t)81 * nc * sizeof(S), cudaMemcpyDeviceToHost, stream));
    if (blocks) CU(cudaMemcpyAsync(blocks, D.blocks, (size_t)81 * nc * sizeof(S), cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    return RBA_OK;
  }
  // ref: qr/linearization_qr.hpp:823-825
  int right_multiply(const void* x, void* y) override {
    if (!linearized || !damping_valid) { g_err = "rba_right_multiply needs rba_linearize + rba_solve first"; return RBA_ERR_STATE; }
    CU(cudaMemcpyAsync(D.z, x, (size_t)9 * nc * sizeof(S), cudaMemcpyHostToDevice, stream));
    CU(cudaMemsetAsync(D.y, 0, (size_t)9 * nc * sizeof(S), stream));  // cameras without observations in this shard are not written
    matvec_launch(D.z, nullptr);
    int rc = matvec_finish(D.z, D.y, last_lambda, nullptr, nullptr); if (rc) return rc;
    CU(cudaMemcpyAsync(y, D.y, (size_t)9 * nc * sizeof(S), cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    CU(cudaGetLastError());
    return RBA_OK;
  }

  int time_matvec(int reps, double* sec) override {
    if (!linearized || !damping_valid) { g_err = "rba_time_matvec needs rba_linearize + rba_solve first"; return RBA_ERR_STATE; }
    matvec_launch(D.p, nullptr);  // warm-up
    int rc = start(ev_mv); if (rc) return rc;
    for (int r = 0; r < reps; ++r) matvec_launch(D.p, nullptr);
    rc = stop(ev_mv); if (rc) return rc;
    CU(cudaStreamSynchronize(stream));
    CU(cudaGetLastError());
    *sec = elapsed(ev_mv) / std::max(reps, 1);
    tm.matvec_time = *sec;
    return RBA_OK;
  }

  int timer_start() override { return start(ev_user); }
  int timer_stop(double* sec) override {
    int rc = stop(ev_user); if (rc) return rc;
    CU(cudaStreamSynchronize(stream));
    *sec = elapsed(ev_user);
    return RBA_OK;
  }
  void* stream_ptr() override { return (void*)stream; }
  int synchronize() override { CU(cudaStreamSynchronize(stream)); return RBA_OK; }

  // reference-layout view of one landmark block (see header)
  int debug_get_block(int lm, void* out, int rows, int cols, void* jls_out) override {
    if (lm < L.lm_begin || lm >= L.lm_end) { g_err = "landmark not in this shard"; return RBA_ERR_INVALID_ARGUMENT; }
    const int sidx = L.sorted_of_lm[lm - L.lm_begin];
    const TileInfo& T = L.tiles[L.tile_of_sorted[sidx]];
    const int n = T.n, G = T.G, KP = T.KP, g = sidx - T.lm_base;
    const int pad = (4 - (9 * n) % 4) % 4, lm_idx = 9 * n + pad, res_idx = lm_idx + 3;
    if (rows != 2 * n + 3 || cols != res_idx + 1) { g_err = "block dims mismatch"; return RBA_ERR_INVALID_ARGUMENT; }
    if (!D.panel) { g_err = "rba_debug_get_block needs operator_form = 0 (no Q2 panels are stored for the implicit operator)"; return RBA_ERR_UNSUPPORTED; }
    CU(cudaStreamSynchronize(stream));
    std::vector<S> panel((size_t)2 * n * KP * 64), rec((size_t)28 * n), lmk(24);
    const int slot0 = T.slot_base + g * n;
    CU(cudaMemcpy(panel.data(), D.panel + T.panel_off, panel.size() * sizeof(S), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(rec.data(), D.q1d + (size_t)28 * slot0, rec.size() * sizeof(S), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(lmk.data(), D.lmk + (size_t)24 * sidx, 24 * sizeof(S), cudaMemcpyDeviceToHost));
    S* o = (S*)out;
    std::fill(o, o + (size_t)rows * cols, S(0));
    for (int c = 0; c < 9 * n; ++c) {
      const int i = c / 9, p = c % 9;
      for (int m = 0; m < 3; ++m) o[(size_t)m * cols + c] = rec[(size_t)28 * i + 9 * m + p];  // damped Q1^T Jp
      const int pr = c / 2, v = c % 2, k = pr / G, j = pr % G, lane = g * G + j;
      for (int r = 0; r < 2 * n; ++r) o[(size_t)(3 + r) * cols + c] = panel[(((size_t)r * KP + k) * 32 + lane) * 2 + v];
    }
    o[0 * cols + lm_idx] = lmk[9]; o[0 * cols + lm_idx + 1] = lmk[10]; o[0 * cols + lm_idx + 2] = lmk[11];
    o[1 * cols + lm_idx + 1] = lmk[12]; o[1 * cols + lm_idx + 2] = lmk[13]; o[2 * cols + lm_idx + 2] = lmk[14];
    for (int m = 0; m < 3; ++m) o[(size_t)m * cols + res_idx] = lmk[15 + m];
    if (jls_out) for (int d = 0; d < 3; ++d) ((S*)jls_out)[d] = lmk[18 + d];
    return RBA_OK;
  }
};

template <class S>
int create_impl(const rba_problem_view* pv, const rba_solver_opts* o, rba_handle** out) {
  if (!pv || !o || !out) { g_err = "null argument"; return RBA_ERR_INVALID_ARGUMENT; }
  if (pv->num_cameras <= 0 || pv->num_landmarks <= 0 || !pv->lm_obs_offset || !pv->obs_cam_idx || !pv->obs_xy) {
    g_err = "empty problem";
    return RBA_ERR_INVALID_ARGUMENT;
  }
  auto* s = new Solver<S>();
  s->scalar_size = sizeof(S);
  int rc = s->init(pv, o);
  if (rc != RBA_OK) { delete s; return rc; }
  *out = s;
  return RBA_OK;
}

}  // namespace rba

extern "C" {

int32_t rba_abi_version(void) { return RBA_ABI_VERSION; }
const char* rba_last_error(void) { return rba::g_err.c_str(); }

void rba_default_solver_opts(rba_solver_opts* o) {
  std::memset(o, 0, sizeof(*o));
  o->use_householder_marginalization = 1;
  o->use_valid_projections_only = 0;
  o->robust_norm = 0;
  o->huber_parameter = 1.0;
  o->jacobi_scaling_epsilon = 0.0;
  o->preconditioner_type = 1;
  o->min_linear_solver_iterations = 0;
  o->max_linear_solver_iterations = 500;
  o->eta = 0.1;
  o->residual_reset_period = 10;
  o->device = -1;
  o->rank = 0;
  o->nranks = 1;
  o->pcg_check_period = 4;
  o->use_cuda_graphs = 0;
  o->power_order = 20;
}

int32_t rba_create_f32(const rba_problem_view* p, const rba_solver_opts* o, rba_handle** out) { return rba::create_impl<float>(p, o, out); }
int32_t rba_create_f64(const rba_problem_view* p, const rba_solver_opts* o, rba_handle** out) { return rba::create_impl<double>(p, o, out); }
int32_t rba_destroy(rba_handle* h) { delete h; return RBA_OK; }
int32_t rba_get_workload_stats(const rba_handle* h, rba_workload_stats* out) { return h->get_stats(out); }
int32_t rba_scalar_size(const rba_handle* h) { return h->scalar_size; }

int32_t rba_partition_landmarks(int32_t nl, const int64_t* off, int32_t nranks, int32_t* bounds) {
  if (nl <= 0 || nranks <= 0 || !off || !bounds) return RBA_ERR_INVALID_ARGUMENT;
  rba::partition_landmarks(nl, off, nranks, bounds);
  return RBA_OK;
}

// ---- BAL loader (host only) ----
struct rba_bal_file {
  rootba_b200::BalProblemSoA<double> p;
  double timings[5] = {0, 0, 0, 0, 0};
};

int32_t rba_bal_load(const char* path, int32_t normalize, double scale, int32_t num_threads, rba_bal_file** out) {
  if (!path || !out) { rba::g_err = "bad arguments"; return RBA_ERR_INVALID_ARGUMENT; }
  *out = nullptr;
  try {
    std::unique_ptr<rba_bal_file> f(new rba_bal_file());
    rootba_b200::LoadTimings t;
    if (rootba_b200::detail::is_bundler_file(path)) f->p = rootba_b200::load_bundler_soa(path, num_threads);  // autodetect_input_type
    else f->p = rootba_b200::load_bal_parallel(path, num_threads, &t);
    const auto t0 = std::chrono::steady_clock::now();
    if (normalize) f->p.normalize(scale);
    f->timings[0] = t.read; f->timings[1] = t.count; f->timings[2] = t.parse; f->timings[3] = t.csr;
    f->timings[4] = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    *out = f.release();
    return RBA_OK;
  } catch (const std::exception& e) {
    rba::g_err = e.what();
    return RBA_ERR_INVALID_ARGUMENT;
  }
}
int32_t rba_bal_filter_obs(rba_bal_file* f, double threshold) {
  if (!f || threshold < 0) { rba::g_err = "bad arguments"; return RBA_ERR_INVALID_ARGUMENT; }  // the reference CHECK_GEs the threshold
  f->p.filter_obs(threshold);
  return RBA_OK;
}
int32_t rba_bal_perturb(rba_bal_file* f, double rotation_sigma, double translation_sigma, double point_sigma, int32_t seed) {
  if (!f || rotation_sigma < 0 || translation_sigma < 0 || point_sigma < 0) { rba::g_err = "bad arguments"; return RBA_ERR_INVALID_ARGUMENT; }  // reference: CHECK_GE
  f->p.perturb(rotation_sigma, translation_sigma, point_sigma, seed);
  return RBA_OK;
}
int32_t rba_bal_dims(const rba_bal_file* f, int32_t* nc, int32_t* nl, int64_t* nobs) {
  if (!f) return RBA_ERR_INVALID_ARGUMENT;
  if (nc) *nc = f->p.nc;
  if (nl) *nl = f->p.nl;
  if (nobs) *nobs = f->p.num_observations();
  return RBA_OK;
}
int32_t rba_bal_copy(const rba_bal_file* f, double* cams, double* lms, int64_t* off, int32_t* oc, double* xy) {
  if (!f) return RBA_ERR_INVALID_ARGUMENT;
  if (cams) std::copy(f->p.cams.begin(), f->p.cams.end(), cams);
  if (lms) std::copy(f->p.lms.begin(), f->p.lms.end(), lms);
  if (off) std::copy(f->p.lm_off.begin(), f->p.lm_off.end(), off);
  if (oc) std::copy(f->p.obs_cam.begin(), f->p.obs_cam.end(), oc);
  if (xy) std::copy(f->p.obs_xy.begin(), f->p.obs_xy.end(), xy);
  return RBA_OK;
}
int32_t rba_bal_load_timings(const rba_bal_file* f, double* out5) {
  if (!f || !out5) return RBA_ERR_INVALID_ARGUMENT;
  std::copy(f->timings, f->timings + 5, out5);
  return RBA_OK;
}
int32_t rba_bal_free(rba_bal_file* f) { delete f; return RBA_OK; }

int32_t rba_layout_selftest(const rba_problem_view* pv, int32_t rank, int32_t nranks, int32_t scalar_size) {
  using namespace rba;
  if (!pv || nranks < 1 || rank < 0 || rank >= nranks) { g_err = "bad arguments"; return RBA_ERR_INVALID_ARGUMENT; }
  Layout L;
  std::string msg = build_layout(pv->num_cameras, pv->num_landmarks, pv->lm_obs_offset, pv->obs_cam_idx, rank, nranks, scalar_size == 4 ? 16 : 10, L);
  if (!msg.empty()) { g_err = msg; return RBA_ERR_INVALID_ARGUMENT; }
  auto fail = [&](const std::string& m) { g_err = "layout selftest: " + m; return RBA_ERR_STATE; };
  // observations <-> slots
  std::vector<char> seen((size_t)L.nobs_local, 0);
  const int64_t obs0 = pv->lm_obs_offset[L.lm_begin];
  long long real_slots = 0;
  for (int s = 0; s < L.nslots; ++s) {
    if (L.slot_lm[s] < 0) { if (L.slot_obs[s] >= 0) return fail("padding slot with an observation"); continue; }
    const long long o = L.slot_obs[s];
    if (o < obs0 || o - obs0 >= L.nobs_local) return fail("slot observation outside the shard");
    if (seen[o - obs0]++) return fail("observation assigned twice");
    if (pv->obs_cam_idx[o] != L.slot_cam[s]) return fail("slot camera mismatch");
    const int lm = L.lm_begin + L.slot_lm[s];
    if (o < pv->lm_obs_offset[lm] || o >= pv->lm_obs_offset[lm + 1]) return fail("slot landmark mismatch");
    ++real_slots;
  }
  if (real_slots != L.nobs_local) return fail("not every observation has a slot");
  // tiles
  std::vector<char> lm_seen((size_t)L.nl_local, 0);
  long long panel = 0;
  for (size_t t = 0; t < L.tiles.size(); ++t) {
    const TileInfo& T = L.tiles[t];
    const int W = 32 / T.G;
    if (T.G != group_size_for(T.n) || T.KP != kp_for(T.n, T.G) || 2 * T.G * T.KP < 9 * T.n) return fail("tile class");
    if (T.panel_off != panel) return fail("panel offsets are not contiguous");
    panel += (long long)2 * T.n * T.KP * 64;
    for (int g = 0; g < W; ++g) {
      const int lm = L.sorted_lm[T.lm_base + g];
      if ((g < T.nvalid) != (lm >= 0)) return fail("nvalid");
      if (lm < 0) continue;
      if (lm_seen[lm]++) return fail("landmark in two tiles");
      if (pv->lm_obs_offset[L.lm_begin + lm + 1] - pv->lm_obs_offset[L.lm_begin + lm] != T.n) return fail("track length of tile");
      for (int i = 0; i < T.n; ++i) {
        const int s = T.slot_base + g * T.n + i;
        if (L.slot_lm[s] != lm || L.slot_obs[s] != pv->lm_obs_offset[L.lm_begin + lm] + i) return fail("slot order inside a landmark");
      }
      if (L.sorted_of_lm[lm] != T.lm_base + g) return fail("sorted_of_lm");
    }
  }
  if (panel != L.panel_scalars) return fail("panel size");
  for (char c : lm_seen) if (!c) return fail("landmark without tile");
  // matvec items: row chunks tile [0, 2n) of every tile exactly once; y slots
  std::vector<int> rows_covered(L.tiles.size(), 0);
  std::vector<char> yslot_used((size_t)L.nyslots, 0);
  for (const MatvecItem& it : L.items) {
    const TileInfo& T = L.tiles[it.tile];
    if (it.nrows <= 0 || it.row0 < 0 || it.row0 + it.nrows > 2 * T.n) return fail("item rows");
    rows_covered[it.tile] += it.nrows;
    for (int k = 0; k < (32 / T.G) * T.n; ++k) {
      if (it.yslot_base + k >= L.nyslots) return fail("y slot range");
      if (yslot_used[it.yslot_base + k]++) return fail("y slot written by two items");
    }
  }
  for (size_t t = 0; t < L.tiles.size(); ++t) if (rows_covered[t] != 2 * L.tiles[t].n) return fail("rows not covered exactly once");
  // camera CSRs
  auto check_csr = [&](const CameraCSR& C, long long expect) -> bool {
    if ((long long)C.slots.size() != expect) return false;
    for (int c = 0; c < pv->num_cameras; ++c) {
      for (int e = C.cam_ptr[c]; e < C.cam_ptr[c + 1]; ++e) if (e > C.cam_ptr[c] && C.slots[e] <= C.slots[e - 1]) return false;
      int covered = 0;
      for (int q = C.cam_item_ptr[c]; q < C.cam_item_ptr[c + 1]; ++q) {
        if (C.items[q].cam != c || C.items[q].begin != C.cam_ptr[c] + covered) return false;
        covered += C.items[q].end - C.items[q].begin;
      }
      if (covered != C.cam_ptr[c + 1] - C.cam_ptr[c]) return false;
    }
    return true;
  };
  if (!check_csr(L.csr_obs, L.nobs_local)) return fail("observation CSR");
  for (int c = 0; c < pv->num_cameras; ++c)
    for (int e = L.csr_obs.cam_ptr[c]; e < L.csr_obs.cam_ptr[c + 1]; ++e)
      if (L.slot_cam[L.csr_obs.slots[e]] != c || L.slot_lm[L.csr_obs.slots[e]] < 0) return fail("observation CSR camera");
  if (!L.csr_y_is_obs) {
    long long expect = 0;
    for (const MatvecItem& it : L.items) expect += (long long)L.tiles[it.tile].nvalid * L.tiles[it.tile].n;
    if (!check_csr(L.csr_y, expect)) return fail("y CSR");
  }
  return RBA_OK;
}

int32_t rba_set_state(rba_handle* h, const void* cams, const void* lms) { return h->set_state(cams, lms); }
int32_t rba_get_state(rba_handle* h, void* cams, void* lms) { return h->get_state(cams, lms); }
int32_t rba_backup(rba_handle* h) { return h->backup(); }
int32_t rba_restore(rba_handle* h) { return h->restore(); }
int32_t rba_compute_error(rba_handle* h, rba_residual_info* out) { return h->compute_error(out); }
int32_t rba_linearize(rba_handle* h) { return h->linearize(); }

#define CHECK_TYPE(h, sz) \
  if ((h)->scalar_size != (sz)) { rba::g_err = "scalar type of the handle does not match the entry point"; return RBA_ERR_INVALID_ARGUMENT; }

int32_t rba_solve_f32(rba_handle* h, float lambda, float* inc, rba_cg_summary* cg) { CHECK_TYPE(h, 4); return h->solve(lambda, inc, cg); }
int32_t rba_solve_f64(rba_handle* h, double lambda, double* inc, rba_cg_summary* cg) { CHECK_TYPE(h, 8); return h->solve(lambda, inc, cg); }
int32_t rba_apply_f32(rba_handle* h, const float* inc, float* l) { CHECK_TYPE(h, 4); return h->apply(inc, l, true); }
int32_t rba_apply_f64(rba_handle* h, const double* inc, double* l) { CHECK_TYPE(h, 8); return h->apply(inc, l, true); }
int32_t rba_lm_step_f32(rba_handle* h, int32_t linearize_first, float lambda, rba_lm_step_result* out) { CHECK_TYPE(h, 4); return h->lm_step(linearize_first != 0, lambda, out); }
int32_t rba_lm_step_f64(rba_handle* h, int32_t linearize_first, double lambda, rba_lm_step_result* out) { CHECK_TYPE(h, 8); return h->lm_step(linearize_first != 0, lambda, out); }
void rba_default_lm_opts(rba_lm_opts* o) {  /* defaults of SolverOptions (solver_options.hpp) */
  o->initial_trust_region_radius = 1e4; o->min_trust_region_radius = 1e-32; o->max_trust_region_radius = 1e16;
  o->min_relative_decrease = 0.0; o->initial_vee = 2.0; o->vee_factor = 2.0; o->function_tolerance = 1e-6;
  o->max_num_iterations = 20; o->optimized_cost = 0;
}
int32_t rba_lm_run_f32(rba_handle* h, const rba_lm_opts* o, int32_t max_steps, rba_lm_iteration* log, int32_t* steps_done, int32_t* terminated, rba_stage_timings* totals) {
  CHECK_TYPE(h, 4); if (!o || !log || !steps_done || !terminated || max_steps < 0) { rba::g_err = "bad arguments"; return RBA_ERR_INVALID_ARGUMENT; }
  return h->lm_run(o, max_steps, log, steps_done, terminated, totals);
}
int32_t rba_lm_run_f64(rba_handle* h, const rba_lm_opts* o, int32_t max_steps, rba_lm_iteration* log, int32_t* steps_done, int32_t* terminated, rba_stage_timings* totals) {
  CHECK_TYPE(h, 8); if (!o || !log || !steps_done || !terminated || max_steps < 0) { rba::g_err = "bad arguments"; return RBA_ERR_INVALID_ARGUMENT; }
  return h->lm_run(o, max_steps, log, steps_done, terminated, totals);
}
int32_t rba_back_substitute_f32(rba_handle* h, const float* inc, float* l) { CHECK_TYPE(h, 4); return h->apply(inc, l, false); }
int32_t rba_back_substitute_f64(rba_handle* h, const double* inc, double* l) { CHECK_TYPE(h, 8); return h->apply(inc, l, false); }
int32_t rba_get_timings(const rba_handle* h, rba_stage_timings* out) { return h->get_timings(out); }
int32_t rba_get_jacobian_scaling(rba_handle* h, void* s, void* d) { return h->get_scaling(s, d); }
int32_t rba_get_rhs(rba_handle* h, void* b) { return h->get_rhs(b); }
int32_t rba_get_preconditioner(rba_handle* h, void* inv, void* blocks) { return h->get_precond(inv, blocks); }
int32_t rba_right_multiply(rba_handle* h, const void* x, void* y) { return h->right_multiply(x, y); }
int32_t rba_debug_get_block(rba_handle* h, int32_t lm, void* out, int32_t rows, int32_t cols, void* jls) {
  return h->debug_get_block(lm, out, rows, cols, jls);
}
int32_t rba_time_matvec(rba_handle* h, int32_t reps, double* sec) { return h->time_matvec(reps, sec); }
int32_t rba_timer_start(rba_handle* h) { return h->timer_start(); }
int32_t rba_timer_stop(rba_handle* h, double* sec) { return h->timer_stop(sec); }
void* rba_stream(rba_handle* h) { return h->stream_ptr(); }
int32_t rba_synchronize(rba_handle* h) { return h->synchronize(); }

int32_t rba_nccl_unique_id(void* out128) {
  rba::NcclApi* api = rba::nccl_api();
  if (!api) { rba::g_err = "libnccl.so.2 could not be loaded"; return RBA_ERR_NCCL; }
  ncclUniqueId id;
  ncclResult_t r = api->GetUniqueId(&id);
  if (r != ncclSuccess) { rba::g_err = std::string("ncclGetUniqueId: ") + api->GetErrorString(r); return RBA_ERR_NCCL; }
  std::memcpy(out128, &id, sizeof(id));
  return RBA_OK;
}
int32_t rba_comm_init(rba_handle* h, const void* uid) { return h->comm_init(uid); }
int32_t rba_ipc_export(rba_handle* h, void* out128) { return h->ipc_export(out128); }
int32_t rba_ipc_import(rba_handle* h, const void* all) { return h->ipc_import(all); }

}  // extern "C"
