// Host-side planner of the fused MLP-chain kernel: turns a chain description into the static job streams
// of csrc/chain_plan.cuh (MMA jobs = weight chunks, loader jobs, epilogue jobs), sizes the rings, and
// proves the plan deadlock-free by simulating it.  No CUDA calls here — the plan is testable on a
// CPU-only box (tests/test_chain_plan_cpu.py).
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "chain_plan.cuh"
#include "common.cuh"

namespace s4g {
namespace {

// ---- cost model (SM cycles, measured with profiles/{umma_bw,issue_cost,tmem_bw}.cu); it only ranks ring
// ---- sizes against each other — correctness never depends on it
constexpr double kWeightLatency = 1100.0;  // L2 -> smem, one 32 KB bulk copy
constexpr double kWeightIssue = 535.0;     // one producer thread issues a bulk copy every ~535 cycles
constexpr double kLoadLatency = 1800.0;    // cp.async of input rows (HBM / L2)
constexpr double kXyzCost = 900.0;         // dependent index -> coordinate loads, synchronous
constexpr double kIssueFixed = 250.0;      // MMA warp: waits + commits + bookkeeping per job
constexpr double kIssuePerMma = 20.0;

struct Block { int kind, c_begin, c_count, layer; };
struct HMma { int blk, acc, k16, koff, n_rows, flags, layer, n_begin, k_begin, n_mma; };
struct HEpi { int kind, acc, blk, layer, relu, c_begin, c_count, aux, pred, same, min_it, coop, sub; };
struct HLoad { int kind, blk, c_begin, c_count, pred, same, min_it, sub; };

struct Draft {
  int S = 0, stages = 0, n_acc = 0, depth = 0;
  std::vector<Block> blocks;
  std::vector<HMma> mma;
  std::vector<HEpi> epi;     // accumulator order = epilogue stream
  std::vector<HLoad> loads;  // production order = loader stream of one tile
};

int round_up(int x, int m) { return (x + m - 1) / m * m; }

// which row-oriented epilogue jobs all 16 warps share: 0 none, 1 all, 2 those whose accumulator is not half of an
// N = 256 pair (a pair is already drained by both groups at once), 3 (default) = 2, but only in chains whose hidden
// layers are all at most 128 wide.  Measured (profiles/ab_chains.py, policy 0 -> 2): the chain that is bound by the
// latency of single-accumulator layers gains (sa0 4.73 -> 4.27 ms); in wide chains the tile tail already overlaps the
// next tile's first layer and the extra barrier traffic of a shared job costs more than the earlier hand-off
// (head chain 1.635 -> 1.72 ms).
thread_local int g_force_coop = -1;  // set by plan_chain for the duration of one planning call (host autotuning)
int coop_policy() {
  if (g_force_coop >= 0) return g_force_coop;
  const char* e = getenv("S4G_EPI_COOP");
  return e ? atoi(e) : 3;
}

// R = row blocks (sub-tiles of 128 rows) per tile.  With R = 2 every layer is emitted for sub-tile 0, then for sub-tile
// 1: the job streams of two 128-row tiles interleaved layer by layer, so that the MMAs of one run while the epilogue
// of the other drains — for narrow chains, whose tile is otherwise a strict MMA -> epilogue -> MMA ping-pong.
bool build_draft(const s4g_chain* ch, const int* relu, int feat_c, int S, bool pair_ok, int R, bool tma_in, Draft& d) {
  const int L = ch->n_layers;
  std::vector<Block> in_desc;
  if (ch->in_mode == IN_ROWS) {
    for (int c = 0; c < ch->cin_pad[0]; c += 128) in_desc.push_back({WK_LOAD_ROWS, c, std::min(128, ch->cin_pad[0] - c), -1});
  } else if (ch->in_mode == IN_XYZ_MLP) {
    in_desc.push_back({WK_LOAD_XYZ, 0, ch->cin_pad[0], -1});
  } else {
    for (int c = 0; c < feat_c; c += 128) in_desc.push_back({WK_LOAD_FEAT, c, std::min(128, feat_c - c), -1});
    in_desc.push_back({WK_LOAD_XYZ, feat_c, 16, -1});
  }
  std::vector<int> cur_sub[2];
  int n_maxpool = 0;
  for (int l = 0; l < L; ++l) {
    const bool last = (l == L - 1);
    const bool transposed = last && ch->out_mode == OUT_MAXPOOL;
    const int width = ch->cout_pad[l];
    std::vector<std::pair<int, int>> nbs;
    for (int n = 0; n < width; n += 128) nbs.push_back({n, std::min(128, width - n)});
    const int nn = (int)nbs.size();
    const int nk = (l == 0) ? (int)in_desc.size() : (int)cur_sub[0].size();
    // N-outer (one output block after the other, each over all K-blocks; the epilogue of block n overlaps
    // the MMAs of block n+1) needs every K-block and all but the last output block resident at once;
    // otherwise K-outer: up to 4 accumulators filled K-block by K-block, inputs released as they go.
    // (the outputs of the LAST N-group — a pair of blocks when pairs are allowed — are written only after
    // every K-block of the layer has been released, so they need no slot of their own)
    const int last_grp = (pair_ok && !transposed && nn >= 2 && nn % 2 == 0 && (d.n_acc % 2 == 0)) ? 2 : 1;
    const int need = nk + (last ? 0 : nn - last_grp);
    const bool n_outer = need <= S;
    if (!n_outer && l > 0 && nn > kAccBlocks) return false;  // a hidden layer cannot be re-read in passes
    if (!n_outer && !last && nn > S) return false;
    const int passes = n_outer ? 1 : (nn + kAccBlocks - 1) / kAccBlocks;
    // With two row blocks the input blocks of BOTH come first in the block order.  The slot protocol waits with a
    // one-bit phase ("the release of block pred in the previous tile"), which is only unambiguous if block pred of the
    // CURRENT tile cannot be released before that wait is made; an epilogue-produced block whose slot predecessor
    // is a loader-produced block of higher index would break that (the loader and the MMA warp run ahead of the
    // epilogue).  Inputs first + S <= blocks per tile rules it out, as in the single-block order.
    std::vector<int> kin_pre[2];
    if (l == 0 && R > 1) {
      if (passes != 1) return false;
      for (int sub = 0; sub < R; ++sub)
        for (const Block& b : in_desc) {
          const int idx = (int)d.blocks.size();
          d.blocks.push_back(b);
          d.loads.push_back({b.kind, idx, b.c_begin, b.c_count, 0, 0, 0, sub});
          kin_pre[sub].push_back(idx);
        }
    }
    for (int sub = 0; sub < R; ++sub) {
    std::vector<int>& cur = cur_sub[sub];
    std::vector<int> produced;
    for (int pass = 0; pass < passes; ++pass) {
      const int nb0 = n_outer ? 0 : pass * kAccBlocks;
      const int nb1 = n_outer ? nn : std::min(nn, nb0 + kAccBlocks);
      std::vector<int> kin;
      if (l == 0 && R > 1) {
        kin = kin_pre[sub];
      } else if (l == 0) {
        for (const Block& b : in_desc) {
          const int idx = (int)d.blocks.size();
          d.blocks.push_back(b);
          d.loads.push_back({b.kind, idx, b.c_begin, b.c_count, 0, 0, 0, sub});
          kin.push_back(idx);
        }
      } else {
        kin = cur;
      }
      const int acc0 = d.n_acc;
      d.n_acc += nb1 - nb0;
      // N-groups: two adjacent full blocks share N = 256 MMAs when their accumulators form an aligned pair
      struct Grp { int nb, cnt; };
      std::vector<Grp> grps;
      for (int nb = nb0; nb < nb1;) {
        const int acc = acc0 + nb - nb0;
        const bool pair = pair_ok && !transposed && (acc % 2 == 0) && nb + 1 < nb1 && nbs[nb].second == 128 &&
                          nbs[nb + 1].second == 128;
        grps.push_back({nb, pair ? 2 : 1});
        nb += pair ? 2 : 1;
      }
      auto emit = [&](size_t gi, int kb) {
        const Grp& g = grps[gi];
        const Block& b = d.blocks[kin[kb]];
        const int steps = b.c_count / 16;
        // <= 32 KB of weights per job; a job on a swizzled (TMA-loaded) input block stays inside one 64-channel half
        const bool swz = tma_in && l == 0 && b.kind != WK_LOAD_XYZ;  // (the xyz block is written by threads: interleaved)
        const int per_job = (g.cnt == 2 || swz) ? 4 : 8;
        for (int ks = 0; ks < steps; ks += per_job) {
          const int k16 = std::min(per_job, steps - ks);
          const bool tail = ks + per_job >= steps;
          int flags = 0;
          if (gi == 0 && ks == 0) flags |= MF_WAIT_ACT;
          if (kb == 0 && ks == 0) flags |= MF_FIRST_K;
          if (kb == nk - 1 && tail) flags |= MF_LAST_K;
          if (gi + 1 == grps.size() && tail) flags |= MF_RELEASE;
          if (transposed) flags |= MF_TRANSPOSED;
          if (g.cnt == 2) flags |= MF_PAIR;
          if (swz) flags |= MF_SWZ;
          const int n_rows = transposed ? 128 : (g.cnt == 2 ? 256 : nbs[g.nb].second);
          d.mma.push_back({kin[kb], acc0 + g.nb - nb0, k16, ks, n_rows, flags, l, nbs[g.nb].first, b.c_begin + ks * 16,
                           transposed ? 128 : n_rows});
        }
      };
      if (n_outer) {
        for (size_t gi = 0; gi < grps.size(); ++gi)
          for (int kb = 0; kb < nk; ++kb) emit(gi, kb);
      } else {
        for (int kb = 0; kb < nk; ++kb)
          for (size_t gi = 0; gi < grps.size(); ++gi) emit(gi, kb);
      }
      std::vector<int> in_pair(nn, 0);
      for (const Grp& g : grps)
        if (g.cnt == 2) in_pair[g.nb] = in_pair[g.nb + 1] = 1;
      int policy = coop_policy();
      if (policy == 3) {
        policy = 2;
        for (int h = 0; h + 1 < L; ++h)
          if (ch->cout_pad[h] > 128) policy = 0;
      }
      for (int nb = nb0; nb < nb1; ++nb) {
        const int acc = acc0 + nb - nb0;
        const int coop = policy == 1 || (policy == 2 && !in_pair[nb]);
        if (!last) {
          const int idx = (int)d.blocks.size();
          d.blocks.push_back({WK_EPI_HIDDEN, nbs[nb].first, nbs[nb].second, l});
          produced.push_back(idx);
          d.epi.push_back({WK_EPI_HIDDEN, acc, idx, l, relu[l], nbs[nb].first, nbs[nb].second, 0, 0, 0, 0, coop, sub});
        } else {
          const int kind = ch->out_mode == OUT_ROWS ? WK_EPI_ROWS : ch->out_mode == OUT_MAXPOOL ? WK_EPI_MAXPOOL : WK_EPI_LOGITS;
          d.epi.push_back({kind, acc, -1, l, relu[l], nbs[nb].first, nbs[nb].second, (n_maxpool++) & 1, 0, 0, 0,
                           kind == WK_EPI_ROWS ? coop : 0, sub});
        }
      }
    }
    cur = produced;
    }
  }
  d.S = S;
  // slot re-use: block b of tile t inherits the slot of block (t * nB + b - S); see chain_plan.cuh
  const int nB = (int)d.blocks.size();
  if (nB > kMaxBlocks) return false;
  auto pred_of = [&](int b, int& pred, int& same, int& min_it) {
    pred = ((b - S) % nB + nB) % nB;
    same = b >= S ? 1 : 0;
    min_it = same ? 0 : (S - b + nB - 1) / nB;
  };
  // The one-bit barrier phase makes "wait for the release of block pred in the previous tile" ambiguous when
  // that block of the CURRENT tile can already be dead, i.e. when pred < b for an epilogue-produced block,
  // which needs more slots than blocks per tile.  Chains with hidden layers therefore keep S <= blocks per tile.
  // The same holds for loader-produced blocks: with S > nB a block inherits its slot from a tile SEVERAL iterations
  // back, its first wait (at iteration min_it) is then up to min_it completions away from the barrier, and a parity
  // wait that far behind passes on the wrong phase — the loader overwrote a block the MMA warp had not read yet and
  // published its slot twice (tiles of a single 64-channel block, e.g. a 64 -> 32 layer, from the 4th tile of a CTA on:
  // mbarrier dead-lock -> trap; found by the tuner on the tiny test model, round 2).  So: S <= blocks per tile, always.
  if (S > nB) return false;
  for (HLoad& l : d.loads) pred_of(l.blk, l.pred, l.same, l.min_it);
  for (HEpi& e : d.epi)
    if (e.kind == WK_EPI_HIDDEN) pred_of(e.blk, e.pred, e.same, e.min_it);
  return (int)d.mma.size() <= kMaxMmaJobs && d.n_acc <= 255 && (int)d.blocks.size() <= 255 &&
         (int)d.epi.size() <= kMaxEpiJobs;
}

double epi_cost(const HEpi& e) {
  const double cols = e.coop ? 0.5 * e.c_count : e.c_count;  // columns per lane quadrant
  switch (e.kind) {
    case WK_EPI_HIDDEN: return 700.0 + 6.0 * cols;  // per group of 8 warps (profiles/chain_prof.py)
    case WK_EPI_ROWS: return 700.0 + 6.5 * cols;
    case WK_EPI_MAXPOOL: return 500.0;
    default: return 500.0;
  }
}

// ---------------------------------------------------------------------------------------------
// Simulation of T tiles: producers, MMA warp, loader warps, epilogue warps as four sequential actors.
// ---------------------------------------------------------------------------------------------
struct Sim {
  const Draft& d;
  int T, nB, nA, nC, nE, nL;
  std::vector<double> act_ready, act_free, issue_t, tm_full, tm_empty, w_full, w_empty;
  int pc_prod = 0, pc_mma = 0, pc_ld = 0, pc_ep[kEpiGroups] = {0, 0};
  double t_prod[2] = {0, 0}, last_arrive = 0, t_mma = 0, pipe = 0, pipe_busy = 0, t_ld = 0, t_ep[kEpiGroups] = {0, 0};
  std::vector<double> tile_end;

  Sim(const Draft& dd, int tiles)
      : d(dd), T(tiles), nB((int)dd.blocks.size()), nA(dd.n_acc), nC((int)dd.mma.size()), nE((int)dd.epi.size()),
        nL((int)dd.loads.size()) {
    act_ready.assign((size_t)T * nB, -1.0);
    act_free = issue_t = act_ready;
    tm_full.assign((size_t)T * nA, -1.0);
    tm_empty = tm_full;
    w_full.assign((size_t)T * nC, -1.0);
    w_empty = w_full;
    tile_end.assign(T, -1.0);
  }

  // time at which the producer of block `blk` of tile `tile` may write: the device waits for the release
  // of `pred` in the same tile, or in the PREVIOUS tile (which implies the true previous occupant)
  double slot_free(int tile, int pred, int same, int min_it) const {
    if (same) return act_free[tile * nB + pred];
    if (tile < min_it) return 0.0;
    return act_free[(tile - 1) * nB + pred];
  }

  bool adv_prod() {
    bool prog = false;
    while (pc_prod < T * nC) {
      const int c = pc_prod;
      double& tp = t_prod[c % kProducers];
      double issue = tp;
      if (c >= d.stages) {
        if (w_empty[c - d.stages] < 0) break;
        issue = std::max(issue, w_empty[c - d.stages]);
      }
      const HMma& j = d.mma[c % nC];
      const double bytes = j.n_rows * j.k16 * 32.0;  // rows x 16 k16 channels x 2 B
      const double arrive = std::max(issue + kWeightLatency, last_arrive + bytes / 64.0);
      w_full[c] = last_arrive = arrive;
      tp = issue + kWeightIssue;
      ++pc_prod;
      prog = true;
    }
    return prog;
  }

  bool adv_mma() {
    bool prog = false;
    while (pc_mma < T * nC) {
      const int tile = pc_mma / nC;
      const HMma& j = d.mma[pc_mma % nC];
      const int p = tile * nB + j.blk, q = tile * nA + j.acc;
      double t = t_mma;
      if (j.flags & MF_WAIT_ACT) {
        if (act_ready[p] < 0) break;
        t = std::max(t, act_ready[p]);
      }
      if ((j.flags & MF_FIRST_K) && q >= kAccBlocks) {
        if (tm_empty[q - kAccBlocks] < 0) break;
        t = std::max(t, tm_empty[q - kAccBlocks]);
        if (j.flags & MF_PAIR) {
          if (tm_empty[q + 1 - kAccBlocks] < 0) break;
          t = std::max(t, tm_empty[q + 1 - kAccBlocks]);
        }
      }
      if (w_full[pc_mma] < 0) break;
      t = std::max(t, w_full[pc_mma]);
      const double issue = t + kIssueFixed + kIssuePerMma * j.k16;
      const double start = std::max(issue, pipe);
      const double dur = j.k16 * std::max(j.n_mma / 2.0, 64.0);  // an M = 128 MMA occupies the pipe >= 64 cycles
      pipe = start + dur;
      pipe_busy += dur;
      w_empty[pc_mma] = pipe;
      if (j.flags & MF_LAST_K) {
        tm_full[q] = pipe;
        if (j.flags & MF_PAIR) tm_full[q + 1] = pipe;
      }
      if (j.flags & MF_RELEASE) act_free[p] = pipe;
      t_mma = issue;
      ++pc_mma;
      prog = true;
    }
    return prog;
  }

  // loader: issues the tile's input blocks in order, at most `depth` cp.async blocks in flight; a block is
  // published when the pipeline is full or — so that publication never waits on a slot — before the
  // loader blocks on a slot that is not free yet (the device drains its pending blocks the same way)
  std::vector<int> pend;  // production indices issued, not yet published
  void publish_front() {
    const int p = pend.front();
    t_ld = std::max(t_ld, issue_t[p] + kLoadLatency) + 40;
    act_ready[p] = t_ld;
    pend.erase(pend.begin());
  }
  bool adv_loader() {
    bool prog = false;
    while (nL && pc_ld < T * nL) {
      const HLoad& l = d.loads[pc_ld % nL];
      const int tile = pc_ld / nL;
      const int p = tile * nB + l.blk;
      if (l.kind != WK_LOAD_XYZ && (int)pend.size() == std::max(1, d.depth)) { publish_front(); prog = true; }
      const double f = slot_free(tile, l.pred, l.same, l.min_it);
      if (f < 0 || f > t_ld) {
        if (!pend.empty()) { while (!pend.empty()) publish_front(); prog = true; }
        if (f < 0) break;
      }
      if (l.kind == WK_LOAD_XYZ) {
        t_ld = std::max(t_ld, f) + kXyzCost + (l.c_count > 16 ? 12.0 * l.c_count : 0.0);  // + the xyz layer itself
        act_ready[p] = t_ld;
      } else {
        t_ld = std::max(t_ld, f) + 30 + 8.0 * l.c_count / 8;
        issue_t[p] = t_ld;
        pend.push_back(p);
      }
      ++pc_ld;
      prog = true;
    }
    if (pc_ld == T * nL && !pend.empty()) { while (!pend.empty()) publish_front(); prog = true; }
    return prog;
  }

  // epilogue group g handles, in order, the accumulators with q % 2 == g
  bool adv_epi() {
    bool prog = false;
    for (int g = 0; g < kEpiGroups; ++g) {
      while (pc_ep[g] < T * nE) {
        const int tile = pc_ep[g] / nE;
        const HEpi& e = d.epi[pc_ep[g] % nE];
        const int q = tile * nA + e.acc;
        if (e.coop) {  // both groups work on it: processed once, when both have arrived
          if (pc_ep[g ^ 1] != pc_ep[g]) break;
          if (g == 1) break;  // group 0 runs it for both
        } else if ((q & 1) != g) { ++pc_ep[g]; prog = true; continue; }
        if (tm_full[q] < 0) break;
        double t = std::max(t_ep[g], tm_full[q]);
        if (e.coop) t = std::max(t, t_ep[1]);
        int p = -1;
        if (e.kind == WK_EPI_HIDDEN) {
          p = tile * nB + e.blk;
          const double f = slot_free(tile, e.pred, e.same, e.min_it);
          if (f < 0) break;
          t = std::max(t, f);
        }
        t_ep[g] = t + epi_cost(e);
        tm_empty[q] = t_ep[g];
        if (p >= 0) act_ready[p] = t_ep[g];
        if (pc_ep[g] % nE == nE - 1) tile_end[tile] = t_ep[g];
        ++pc_ep[g];
        if (e.coop) { t_ep[1] = t_ep[0]; ++pc_ep[1]; }
        prog = true;
      }
    }
    return prog;
  }

  bool run() {
    for (;;) {
      bool prog = adv_prod();
      prog |= adv_mma();
      prog |= adv_loader();
      prog |= adv_epi();
      if (!prog) break;
    }
    return pc_mma == T * nC && pc_ep[0] == T * nE && pc_ep[1] == T * nE;
  }
};

struct Candidate {
  Draft d;
  double cycles = 0, mma_cycles = 0;
  bool ok = false;
};

void evaluate(Candidate& c) {
  c.ok = false;
  if ((int)c.d.loads.size() > kMaxLoadJobs) return;
  const int T = 6;
  Sim sim(c.d, T);
  if (!sim.run()) return;
  c.ok = true;
  c.cycles = (sim.tile_end[T - 1] - sim.tile_end[1]) / (T - 2);
  c.mma_cycles = sim.pipe_busy / T;
}

}  // namespace

int plan_chain(s4g_chain* ch, int n_layers, const int* cin, const int* cout, const int* relu, int in_mode, int feat_c,
               int out_mode, int out_c, int group, int sigmoid, int force_slots, int force_pairs, int force_coop, int subs, int tma_in) {
  const bool gathered = in_mode == IN_GATHER || in_mode == IN_GATHER_EDGE;
  S4G_CHECK_ARG(!tma_in || (in_mode == IN_ROWS && out_mode != OUT_MAXPOOL && cin[0] % 64 == 0) ||
                    (gathered && out_mode == OUT_MAXPOOL && n_layers > 1 && feat_c > 0 && feat_c % 64 == 0 &&
                     group % 4 == 0),
                "mlp_chain: TMA input needs row input with a multiple of 64 channels and no max-pool, or a gathered "
                "max-pool chain of >= 2 layers over a feature table of a multiple of 64 channels, group % 4 == 0");
  S4G_CHECK_ARG(subs == 1 || subs == 2, "mlp_chain: 1 or 2 row blocks per tile");
  struct CoopScope {  // force_coop: -1 = default policy, 0..2 = see coop_policy()
    explicit CoopScope(int v) { g_force_coop = v; }
    ~CoopScope() { g_force_coop = -1; }
  } coop_scope(force_coop);
  memset(ch, 0, sizeof(*ch));
  S4G_CHECK_ARG(n_layers >= 1 && n_layers <= kMaxLayers, "mlp_chain: 1..%d layers supported", kMaxLayers);
  S4G_CHECK_ARG(in_mode == IN_ROWS || gathered || in_mode == IN_XYZ_MLP, "mlp_chain: bad in_mode");
  S4G_CHECK_ARG(out_mode >= OUT_ROWS && out_mode <= OUT_LOGITS, "mlp_chain: bad out_mode");
  // the per-group term is added by the hidden epilogue: layer 0 must not be the transposed max-pool layer
  S4G_CHECK_ARG(in_mode != IN_GATHER_EDGE || (out_mode == OUT_MAXPOOL && n_layers > 1 && feat_c > 0),
                "mlp_chain: an edge chain is a gathered max-pool chain of >= 2 layers over a feature table");
  ch->n_layers = n_layers;
  ch->in_mode = in_mode;
  ch->out_mode = out_mode;
  const int L = n_layers;
  for (int l = 0; l < L; ++l) {
    S4G_CHECK_ARG(cin[l] > 0 && cout[l] > 0, "mlp_chain: bad layer width");
    if (l > 0) S4G_CHECK_ARG(cin[l] == cout[l - 1], "mlp_chain: layer %d input width != previous output width", l);
    ch->cin_pad[l] = round_up(cin[l], 16);
    ch->cout_pad[l] = round_up(cout[l], 16);
  }
  if (gathered) {
    S4G_CHECK_ARG(feat_c % 16 == 0 && cin[0] == feat_c + 3, "mlp_chain: gather input must be feat_c(%%16==0) + 3 xyz");
    ch->cin_pad[0] = feat_c + 16;
  } else if (in_mode == IN_XYZ_MLP) {
    S4G_CHECK_ARG(feat_c == 0 && cin[0] % 16 == 0 && cin[0] <= 128,
                  "mlp_chain: the CUDA-core xyz layer needs feat_c == 0 and an output width that is a multiple of 16, <= 128");
  } else {
    S4G_CHECK_ARG(cin[0] % 8 == 0, "mlp_chain: row input width must be a multiple of 8");
  }
  for (int l = 0; l + 1 < L; ++l)
    S4G_CHECK_ARG(ch->cout_pad[l] == cout[l] && cout[l] <= 512, "mlp_chain: hidden width must be a multiple of 16, <= 512");
  if (out_mode == OUT_MAXPOOL) {
    ch->cout_pad[L - 1] = round_up(cout[L - 1], 128);
    S4G_CHECK_ARG(group == 8 || group == 16 || group == 32 || group == 64,
                  "mlp_chain: max-pool group (neighbours per centroid) must be 8, 16, 32 or 64");
  } else if (out_mode == OUT_LOGITS) {
    S4G_CHECK_ARG(cout[L - 1] <= 16, "mlp_chain: logits layer supports <= 16 outputs");
    ch->cout_pad[L - 1] = 16;
  } else {
    S4G_CHECK_ARG(cout[L - 1] % 16 == 0, "mlp_chain: row output width must be a multiple of 16");
  }

  const int kSmemBudget = 227 * 1024 - 1024;  // barriers + TMEM slot live in the last KB
  Candidate best;
  // force_slots > 0 restricts the search to that many activation slots (the rest of shared memory goes to weight
  // stages): the simulation ranks slot counts imperfectly — the set-abstraction level 2 chain runs 23 % faster with 5
  // slots than with the 3 it prefers — so the host can time the alternatives and pin the best (engine.py autotune)
  for (int S = kMaxSlots; S >= 1; --S) {
    if (force_slots > 0 && S != force_slots) continue;
    int stages = (kSmemBudget - S * kSlotBytes) / kStageBytes;
    if (stages < 2) continue;
    stages = std::min(stages, kMaxStages);
    for (int pair_ok = 1; pair_ok >= 0; --pair_ok) {
      if (force_pairs >= 0 && pair_ok != force_pairs) continue;  // -1 = both, 0 = N <= 128 only, 1 = N = 256 pairs
      for (int depth = 3; depth >= 1; --depth) {
        Candidate c;
        if (!build_draft(ch, relu, feat_c, S, pair_ok != 0, subs, tma_in != 0, c.d)) continue;
        if (pair_ok && (c.d.n_acc & 1)) continue;  // pairs need tile-invariant accumulator parity
        c.d.stages = stages;
        c.d.depth = depth;
        evaluate(c);
        if (c.ok && (!best.ok || c.cycles < best.cycles * 0.995)) best = c;
      }
    }
  }
  S4G_CHECK_ARG(best.ok, "mlp_chain: no deadlock-free plan fits on chip for this chain shape");

  ChainParams& p = ch->prm;
  const Draft& d = best.d;
  const int S = d.S;
  p.n_mma = (int)d.mma.size();
  size_t wb = 0;
  for (int j = 0; j < p.n_mma; ++j) {
    const HMma& m = d.mma[j];
    p.mma[j] = {(uint8_t)(m.blk % S), (uint8_t)(m.blk / S), (uint8_t)m.acc, (uint8_t)m.k16, (uint8_t)m.koff,
                (uint8_t)(m.n_rows / 8), (uint8_t)m.flags, (uint8_t)m.blk};
    ch->chunk[j] = {m.layer, m.n_begin, m.n_rows, m.k_begin, m.k16 * 16};
    wb += (size_t)m.n_rows * m.k16 * 32;
  }
  p.n_ld = (int)d.loads.size();
  for (int j = 0; j < p.n_ld; ++j) {
    const HLoad& l = d.loads[j];
    p.ld[j] = {(uint8_t)l.kind, (uint8_t)l.same, (uint8_t)(l.blk % S), (uint8_t)(l.blk / S), 0, 0, 0, (uint8_t)l.pred,
               (uint16_t)l.c_begin, (uint16_t)l.c_count, (uint8_t)l.min_it, 0, (uint8_t)l.sub, {0}};
  }
  p.load_depth = std::max(1, d.depth);
  p.n_ep = (int)d.epi.size();
  for (int j = 0; j < p.n_ep; ++j) {
    const HEpi& e = d.epi[j];
    const int blk = e.blk < 0 ? 0 : e.blk;
    p.ep[j] = {(uint8_t)e.kind, (uint8_t)e.same, (uint8_t)(blk % S), (uint8_t)(blk / S), (uint8_t)e.acc, (uint8_t)e.layer,
               (uint8_t)e.relu, (uint8_t)e.pred, (uint16_t)e.c_begin, (uint16_t)e.c_count, (uint8_t)e.min_it,
               (uint8_t)e.coop, (uint8_t)e.sub, {0}};
  }
  const int nB = (int)d.blocks.size();
  p.n_act_mod = nB % S;
  p.n_act_div = nB / S;
  p.n_acc = d.n_acc;
  p.slots = S;
  p.stages = d.stages;
  p.in_mode = in_mode;
  p.subs = subs;
  p.tma_in = tma_in ? 1 : 0;
  p.feat_c = feat_c;
  p.out_c = out_c;
  p.group = group > 0 ? group : 1;
  p.sigmoid = sigmoid;
  p.term_c = in_mode == IN_GATHER_EDGE ? cout[0] : 0;
  ch->w_bytes = wb;
  ch->smem_bytes = (size_t)S * kSlotBytes + (size_t)d.stages * kStageBytes + 1024;
  ch->sim_cycles_per_tile = best.cycles;
  ch->mma_cycles_per_tile = best.mma_cycles;
  ch->load_depth = d.depth;
  return S4G_OK;
}

}  // namespace s4g

// Human-readable dump of a plan (debugging / tests): returns the number of bytes written.
extern "C" int s4g_chain_describe(const s4g_chain* ch, char* buf, int cap) {
  if (!ch || !buf || cap <= 0) return 0;
  static const char* kinds[] = {"LOAD_ROWS", "LOAD_FEAT", "LOAD_DONE", "LOAD_XYZ", "?", "EPI_HIDDEN", "EPI_ROWS",
                                "EPI_MAXPOOL", "EPI_LOGITS"};
  const s4g::ChainParams& p = ch->prm;
  std::string s;
  char line[256];
  snprintf(line, sizeof line,
           "slots=%d stages=%d smem=%zu n_mma=%d n_ld=%d n_ep=%d n_act=%d n_acc=%d w_bytes=%zu depth=%d sim=%.0f cyc/tile mma=%.0f\n",
           p.slots, p.stages, ch->smem_bytes, p.n_mma, p.n_ld, p.n_ep, p.n_act_div * p.slots + p.n_act_mod, p.n_acc,
           ch->w_bytes, ch->load_depth, ch->sim_cycles_per_tile, ch->mma_cycles_per_tile);
  s += line;
  for (int j = 0; j < p.n_mma; ++j) {
    const s4g::MmaJob& m = p.mma[j];
    snprintf(line, sizeof line, "  mma %3d: blk=%d acc=%d k16=%d koff=%d n=%d flags=%s%s%s%s%s%s  L%d n0=%d k0=%d\n", j,
             m.blk_div * p.slots + m.blk_mod, m.acc, m.k16, m.koff, m.n8 * 8, (m.flags & s4g::MF_WAIT_ACT) ? "W" : "-",
             (m.flags & s4g::MF_FIRST_K) ? "F" : "-", (m.flags & s4g::MF_LAST_K) ? "L" : "-",
             (m.flags & s4g::MF_RELEASE) ? "R" : "-", (m.flags & s4g::MF_TRANSPOSED) ? "T" : "-",
             (m.flags & s4g::MF_PAIR) ? "P" : "-", ch->chunk[j].layer, ch->chunk[j].n_begin, ch->chunk[j].k_begin);

    s += line;
  }
  for (int j = 0; j < p.n_ld; ++j) {
    const s4g::WorkerJob& w = p.ld[j];
    snprintf(line, sizeof line, "  ld %3d: %-11s blk=%d c=[%d,+%d) after blk %d of %s tile (from it %d)\n", j, kinds[w.kind],
             w.blk_div * p.slots + w.blk_mod, w.c_begin, w.c_count, w.pred, w.same ? "this" : "the previous", w.min_it);
    s += line;
  }
  for (int j = 0; j < p.n_ep; ++j) {
    const s4g::WorkerJob& w = p.ep[j];
    snprintf(line, sizeof line, "  ep %3d: %-11s blk=%d acc=%d L%d c=[%d,+%d)\n", j, kinds[w.kind],
             w.blk_div * p.slots + w.blk_mod, w.acc, w.layer, w.c_begin, w.c_count);
    s += line;
  }
  const int n = (int)std::min<size_t>(s.size(), (size_t)cap - 1);
  memcpy(buf, s.data(), n);
  buf[n] = 0;
  return n;
}
