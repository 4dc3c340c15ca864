// Job streams of the fused tcgen05 MLP-chain kernel (csrc/mlp_chain.cu), shared by the host planner
// (csrc/chain_plan.cu) and the device interpreter.
//
// One CTA walks 128-row tiles through a whole shared-MLP chain.  Four roles run STATIC per-tile job
// streams, coupled only through mbarriers:
//   * two TMA producer warps stream one bf16 weight chunk (<= 32 KB) per MMA job into a shared-memory ring;
//   * the MMA warp issues, per job, up to 8 tcgen05.mma (M = 128, N <= 256, K = 16) that multiply (part
//     of) one activation K-block (a 32 KB shared-memory "slot") by that weight chunk into one 128-column
//     TMEM accumulator block, or into two adjacent ones (N = 256: twice the tensor work per instruction —
//     the issuing thread, not the tensor pipe, is the scarce resource; see profiles/issue_cost.cu);
//   * 2 loader warps (each thread owns two tile rows) stage the layer-0 input K-blocks: cp.async of contiguous
//     rows or of gathered neighbour rows, and the relative-xyz block of a set-abstraction layer.  They run
//     ahead of the MMA warp by as many blocks as the slot ring allows, i.e. they prefetch the next tile;
//   * 16 epilogue warps in two groups of 8 (two per TMEM lane quadrant, 64 columns each); group g drains the
//     accumulators with q % 2 == g, so the two blocks of an N = 256 pair are drained concurrently: + shift, ReLU, bf16 ->
//     the next layer's K-block slot, or the chain's output (rows / max-pooled groups / logits).  Jobs marked `coop`
//     are drained by all 16 warps (four per lane quadrant, 32 columns each): the block is ready in half the time,
//     which is what the next layer's first MMA waits for.
// Activation blocks and accumulators live in RINGS indexed by their production order, so the streams are
// identical for every tile and every wait is "the n-th completion of barrier b":
//   activation block p (p-th produced, across tiles)  -> slot p % S, use p / S
//   accumulator q                                      -> TMEM columns 128 * (q % 4), use q / 4
//   weight chunk c                                     -> ring stage c % stages, use c / stages
// mbarrier waits only carry one bit of phase, so a waiter must never be two completions away from the
// barrier.  Producer/consumer pairs that alternate strictly satisfy this (weight ring, TMEM ring, and the
// MMA warp, which reads every block in order).  Slot RE-USE does not — the loader may run a tile ahead of
// the epilogue groups that produced the slot's previous block — so the release of a block is signalled
// on a barrier of its own, blk_free[b] for tile-relative block b: it completes exactly once per tile, and
// the producer of the block that inherits the slot waits for the completion of its own tile (previous
// block in the same tile) or of the tile before (which implies every older one).
// A block's slot is fixed by its index, so no role can take a resource another one needs: deadlock
// freedom depends only on the dependency graph, which the planner checks by simulating the streams
// (a Kahn network: if one schedule completes, every schedule does).
#pragma once
#include <cuda.h>
#include <stdint.h>

namespace s4g {

constexpr int kTileRows = 128;
constexpr int kEpiWarps = 16;                     // warps 0..15
constexpr int kEpiGroups = 2;                     // group g = warps 8g..8g+7 drains accumulators q % 2 == g
constexpr int kEpiGroupWarps = kEpiWarps / kEpiGroups;
constexpr int kLoadWarps = 2;                     // warps 16, 17: each thread stages rows r and r + 64
constexpr int kLoadWarp0 = kEpiWarps;
constexpr int kMmaWarp = kEpiWarps + kLoadWarps;  // warp 18
constexpr int kProducerWarp = kMmaWarp + 1;       // warps 19, 20 (even / odd chunks): one thread can only issue
constexpr int kProducers = 1;                     // a bulk copy every ~530 cycles, whatever its size
constexpr int kChainThreads = 32 * (kEpiWarps + kLoadWarps + 1 + kProducers);
constexpr int kSlotBytes = 32768;   // one activation K-block: 128 rows x 128 channels bf16, [16 pieces][128 rows][16 B]
constexpr int kStageBytes = 32768;  // one weight chunk: 128 rows x 128 channels or 256 rows x 64 channels bf16
constexpr int kAccBlocks = 4;       // TMEM: 4 accumulator blocks of 128 fp32 columns
constexpr int kMaxSlots = 6;
constexpr int kMaxStages = 6;
constexpr int kMaxMmaJobs = 128;
constexpr int kMaxLoadJobs = 64;
constexpr int kMaxEpiJobs = 32;
constexpr int kMaxLayers = 6;
constexpr int kMaxBlocks = 32;  // activation blocks per tile

// IN_XYZ_MLP: gathered input without features whose 3 -> cin[0] first layer (K = 3: 81 % of a K = 16 MMA step
// would be padding, and its epilogue a whole MMA -> epilogue -> MMA round trip) is computed by the loader warps
// on the CUDA cores in fp32, straight into the activation block the chain's layer 0 reads
// IN_GATHER_EDGE: IN_GATHER whose layer-0 epilogue also adds a per-group bf16 term term[row / K][col] to the shift, in
// fp32, before the ReLU and the rounding — the centroid part -W_b f_c of an edge level (EdgeQueryGrouper's rows
// [x_j - x_c | f_j | f_j - f_c] multiply as [W_x | W_a + W_b] [x_j - x_c ; f_j] - W_b f_c).  Planned exactly like
// IN_GATHER; a mode of its own so that its kernels and tuned plans never mix with the plain chains'.
enum InMode { IN_ROWS = 0, IN_GATHER = 1, IN_XYZ_MLP = 5, IN_GATHER_EDGE = 6 };
enum OutMode { OUT_ROWS = 2, OUT_MAXPOOL = 3, OUT_LOGITS = 4 };

// MF_PAIR: the job's MMAs are N = 256 wide and fill accumulators acc and acc + 1 (adjacent TMEM blocks)
// MF_SWZ: the activation block read is a TMA-loaded INPUT block in the 128-byte-swizzled K-major layout (two 16 KB halves
// of 64 channels, rows 128 B apart) instead of the interleaved layout the epilogue writes
enum MmaFlags { MF_WAIT_ACT = 1, MF_FIRST_K = 2, MF_LAST_K = 4, MF_RELEASE = 8, MF_TRANSPOSED = 16, MF_PAIR = 32, MF_SWZ = 64 };

struct MmaJob {      // one weight chunk x one activation K-block (part) -> one accumulator block (or pair)
  uint8_t blk_mod;   // activation block read: tile-relative production index i, as i % S ...
  uint8_t blk_div;   //                                                        ... and i / S
  uint8_t acc;       // tile-relative accumulator index
  uint8_t k16;       // K = 16 steps in this chunk (1..8; 1..4 for a pair)
  uint8_t koff;      // first K = 16 step inside the activation block
  uint8_t n8;        // weight-chunk rows / 8  (= MMA N / 8 <= 32, or 16 = the 128 output channels when transposed)
  uint8_t flags;     // MmaFlags
  uint8_t blk;       // tile-relative index of the activation block read (MF_RELEASE commits blk_free[blk])
};

enum WorkerKind {
  WK_LOAD_ROWS = 0,   // loader: cp.async a K-block of contiguous input rows (published once landed)
  WK_LOAD_FEAT = 1,   // loader: cp.async a K-block of gathered neighbour feature rows
  WK_LOAD_XYZ = 3,    // loader: build and publish the 16-channel relative-xyz block (synchronous); IN_XYZ_MLP: the
                      //         c_count-channel output of the xyz layer, ReLU(W (x - c) + shift), instead
  WK_EPI_HIDDEN = 5,  // epilogue: accumulator -> +shift, ReLU, bf16 -> activation block
  WK_EPI_ROWS = 6,    // epilogue: accumulator -> bf16 rows in global memory
  WK_EPI_MAXPOOL = 7, // epilogue: transposed accumulator -> max over each group of columns -> bf16 [group][channel]
  WK_EPI_LOGITS = 8   // epilogue: 16-column accumulator -> fp32 channel-first logits (+bias, optional sigmoid)
};

struct WorkerJob {
  uint8_t kind;
  uint8_t same;      // producers: 1 = the slot's previous block `pred` belongs to the same tile
  uint8_t blk_mod;   // activation block produced (loads, EPI_HIDDEN), relative to the job's tile
  uint8_t blk_div;
  uint8_t acc;       // accumulator consumed (epilogues)
  uint8_t layer;     // epilogues: layer whose shift vector applies
  uint8_t relu;
  uint8_t pred;      // producers: tile-relative index of the block that last held this block's slot
  uint16_t c_begin;  // loads: first input channel; epilogues: first output channel of the block
  uint16_t c_count;  // channels / columns in the block (multiple of 8 for loads, of 16 for epilogues)
  uint8_t min_it;    // producers, same == 0: first tile iteration of the CTA at which a previous block exists
  uint8_t coop;      // EPI_HIDDEN / EPI_ROWS: 1 = all 16 epilogue warps drain this accumulator (32 columns each)
  uint8_t sub;       // row block (sub-tile of 128 rows) of the tile this job works on: 0, or 1 when the tile has two
  uint8_t pad[1];
};

struct ChainParams {
  MmaJob mma[kMaxMmaJobs];
  WorkerJob ld[kMaxLoadJobs];
  WorkerJob ep[kMaxEpiJobs];
  int n_mma, n_ld, n_ep;
  int n_act_mod, n_act_div;  // activation blocks produced per tile, as n % S and n / S
  int n_acc;                 // accumulators per tile
  int slots, stages;
  int load_depth;            // cp.async input blocks a loader thread keeps in flight (1..3)
  int subs;                  // row blocks per tile (1 or 2): a tile is 128 * subs rows
  int tma_in;                // IN_ROWS: input blocks arrive by TMA tensor copies (in_map) in the swizzled layout
  alignas(64) CUtensorMap in_map;  // 2-D map of the input rows [P][in_stride] bf16, box 64 channels x 128 rows, 128 B swizzle
  const void* weights;       // packed chunk stream of one tile, in MMA-job order
  const float* bias[kMaxLayers];
  int P;                     // rows (positions)
  // input
  int in_mode;
  const void* in_rows;       // IN_ROWS: bf16 [P][in_stride]
  int in_stride;
  const void* feat;          // IN_GATHER: bf16 [B*N][feat_c] (null when feat_c == 0)
  int feat_c;
  float xyz_w[128 * 4];      // IN_XYZ_MLP: [cin[0]][4] fp32 = (w_x, w_y, w_z, shift) of the xyz layer (BN folded);
  int xyz_relu;              //   in kernel-parameter space: every lane reads the same entry (constant-bank broadcast)
  int xyz_set;
  const float* xyz;          // (B,3,N)
  const float* ctr;          // (B,3,M)
  const int* nbr;            // (B,M,K)
  int N, M, K;
  // output
  void* out;
  int out_c;                 // real output channels
  int group;                 // MAXPOOL: rows per group
  int n_points;              // LOGITS: points per batch element
  int sigmoid;
  long long* prof;           // optional: 16 cycle counters per CTA (see s4g_chain_set_profile); null = off
  // IN_GATHER_EDGE: bf16 [P / K][term_c] per-group term of layer 0 (term_c = layer 0's output width)
  const void* term;
  int term_c;
};

}  // namespace s4g

// host-side description of a planned chain
struct s4g_chain {
  s4g::ChainParams prm;
  int n_layers;
  int cin_pad[s4g::kMaxLayers], cout_pad[s4g::kMaxLayers];
  int in_mode, out_mode;
  size_t smem_bytes;
  size_t w_bytes;
  // per MMA job: which slice of which layer's weight matrix its chunk holds
  struct ChunkSrc { int layer, n_begin, n_rows, k_begin, k_count; } chunk[s4g::kMaxMmaJobs];
  double sim_cycles_per_tile;  // planner's estimate (SM cycles)
  double mma_cycles_per_tile;  // tensor-pipe busy cycles per tile
  int load_depth;              // cp.async blocks in flight per loader thread
};

namespace s4g {
// Plans the chain: fills ch->prm job streams, ring sizes, chunk sources.  Returns S4G_OK or sets the error.
int plan_chain(s4g_chain* ch, int n_layers, const int* cin, const int* cout, const int* relu, int in_mode, int feat_c,
               int out_mode, int out_c, int group, int sigmoid, int force_slots = 0, int force_pairs = -1,
               int force_coop = -1, int subs = 1, int tma_in = 0);
}  // namespace s4g
