// Generic batched kernels, templated on a per-game rule core ("Rules").  One lane = one State.
// All kernels are HBM-streaming: one coalesced load of the packed state per lane, a handful of
// integer ops, coalesced stores.  Grid = ceil(n / block); blocks of 256 threads.
#pragma once
#include <new>

#include "common.cuh"

namespace b2s {

constexpr int kBlock = 256;

extern long long g_launches;   // api.cu

// Programmatic dependent launch (sm_90+): a kernel launched with the programmatic-stream-serialization
// attribute may start while its predecessor drains; pdl_wait() blocks until the predecessor has fully
// completed and flushed (so data dependencies between consecutive steps stay intact), pdl_launch_dependents()
// lets the successor's CTAs be scheduled as soon as this grid has issued its loads.  Both are no-ops when the
// kernel was launched normally.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline void launch_pdl(void (*kernel)(KArgs...), unsigned grid, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kBlock);
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- kernels -------------------------------------------------------------------------------------

template <class R>
__global__ void __launch_bounds__(kBlock) k_reset(Ctx ctx, typename R::Cfg cfg, long long n) {
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i == 0) { ctx.err->count = 0; ctx.err->first = 0x7fffffffffffffffLL; }
  if (i >= n) return;
  typename R::S s;
  R::init(s, cfg, ctx, i);
  R::store(s, ctx, i);
}

// State::ApplyAction over the batch (spiel.cc:441-451).  Each thread owns ILP lanes, block-strided so every
// access stays coalesced; all loads (action + packed state) are issued before any compute so that a thread
// has ILP independent 128-bit requests in flight (the kernel is a pure HBM stream).
template <class R, int ILP>
__global__ void __launch_bounds__(kBlock, R::kMinBlocks) k_apply(Ctx ctx, typename R::Cfg cfg, const int* __restrict__ actions, long long n) {
  pdl_wait();
  long long base = (long long)blockIdx.x * (kBlock * ILP) + threadIdx.x;
  int a[ILP];
  typename R::S s[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    a[j] = -1;
    if (i < n) { a[j] = __ldg(actions + i); R::load(s[j], ctx, i); }
  }
  pdl_launch_dependents();
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    if (a[j] == -1) continue;
    if (R::terminal(s[j], cfg) || !R::apply(s[j], a[j], cfg, ctx, i)) { flag_error(ctx.err, ctx.lane0 + i); continue; }
    R::store(s[j], ctx, i);
  }
}

// Coalesced store of multi-word legal masks.  A warp owns 32 consecutive lanes, whose mask words are one contiguous range of
// the output, but written lane by lane (mask[i * W + w] in a loop over w) every store instruction scatters over 32 sectors —
// for breakthrough (W = 24) that, not the mask arithmetic, was the kernel's limit (ncu, profiles/r02_item9: 2 % of DRAM
// bandwidth, 15 % SM busy, 40 us for 262k lanes).  The warp stages its 32 x W words in shared memory (row stride odd: no
// bank conflicts) and writes the range with fully coalesced 128-byte stores.  Every lane of the warp must call (active =
// false for lanes past n); W <= MAXW.  `first` = lane index of the warp's lane 0, `n` = lanes in the batch.
template <int MAXW>
struct MaskStage {
  static constexpr int kRow = MAXW | 1;
  u32 w[kBlock / 32][32 * kRow];
};
template <int MAXW>
__device__ __forceinline__ void store_masks_coalesced(u32* __restrict__ mask, long long first, long long n, bool active, int W,
                                                      const u32* m, MaskStage<MAXW>& stage) {
  const int lane = threadIdx.x & 31;
  u32* st = stage.w[threadIdx.x >> 5];
  if (active) {
#pragma unroll
    for (int k = 0; k < MAXW; ++k) if (k < W) st[lane * MaskStage<MAXW>::kRow + k] = m[k];
  }
  __syncwarp();
  const long long left = n - first;
  const int total = (int)(left < 32 ? left : 32) * W;       // words this warp owns
  int q = lane / W, r = lane - q * W;                        // flat word index f = q * W + r, advanced by 32 per iteration
  const int dq = 32 / W, dr = 32 - dq * W;
  u32* out = mask + first * W;
  for (int f = lane; f < total; f += 32) {
    out[f] = st[q * MaskStage<MAXW>::kRow + r];
    q += dq; r += dr;
    if (r >= W) { r -= W; ++q; }
  }
  __syncwarp();
}

template <class R, int ILP>
__global__ void __launch_bounds__(kBlock) k_legal_mask(Ctx ctx, typename R::Cfg cfg, u32* __restrict__ mask, int mask_words, long long n) {
  long long base = (long long)blockIdx.x * (kBlock * ILP) + threadIdx.x;
  typename R::S s[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    if (i < n) R::load(s[j], ctx, i);
  }
  __shared__ MaskStage<R::kMaskWords == 1 ? 0 : R::kMaskWords> stage;
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    u32 m[R::kMaskWords];
    if (i < n) R::legal(s[j], cfg, m);
    if (R::kMaskWords == 1) {
      if (i < n) mask[i] = m[0];
    } else {
      store_masks_coalesced(mask, i - (threadIdx.x & 31), n, i < n, mask_words, m, stage);
    }
  }
}

template <class R>
__global__ void __launch_bounds__(kBlock) k_legal_list(Ctx ctx, typename R::Cfg cfg, short* __restrict__ out, int* __restrict__ counts, int stride, int mask_words, long long n) {
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  typename R::S s;
  R::load(s, ctx, i);
  u32 m[R::kMaskWords];
  R::legal(s, cfg, m);
  int k = 0;
  for (int w = 0; w < mask_words; ++w) {
    u32 bits = m[w];
    while (bits) {
      int b = __ffs(bits) - 1;
      bits &= bits - 1;
      if (k < stride) out[i * stride + k] = (short)(w * 32 + b);
      ++k;
    }
  }
  counts[i] = k;
}

// Returns row i of a [n][num_players] float buffer.  Two players: one 8-byte store per lane when the buffer allows it; the
// C ABI promises only float (4-byte) alignment, so a buffer at an odd float offset takes two 4-byte stores (the test is on
// the base pointer, hence uniform over the launch).
template <class R>
__device__ __forceinline__ void store_returns(float* __restrict__ rets, long long i, const float* r, const typename R::Cfg& cfg) {
  if (R::kPlayers == 2) {
    if (((unsigned long long)rets & 7ull) == 0) reinterpret_cast<float2*>(rets)[i] = make_float2(r[0], r[1]);
    else { rets[2 * i] = r[0]; rets[2 * i + 1] = r[1]; }
  } else {
    const int np = rule_num_players<R>(cfg);
    for (int p = 0; p < np; ++p) rets[i * np + p] = r[p];
  }
}

template <class R, int ILP>
__global__ void __launch_bounds__(kBlock) k_status(Ctx ctx, typename R::Cfg cfg, signed char* __restrict__ cur, unsigned char* __restrict__ term, float* __restrict__ rets, long long n) {
  long long base = (long long)blockIdx.x * (kBlock * ILP) + threadIdx.x;
  typename R::S s[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    if (i < n) R::load(s[j], ctx, i);
  }
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    if (i >= n) continue;
    int cp = R::cur_player(s[j], cfg);
    if (cur) cur[i] = (signed char)cp;
    if (term) term[i] = cp == kTerminalPlayerId ? 1 : 0;
    if (rets) {
      float r[R::kPlayers];
      R::returns(s[j], cfg, r);
      store_returns<R>(rets, i, r, cfg);
    }
  }
}

// ApplyAction + IsTerminal + Returns + next LegalActionsMask in one pass.
template <class R, int ILP>
__global__ void __launch_bounds__(kBlock) k_step_fused(Ctx ctx, typename R::Cfg cfg, const int* __restrict__ actions, u32* __restrict__ mask, int mask_words, unsigned char* __restrict__ term, float* __restrict__ rets, long long n) {
  pdl_wait();
  long long base = (long long)blockIdx.x * (kBlock * ILP) + threadIdx.x;
  int a[ILP];
  typename R::S s[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    a[j] = -1;
    if (i < n) { a[j] = __ldg(actions + i); R::load(s[j], ctx, i); }
  }
  pdl_launch_dependents();
  __shared__ MaskStage<R::kMaskWords == 1 ? 0 : R::kMaskWords> stage;
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    const bool live = i < n;
    u32 m[R::kMaskWords];
    if (live) {
      if (a[j] != -1) {
        if (R::terminal(s[j], cfg) || !R::apply(s[j], a[j], cfg, ctx, i)) flag_error(ctx.err, ctx.lane0 + i);
        else R::store(s[j], ctx, i);
      }
      bool t = R::terminal(s[j], cfg);
      if (term) term[i] = t ? 1 : 0;
      if (rets) {
        float r[R::kPlayers];
        R::returns(s[j], cfg, r);
        store_returns<R>(rets, i, r, cfg);
      }
      if (mask) {
        if (t) { for (int w = 0; w < R::kMaskWords; ++w) m[w] = 0; }
        else R::legal_nonterminal(s[j], cfg, m);
      }
    }
    if (mask) {                                            // uniform over the grid
      if (R::kMaskWords == 1) { if (live) mask[i] = m[0]; }
      else store_masks_coalesced(mask, i - (threadIdx.x & 31), n, live, mask_words, m, stage);
    }
  }
}

// Compact env step for host-driven loops (b2s_step_fused_host_compact): the same apply -> terminal -> returns -> next legal
// mask pass as k_step_fused with byte-wide I/O, because through PCIe the bytes per lane ARE the cost.  Actions are AT
// (unsigned char: 0xFF = leave the lane untouched; int: -1).  One status byte per lane:
//   bit 7      IsTerminal
//   terminal:  bits 0-1 = outcome (0 draw / no winner, 1 player 0 won, 2 player 1 won) — win/loss/draw games only
//   otherwise: bits 0-6 = LegalActionsMask when the game has <= 7 distinct actions (connect_four <= 7 columns), else 0
// Games with more actions get their mask words through `mask` (nullable), exactly as k_step_fused writes them.
template <class R, int ILP, class AT>
__global__ void __launch_bounds__(kBlock) k_step_compact(Ctx ctx, typename R::Cfg cfg, const AT* __restrict__ actions, unsigned char* __restrict__ status,
                                                         u32* __restrict__ mask, int mask_words, int small_mask, long long n) {
  pdl_wait();
  long long base = (long long)blockIdx.x * (kBlock * ILP) + threadIdx.x;
  int a[ILP];
  typename R::S s[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    a[j] = -1;
    if (i < n) {
      AT raw = __ldg(actions + i);
      a[j] = (sizeof(AT) == 1 && (unsigned char)raw == 0xFFu) ? -1 : (int)raw;
      R::load(s[j], ctx, i);
    }
  }
  pdl_launch_dependents();
  __shared__ MaskStage<R::kMaskWords == 1 ? 0 : R::kMaskWords> stage;
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    const bool live = i < n;
    u32 m[R::kMaskWords];
    if (live) {
      if (a[j] != -1) {
        if (R::terminal(s[j], cfg) || !R::apply(s[j], a[j], cfg, ctx, i)) flag_error(ctx.err, ctx.lane0 + i);
        else R::store(s[j], ctx, i);
      }
      bool t = R::terminal(s[j], cfg);
      unsigned st = 0;
      if (t) {
        float r[R::kPlayers];
        R::returns(s[j], cfg, r);
        st = 0x80u | (r[0] > 0.f ? 1u : (r[0] < 0.f ? 2u : 0u));
        for (int w = 0; w < R::kMaskWords; ++w) m[w] = 0;
      } else if (small_mask || mask) {
        R::legal_nonterminal(s[j], cfg, m);
        if (small_mask) st = m[0] & 0x7Fu;
      }
      status[i] = (unsigned char)st;
    }
    if (mask) {                                            // uniform over the grid
      if (R::kMaskWords == 1) { if (live) mask[i] = m[0]; }
      else store_masks_coalesced(mask, i - (threadIdx.x & 31), n, live, mask_words, m, stage);
    }
  }
}

// R::kObsBitPacked (optional): ObsPack is the tensor as a flat little-endian bit string in output order
template <class R> constexpr auto obs_bitpacked(int) -> decltype(R::kObsBitPacked) { return R::kObsBitPacked; }
template <class R> constexpr bool obs_bitpacked(long) { return false; }

// ObservationTensor / InformationStateTensor.  A warp owns 32 consecutive lanes: every thread packs
// its own state's tensor into shared memory (game-specific compact form), then the warp streams the
// 32*size floats of its tile out as fully coalesced 16-byte stores.
template <class R>
__global__ void __launch_bounds__(kBlock) k_obs(Ctx ctx, typename R::Cfg cfg, int player, int which, int zero_terminal, float* __restrict__ out, int size, u32 magic, long long n) {
  __shared__ typename R::ObsPack packs[kBlock];
  __shared__ unsigned char dead_flags[kBlock];      // zero_terminal: lanes whose tensor is all-zero padding
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (i < n) {
    typename R::S s;
    R::load(s, ctx, i);
    if (zero_terminal) dead_flags[threadIdx.x] = R::terminal(s, cfg) ? 1 : 0;
    int pl = player;
    if (pl < 0) { pl = R::cur_player(s, cfg); if (pl < 0) pl = 0; }
    R::obs_pack(s, cfg, pl, which, packs[threadIdx.x]);
  }
  __syncwarp();
  long long tile0 = ((long long)blockIdx.x * kBlock + warp * 32);   // first lane of this warp's tile
  if (tile0 >= n) return;
  int lanes_here = (int)((n - tile0) < 32 ? (n - tile0) : 32);
  int total = lanes_here * size;                                       // floats in this tile
  float* base = out + tile0 * size;
  // The tile is emitted as 16-byte stores, so the vector part must start on a 16-byte boundary.  tile0 * size * 4 is a
  // multiple of 16 (tile0 is a multiple of 32), but `out` itself need not be (a caller pointer, or row t of the
  // trajectory recorder at offset t*n*F floats): the first `peel` floats of the tile are written as scalars.
  const int peel = (int)(((16u - (unsigned)((unsigned long long)base & 15ull)) & 15u) >> 2);
  const typename R::ObsPack* wp = packs + warp * 32;
  const unsigned char* dead = dead_flags + warp * 32;
  const int head = peel < total ? peel : total;
  if (lane < head) {
    int st = (int)(((u64)lane * magic) >> 32);
    base[lane] = (zero_terminal && dead[st]) ? 0.f : R::obs_elem(wp[st], cfg, lane - st * size);
  }
  int nvec = (total - head) >> 2;
  float4* vbase = reinterpret_cast<float4*>(base + head);
  for (int q = lane; q < nvec; q += 32) {
    int e0 = head + (q << 2);
    int st = (int)(((u64)e0 * magic) >> 32);         // e0 / size (magic verified on the host for the range)
    int within = e0 - st * size;
    float v[4];
    if (obs_bitpacked<R>(0) && within + 4 <= size) {
      // 0/1 tensors kept as a flat bit string in output order: one funnel shift yields the four bits of this float4
      const u32* b = reinterpret_cast<const u32*>(&wp[st]);
      int wi = within >> 5, sh = within & 31;
      u32 lo = b[wi], hi = sh > 28 ? b[wi + 1] : 0u;    // (within+3)>>5 == wi+1 exactly when sh > 28: in range
      u32 nib = __funnelshift_r(lo, hi, sh);
      if (zero_terminal && dead[st]) nib = 0;
      v[0] = (float)(nib & 1u); v[1] = (float)((nib >> 1) & 1u); v[2] = (float)((nib >> 2) & 1u); v[3] = (float)((nib >> 3) & 1u);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[j] = (zero_terminal && dead[st]) ? 0.f : R::obs_elem(wp[st], cfg, within);
        if (++within == size) { within = 0; ++st; }     // a float4 may straddle two lanes' tensors
      }
    }
    vbase[q] = make_float4(v[0], v[1], v[2], v[3]);
  }
  for (int e = head + (nvec << 2) + lane; e < total; e += 32) {        // ragged tail of the last tile
    int st = (int)(((u64)e * magic) >> 32);
    base[e] = (zero_terminal && dead[st]) ? 0.f : R::obs_elem(wp[st], cfg, e - st * size);
  }
}

// Random playout to terminal (mcts.cc:43-72 inner loop; benchmark_game.cc:32-115).
template <class R>
__global__ void __launch_bounds__(kBlock) k_rollout(Ctx ctx, typename R::Cfg cfg, u64 seed, long long lane_offset, int mask_words, int max_plies, float* __restrict__ rets, int* __restrict__ plies, long long n) {
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  typename R::S s;
  R::load(s, ctx, i);
  int ply = 0;
  while (!R::terminal(s, cfg) && ply < max_plies) {
    auto draw = [&](u32 b, u32 n) { return philox_uniform(seed, (u64)(i + lane_offset), b, n); };
    playout_step<R>(s, cfg, ctx, i, mask_words, draw, (u32)ply);
    ++ply;
  }
  R::store(s, ctx, i);
  if (plies) plies[i] = ply;
  if (rets) {
    float r[R::kPlayers];
    R::returns(s, cfg, r);
    const int np = rule_num_players<R>(cfg);
    for (int p = 0; p < np; ++p) rets[i * np + p] = r[p];
  }
}

// ---- self-play trajectory recorder (algorithms/trajectories.cc RecordTrajectory :140-200) -------------------
// The reference plays one episode at a time and pads afterwards; here every lane advances by one *decision* per
// launch, so step t of all episodes is written as one coalesced [n]-row of the time-major outputs.  Chance nodes
// are sampled and applied but not recorded (trajectories.cc:152-157).  Random numbers, lane g = lane_offset + i:
//   decision of step t      k = philox_uniform(seed, g, 64 (t+1),         #legal)  -> k-th legal action (ascending)
//   j-th chance node after   k = philox_uniform(seed, g, 64 (t+1) + 1 + j, #outcomes)   (before step 0: 64*0 + 1 + j)
// (uniform policy = GetUniformPolicy; the chance distributions of kuhn / leduc are uniform over the listed outcomes).
template <class R>
__device__ __forceinline__ void traj_resolve_chance(typename R::S& s, const typename R::Cfg& cfg, const Ctx& ctx, long long i,
                                                    u64 seed, u64 g, int mask_words, u32 b0) {
  u32 j = 0;
  while (R::cur_player(s, cfg) == kChancePlayerId) {
    u32 m[R::kMaskWords];
    R::legal_nonterminal(s, cfg, m);
    int cnt = 0;
    for (int w = 0; w < mask_words; ++w) cnt += __popc(m[w]);
    int a = nth_set_bit(m, mask_words, (int)philox_uniform(seed, g, b0 + 1u + j, (u32)cnt));
    apply_known_legal<R>(s, a, cfg, ctx, i);
    ++j;
  }
}

template <class R>
__global__ void __launch_bounds__(kBlock) k_traj_begin(Ctx ctx, typename R::Cfg cfg, u64 seed, long long lane_offset, int mask_words, int* __restrict__ lengths, long long n) {
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  if (lengths) lengths[i] = 0;
  typename R::S s;
  R::load(s, ctx, i);
  if (R::cur_player(s, cfg) != kChancePlayerId) return;
  traj_resolve_chance<R>(s, cfg, ctx, i, seed, (u64)(i + lane_offset), mask_words, 0u);
  R::store(s, ctx, i);
}

// Zero-copy form of k_step_compact for pinned, device-mapped host buffers (b2s_step_fused_host_compact): the kernel reads the
// action bytes straight from host memory and writes the status bytes straight back, so a step is ONE launch and the bytes
// cross PCIe under the kernel's own load / store parallelism — no DMA-engine copies, whose fixed set-up (~10-15 us each way)
// is most of a 1M-lane step whose payload is 1 MiB each way.  PCIe wants large requests: a block moves its kBlock * ILP
// action bytes with 16-byte loads into shared memory (one 64-thread slice of the block, 1 KiB contiguous per block), works
// from there, and writes its status bytes back the same way.  `actions` / `status` are device-visible addresses of the host
// buffers, 16-byte aligned.
template <class R, int ILP>
__global__ void __launch_bounds__(kBlock) k_step_compact_zc(Ctx ctx, typename R::Cfg cfg, const unsigned char* __restrict__ actions,
                                                            unsigned char* __restrict__ status, int small_mask, long long n) {
  __shared__ __align__(16) unsigned char act_s[kBlock * ILP];
  __shared__ __align__(16) unsigned char st_s[kBlock * ILP];
  const long long b0 = (long long)blockIdx.x * (kBlock * ILP);
  const long long left = n - b0;
  const int here = (int)(left < kBlock * ILP ? left : kBlock * ILP);       // lanes of this block
  const int vec = threadIdx.x * 16;
  if (vec < here) {
    if (vec + 16 <= here) *reinterpret_cast<uint4*>(act_s + vec) = *reinterpret_cast<const uint4*>(actions + b0 + vec);
    else for (int k = vec; k < here; ++k) act_s[k] = actions[b0 + k];
  }
  long long base = b0 + threadIdx.x;
  typename R::S s[ILP];
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    if (i < n) R::load(s[j], ctx, i);
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < ILP; ++j) {
    long long i = base + (long long)j * kBlock;
    if (i >= n) continue;
    const unsigned raw = act_s[threadIdx.x + j * kBlock];
    if (raw != 0xFFu) {
      if (R::terminal(s[j], cfg) || !R::apply(s[j], (int)raw, cfg, ctx, i)) flag_error(ctx.err, ctx.lane0 + i);
      else R::store(s[j], ctx, i);
    }
    unsigned st = 0;
    if (R::terminal(s[j], cfg)) {
      float r[R::kPlayers];
      R::returns(s[j], cfg, r);
      st = 0x80u | (r[0] > 0.f ? 1u : (r[0] < 0.f ? 2u : 0u));
    } else if (small_mask) {
      u32 m[R::kMaskWords];
      R::legal_nonterminal(s[j], cfg, m);
      st = m[0] & 0x7Fu;
    }
    st_s[threadIdx.x + j * kBlock] = (unsigned char)st;
  }
  __syncthreads();
  if (vec < here) {
    if (vec + 16 <= here) *reinterpret_cast<uint4*>(status + b0 + vec) = *reinterpret_cast<const uint4*>(st_s + vec);
    else for (int k = vec; k < here; ++k) status[b0 + k] = st_s[k];
  }
}

struct TrajStepOut {          // row t of the time-major outputs; any pointer may be null
  u32* mask;                  // [n][mask_words]
  int* actions;               // [n]
  signed char* players;       // [n]
  unsigned char* valid;       // [n]
  unsigned char* next_is_terminal;   // [n]
  int* lengths;               // [n] (not a row: set to t+1 by the step that ends the episode)
};

template <class R>
__global__ void __launch_bounds__(kBlock) k_traj_step(Ctx ctx, typename R::Cfg cfg, u64 seed, long long lane_offset, int t, int mask_words, int num_actions, TrajStepOut o, long long n) {
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  const bool live = i < n;
  __shared__ MaskStage<R::kMaskWords == 1 ? 0 : R::kMaskWords> stage;
  typename R::S s;
  u32 m[R::kMaskWords];
  int a = 0, pl = 0;
  unsigned char valid = 0, nit = 0;
  if (live) {
    R::load(s, ctx, i);
    if (R::terminal(s, cfg)) {
      // padding as BatchedTrajectory::ResizeFields (trajectories.cc:62-96): legal mask all ones, everything else 0
      for (int w = 0; w < R::kMaskWords; ++w) {
        int bits = num_actions - 32 * w;
        m[w] = bits >= 32 ? 0xffffffffu : (bits > 0 ? (1u << bits) - 1u : 0u);
      }
    } else {
      const u64 g = (u64)(i + lane_offset);
      const u32 b0 = 64u * (u32)(t + 1);
      R::legal_nonterminal(s, cfg, m);
      int cnt = 0;
      for (int w = 0; w < mask_words; ++w) cnt += __popc(m[w]);
      a = nth_set_bit(m, mask_words, (int)philox_uniform(seed, g, b0, (u32)cnt));
      pl = R::cur_player(s, cfg);
      valid = 1;
      apply_known_legal<R>(s, a, cfg, ctx, i);
      traj_resolve_chance<R>(s, cfg, ctx, i, seed, g, mask_words, b0);
      nit = R::terminal(s, cfg) ? 1 : 0;
      R::store(s, ctx, i);
      if (nit && o.lengths) o.lengths[i] = t + 1;
    }
  }
  if (o.mask) {                                            // uniform over the grid
    if (R::kMaskWords == 1) { if (live) o.mask[i] = m[0]; }
    else store_masks_coalesced(o.mask, i - (threadIdx.x & 31), n, live, mask_words, m, stage);
  }
  if (!live) return;
  if (o.actions) o.actions[i] = a;
  if (o.players) o.players[i] = (signed char)pl;
  if (o.valid) o.valid[i] = valid;
  if (o.next_is_terminal) o.next_is_terminal[i] = nit;
}

// Terminal Returns() of every episode (trajectories.cc:190); an episode still running after the last recorded
// step is an error (the reference CHECKs max_unroll_length >= the longest episode, trajectories.cc:64-68).
template <class R>
__global__ void __launch_bounds__(kBlock) k_traj_finish(Ctx ctx, typename R::Cfg cfg, float* __restrict__ rewards, long long n) {
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  typename R::S s;
  R::load(s, ctx, i);
  if (!R::terminal(s, cfg)) flag_error(ctx.err, i);
  if (rewards) {
    float r[R::kPlayers];
    R::returns(s, cfg, r);
    const int np = rule_num_players<R>(cfg);
    for (int p = 0; p < np; ++p) rewards[i * np + p] = r[p];
  }
}

// Clone: copy lane `src` of one batch into lanes [dst0, dst0+count) of another.
template <class R>
__global__ void __launch_bounds__(kBlock) k_broadcast(Ctx dst, long long dst0, long long count, Ctx srcctx, long long src, typename R::Cfg cfg) {
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= count) return;
  typename R::S s;
  R::load(s, srcctx, src);
  R::store(s, dst, dst0 + i);
  R::copy_history(dst, dst0 + i, srcctx, src, s, cfg);
}

// Clone a lane range: dst[dst0 + i] = src[src0 + i].
template <class R>
__global__ void __launch_bounds__(kBlock) k_copy(Ctx dst, long long dst0, Ctx srcctx, long long src0, long long count, typename R::Cfg cfg) {
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= count) return;
  typename R::S s;
  R::load(s, srcctx, src0 + i);
  R::store(s, dst, dst0 + i);
  R::copy_history(dst, dst0 + i, srcctx, src0 + i, s, cfg);
}

// Gather-clone: dst[i] = src[src_lanes[i]] (tree expansion: one child lane per (parent, action) pair).
template <class R>
__global__ void __launch_bounds__(kBlock) k_gather(Ctx dst, Ctx srcctx, const long long* __restrict__ src_lanes, long long count, typename R::Cfg cfg) {
  long long i = (long long)blockIdx.x * kBlock + threadIdx.x;
  if (i >= count) return;
  long long sl = src_lanes[i];
  if (sl < 0 || sl >= srcctx.cap) { flag_error(dst.err, i); return; }
  typename R::S s;
  R::load(s, srcctx, sl);
  R::store(s, dst, i);
  R::copy_history(dst, i, srcctx, sl, s, cfg);
}

// ---- host-side per-game dispatch table --------------------------------------------------------------

struct Batch;   // api.cu

// optional per-game device-side tables (e.g. go's Zobrist keys): R::device_init() if the rule core has one
template <class R> auto call_device_init(int) -> decltype(R::device_init(), void()) { R::device_init(); }
template <class R> void call_device_init(long) {}

struct GameOps {
  virtual ~GameOps() {}
  virtual void device_init() = 0;     // called with the batch's device current
  virtual const char* configure(const b2s_params& p, b2s_game_info& gi) = 0;
  virtual size_t chunk_bytes() const = 0;
  virtual int chunks() const = 0;
  virtual void reset(const Ctx&, long long n, cudaStream_t) = 0;
  virtual void apply(const Ctx&, const int* a, long long n, cudaStream_t) = 0;
  virtual void legal_mask(const Ctx&, u32* m, long long n, cudaStream_t) = 0;
  virtual void legal_list(const Ctx&, short* out, int* counts, int stride, long long n, cudaStream_t) = 0;
  virtual void status(const Ctx&, signed char* cur, unsigned char* term, float* rets, long long n, cudaStream_t) = 0;
  virtual const char* obs(const Ctx&, int player, int which, int zero_terminal, float* out, long long n, cudaStream_t) = 0;
  virtual void step_fused(const Ctx&, const int* a, u32* m, unsigned char* term, float* rets, long long n, cudaStream_t) = 0;
  virtual void step_compact(const Ctx&, const void* a, int action_bytes, unsigned char* status, u32* m, long long n, cudaStream_t) = 0;
  // uint8 actions and status bytes in device-mapped HOST memory, no mask words (k_step_compact_zc)
  virtual void step_compact_zero_copy(const Ctx&, const unsigned char* a_host, unsigned char* status_host, long long n, cudaStream_t) = 0;
  virtual void rollout(const Ctx&, u64 seed, long long lane_offset, float* rets, int* plies, long long n, cudaStream_t) = 0;
  virtual void broadcast(const Ctx& dst, long long dst0, long long count, const Ctx& src, long long srclane, cudaStream_t) = 0;
  virtual void copy(const Ctx& dst, long long dst0, const Ctx& src, long long src0, long long count, cudaStream_t) = 0;
  virtual void gather(const Ctx& dst, const Ctx& src, const long long* src_lanes, long long count, cudaStream_t) = 0;
  virtual void traj_begin(const Ctx&, u64 seed, long long lane_offset, int* lengths, long long n, cudaStream_t) = 0;
  virtual void traj_step(const Ctx&, u64 seed, long long lane_offset, int t, const TrajStepOut& o, long long n, cudaStream_t) = 0;
  virtual void traj_finish(const Ctx&, float* rewards, long long n, cudaStream_t) = 0;
  // MCTS over n roots (mcts.cuh); returns an error string when the game has no device MCTS
  virtual const char* mcts(const Ctx& roots, const Ctx& work, long long n, const struct MctsArgs& args, cudaStream_t) = 0;
  b2s_game_info info;
};

inline unsigned grid_for(long long n, int ilp = 1) { return (unsigned)((n + (long long)kBlock * ilp - 1) / ((long long)kBlock * ilp)); }

// magic M with floor(e*M >> 32) == e / d for all 0 <= e < limit (checked exhaustively).
inline bool make_magic(int d, int limit, u32* out) {
  u64 M = ((1ull << 32) + d - 1) / d;
  if (M >> 32) { if (d == 1) { *out = 0; return false; } }
  for (int e = 0; e < limit; ++e)
    if ((int)(((u64)e * M) >> 32) != e / d) return false;
  *out = (u32)M;
  return true;
}

template <class R>
struct GameOpsT : GameOps {
  typename R::Cfg cfg;
  const char* configure(const b2s_params& p, b2s_game_info& gi) override {
    const char* e = R::make_cfg(p, cfg, gi);
    if (e) return e;
    int width = gi.num_distinct_actions > gi.max_chance_outcomes ? gi.num_distinct_actions : gi.max_chance_outcomes;
    gi.mask_words = (width + 31) / 32;
    if (gi.mask_words > R::kMaskWords) return "action space too large for the device path";
    gi.state_bytes = (int)(sizeof(typename R::Chunk) * R::kChunks);
    gi.game_id = R::kGameId;
    info = gi;
    return nullptr;
  }
  void device_init() override { call_device_init<R>(0); }
  size_t chunk_bytes() const override { return sizeof(typename R::Chunk); }
  int chunks() const override { return R::kChunks; }
  void reset(const Ctx& c, long long n, cudaStream_t st) override {
    long long m = n > 0 ? n : 1;
    k_reset<R><<<grid_for(m), kBlock, 0, st>>>(c, cfg, n); ++g_launches;
  }
  void apply(const Ctx& c, const int* a, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    launch_pdl(k_apply<R, R::kIlp>, grid_for(n, R::kIlp), st, c, cfg, a, n); ++g_launches;
  }
  void legal_mask(const Ctx& c, u32* m, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    k_legal_mask<R, R::kIlp><<<grid_for(n, R::kIlp), kBlock, 0, st>>>(c, cfg, m, info.mask_words, n); ++g_launches;
  }
  void legal_list(const Ctx& c, short* out, int* counts, int stride, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    k_legal_list<R><<<grid_for(n), kBlock, 0, st>>>(c, cfg, out, counts, stride, info.mask_words, n); ++g_launches;
  }
  void status(const Ctx& c, signed char* cur, unsigned char* term, float* rets, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    k_status<R, R::kIlp><<<grid_for(n, R::kIlp), kBlock, 0, st>>>(c, cfg, cur, term, rets, n); ++g_launches;
  }
  const char* obs(const Ctx& c, int player, int which, int zero_terminal, float* out, long long n, cudaStream_t st) override {
    int size = which == 0 ? info.observation_tensor_size : info.information_state_tensor_size;
    if (size <= 0) return "game provides no such tensor";
    if (which == 1 && !R::kHasInfoState) return "game provides no information state tensor";
    if (n <= 0) return nullptr;
    u32 magic;
    if (!make_magic(size, 32 * size, &magic)) return "internal: no division magic";
    k_obs<R><<<grid_for(n), kBlock, 0, st>>>(c, cfg, player, which, zero_terminal, out, size, magic, n); ++g_launches;
    return nullptr;
  }
  void step_fused(const Ctx& c, const int* a, u32* m, unsigned char* term, float* rets, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    launch_pdl(k_step_fused<R, R::kIlp>, grid_for(n, R::kIlp), st, c, cfg, a, m, info.mask_words, term, rets, n); ++g_launches;
  }
  void step_compact(const Ctx& c, const void* a, int action_bytes, unsigned char* status, u32* m, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    const int small_mask = info.num_distinct_actions <= 7 ? 1 : 0;
    if (action_bytes == 1)
      launch_pdl(k_step_compact<R, R::kIlp, unsigned char>, grid_for(n, R::kIlp), st, c, cfg, (const unsigned char*)a, status, m, info.mask_words, small_mask, n);
    else
      launch_pdl(k_step_compact<R, R::kIlp, int>, grid_for(n, R::kIlp), st, c, cfg, (const int*)a, status, m, info.mask_words, small_mask, n);
    ++g_launches;
  }
  void step_compact_zero_copy(const Ctx& c, const unsigned char* a_host, unsigned char* status_host, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    const int small_mask = info.num_distinct_actions <= 7 ? 1 : 0;
    k_step_compact_zc<R, R::kIlp><<<grid_for(n, R::kIlp), kBlock, 0, st>>>(c, cfg, a_host, status_host, small_mask, n); ++g_launches;
  }
  void rollout(const Ctx& c, u64 seed, long long lane_offset, float* rets, int* plies, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    k_rollout<R><<<grid_for(n), kBlock, 0, st>>>(c, cfg, seed, lane_offset, info.mask_words, info.max_game_length + 4, rets, plies, n); ++g_launches;
  }
  void broadcast(const Ctx& dst, long long dst0, long long count, const Ctx& src, long long srclane, cudaStream_t st) override {
    if (count <= 0) return;
    k_broadcast<R><<<grid_for(count), kBlock, 0, st>>>(dst, dst0, count, src, srclane, cfg); ++g_launches;
  }
  void traj_begin(const Ctx& c, u64 seed, long long lane_offset, int* lengths, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    k_traj_begin<R><<<grid_for(n), kBlock, 0, st>>>(c, cfg, seed, lane_offset, info.mask_words, lengths, n); ++g_launches;
  }
  void traj_step(const Ctx& c, u64 seed, long long lane_offset, int t, const TrajStepOut& o, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    k_traj_step<R><<<grid_for(n), kBlock, 0, st>>>(c, cfg, seed, lane_offset, t, info.mask_words, info.num_distinct_actions, o, n); ++g_launches;
  }
  void traj_finish(const Ctx& c, float* rewards, long long n, cudaStream_t st) override {
    if (n <= 0) return;
    k_traj_finish<R><<<grid_for(n), kBlock, 0, st>>>(c, cfg, rewards, n); ++g_launches;
  }
  const char* mcts(const Ctx& roots, const Ctx& work, long long n, const MctsArgs& args, cudaStream_t st) override;
  void gather(const Ctx& dst, const Ctx& src, const long long* src_lanes, long long count, cudaStream_t st) override {
    if (count <= 0) return;
    k_gather<R><<<grid_for(count), kBlock, 0, st>>>(dst, src, src_lanes, count, cfg); ++g_launches;
  }
  void copy(const Ctx& dst, long long dst0, const Ctx& src, long long src0, long long count, cudaStream_t st) override {
    if (count <= 0) return;
    k_copy<R><<<grid_for(count), kBlock, 0, st>>>(dst, dst0, src, src0, count, cfg); ++g_launches;
  }
};

}  // namespace b2s
#include "mcts.cuh"
namespace b2s {
template <class R>
const char* GameOpsT<R>::mcts(const Ctx& roots, const Ctx& work, long long n, const MctsArgs& args, cudaStream_t st) {
  if constexpr (R::kMaxPath > 0) {
    if (info.max_game_length + 2 > R::kMaxPath) return "mcts: max_game_length too large for the device search path stack";
    if (info.min_utility != -1.0 || info.max_utility != 1.0) return "mcts: the device search needs win / loss / draw returns";
    if (n <= 0) return nullptr;
    MctsArgs a = args;
    a.num_actions = info.num_distinct_actions;
    a.mask_words = info.mask_words;
    a.max_plies = info.max_game_length + 4;
    a.max_utility = info.max_utility;
    const unsigned grid = (unsigned)((n + 127) / 128);
    // many trees: cap registers (6 CTAs of 128 threads per SM) so more warps are resident; few trees (deep
    // searches are memory-limited to a few thousand roots): let the compiler keep everything in registers
    if (a.compact) {
      if (n >= 100000) k_mcts<R, StatsC, R::kMaxPath, 6><<<grid, 128, 0, st>>>(roots, work, cfg, a, n);
      else k_mcts<R, StatsC, R::kMaxPath, 4><<<grid, 128, 0, st>>>(roots, work, cfg, a, n);
    } else {
      k_mcts<R, StatsW, R::kMaxPath, 4><<<grid, 128, 0, st>>>(roots, work, cfg, a, n);
    }
    ++g_launches;
    return nullptr;
  } else {
    return "mcts: games with chance nodes / imperfect information have no device MCTS";
  }
}

// one factory per game, defined in game_<name>.cu
GameOps* make_ops_tic_tac_toe();
GameOps* make_ops_connect_four();
GameOps* make_ops_breakthrough();
GameOps* make_ops_hex();
GameOps* make_ops_go();
GameOps* make_ops_kuhn_poker();
GameOps* make_ops_leduc_poker();
GameOps* make_ops_leduc_poker_n();   // players = 3..4
GameOps* make_ops_mnk();
GameOps* make_ops_othello();
GameOps* make_ops_y();
GameOps* make_ops_havannah();

}  // namespace b2s
