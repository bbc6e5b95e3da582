// imb_disc.cu -- stage 3 of the GAIL/AIRL round: the discriminator update, fused.
//
// Replaces (reference, paths relative to imitation's src/imitation): rewards/reward_nets.py:441-457
// (BasicRewardNet.forward), :701-736 (ShapedRewardNet.forward), util/networks.py:79-134
// (RunningNorm), algorithms/adversarial/common.py:353-372 (BCE-with-logits, backward, Adam)
// and :27-92 (compute_train_stats).
//
// Kernels (no spinning grid barriers -- every dependency is a kernel boundary or the
// "last block done" ticket, so a bug cannot hang the GPU):
//   k_norm_stats        RunningNorm.update_stats for a list of up to three jobs (one normaliser each;
//                       blockIdx.y = job): per-chunk (mean, M2) per input feature, then the last CTA
//                       Chan-merges each job's chunks in a fixed order and folds the jobs into their
//                       running statistics in job order -- or, for a one-job launch, appends the batch
//                       moments to a deferred slot list.
//   k_norm_fold         folds deferred slots into the running statistics, in order.
//   k_disc_fwdbwd<R>    fp32-FFMA forward / BCE / backward: persistent CTAs over R-row tiles of the
//                       feature-major batch staged by cp.async.bulk, tiled contractions of
//                       imb_tile.cuh; one partial [gradient | statistics] row per CTA.
//   k_disc_fwdbwd_tc    the same on the tcgen05 tensor cores (imb_disc_tc.cuh), used whenever the
//                       network shape fits it.
//   k_disc_reduce       warp-per-parameter deterministic sum of the per-CTA partials.
//   k_disc_adam         torch.optim.Adam / AdamW step + the 9 train statistics.
//   k_disc_reduce_adam  both in one launch: the last block to finish the reduction runs the step.
//   k_pref_loss         preference comparisons: Boltzmann probability, cross entropy and its gradient.
//   k_reward_fwd<H>     forward only (reward relabel / predict), thread per row.
//   k_reward_norm_scan  NormalizedRewardNet.predict_processed over consecutive env steps.
//   k_stats_publish, k_set_rows, k_set_meta, k_state_add: small bookkeeping kernels.
#include <stdlib.h>

#include "imb_common.cuh"
#include "imb_mlp.cuh"
#include "imb_tile.cuh"

thread_local char g_imb_err[512] = {0};

extern "C" int imb_version(void) { return 1; }
extern "C" const char* imb_last_error(void) { return g_imb_err; }

namespace {

constexpr int NORM_CHUNK = 512;       // rows per CTA in k_norm_stats
constexpr int NORM_PS = 2 * IMB_MAX_DIN + 4;  // floats per chunk record of k_norm_stats: mean | M2 | n
constexpr int MAXG = 296;             // max CTAs of k_disc_fwdbwd (2 per SM)

// ---- workspace layout (floats) -----------------------------------------------------------------
struct WsLayout {
  int64_t gacc;      // [P] accumulated gradient
  int64_t stats;     // [16] reduced sums of the last minibatch
  int64_t meta;      // [16] ints: grid of the last fwdbwd launch, n rows, n_expert
  int64_t snap;      // [2*IMB_MAX_DIN] potential-norm stats after the first (next_obs) update
  int64_t ticket;    // [16] uint tickets
  int64_t normpart;  // [MAXCHUNKS][NORM_PS]
  int64_t partial;   // [MAXG][P + 16]
  int64_t total;
};
constexpr int MAXCHUNKS = 16384;  // up to 8M rows per norm launch
__host__ __device__ inline int64_t part_stride(int P) { return (int64_t)((P + 16 + 31) / 32) * 32; }
inline WsLayout ws_layout(int P) {
  WsLayout w;
  int64_t o = 0;
  w.gacc = o;
  o += (P + 31) / 32 * 32;
  w.stats = o;
  o += 32;
  w.meta = o;
  o += 32;
  w.snap = o;
  o += 2 * IMB_MAX_DIN;
  w.ticket = o;
  o += 32;
  w.normpart = o;
  o += (int64_t)MAXCHUNKS * NORM_PS;
  w.partial = o;
  o += (int64_t)MAXG * part_stride(P);
  w.total = o;
  return w;
}

// ---- RunningNorm statistics ----------------------------------------------------------------------
// One RunningNorm.update_stats per job.  A shaped net updates its potential's normaliser twice per training forward
// (next_obs, then obs -- reward_nets.py:708-710), so two jobs may share one normaliser.
struct NormJob {
  int din;
  short row[IMB_MAX_DIN];  // batch feature rows
  float* rmv;              // running [mean | var] of the job's normaliser
  int32_t* cnt;
  float* snap;             // optional copy of the statistics after this job's fold
};
struct NormJobs {
  int njobs;
  NormJob job[3];
};

// exact two-pass (mean, M2) of the cn values at src, by one warp
__device__ __forceinline__ void chunk_moments(const float* src, int cn, int lane, float& mean, float& m2) {
  float s = 0.f;
  for (int i = lane; i < cn; i += 32) s += src[i];
  s = warp_sum(s);
  mean = s / (float)cn;
  m2 = 0.f;
  for (int i = lane; i < cn; i += 32) {
    float dlt = src[i] - mean;
    m2 = fmaf(dlt, dlt, m2);
  }
  m2 = warp_sum(m2);
}

// Chan et al. merge of feature k over the nchunks chunk records at `part`, by one warp: every lane merges its chunks
// (lane, lane + 32, ...) in index order, then the 32 lane results are merged by a fixed butterfly (deterministic; a
// single thread walking all chunks cost more than the statistics themselves once the chunks became small enough to fill
// the GPU).  Every lane ends with (n, mean, M2) of the whole batch.
__device__ __forceinline__ void chan_merge_chunks(const float* part, int nchunks, int k, int lane, float& na, float& ma,
                                                  float& m2a) {
  na = 0.f;
  ma = 0.f;
  m2a = 0.f;
  for (int c = lane; c < nchunks; c += 32) {
    const float* p = part + (int64_t)c * NORM_PS;
    const float nb = __ldcg(p + 2 * IMB_MAX_DIN), mb = __ldcg(p + k), m2b = __ldcg(p + IMB_MAX_DIN + k);
    const float nt = na + nb;
    const float dlt = mb - ma;
    ma = ma + dlt * (nb / nt);
    m2a = m2a + m2b + dlt * dlt * (na * nb / nt);
    na = nt;
  }
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float nb = __shfl_xor_sync(0xffffffffu, na, o), mb = __shfl_xor_sync(0xffffffffu, ma, o),
                m2b = __shfl_xor_sync(0xffffffffu, m2a, o);
    // merge (lower lane, higher lane) in that order on both sides so the pair agrees bit for bit
    const bool lowme = (lane & o) == 0;
    const float n1 = lowme ? na : nb, m1 = lowme ? ma : mb, q1 = lowme ? m2a : m2b;
    const float n2 = lowme ? nb : na, m2v = lowme ? mb : ma, q2 = lowme ? m2b : m2a;
    const float nt = n1 + n2;
    if (nt > 0.f) {
      const float dlt = m2v - m1;
      ma = m1 + dlt * (n2 / nt);
      m2a = q1 + q2 + dlt * dlt * (n1 * n2 / nt);
    }
    na = nt;
  }
}

// fold batch moments (b_mean, biased b_var, b_n rows) into running statistics over cnt earlier rows with
// RunningNorm.update_stats' arithmetic (util/networks.py:121-134).  nvcc contracts `var * cnt + b_var * b_n` per call
// site: fma(b_var, b_n, var * cnt) in k_norm_stats, fma(var, cnt, b_var * b_n) in k_norm_fold, so an immediate and a
// deferred fold of the same batch can differ in the last bit of the variance.
__device__ __forceinline__ void fold_moments(float& mean, float& var, float cnt, float b_mean, float b_var, float b_n) {
  const float tot = cnt + b_n;
  const float delta = b_mean - mean;
  mean += delta * b_n / tot;
  var *= cnt;
  var += b_var * b_n;
  var += delta * delta * cnt * b_n / tot;
  var /= tot;
}

// One CTA per chunk_rows rows of job blockIdx.y; warp w handles features w, w+nw, ...  The last CTA of the grid merges
// each job's chunks and folds the jobs into their running statistics in job order (a later job may read what an earlier
// one wrote).  Deferred mode, for one-job launches only: the batch moments go to the next free slot of `defer` ([0] =
// slot counter, slots of 2 * din + 1 floats: mean | biased variance | n) instead of into the running statistics;
// k_norm_fold applies them later, in order.
__global__ void __launch_bounds__(256) k_norm_stats(NormJobs J, const float* __restrict__ batch, int64_t ld, int64_t n,
                                                    int chunk_rows, float* __restrict__ part,
                                                    unsigned int* __restrict__ ticket, float* __restrict__ defer,
                                                    int defer_cap) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  const int nchunks = gridDim.x;
  const NormJob& L = J.job[blockIdx.y];
  const int64_t r0 = (int64_t)blockIdx.x * chunk_rows;
  const int64_t r1 = min(n, r0 + (int64_t)chunk_rows);
  const int cn = (int)(r1 - r0);
  float* my = part + ((int64_t)blockIdx.y * nchunks + blockIdx.x) * NORM_PS;
  for (int k = warp; k < L.din; k += nw) {
    float mean, m2;
    chunk_moments(batch + (int64_t)L.row[k] * ld + r0, cn, lane, mean, m2);
    if (lane == 0) {
      my[k] = mean;
      my[IMB_MAX_DIN + k] = m2;
    }
  }
  if (threadIdx.x == 0) my[2 * IMB_MAX_DIN] = (float)cn;
  __threadfence();
  __shared__ bool is_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned int t = atomicAdd(ticket, 1u);
    is_last = (t == gridDim.x * gridDim.y - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  float* slot = nullptr;
  if (defer) {
    int k = (int)defer[0];
    if (k >= defer_cap) k = defer_cap - 1;  // (host folds long before this; never overrun)
    slot = defer + 4 + (int64_t)k * (2 * J.job[0].din + 1);
  }
  for (int job = 0; job < J.njobs; ++job) {
    const NormJob& Lj = J.job[job];
    const int32_t old_count = slot ? 0 : *Lj.cnt;
    for (int k = warp; k < Lj.din; k += nw) {
      float na, ma, m2a;
      chan_merge_chunks(part + (int64_t)job * nchunks * NORM_PS, nchunks, k, lane, na, ma, m2a);
      if (lane == 0 && slot) {
        slot[k] = ma;
        slot[Lj.din + k] = m2a / na;
      } else if (lane == 0) {
        float mean = Lj.rmv[k], var = Lj.rmv[Lj.din + k];
        fold_moments(mean, var, (float)old_count, ma, m2a / na, na);
        Lj.rmv[k] = mean;
        Lj.rmv[Lj.din + k] = var;
        if (Lj.snap) {
          Lj.snap[k] = mean;
          Lj.snap[Lj.din + k] = var;
        }
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      if (slot) {
        slot[2 * Lj.din] = (float)n;
        defer[0] += 1.0f;
      } else {
        *Lj.cnt = old_count + (int32_t)n;
      }
    }
    __syncthreads();  // the next job may fold into the same normaliser: count and statistics are in place
  }
  if (threadIdx.x == 0) *ticket = 0u;  // re-arm for the next launch
}

// fold the deferred batch moments into the running statistics, slot by slot
__global__ void k_norm_fold(int din, float* __restrict__ defer, float* __restrict__ run_mean_var,
                            int32_t* __restrict__ count, int k_fixed) {
  const int K = k_fixed > 0 ? k_fixed : (int)defer[0];
  const int k = threadIdx.x;
  int32_t cnt_i = *count;
  if (k < din) {
    float mean = run_mean_var[k], var = run_mean_var[din + k];
    int32_t c = cnt_i;
    for (int sidx = 0; sidx < K; ++sidx) {
      const float* slot = defer + 4 + (int64_t)sidx * (2 * din + 1);
      const float b_n = slot[2 * din];
      fold_moments(mean, var, (float)c, slot[k], slot[din + k], b_n);
      c += (int32_t)b_n;
    }
    run_mean_var[k] = mean;
    run_mean_var[din + k] = var;
  }
  __syncthreads();
  if (k == 0) {
    for (int sidx = 0; sidx < K; ++sidx) cnt_i += (int32_t)defer[4 + (int64_t)sidx * (2 * din + 1) + 2 * din];
    *count = cnt_i;
    if (k_fixed <= 0) defer[0] = 0.f;
  }
}

// ---- the fused forward / BCE / backward kernel (tiled-GEMM form, see imb_tile.cuh) ------------------
// Dynamic shared memory (floats):
//   [image per pass][AW: 4 slices x P][stage: nstage x RS][XN: KP x RS][H1, H2, DZ1: JP x RS each]
//   [lg, gv, gp, dv, lpv: R each]
template <int R>
__global__ void __launch_bounds__(R, 256 / R) k_disc_fwdbwd(const DiscLaunch L, const float* __restrict__ params,
                                                      const float* __restrict__ batch, int64_t ld, int64_t n,
                                                      int64_t n_expert, float loss_scale,
                                                      const float* __restrict__ grad_out,
                                                      float* __restrict__ logits_out, float* __restrict__ partial,
                                                      int* __restrict__ meta, int JP, int KP, int img_sz, int aw_off, int st_off, int xn_off,
                                                      int t_off, int v_off, int nsl) {
  // one thread per tile row: R threads, warp w -> column group w % 4 (8 columns) and row half w / 4
  constexpr int NQ = 1;
  constexpr int NTK = R;
  constexpr int RS = R + TILE_PAD;
  extern __shared__ __align__(128) float smem[];
  __shared__ __align__(8) uint64_t bar;
  __shared__ float red[64];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cg = warp & 3, grp = warp >> 2, tg = tid & 127;
  float* AW = smem + aw_off;
  float* xs = smem + st_off;
  float* XN = smem + xn_off;
  float* H1 = smem + t_off;
  float* H2 = H1 + JP * RS;
  float* DZ1 = H2 + JP * RS;
  float* lg = smem + v_off;
  float* gv = lg + R;
  float* gp = gv + R;
  float* dv = gp + R;
  float* lpv = dv + R;
  const int P = L.P;

  for (int p = 0; p < L.npass; ++p)
    load_timg(smem + p * img_sz, L.pass[p], JP, params, L.pass[p].has_norm ? L.pass[p].norm : nullptr, L.pass[p].eps);
  for (int i = tid; i < nsl * P; i += NTK) AW[i] = 0.f;
  if (tid == 0) {
    mbar_init(&bar, 1);
    mbar_fence_init();
    if (blockIdx.x == 0) {  // launch record for k_disc_reduce / k_disc_adam (stats of the LAST minibatch)
      meta[0] = (int)gridDim.x;
      meta[1] = (int)n;
      meta[2] = (int)n_expert;
      reinterpret_cast<float*>(meta)[3] = loss_scale;
    }
  }
  __syncthreads();

  const int64_t ntiles = (n + R - 1) / R;
  auto issue = [&](int64_t tile) {
    int64_t cnt = ld - tile * R;  // floats available in each feature row from this tile's start
    if (cnt > R) cnt = R;
    mbar_expect_tx(&bar, (uint32_t)(L.nstage * cnt * 4));
    for (int s = 0; s < L.nstage; ++s)
      bulk_g2s(xs + s * RS, batch + (int64_t)L.stage_row[s] * ld + tile * R, (uint32_t)(cnt * 4), &bar);
  };
  uint32_t phase = 0;
  if (tid == 0 && (int64_t)blockIdx.x < ntiles) issue(blockIdx.x);

  int rq[NQ];
  rq[0] = grp * 128 + lane * 4;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  float s_loss = 0.f, s_ent = 0.f;
  int c_exp = 0, c_gen = 0, c_pred_exp = 0;

  // one MLP forward over the tile for pass `p`: builds XN, H1, H2 and returns nothing; the per-row
  // output is accumulated into lg[] (scaled by the pass coefficient) when `accumulate` is set.
  auto forward_pass = [&](int p, int nv, bool accumulate, bool first) {
    const PassDesc& Pd = L.pass[p];
    const float* img = smem + p * img_sz;
    const int din = Pd.din;
    const float* mean = img + TImg::mean(din, JP);
    const float* istd = img + TImg::istd(din, JP);
    // normalised inputs, feature-major; rows >= nv and features >= din are zero
    for (int i = tid; i < KP * (R / 4); i += NTK) {
      const int k = i / (R / 4), r4 = (i - k * (R / 4)) * 4;
      float4 v = zero4;
      if (k < din) {
        const float4 x = ld4(xs + Pd.in_slot[k] * RS + r4);
        const float m = mean[k], is = istd[k];
        v.x = (r4 + 0 < nv) ? (x.x - m) * is : 0.f;
        v.y = (r4 + 1 < nv) ? (x.y - m) * is : 0.f;
        v.z = (r4 + 2 < nv) ? (x.z - m) * is : 0.f;
        v.w = (r4 + 3 < nv) ? (x.w - m) * is : 0.f;
      }
      st4(XN + k * RS + r4, v);
    }
    __syncthreads();
    const float* HL = XN;
    int hl = din;
    float4 gq[NQ];
#pragma unroll
    for (int q = 0; q < NQ; ++q) gq[q] = zero4;
    if (Pd.n_hidden >= 1) {
      for (int jh = 0; jh < JP / 32; ++jh) {
        const int j0 = jh * 32 + cg * 8;
        float acc[NQ * 4][8];
#pragma unroll
        for (int a = 0; a < NQ * 4; ++a)
#pragma unroll
          for (int t = 0; t < 8; ++t) acc[a][t] = 0.f;
        gemm_acc<NQ, false>(acc, XN, RS, rq, img + TImg::w1t(din, JP), JP, j0, din, gq, nullptr);
        const float* b1 = img + TImg::b1(din, JP);
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          const float b = b1[j0 + t];
#pragma unroll
          for (int q = 0; q < NQ; ++q)
            st4(H1 + (j0 + t) * RS + rq[q],
                make_float4(fmaxf(acc[q * 4 + 0][t] + b, 0.f), fmaxf(acc[q * 4 + 1][t] + b, 0.f),
                            fmaxf(acc[q * 4 + 2][t] + b, 0.f), fmaxf(acc[q * 4 + 3][t] + b, 0.f)));
        }
      }
      __syncthreads();
      HL = H1;
      hl = Pd.h1;
    }
    if (Pd.n_hidden >= 2) {
      for (int jh = 0; jh < JP / 32; ++jh) {
        const int j0 = jh * 32 + cg * 8;
        float acc[NQ * 4][8];
#pragma unroll
        for (int a = 0; a < NQ * 4; ++a)
#pragma unroll
          for (int t = 0; t < 8; ++t) acc[a][t] = 0.f;
        gemm_acc<NQ, false>(acc, H1, RS, rq, img + TImg::w2t(din, JP), JP, j0, Pd.h1, gq, nullptr);
        const float* b2 = img + TImg::b2(din, JP);
#pragma unroll
        for (int t = 0; t < 8; ++t) {
          const float b = b2[j0 + t];
#pragma unroll
          for (int q = 0; q < NQ; ++q)
            st4(H2 + (j0 + t) * RS + rq[q],
                make_float4(fmaxf(acc[q * 4 + 0][t] + b, 0.f), fmaxf(acc[q * 4 + 1][t] + b, 0.f),
                            fmaxf(acc[q * 4 + 2][t] + b, 0.f), fmaxf(acc[q * 4 + 3][t] + b, 0.f)));
        }
      }
      __syncthreads();
      HL = H2;
      hl = Pd.h2;
    }
    if (accumulate) {
      const float* wf = img + TImg::wf(din, JP);
      const float bf = img[TImg::bf(din, JP)];
      for (int r = tid; r < R; r += NTK) {
        float o = bf;
        for (int j = 0; j < hl; ++j) o = fmaf(wf[j], HL[j * RS + r], o);
        const float c = pass_coef(Pd.coef_kind, L.gamma, dv[r]);
        lg[r] = first ? c * o : fmaf(c, o, lg[r]);
      }
      __syncthreads();
    }
  };

  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    mbar_wait(&bar, phase);
    phase ^= 1u;
    const int nv = (int)min((int64_t)R, n - tile * R);
    for (int r = tid; r < R; r += NTK) {
      dv[r] = (L.done_slot >= 0 && r < nv) ? xs[L.done_slot * RS + r] : 0.f;
      lpv[r] = (L.logp_slot >= 0 && r < nv) ? xs[L.logp_slot * RS + r] : 0.f;
    }
    __syncthreads();
    // ---- logits: forward over all passes (the last pass's tiles stay valid for its backward) -------
    for (int p = 0; p < L.npass; ++p) forward_pass(p, nv, true, p == 0);
    // stage is free once the last forward that reads it is done -- unless passes are recomputed below
    const bool recompute = L.npass > 1;
    const int64_t next = tile + gridDim.x;
    if (!recompute && tid == 0 && next < ntiles) issue(next);
    // ---- dL/dlogit per row + statistics -------------------------------------------------------------
    for (int r = tid; r < R; r += NTK) {
      float g = 0.f;
      if (r < nv) {
        const int64_t row = tile * R + r;
        const float logit = lg[r] - lpv[r];
        if (logits_out) logits_out[row] = logit;
        if (grad_out) {
          g = grad_out[row];
        } else {
          const float y = (row < n_expert) ? 1.f : 0.f;
          const float sg = sigmoid_f(logit);
          const float sp = fmaxf(logit, 0.f) + log1pf(expf(-fabsf(logit)));
          s_loss += sp - logit * y;
          s_ent += sp - logit * sg;
          const bool pred_exp = !(logit < 0.f);
          c_pred_exp += pred_exp;
          if (y > 0.5f) c_exp += pred_exp; else c_gen += !pred_exp;
          g = (sg - y) * loss_scale;
        }
      }
      gv[r] = g;
    }
    __syncthreads();

    // ---- backward + weight gradients, pass by pass ---------------------------------------------------
    for (int pi = 0; pi < L.npass; ++pi) {
      const int p = L.npass - 1 - pi;  // last pass first: its forward tiles are still in shared memory
      if (pi > 0) forward_pass(p, nv, false, false);
      if (recompute && pi == L.npass - 1 && tid == 0 && next < ntiles) issue(next);
      const PassDesc& Pd = L.pass[p];
      const float* img = smem + p * img_sz;
      const int din = Pd.din;
      const float* wf = img + TImg::wf(din, JP);
      for (int r = tid; r < R; r += NTK) gp[r] = gv[r] * pass_coef(Pd.coef_kind, L.gamma, dv[r]);
      __syncthreads();
      float* A0 = AW;  // slice 0 accumulators
      const int h1w = Pd.h1, h2w = Pd.h2;
      const int off_w1 = Pd.param_off, off_b1 = off_w1 + h1w * din, off_w2 = off_b1 + h1w;
      const int off_b2 = off_w2 + ((Pd.n_hidden == 2) ? h2w * h1w : 0);
      const int off_wf = (Pd.n_hidden == 2) ? off_b2 + h2w : (Pd.n_hidden == 1 ? off_w2 : Pd.param_off);
      const int hl = (Pd.n_hidden == 2) ? h2w : (Pd.n_hidden == 1 ? h1w : din);
      const float* HL = (Pd.n_hidden == 2) ? H2 : (Pd.n_hidden == 1 ? H1 : XN);
      // dL/dz1 tile
      if (Pd.n_hidden == 2) {
        float4 gq[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) gq[q] = ld4(gp + rq[q]);
        for (int jh = 0; jh < JP / 32; ++jh) {
          const int i0 = jh * 32 + cg * 8;
          float acc[NQ * 4][8];
#pragma unroll
          for (int a = 0; a < NQ * 4; ++a)
#pragma unroll
            for (int t = 0; t < 8; ++t) acc[a][t] = 0.f;
          gemm_acc<NQ, true>(acc, H2, RS, rq, img + TImg::w2(din, JP), JP, i0, h2w, gq, wf);
#pragma unroll
          for (int t = 0; t < 8; ++t)
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
              const float4 h = ld4(H1 + (i0 + t) * RS + rq[q]);
              st4(DZ1 + (i0 + t) * RS + rq[q],
                  make_float4(h.x > 0.f ? acc[q * 4 + 0][t] : 0.f, h.y > 0.f ? acc[q * 4 + 1][t] : 0.f,
                              h.z > 0.f ? acc[q * 4 + 2][t] : 0.f, h.w > 0.f ? acc[q * 4 + 3][t] : 0.f));
            }
        }
      } else if (Pd.n_hidden == 1) {
        for (int i = tid; i < JP * (R / 4); i += NTK) {
          const int j = i / (R / 4), r4 = (i - j * (R / 4)) * 4;
          const float4 h = ld4(H1 + j * RS + r4), g = ld4(gp + r4);
          const float w = wf[j];
          st4(DZ1 + j * RS + r4, make_float4(h.x > 0.f ? g.x * w : 0.f, h.y > 0.f ? g.y * w : 0.f,
                                             h.z > 0.f ? g.z * w : 0.f, h.w > 0.f ? g.w * w : 0.f));
        }
      }
      __syncthreads();
      const int jl = lane & 7, il = lane >> 3;
      // weight gradients: a group of 4 warps (128 threads) per contraction; with two groups (R = 256)
      // dW2 and dW1 run concurrently, each split into row slices with private accumulators.
      constexpr int NGRP = R / 128;
      // R = 256: two 128-thread groups run dW2 and dW1 concurrently (4 row slices each).
      // R = 128: 32-wide nets split the CTA 64/64 (dW2 | dW1, 2 slices each); otherwise sequential.
      const bool split64 = (NGRP == 1) && JP == 32 && Pd.n_hidden == 2;
      const int wg = split64 ? (tid >> 6) : grp;        // which contraction group this thread is in
      const int tgw = split64 ? (tid & 63) : tg;        // thread index inside the group
      const int gthreads = split64 ? 64 : 128;
      const bool do_w2 = Pd.n_hidden == 2 && ((NGRP == 1 && !split64) || wg == 0);
      const bool do_w1 = Pd.n_hidden >= 1 && ((NGRP == 1 && !split64) || wg == (Pd.n_hidden == 2 ? 1 : 0));
      if (do_w2) {
        const int nblk = (JP / 32) * (JP / 32), ntl = nblk * 32;
        const int slices = min(gthreads / ntl, nsl);
        const int lt = tgw % ntl, sl = tgw / ntl, blk = lt >> 5;
        const int jb = (blk % (JP / 32)) * 32, ib = (blk / (JP / 32)) * 32;
        float acc[4][8], bacc[4], sj[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          bacc[jj] = 0.f;
          sj[jj] = wf[jb + jl + 8 * jj];
#pragma unroll
          for (int ii = 0; ii < 8; ++ii) acc[jj][ii] = 0.f;
        }
        const int rows = R / slices;
        if (sl < slices)
          wgrad_acc<true>(acc, bacc, H2, H1, RS, jb + jl, ib + il, sl * rows, (sl + 1) * rows, gp, sj);
        float* A = A0 + (sl < slices ? sl : 0) * P;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const int j = jb + jl + 8 * jj;
          if (j < h2w) {
#pragma unroll
            for (int ii = 0; ii < 8; ++ii) {
              const int i = ib + il + 4 * ii;
              if (i < h1w) A[off_w2 + j * h1w + i] += acc[jj][ii];
            }
            if (il == 0 && ib == 0) A[off_b2 + j] += bacc[jj];
          }
        }
      }
      if (do_w1) {
        const int nblk = (JP / 32) * (KP / 32), ntl = nblk * 32;
        const int slices = min(gthreads / ntl, nsl);
        const int lt = tgw % ntl, sl = tgw / ntl, blk = lt >> 5;
        const int jb = (blk % (JP / 32)) * 32, ib = (blk / (JP / 32)) * 32;
        float acc[4][8], bacc[4];
        const float sj[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          bacc[jj] = 0.f;
#pragma unroll
          for (int ii = 0; ii < 8; ++ii) acc[jj][ii] = 0.f;
        }
        const int rows = R / slices;
        if (sl < slices)
          wgrad_acc<false>(acc, bacc, DZ1, XN, RS, jb + jl, ib + il, sl * rows, (sl + 1) * rows, nullptr, sj);
        float* A = A0 + (sl < slices ? sl : 0) * P;
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) {
          const int j = jb + jl + 8 * jj;
          if (j < h1w) {
#pragma unroll
            for (int ii = 0; ii < 8; ++ii) {
              const int kk = ib + il + 4 * ii;
              if (kk < din) A[off_w1 + j * din + kk] += acc[jj][ii];
            }
            if (il == 0 && ib == 0) A[off_b1 + j] += bacc[jj];
          }
        }
      }
      // dwf / dbf: thread j sums its feature row against gp (slice 1 accumulators keep owners unique)
      {
        float* A = A0 + 1 * P;
        for (int j = tid; j <= hl; j += NTK) {
          float acc = 0.f;
          if (j < hl) {
            for (int r = 0; r < R; r += 4) {
              const float4 h = ld4(HL + j * RS + r), g = ld4(gp + r);
              acc = fmaf(h.x, g.x, acc);
              acc = fmaf(h.y, g.y, acc);
              acc = fmaf(h.z, g.z, acc);
              acc = fmaf(h.w, g.w, acc);
            }
          } else {
            for (int r = 0; r < R; r += 4) {
              const float4 g = ld4(gp + r);
              acc += (g.x + g.y) + (g.z + g.w);
            }
          }
          A[off_wf + j] += acc;
        }
      }
      __syncthreads();
    }
  }

  // ---- per-CTA partials: gradients (slices summed in fixed order) + statistics ----------------------
  float* my = partial + (int64_t)blockIdx.x * part_stride(P);
  for (int i = tid; i < P; i += NTK) {
    float v = AW[i];
    for (int s2 = 1; s2 < nsl; ++s2) v += AW[s2 * P + i];
    my[i] = v;
  }
  s_loss = warp_sum(s_loss);
  s_ent = warp_sum(s_ent);
  c_exp = warp_sum_i(c_exp);
  c_gen = warp_sum_i(c_gen);
  c_pred_exp = warp_sum_i(c_pred_exp);
  if (lane == 0) {
    red[warp * 5 + 0] = s_loss;
    red[warp * 5 + 1] = s_ent;
    red[warp * 5 + 2] = (float)c_exp;
    red[warp * 5 + 3] = (float)c_gen;
    red[warp * 5 + 4] = (float)c_pred_exp;
  }
  __syncthreads();
  if (tid < 5) {
    float v = 0.f;
    for (int w = 0; w < NTK / 32; ++w) v += red[w * 5 + tid];
    my[P + tid] = v;
  }
}

}  // namespace
#include "imb_disc_tc.cuh"
namespace {

// ---- deterministic reduction of the per-CTA partials -----------------------------------------
// warp per parameter (and per statistic): lanes stride over the G partial rows, shuffle-reduce.  Parameter sums are
// added to the gradient accumulator (and copied to grad_out_flat if given); statistic sums replace the previous ones.
__device__ __forceinline__ void reduce_partials(int P, int G, const float* __restrict__ partial, float* __restrict__ gacc,
                                                float* __restrict__ stats, float* __restrict__ grad_out_flat) {
  const int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  const int64_t ps = part_stride(P);
  for (int p = gw; p < P + 5; p += nwarps) {
    float acc = 0.f;
    for (int c = lane; c < G; c += 32) acc += partial[(int64_t)c * ps + p];
    acc = warp_sum(acc);
    if (lane == 0) {
      if (p < P) {
        const float v = gacc[p] + acc;
        gacc[p] = v;
        if (grad_out_flat) grad_out_flat[p] = v;
      } else {
        stats[p - P] = acc;  // statistics of the LAST minibatch only (common.py:376-381)
      }
    }
  }
}

__global__ void __launch_bounds__(256) k_disc_reduce(int P, int G, const float* __restrict__ partial,
                                                    float* __restrict__ gacc, float* __restrict__ stats,
                                                    float* __restrict__ grad_out_flat) {
  reduce_partials(P, G, partial, gacc, stats, grad_out_flat);
}

// beta^n for an integer step count by repeated squaring (pow(double, double) costs microseconds on one thread)
__device__ __forceinline__ double dpowi(double b, int64_t n) {
  double r = 1.0;
  while (n > 0) {
    if (n & 1) r *= b;
    b *= b;
    n >>= 1;
  }
  return r;
}

// torch.optim.Adam / AdamW step by one block: thread 0 computes the bias corrections and commits the step counter, then
// the block strides over the P elements.  grad is read through L2: in k_disc_reduce_adam other blocks wrote it.
__device__ __forceinline__ void adam_step(int P, const imb_adam& opt, float* __restrict__ params, float* __restrict__ m,
                                          float* __restrict__ v, const float* grad, float grad_div,
                                          int64_t* __restrict__ step_io) {
  // bias corrections in double like torch's Python-scalar arithmetic (torch/optim/adam.py)
  __shared__ float s_bc[2];
  if (threadIdx.x == 0) {
    const int64_t step = *step_io + 1;
    const double bc1d = 1.0 - dpowi((double)opt.beta1, step);
    const double bc2d = 1.0 - dpowi((double)opt.beta2, step);
    s_bc[0] = (float)((double)opt.lr / bc1d);
    s_bc[1] = (float)sqrt(bc2d);
    *step_io = step;
  }
  __syncthreads();
  const float step_size = s_bc[0], bc2_sqrt = s_bc[1];
  for (int i = threadIdx.x; i < P; i += blockDim.x) {
    const float g = __ldcg(grad + i) / grad_div;
    const float mi = m[i] + (g - m[i]) * (1.0f - opt.beta1);        // torch: exp_avg.lerp_(grad, 1-beta1)
    const float vi = v[i] * opt.beta2 + (1.0f - opt.beta2) * g * g;  // exp_avg_sq.mul_(b2).addcmul_(g,g,1-b2)
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + opt.eps;
    const float pw = opt.weight_decay > 0.f ? params[i] * (1.0f - opt.lr * opt.weight_decay) : params[i];  // AdamW
    params[i] = pw - step_size * (mi / denom);
  }
}

// the nine statistics of compute_train_stats (common.py:27-92), by one thread, from the reduced sums of the last
// minibatch and its launch record (meta: n rows, n_expert, loss scale).  stats is read through L2: in
// k_disc_reduce_adam other blocks wrote it.
__device__ __forceinline__ void write_train_stats(const float* stats, const int* meta, float* stats_out) {
  const float n = (float)meta[1], n_exp = (float)meta[2], n_gen = n - n_exp;
  const float loss_sum = __ldcg(stats + 0), ent_sum = __ldcg(stats + 1), c_exp = __ldcg(stats + 2),
              c_gen = __ldcg(stats + 3), c_pred = __ldcg(stats + 4);
  const float nanv = __int_as_float(0x7fc00000);
  stats_out[0] = loss_sum * reinterpret_cast<const float*>(meta)[3];  // disc_loss (scaled minibatch mean)
  stats_out[1] = n > 0 ? (c_exp + c_gen) / n : nanv;                  // disc_acc
  stats_out[2] = n_exp >= 1 ? c_exp / n_exp : nanv;                   // disc_acc_expert
  stats_out[3] = c_gen / fmaxf(1.f, n_gen);                           // disc_acc_gen
  stats_out[4] = n > 0 ? ent_sum / n : nanv;                          // disc_entropy
  stats_out[5] = n > 0 ? n_exp / n : nanv;                            // disc_proportion_expert_true
  stats_out[6] = n > 0 ? c_pred / n : nanv;                           // disc_proportion_expert_pred
  stats_out[7] = n_exp;
  stats_out[8] = n_gen;
}

// single block: P <= ~8.5k parameters = a handful of iterations per thread.
__global__ void __launch_bounds__(1024) k_disc_adam(int P, imb_adam opt, float* __restrict__ params,
                                                  float* __restrict__ m, float* __restrict__ v,
                                                  const float* __restrict__ grad, float grad_div,
                                                  const float* __restrict__ stats, const int* __restrict__ meta,
                                                  int64_t* __restrict__ step_io,
                                                  float* __restrict__ stats_out) {
  adam_step(P, opt, params, m, v, grad, grad_div, step_io);
  if (threadIdx.x == 0 && stats_out) write_train_stats(stats, meta, stats_out);
}

// reduce + Adam in one launch (the last minibatch of an update): every block reduces its share of the partials
// like k_disc_reduce; the last block to finish (ticket) runs the optimiser step and the statistics.
__global__ void __launch_bounds__(256) k_disc_reduce_adam(int P, int G, const float* __restrict__ partial,
                                                         float* __restrict__ gacc, float* __restrict__ stats,
                                                         imb_adam opt, float* __restrict__ params,
                                                         float* __restrict__ m, float* __restrict__ v, float grad_div,
                                                         const int* __restrict__ meta, int64_t* __restrict__ step_io,
                                                         float* __restrict__ stats_out,
                                                         unsigned int* __restrict__ ticket) {
  reduce_partials(P, G, partial, gacc, stats, nullptr);
  __threadfence();
  __shared__ bool is_last;
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(ticket, 1u);
    is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  if (threadIdx.x == 0) *ticket = 0u;  // re-arm for the next launch
  adam_step(P, opt, params, m, v, gacc, grad_div, step_io);
  if (threadIdx.x == 0 && stats_out) write_train_stats(stats, meta, stats_out);
}

// ---- preference comparisons: fragment returns -> Boltzmann probability -> cross entropy (+ its gradient) -------------
// Warp per fragment pair: lanes stride over the L time steps (coalesced: a fragment's rewards are contiguous), shuffle
// reduction of the discounted difference, lane-parallel write of the 2 L gradient entries.  The minibatch sums (loss,
// accuracy) are accumulated per CTA and added to the statistics accumulator with one atomic each; a minibatch is a few
// hundred pairs, so the order-dependent rounding of those atomics only touches the logged means (1e-7 relative).
__global__ void __launch_bounds__(256) k_pref_loss(const float* __restrict__ rews, int P, int L,
                                                  const float* __restrict__ prefs, float noise_prob, float discount,
                                                  float threshold, float grad_scale, float* __restrict__ grad_rews,
                                                  float* __restrict__ probs_out, float* __restrict__ stats_acc) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  __shared__ float s_loss[8], s_acc[8];
  float w_loss = 0.f, w_acc = 0.f;
  const float inv_P = 1.0f / (float)P;
  for (int pr = blockIdx.x * nw + warp; pr < P; pr += gridDim.x * nw) {
    const float* r1 = rews + (int64_t)pr * L;
    const float* r2 = rews + ((int64_t)P + pr) * L;
    float s = 0.f;
    if (discount == 1.0f) {
      for (int t = lane; t < L; t += 32) s += r2[t] - r1[t];
    } else {
      for (int t = lane; t < L; t += 32) s = fmaf(powf(discount, (float)t), r2[t] - r1[t], s);
    }
    s = warp_sum(s);
    const bool clipped = s < -threshold || s > threshold;  // th.clip passes the gradient on [min, max] only
    const float d = fminf(fmaxf(s, -threshold), threshold);
    const float ed = expf(d);
    const float m = 1.0f / (1.0f + ed);
    const float p = noise_prob * 0.5f + (1.0f - noise_prob) * m;
    const float y = prefs[pr];
    // F.binary_cross_entropy: logs clamped at -100; backward (p - y) / max(p (1 - p), 1e-12)
    const float lp = fmaxf(logf(p), -100.0f), l1p = fmaxf(log1pf(-p), -100.0f);
    const float loss = -(y * lp + (1.0f - y) * l1p);
    const float dl_dp = (p - y) / fmaxf(p * (1.0f - p), 1e-12f) * inv_P;
    const float dp_dd = -(1.0f - noise_prob) * m * m * ed;  // = -(1 - noise) m (1 - m), without the cancellation in 1 - m
    const float g = clipped ? 0.f : grad_scale * dl_dp * dp_dd;  // d loss / d (returns difference)
    if (grad_rews) {
      float* g1 = grad_rews + (int64_t)pr * L;
      float* g2 = grad_rews + ((int64_t)P + pr) * L;
      for (int t = lane; t < L; t += 32) {
        const float w = discount == 1.0f ? g : g * powf(discount, (float)t);
        g1[t] = -w;
        g2[t] = w;
      }
    }
    if (lane == 0) {
      if (probs_out) probs_out[pr] = p;
      w_loss += loss;
      w_acc += ((p > 0.5f) == (y > 0.5f)) ? 1.f : 0.f;
    }
  }
  if (!stats_acc) return;
  if (lane == 0) {
    s_loss[warp] = w_loss;
    s_acc[warp] = w_acc;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, b = 0.f;
    for (int w = 0; w < nw; ++w) {
      a += s_loss[w];
      b += s_acc[w];
    }
    atomicAdd(stats_acc + 0, a * inv_P);
    atomicAdd(stats_acc + 1, b * inv_P);
    if (blockIdx.x == 0) atomicAdd(stats_acc + 2, 1.0f);
  }
}

__global__ void k_state_add(int64_t* state, int idx, int64_t v) { state[idx] += v; }

// statistics -> host-mapped pinned memory, followed by a sequence word (system-scope fence in between): the host polls
// the word instead of issuing a D2H copy and synchronising on an event (one PCIe posted write burst per update)
__global__ void k_stats_publish(const float* __restrict__ stats_dev, int n, float* host, const int64_t* __restrict__ state,
                                int state_idx) {
  const int lane = threadIdx.x;
  if (lane < n) host[lane] = stats_dev[lane];
  __threadfence_system();
  __syncwarp();
  if (lane == 0) reinterpret_cast<volatile int*>(host)[15] = (int)state[state_idx];
}
__global__ void k_set_meta(int* meta, int G, int64_t n, int64_t n_expert, float loss_scale) {
  meta[0] = G;
  meta[1] = (int)n;
  meta[2] = (int)n_expert;
  reinterpret_cast<float*>(meta)[3] = loss_scale;
}

// ---- forward only (reward relabel / predict) ---------------------------------------------------
// thread per row straight from global memory (coalesced over rows for each feature).
template <int H>
__global__ void __launch_bounds__(NT) k_reward_fwd(const DiscLaunch L, const float* __restrict__ params,
                                                  const float* __restrict__ batch, int64_t ld, int64_t n,
                                                  int out_mode, float* __restrict__ out, int img1_off, int xn_off,
                                                  int xn_ld) {
  extern __shared__ __align__(128) float smem[];
  float* img[MAX_PASS] = {smem, smem + img1_off, smem + img1_off};
  float* XN = smem + xn_off;
  const int tid = threadIdx.x;
  load_mlp<H>(img[0], L.pass[0], params);
  float* mean2 = nullptr;
  float* istd2 = nullptr;
  if (L.npass == 3) {
    load_mlp<H>(img[1], L.pass[1], params);
    const int din = L.pass[2].din;
    mean2 = img[1] + MlpSm<H>::size(din);
    istd2 = mean2 + IMB_MAX_DIN;
    for (int i = tid; i < din; i += NT) {
      if (L.pass[2].has_norm) {
        mean2[i] = L.pass[2].norm[i];
        istd2[i] = 1.0f / sqrtf(L.pass[2].norm[din + i] + L.pass[2].eps);
      } else {
        mean2[i] = 0.f;
        istd2[i] = 1.f;
      }
    }
  }
  __syncthreads();
  float h1[H], h2[H];
  for (int64_t row = (int64_t)blockIdx.x * NT + tid; row < n; row += (int64_t)gridDim.x * NT) {
    const float done = (L.done_slot >= 0) ? batch[(int64_t)L.stage_row[L.done_slot] * ld + row] : 0.f;
    float logit = 0.f;
    for (int p = 0; p < L.npass; ++p) {
      const PassDesc& P = L.pass[p];
      const float* mean = (p == 2) ? mean2 : img[p] + MlpSm<H>::mean_off(P.din);
      const float* istd = (p == 2) ? istd2 : img[p] + MlpSm<H>::istd_off(P.din);
      float* xn = XN + tid * xn_ld;
      for (int k = 0; k < P.din; ++k)
        xn[k] = (batch[(int64_t)L.stage_row[P.in_slot[k]] * ld + row] - mean[k]) * istd[k];
      const float o = mlp_forward_row<H, false>(img[p], P, xn, h1, h2);
      logit = fmaf(pass_coef(P.coef_kind, L.gamma, done), o, logit);
    }
    if (out_mode >= 1 && L.logp_slot >= 0) logit -= batch[(int64_t)L.stage_row[L.logp_slot] * ld + row];
    out[row] = (out_mode == 2) ? softplus_f(logit) : logit;
  }
}

// ---- NormalizedRewardNet.predict_processed over consecutive env steps ---------------------------
// single CTA: for t in steps: normalise the E rewards of step t with the running stats, then merge
// step t's raw rewards into the stats (reward_nets.py:637-671 + networks.py:111-134).
__global__ void __launch_bounds__(1024) k_reward_norm_scan(float* __restrict__ rews, int64_t E, int64_t T,
                                                          int64_t step_stride, int64_t env_stride,
                                                          float* __restrict__ mv, int32_t* __restrict__ count,
                                                          float eps, int update) {
  __shared__ float red[64];
  __shared__ float bc[2];
  float mean = mv[0], var = mv[1];
  int32_t cnt = *count;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = blockDim.x >> 5;
  for (int64_t t = 0; t < T; ++t) {
    float* r = rews + t * step_stride;
    const float istd = 1.0f / sqrtf(var + eps);
    float s = 0.f;
    for (int64_t e = tid; e < E; e += blockDim.x) s += r[e * env_stride];
    s = warp_sum(s);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    if (tid == 0) {
      float a = 0.f;
      for (int w = 0; w < nw; ++w) a += red[w];
      bc[0] = a / (float)E;
    }
    __syncthreads();
    const float bmean = bc[0];
    float m2 = 0.f;
    for (int64_t e = tid; e < E; e += blockDim.x) {
      const float v = r[e * env_stride];
      const float dlt = v - bmean;
      m2 = fmaf(dlt, dlt, m2);
      r[e * env_stride] = (v - mean) * istd;  // normalise with the stats BEFORE this step's update
    }
    m2 = warp_sum(m2);
    if (lane == 0) red[32 + warp] = m2;
    __syncthreads();
    if (tid == 0) {
      float a = 0.f;
      for (int w = 0; w < nw; ++w) a += red[32 + w];
      bc[1] = a / (float)E;
    }
    __syncthreads();
    if (update) {
      fold_moments(mean, var, (float)cnt, bmean, bc[1], (float)E);
      cnt += (int32_t)E;
    }
    __syncthreads();
  }
  if (tid == 0 && update) {
    mv[0] = mean;
    mv[1] = var;
    *count = cnt;
  }
}

// ---- host-side launch helpers -----------------------------------------------------------------
template <int H>
struct SmemPlan {
  int img1_off, xn_off, xn_ld, total_floats;
};
template <int H>
SmemPlan<H> plan_smem(const DiscLaunch& L, bool) {
  SmemPlan<H> s;
  auto al = [](int x) { return (x + 31) / 32 * 32; };
  int o = al(MlpSm<H>::size(L.pass[0].din));
  s.img1_off = o;
  if (L.npass == 3) o += al(MlpSm<H>::size(L.pass[1].din) + 2 * IMB_MAX_DIN);
  int maxdin = 0;
  for (int p = 0; p < L.npass; ++p) maxdin = L.pass[p].din > maxdin ? L.pass[p].din : maxdin;
  s.xn_ld = maxdin | 1;
  s.xn_off = o;
  o += al(NT * s.xn_ld);
  s.total_floats = o;
  return s;
}

inline int pick_H(const DiscLaunch& L) {
  int h = 0;
  for (int p = 0; p < L.npass; ++p) {
    if (L.pass[p].n_hidden >= 1 && L.pass[p].h1 > h) h = L.pass[p].h1;
    if (L.pass[p].n_hidden >= 2 && L.pass[p].h2 > h) h = L.pass[p].h2;
  }
  return h <= 32 ? 32 : 64;
}

}  // namespace

extern "C" int64_t imb_disc_workspace_floats(const imb_disc_desc* d) { return ws_layout(d->n_params).total; }

// RunningNorm updates of the jobs in J from batch rows [0, n): one launch when the chunk table holds every job's chunks,
// else one launch per job, in job order
static int norm_stats(const NormJobs& J, const float* batch, int64_t ld, int64_t n, float* defer, int defer_cap,
                      float* ws, const WsLayout& w, cudaStream_t st) {
  // chunk size: small enough to fill the GPU at the tuned batch sizes (16 384 rows -> 128 CTAs), larger for the
  // multi-million-row sweeps so the chunk table stays bounded
  const int chunk_rows = n <= (int64_t)128 * 2048 ? 128 : NORM_CHUNK;
  const int chunks = (int)((n + chunk_rows - 1) / chunk_rows);
  IMB_REQUIRE(chunks >= 1 && chunks <= MAXCHUNKS, "norm update: n=%lld out of range", (long long)n);
  float* part = ws + w.normpart;
  unsigned int* ticket = reinterpret_cast<unsigned int*>(ws + w.ticket);
  if ((int64_t)chunks * J.njobs <= MAXCHUNKS) {
    k_norm_stats<<<dim3(chunks, J.njobs), 256, 0, st>>>(J, batch, ld, n, chunk_rows, part, ticket, defer, defer_cap);
    IMB_CHECK_LAUNCH("k_norm_stats");
    return 0;
  }
  for (int j = 0; j < J.njobs; ++j) {
    NormJobs one{};
    one.njobs = 1;
    one.job[0] = J.job[j];
    k_norm_stats<<<chunks, 256, 0, st>>>(one, batch, ld, n, chunk_rows, part, ticket, defer, defer_cap);
    IMB_CHECK_LAUNCH("k_norm_stats");
  }
  return 0;
}

extern "C" int imb_disc_norm_update(const imb_disc_desc* d, const float* batch, int64_t ld, int64_t n,
                                    float* norm_state, int32_t* norm_count, float* ws, void* stream) {
  IMB_REQUIRE(n >= 1, "norm update needs n >= 1");
  const WsLayout w = ws_layout(d->n_params);
  DiscLaunch L;
  if (int rc = build_launch(d, norm_state, nullptr, L)) return rc;
  // the base normaliser, then for a shaped net the potential's with next_obs and then with obs (reference order, both on
  // the same RunningNorm; the Phi(s') pass of the forward reads the snapshot taken between the two)
  NormJobs J{};
  auto add = [&](const imb_mlp& m, int pass, float* snap) {
    NormJob& j = J.job[J.njobs++];
    j.din = m.din;
    for (int k = 0; k < m.din; ++k) j.row[k] = L.stage_row[L.pass[pass].in_slot[k]];
    j.rmv = norm_state + m.norm_off;
    j.cnt = norm_count + m.count_idx;
    j.snap = snap;
  };
  if (d->base.has_norm) add(d->base, 0, nullptr);
  if (d->shaped && d->potential.has_norm) {
    add(d->potential, 1, ws + w.snap);
    add(d->potential, 2, nullptr);
  }
  if (J.njobs == 0) return 0;
  return norm_stats(J, batch, ld, n, nullptr, 0, ws, w, (cudaStream_t)stream);
}

extern "C" int imb_norm_batch_stats(const imb_disc_desc* d, const float* batch, int64_t ld, int64_t n, int row0, int din,
                                    float* norm_state, int32_t* norm_count, float* defer, int defer_cap, float* ws,
                                    void* stream) {
  IMB_REQUIRE(n >= 1 && din >= 1 && din <= IMB_MAX_DIN, "norm batch stats: bad sizes");
  IMB_REQUIRE(defer == nullptr || defer_cap >= 1, "norm batch stats: defer_cap");
  NormJobs J{};
  J.njobs = 1;
  J.job[0].din = din;
  for (int k = 0; k < din; ++k) J.job[0].row[k] = (short)(row0 + k);
  J.job[0].rmv = norm_state;
  J.job[0].cnt = norm_count;
  return norm_stats(J, batch, ld, n, defer, defer_cap, ws, ws_layout(d->n_params), (cudaStream_t)stream);
}

extern "C" int imb_norm_fold(int din, float* defer, float* norm_state, int32_t* norm_count, int n_slots, void* stream) {
  IMB_REQUIRE(din >= 1 && din <= IMB_MAX_DIN, "norm fold: din");
  k_norm_fold<<<1, 64, 0, (cudaStream_t)stream>>>(din, defer, norm_state, norm_count, n_slots);
  IMB_CHECK_LAUNCH("k_norm_fold");
  return 0;
}

// multi-GPU: the statistics of the last minibatch were summed over the ranks -> the row counts k_disc_adam divides by
// are the global ones
__global__ void k_set_rows(int* meta, int64_t n, int64_t n_expert) {
  meta[1] = (int)n;
  meta[2] = (int)n_expert;
}
extern "C" int imb_disc_set_rows(const imb_disc_desc* d, float* ws, int64_t n, int64_t n_expert, void* stream) {
  const WsLayout w = ws_layout(d->n_params);
  k_set_rows<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<int*>(ws + w.meta), n, n_expert);
  IMB_CHECK_LAUNCH("k_set_rows");
  return 0;
}

extern "C" int imb_stats_publish(const float* stats_dev, int n, float* host_mapped, const int64_t* state, int state_idx,
                                 void* stream) {
  IMB_REQUIRE(n >= 1 && n <= 15 && state_idx >= 0 && state_idx < IMB_ST_WORDS, "stats publish: bad sizes");
  k_stats_publish<<<1, 32, 0, (cudaStream_t)stream>>>(stats_dev, n, host_mapped, state, state_idx);
  IMB_CHECK_LAUNCH("k_stats_publish");
  return 0;
}

struct TPlan {
  int JP, KP, img_sz, aw_off, st_off, xn_off, t_off, v_off, nsl, total;
};
static TPlan plan_tiled(const DiscLaunch& L, int R) {
  TPlan t;
  auto al = [](int x) { return (x + 31) / 32 * 32; };
  const int RS = R + TILE_PAD;
  int h = 1, dmax = 1;
  for (int p = 0; p < L.npass; ++p) {
    if (L.pass[p].n_hidden >= 1 && L.pass[p].h1 > h) h = L.pass[p].h1;
    if (L.pass[p].n_hidden >= 2 && L.pass[p].h2 > h) h = L.pass[p].h2;
    if (L.pass[p].din > dmax) dmax = L.pass[p].din;
  }
  t.JP = h <= 32 ? 32 : 64;
  t.KP = dmax <= 32 ? 32 : 64;
  t.img_sz = al(TImg::size(dmax, t.JP));
  int o = L.npass * t.img_sz;
  t.nsl = (t.JP == 32 && R == 256) ? 4 : 2;  // row slices of the weight-gradient phase (>= 2: slice 1 holds dwf)
  t.aw_off = o;
  o += al(t.nsl * L.P);
  t.st_off = o;
  o += al(L.nstage * RS);
  t.xn_off = o;
  o += al(t.KP * RS);
  t.t_off = o;
  o += al(3 * t.JP * RS);
  t.v_off = o;
  o += al(5 * R);
  t.total = o;
  return t;
}

template <int R>
static int launch_fwdbwd(const DiscLaunch& L, const TPlan& t, const float* params, const float* batch, int64_t ld,
                         int64_t n, int64_t n_expert, float loss_scale, const float* grad_out, float* logits_out,
                         float* ws, const WsLayout& w, cudaStream_t st, int ctas_per_sm) {
  const size_t bytes = (size_t)t.total * 4;
  static size_t attr_bytes = 0;
  if (bytes > attr_bytes) {
    cudaError_t e = cudaFuncSetAttribute(k_disc_fwdbwd<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) IMB_FAIL(-2, "cudaFuncSetAttribute(%zu): %s", bytes, cudaGetErrorString(e));
    attr_bytes = bytes;
  }
  const int64_t ntiles = (n + R - 1) / R;
  int64_t G = (int64_t)imb_num_sms() * ctas_per_sm;
  if (G > MAXG) G = MAXG;
  if (G > ntiles) G = ntiles;
  k_disc_fwdbwd<R><<<(int)G, R, bytes, st>>>(L, params, batch, ld, n, n_expert, loss_scale, grad_out, logits_out,
                                               ws + w.partial, reinterpret_cast<int*>(ws + w.meta), t.JP, t.KP, t.img_sz, t.aw_off, t.st_off, t.xn_off,
                                               t.t_off, t.v_off, t.nsl);
  IMB_CHECK_LAUNCH("k_disc_fwdbwd");
  return (int)G;
}

// host mirror of the grid chosen by the last fwd/bwd launch (stream-ordered use only)
static thread_local int g_last_grid = 0;

extern "C" int imb_disc_fwd_bwd(const imb_disc_desc* d, const float* params, const float* norm_state,
                                const float* batch, int64_t ld, int64_t n, int64_t n_expert, float loss_scale,
                                const float* grad_out, float* logits_out, int flags, float* ws, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  IMB_REQUIRE(n >= 1, "fwd_bwd needs n >= 1");
  IMB_REQUIRE(ld % 4 == 0 && ld >= (n + IMB_TILE_ROWS - 1) / IMB_TILE_ROWS * IMB_TILE_ROWS,
              "batch leading dimension must cover n rounded up to %d rows", IMB_TILE_ROWS);
  const WsLayout w = ws_layout(d->n_params);
  DiscLaunch L;
  // in training mode the Phi(s') pass uses the stats snapshot taken between the two norm updates
  const bool snap = d->shaped && d->potential.has_norm && (flags & IMB_F_TRAIN_NORM);
  if (int rc = build_launch(d, norm_state, snap ? ws + w.snap : nullptr, L)) return rc;
  if (flags & IMB_F_ZERO_GRAD) {
    cudaError_t e = cudaMemsetAsync(ws + w.gacc, 0, sizeof(float) * d->n_params, st);
    if (e != cudaSuccess) IMB_FAIL(-2, "memset: %s", cudaGetErrorString(e));
  }
  // Tensor-core path (tcgen05 / TMEM, 3xTF32 split) whenever the network shape fits it
  if (!(flags & IMB_F_NO_TENSOR) && tc_applicable(L)) {
    const TcPlan T = tc_plan(L);
    const size_t bytes = (size_t)T.total * 4 + 1024;
    static bool attr_set = false;
    static int cw = 8;
    if (!attr_set) {
      if (const char* e = getenv("IMB_TC_CW")) cw = atoi(e) == 16 ? 16 : 8;  // (tuning knob: columns per epilogue thread)
      cudaError_t e1 = cudaFuncSetAttribute(k_disc_fwdbwd_tc<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IMB_SMEM_MAX);
      cudaError_t e2 = cudaFuncSetAttribute(k_disc_fwdbwd_tc<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)IMB_SMEM_MAX);
      if (e1 != cudaSuccess || e2 != cudaSuccess) IMB_FAIL(-2, "cudaFuncSetAttribute(tc): %s", cudaGetErrorString(e1 != cudaSuccess ? e1 : e2));
      attr_set = true;
    }
    IMB_REQUIRE(bytes <= IMB_SMEM_MAX, "tensor-core disc kernel: %zu B of shared memory", bytes);
    const int64_t ntiles = (n + 127) / 128;
    int64_t Gt = imb_num_sms();
    if (Gt > MAXG) Gt = MAXG;
    if (Gt > ntiles) Gt = ntiles;
    if (cw == 8)
      k_disc_fwdbwd_tc<8><<<(int)Gt, TcCfg<8>::THREADS, bytes, st>>>(L, T, params, batch, ld, n, n_expert, loss_scale, grad_out, logits_out,
                                                        ws + w.partial, reinterpret_cast<int*>(ws + w.meta),
                                                        part_stride(d->n_params));
    else
      k_disc_fwdbwd_tc<16><<<(int)Gt, TcCfg<16>::THREADS, bytes, st>>>(L, T, params, batch, ld, n, n_expert, loss_scale, grad_out, logits_out,
                                                         ws + w.partial, reinterpret_cast<int*>(ws + w.meta),
                                                         part_stride(d->n_params));
    IMB_CHECK_LAUNCH("k_disc_fwdbwd_tc");
    g_last_grid = (int)Gt;
    return 0;
  }
  // Preferred: 128-row tiles with TWO resident CTAs per SM (independent CTAs overlap each other's
  // barriers and epilogues); else one 256-row CTA; else one 128-row CTA.
  TPlan t256 = plan_tiled(L, 256), t128 = plan_tiled(L, 128);
  int G;
  if (2 * ((size_t)t128.total * 4 + 1024 + 512) <= 228 * 1024)
    G = launch_fwdbwd<128>(L, t128, params, batch, ld, n, n_expert, loss_scale, grad_out, logits_out, ws, w, st, 2);
  else if ((size_t)t256.total * 4 <= IMB_SMEM_MAX && n > 128)
    G = launch_fwdbwd<256>(L, t256, params, batch, ld, n, n_expert, loss_scale, grad_out, logits_out, ws, w, st, 1);
  else if ((size_t)t128.total * 4 <= IMB_SMEM_MAX)
    G = launch_fwdbwd<128>(L, t128, params, batch, ld, n, n_expert, loss_scale, grad_out, logits_out, ws, w, st, 1);
  else
    IMB_FAIL(-1, "discriminator too large for the fused kernel (%zu B of shared memory)", (size_t)t128.total * 4);
  if (G < 0) return G;
  g_last_grid = G;
  return 0;
}

// grid of k_disc_reduce / k_disc_reduce_adam: a warp per parameter and per statistic, at most two 256-thread blocks per SM
static int reduce_blocks(int P) {
  const int blocks = ((P + 5) * 32 + 255) / 256;
  return blocks < 2 * imb_num_sms() ? blocks : 2 * imb_num_sms();
}

extern "C" int imb_disc_reduce(const imb_disc_desc* d, float* ws, float* grad_out_flat, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const WsLayout w = ws_layout(d->n_params);
  IMB_REQUIRE(g_last_grid > 0, "imb_disc_reduce called before imb_disc_fwd_bwd");
  const int P = d->n_params;
  k_disc_reduce<<<reduce_blocks(P), 256, 0, st>>>(P, g_last_grid, ws + w.partial, ws + w.gacc, ws + w.stats,
                                                   grad_out_flat);
  IMB_CHECK_LAUNCH("k_disc_reduce");
  return 0;
}

extern "C" int imb_disc_adam(const imb_disc_desc* d, const imb_adam* opt, float* params, float* exp_avg,
                             float* exp_avg_sq, const float* grad_flat_or_null, float grad_div, float* ws,
                             int64_t* state, float* stats_out, void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const WsLayout w = ws_layout(d->n_params);
  const int P = d->n_params;
  const float* grad = grad_flat_or_null ? grad_flat_or_null : ws + w.gacc;
  // loss statistic: sum * loss_scale recorded by the last fwd/bwd launch (meta[3])
  k_disc_adam<<<1, 1024, 0, st>>>(P, *opt, params, exp_avg, exp_avg_sq, grad, grad_div, ws + w.stats,
                                  reinterpret_cast<const int*>(ws + w.meta), state + IMB_ST_DISC_STEP, stats_out);
  IMB_CHECK_LAUNCH("k_disc_adam");
  return 0;
}

extern "C" int imb_disc_reduce_adam(const imb_disc_desc* d, const imb_adam* opt, float* params, float* exp_avg,
                                    float* exp_avg_sq, float grad_div, float* ws, int64_t* state, float* stats_out,
                                    void* stream) {
  cudaStream_t st = (cudaStream_t)stream;
  const WsLayout w = ws_layout(d->n_params);
  IMB_REQUIRE(g_last_grid > 0, "imb_disc_reduce_adam called before imb_disc_fwd_bwd");
  const int P = d->n_params;
  k_disc_reduce_adam<<<reduce_blocks(P), 256, 0, st>>>(P, g_last_grid, ws + w.partial, ws + w.gacc, ws + w.stats, *opt,
                                                        params, exp_avg, exp_avg_sq, grad_div,
                                                        reinterpret_cast<const int*>(ws + w.meta),
                                                        state + IMB_ST_DISC_STEP, stats_out,
                                                        reinterpret_cast<unsigned int*>(ws + w.ticket) + 8);
  IMB_CHECK_LAUNCH("k_disc_reduce_adam");
  return 0;
}

template <int H>
static int launch_fwd(const DiscLaunch& L, const float* params, const float* batch, int64_t ld, int64_t n,
                      int out_mode, float* out, cudaStream_t st) {
  const SmemPlan<H> s = plan_smem<H>(L, false);
  const size_t bytes = (size_t)s.total_floats * 4;
  IMB_REQUIRE(bytes <= IMB_SMEM_MAX, "reward net too large for the fused kernel (%zu B smem)", bytes);
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(k_reward_fwd<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, IMB_SMEM_MAX);
    if (e != cudaSuccess) IMB_FAIL(-2, "cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  int64_t blocks = (n + NT - 1) / NT;
  const int64_t cap = (int64_t)imb_num_sms() * 4;
  if (blocks > cap) blocks = cap;
  k_reward_fwd<H><<<(int)blocks, NT, bytes, st>>>(L, params, batch, ld, n, out_mode, out, s.img1_off, s.xn_off,
                                                   s.xn_ld);
  IMB_CHECK_LAUNCH("k_reward_fwd");
  return 0;
}

extern "C" int imb_reward_forward(const imb_disc_desc* d, const float* params, const float* norm_state,
                                  const float* batch, int64_t ld, int64_t n, int out_mode, float* out,
                                  void* stream) {
  if (n <= 0) return 0;
  DiscLaunch L;
  imb_disc_desc dd = *d;
  if (out_mode == 0) dd.subtract_logp = 0;
  if (int rc = build_launch(&dd, norm_state, nullptr, L)) return rc;
  return (pick_H(L) == 32) ? launch_fwd<32>(L, params, batch, ld, n, out_mode, out, (cudaStream_t)stream)
                           : launch_fwd<64>(L, params, batch, ld, n, out_mode, out, (cudaStream_t)stream);
}

extern "C" int imb_reward_norm_scan(float* rews, int64_t n_envs, int64_t n_steps, int64_t step_stride,
                                    int64_t env_stride, float* norm_state2, int32_t* norm_count, float eps,
                                    int update_stats, void* stream) {
  IMB_REQUIRE(n_envs >= 1 && n_steps >= 0, "bad sizes");
  if (n_steps == 0) return 0;
  int threads = 1024;
  while (threads > 32 && threads / 2 >= n_envs) threads /= 2;
  k_reward_norm_scan<<<1, threads, 0, (cudaStream_t)stream>>>(rews, n_envs, n_steps, step_stride, env_stride,
                                                              norm_state2, norm_count, eps, update_stats);
  IMB_CHECK_LAUNCH("k_reward_norm_scan");
  return 0;
}

extern "C" int imb_pref_loss(const float* rews, int64_t n_pairs, int32_t frag_len, const float* prefs, float noise_prob,
                             float discount, float threshold, float grad_scale, float* grad_rews, float* probs_out,
                             float* stats_acc, int32_t stats_slot, void* stream) {
  IMB_REQUIRE(n_pairs >= 1 && n_pairs < (1ll << 30) && frag_len >= 1, "imb_pref_loss: bad sizes");
  IMB_REQUIRE(stats_slot >= 0, "imb_pref_loss: bad statistics slot");
  int64_t blocks = (n_pairs + 7) / 8;
  if (blocks > 4 * imb_num_sms()) blocks = 4 * imb_num_sms();
  k_pref_loss<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(rews, (int)n_pairs, frag_len, prefs, noise_prob, discount,
                                                             threshold, grad_scale, grad_rews, probs_out,
                                                             stats_acc ? stats_acc + 4 * stats_slot : nullptr);
  IMB_CHECK_LAUNCH("k_pref_loss");
  return 0;
}

extern "C" int imb_state_init(int64_t* state, void* stream) {
  cudaError_t e = cudaMemsetAsync(state, 0, sizeof(int64_t) * IMB_ST_WORDS, (cudaStream_t)stream);
  if (e != cudaSuccess) IMB_FAIL(-2, "memset: %s", cudaGetErrorString(e));
  return 0;
}
