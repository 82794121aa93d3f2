// plan.cu -- the launch policy of the fused step (prologue kernel -> marching kernel -> epilogue kernel): which kernel
// instance runs, how its work is cut into warp tasks and how the prologue's grid is laid out.  Host code only; the
// launchers take the plan as it is.  The numbers were calibrated on B200 (DESIGN.md §4, profiles/README.md).
#include <stdlib.h>

#include "common.cuh"
#include "kernels.h"

namespace {

// Test hooks that force a launch variant (tests/test_gpu_parity.py); `unset` when the variable is not set.
//   SFM_HSEG       task height of either marching kernel
//   SFM_SSIM_NW    1 or 2 warps per SSIM CTA
//   SFM_SSIM_SREC  SSIM forward records in shared memory (1) or registers (0)
// A value the plan's mode has no kernel instance for is ignored.
int test_hook(const char* name, int unset) {
  const char* e = getenv(name);
  return e ? atoi(e) : unset;
}

// Task table of either marching kernel: scale s is cut into ceil(rows[s] / hseg) segments per snippet and, with
// `strips`, each segment into nstrip[s] column strips.
SfmTaskTable task_table(int B, int ns, int hseg, const int* nstrip, const int* rows, bool strips) {
  SfmTaskTable t{};
  t.hseg = hseg;
  int total = 0;
  for (int s = 0; s < SFM_MAX_SCALES; ++s) {
    t.task_begin[s] = total;
    if (s < ns) {
      t.nstrip[s] = nstrip[s];
      t.nseg[s] = (rows[s] + hseg - 1) / hseg;
      total += B * (strips ? nstrip[s] : 1) * t.nseg[s];
    } else {
      t.nstrip[s] = t.nseg[s] = 1;
    }
  }
  t.task_begin[SFM_MAX_SCALES] = total;
  return t;
}

// L1 marching kernel: a task is hseg runs of 32 pixels; the task length is halved until there are enough warps
// (~12 per scheduler), but not below 4 runs, where the prologue / flush of a task dominates (measured).
void plan_l1(SfmStepPlan& q, const SfmDesc* d, int num_sms) {
  int runs[SFM_MAX_SCALES];
  for (int s = 0; s < d->n_scales; ++s) runs[s] = (sfm_step_h(d, s) * sfm_step_w(d, s) + 31) / 32;
  const long long want_warps = (long long)num_sms * 4 * 12;
  int hseg = 32;
  while (task_table(d->B, d->n_scales, hseg, runs, runs, false).task_begin[SFM_MAX_SCALES] < want_warps && hseg > 4) hseg >>= 1;
  const int forced = test_hook("SFM_HSEG", 0);
  if (forced > 0) hseg = forced;
  q.tasks = task_table(d->B, d->n_scales, hseg, runs, runs, false);
}

// Instructions a SSIM task of h rows issues per source, in full row steps: it marches h + 4 steps and runs refill + A + B
// on all of them, C + D on h + 2 and E + F on h (ssim_march.cuh, RowStages).  The stage shares of a full step are
// those of the SASS of the row loop (tools/sass_loop.py on instances whose loop runs only A + B, or only A..D): 0.33 /
// 0.22 / 0.45 in the register-record instance, 0.40 / 0.17 / 0.43 in the shared-memory-record one.
double ssim_task_steps(int h) { return 0.35 * (h + 4) + 0.2 * (h + 2) + 0.45 * h; }

// SSIM marching kernel.  Task height (rows per strip segment), cost model calibrated on B200 (tools/time_graph.py
// sweeps, DESIGN.md): a task costs ssim_task_steps(hseg) row steps per source; up to SFM_SSIM_MIN_WARPS single-warp
// CTAs are resident per SM, i.e. 3 per scheduler.  Above one wave the time is waves x steps; below one wave the
// busiest scheduler holds w = ceil(tasks / schedulers) warps and runs them at a relative issue efficiency of
// 0.66 / 0.9 / 1.0 for w = 1 / 2 / 3 (a lone warp cannot hide its own latencies).
// Example cfg2 (B=4, 128x416, register records): NW = 2, hseg 19 -> 588 tasks, w = 1, 20.8 steps: cost 44.2;
// hseg 20 -> 588 tasks, 21.8 steps: 46.3; shared-memory records, hseg 13 -> 824 tasks, w = 2, 14.8 steps: 46.6; NW = 1,
// hseg 10 -> 1084 tasks, w = 2, 2 x 11.8 steps: 47.7.
// With two sources and a sub-wave grid the sources can also be split over the two warps of a CTA (NW = 2): a task
// is then one pass long and there are twice as many warps, so the same occupancy is reached with taller segments
// (fewer halo rows); the per-row CTA barrier is charged 5 %.
void plan_ssim(SfmStepPlan& q, const SfmDesc* d, int num_sms) {
  const int B = d->B, S = d->S, ns = d->n_scales;
  int hs[SFM_MAX_SCALES], strips[SFM_MAX_SCALES];
  for (int s = 0; s < ns; ++s) {
    hs[s] = sfm_step_h(d, s);
    strips[s] = (sfm_step_w(d, s) + SFM_SSIM_IW - 1) / SFM_SSIM_IW;
  }
  // the register-record and source-split instances exist for the plain gradient mode only (no image gradients, no
  // per-pixel terms)
  const bool may_reg = q.grad && !q.debug && !q.raw && !q.img && !q.pix;
  const bool may_split = may_reg && S == 2;
  int hseg = 64, nw = 1;
  bool srec = true;
  const long long sched = (long long)num_sms * 4, slots = (long long)num_sms * SFM_SSIM_MIN_WARPS;
  const long long slots_reg = (long long)num_sms * SFM_SSIM_REG_MIN_WARPS;
  double best = 1e300;
  for (int var = 0; var <= (may_reg ? 1 : 0); ++var)
    for (int cand = 1; cand <= (may_split ? 2 : 1); ++cand)
      for (int h = 8; h <= 64; ++h) {
        const long long n = task_table(B, ns, h, strips, hs, true).task_begin[SFM_MAX_SCALES];
        const long long warps = n * cand;
        const double rows = ssim_task_steps(h) * (cand == 1 ? S : 1) * (cand == 1 ? 1.0 : 1.05);
        double cost;
        if (var == 1) {
          // register-record instances: 2 warps per scheduler at most, 9 % faster per row; only while the whole grid is
          // resident at once (above that the shared-memory instances' third warp per scheduler wins: measured at cfg5)
          if (warps > slots_reg) continue;
          const long long w = (warps + sched - 1) / sched;
          cost = 0.91 * rows * (double)w / (w <= 1 ? 0.66 : 0.9);
        } else if (warps > slots) {
          cost = rows * 3.0 * (double)((warps + slots - 1) / slots);
        } else {
          const long long w = (warps + sched - 1) / sched;
          cost = rows * (double)w / (w <= 1 ? 0.66 : w == 2 ? 0.9 : 1.0);
        }
        if (cost < best || (cost == best && cand == nw)) { best = cost; hseg = h; nw = cand; srec = (var == 0); }
      }
  if (srec && nw == 1) {
    // Grids of many waves: the time follows the total number of row steps (measured at cfg5 before the stage schedule
    // of RowStages: 64 / 86 / 128 rows per segment -> 934 / 933 / 912 us for 276 / 276 / 270 row steps per strip), so
    // a taller segment -- fewer halo rows, fewer task flushes -- is taken when it saves at least 1 % of the steps and
    // still leaves three waves of tasks.
    auto work = [&](int h, long long* n_out) {
      long long n = 0;
      double wk = 0.0;
      for (int s = 0; s < ns; ++s) {
        const long long st = (long long)B * strips[s];
        const int full = hs[s] / h, rem = hs[s] - full * h;
        n += st * (full + (rem ? 1 : 0));
        wk += (double)st * (full * ssim_task_steps(h) + (rem ? ssim_task_steps(rem) : 0.0));
      }
      *n_out = n;
      return wk;
    };
    long long n0 = 0;
    double w0 = work(hseg, &n0);
    if (n0 > 3 * slots)
      for (int h2 : {96, 128, 192, 256}) {
        long long n2 = 0;
        const double w2 = work(h2, &n2);
        if (n2 >= 3 * slots && w2 < 0.99 * w0) { hseg = h2; w0 = w2; }
      }
  }
  const int forced_h = test_hook("SFM_HSEG", 0), forced_nw = test_hook("SFM_SSIM_NW", -1);
  const int forced_srec = test_hook("SFM_SSIM_SREC", -1);
  if (forced_h > 0) hseg = forced_h;
  if (forced_nw == 1 || (forced_nw == 2 && may_split)) nw = forced_nw;
  if (forced_srec == 1 || (forced_srec == 0 && may_reg)) srec = forced_srec != 0;
  q.nw = nw;
  q.srec = srec;
  q.tasks = task_table(B, ns, hseg, strips, hs, true);
}

// Second-order smoothness tasks of the prologue: their segment height comes from sfm_smooth_plan, which the workspace
// layout shares, so it does not depend on the device.
void plan_smooth(SfmSmoothParams& m, const SfmDesc* d) {
  m.ns = d->n_scales;
  sfm_smooth_plan(d->B, d->n_scales, d->H, d->W, &m.hseg);
  int total = 0;
  for (int s = 0; s < SFM_MAX_SCALES; ++s) {
    m.tile_begin[s] = total;
    if (s < d->n_scales) {
      m.h[s] = d->H >> s;
      m.w[s] = d->W >> s;
      m.tiles_x[s] = (m.w[s] + SFM_SMOOTH_IW - 1) / SFM_SMOOTH_IW;
      m.tiles_y[s] = (m.h[s] + m.hseg - 1) / m.hseg;
      total += d->B * m.tiles_x[s] * m.tiles_y[s];
    } else {
      m.tiles_x[s] = m.tiles_y[s] = 1;
    }
  }
  m.tile_begin[SFM_MAX_SCALES] = total;
  m.n_tasks = total;
  m.n_ctas = (total + 7) / 8;
}

int pyramid_ctas(const SfmDesc* d, int band) { return d->B * (1 + d->S) * ((d->H + band - 1) / band); }

}  // namespace

// Full-resolution rows per pyramid CTA of the prologue: 8, or 4 / 2 while the grid would not fill the chip twice (small
// batches are latency-bound there: a thread walks band/2 rows of scale 1, so shorter bands mean shorter walks).
int sfm_plan_band(const SfmDesc* d) {
  int band = 8;
  while (band > 2 && pyramid_ctas(d, band) < SFM_REF_SMS * 2) band >>= 1;
  return band;
}

SfmStepPlan sfm_plan_step(const SfmDesc* d, int mode, int num_sms) {
  SfmStepPlan q{};
  q.ssim = (mode & SFM_MODE_SSIM) != 0;
  q.exp = (mode & SFM_MODE_EXP) != 0;
  q.grad = (mode & SFM_MODE_GRAD) != 0;
  q.debug = (mode & SFM_MODE_DEBUG) != 0;
  q.img = q.grad && !q.debug && (mode & SFM_MODE_IMG) != 0;
  q.pix = !q.debug && !q.img && (mode & SFM_MODE_PIX) != 0;
  q.minrep = q.pix && (mode & SFM_MODE_MINREP) != 0;
  // under SFM_FLAG_FULL_RES_MULTISCALE the upsample kernel activates the raw scales >= 1 and the march sees bit 0 only
  q.raw = (sfm_full_res(d) ? d->raw_disp_scales & 1u : d->raw_disp_scales) != 0;
  const bool smooth = (mode & SFM_MODE_SMOOTH) != 0;
  q.accum = q.grad && smooth;
  q.edge_smooth = smooth && (d->flags & SFM_FLAG_EDGE_AWARE_SMOOTH);
  q.nw = 1;
  q.srec = true;
  if (q.ssim) plan_ssim(q, d, num_sms);
  else plan_l1(q, d, num_sms);
  if (q.minrep) {
    // the forward march ahead of the select kernel: the per-pixel instance of the forward mode, planned as such
    SfmStepPlan f = q;
    f.grad = f.accum = false;
    if (f.ssim) plan_ssim(f, d, num_sms);
    else plan_l1(f, d, num_sms);
    q.pre_tasks = f.tasks;
  }
  if (smooth && !q.edge_smooth) plan_smooth(q.smooth, d);
  // the long, issue-bound smoothness CTAs are spread over the first 75 % of the pyramid + smoothness blocks: they start
  // early and the short, memory-bound pyramid CTAs fill the SMs around them and run on alone at the end
  q.band = sfm_plan_band(d);
  // under SFM_FLAG_FULL_RES_MULTISCALE only the edge-aware smoothness reads the pyramid; without it the prologue has none
  const bool pyramid = !(d->flags & SFM_FLAG_REUSE_PYRAMID) && d->n_scales > 1 && (!sfm_full_res(d) || q.edge_smooth);
  const long long mix = ((long long)(pyramid ? pyramid_ctas(d, q.band) : 0) + q.smooth.n_ctas) * 75 / 100;
  q.n_mix_region = (int)(mix < q.smooth.n_ctas ? q.smooth.n_ctas : mix);
  return q;
}
