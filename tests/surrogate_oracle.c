/* surrogate_oracle.c — TEST INFRASTRUCTURE.  CPU restatement of the near-miss measures of the
 * closed-loop rollouts, specified in include/pp.h (pp_rollouts_set_surrogate), for the parity
 * tests (tests/test_surrogate*.py, which compile it with the oracle's flags: -O2
 * -ffp-contract=off).
 *
 * It is built on the oracle and on the monitor's restatement: incident_oracle.c (which includes
 * the whole of oracle/pp_oracle.c) positions the cars as the collision check does.  Only + - * /.
 */
#include "incident_oracle.c"

/* an empty record: minima +inf, no tick, empty histograms */
void ppo_sim_surrogate_init(const pp_rollout_surrogate *s, int64_t n) {
  const int MB = PP_SSM_MEASURES * PP_SSM_BINS;
  for (int64_t r = 0; r < n; r++) {
    s->min_ttc_front[r] = s->min_ttc_rear[r] = s->min_thw[r] = INFINITY;
    s->min_ttc_front_tick[r] = -1;
    for (int e = 0; e < MB; e++) s->time_hist[r * MB + e] = 0;
  }
}

/* the bin of a value >= +0: the number of edges at or below it (PP_SSM_BINS: not counted) */
static int ssm_bin(double v) {
  static const double e[PP_SSM_BINS] = PP_SSM_EDGES;
  int b = 0;
  for (int i = 0; i < PP_SSM_BINS; i++)
    if (!(v < e[i])) b++;
  return b;
}

/* Step the record by one tick: the tick's frames (the ego E) and plans (its driven points), and
 * the car states after the tick; the tick counted is after->tick - 1. */
void ppo_sim_surrogate(ppo_map *m, const pp_rollout_surrogate *s, int64_t n, int32_t c,
                       int32_t consume_k, const pp_frames *fr, const pp_plans *pl,
                       const pp_rollout_state *after) {
  const int64_t t = after->tick - 1;
  for (int64_t r = 0; r < n; r++) {
    const int np = pl->n_points[r];
    const int k = consume_k < np ? consume_k : np;
    const double ex = fr->ego_x[r], ey = fr->ego_y[r];
    double px = ex, py = ey, ux = 0.0, uy = 0.0;
    if (k > 0) {
      px = pl->next_x[r * PP_PATH_LEN + k - 1];
      py = pl->next_y[r * PP_PATH_LEN + k - 1];
      ux = (px - ex) * 50.0 / k;
      uy = (py - ey) * 50.0 / k;
    }
    double val[PP_SSM_MEASURES] = {INFINITY, INFINITY, INFINITY};
    for (int j = 0; j < c; j++) {
      const int64_t q = r * c + j;
      double cx, cy, tx, ty;
      sim_car_pose(m, after->car_lane[q], after->car_wp[q], after->car_ratio[q], &cx, &cy, &tx, &ty);
      const double v = after->car_speed[q];
      const double dx = cx - px, dy = cy - py;
      const double along = dx * tx + dy * ty;
      const double across = dx * ty - dy * tx;
      if (!(fabs(across) < PP_INC_CAR_HALF_WIDTH)) continue;
      const double ut = ux * tx + uy * ty;
      if (along >= PP_INC_CAR_HALF_LEN) {
        const double gap = along - PP_INC_CAR_HALF_LEN;
        const double w = ut - v;
        if (w > 0 && gap / w < val[PP_SSM_TTC_FRONT]) val[PP_SSM_TTC_FRONT] = gap / w;
        if (ut > 0 && gap / ut < val[PP_SSM_THW]) val[PP_SSM_THW] = gap / ut;
      } else if (along <= -PP_INC_CAR_HALF_LEN) {
        const double gap = -along - PP_INC_CAR_HALF_LEN;
        const double w = v - ut;
        if (w > 0 && gap / w < val[PP_SSM_TTC_REAR]) val[PP_SSM_TTC_REAR] = gap / w;
      }
    }
    double *const mins[PP_SSM_MEASURES] = {s->min_ttc_front, s->min_ttc_rear, s->min_thw};
    for (int mm = 0; mm < PP_SSM_MEASURES; mm++) {
      const int b = ssm_bin(val[mm]);
      if (b < PP_SSM_BINS) s->time_hist[(r * PP_SSM_MEASURES + mm) * PP_SSM_BINS + b] += k > 0 ? k : 1;
      if (val[mm] < mins[mm][r]) {
        mins[mm][r] = val[mm];
        if (mm == PP_SSM_TTC_FRONT) s->min_ttc_front_tick[r] = t;
      }
    }
  }
}
