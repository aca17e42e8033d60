/* traffic_oracle.c — TEST INFRASTRUCTURE.  CPU restatement of the IDM traffic model of the
 * closed-loop rollouts, specified in include/pp.h (PP_TRAFFIC_IDM), for the parity tests
 * (tests/test_traffic*.py, which compile it with the oracle's flags: -O2 -ffp-contract=off).
 *
 * It is built on the oracle and on the monitor's restatement: incident_oracle.c (which includes
 * the whole of oracle/pp_oracle.c) gives the reference completion the monitor's lateral check
 * uses, so the ego's lane state comes from the oracle's own init_reference / lane_match; the
 * step reuses the oracle's ppo_sim_advance for the ego, the kept path and the respawns, and its
 * sim_walk segment carry.  Only + - * / and sqrt.
 */
#include "incident_oracle.c"

/* cum(L, w) = sum of the lane lengths of segments 0 .. w-1, in ascending w: [3][n + 1] */
void ppo_traffic_cum(const ppo_map *m, double *cum) {
  for (int lane = 0; lane < 3; lane++) {
    double acc = 0.0;
    cum[lane * (m->n + 1)] = 0.0;
    for (int w = 0; w < m->n; w++) {
      acc += m->t[(size_t)w * PP_MAP_STRIDE + 10 + lane];
      cum[lane * (m->n + 1) + w + 1] = acc;
    }
  }
}

/* the ego's lane state (lanes, S[3]) from its reference and lane match */
static void ego_lane_state(const ppo_map *m, const double *cum, const refstate *rs, double px,
                           double py, int32_t *lanes, double *s3) {
  double ms = 0, md = 0;
  int lane = 0, mwp = 0;
  const int ok = lane_match(m, rs, px, py, &ms, &md, &lane, &mwp);
  int w = rs->wp % m->n;
  if (w < 0) w += m->n;
  *lanes = 0;
  for (int L = 0; L < 3; L++) {
    if (ok && fabs(md - (4.0 * L + 2.0)) < PP_TRF_EGO_CORRIDOR) *lanes |= 1 << L;
    s3[L] = cum[L * (m->n + 1) + w] + rs->ratio[L] * lane_length(m, rs->wp, L);
  }
}

/* Selecting the model: v0 = the current speed, acc = 0, the ego's lane state from the full
 * reference search at its pose. */
void ppo_traffic_init(ppo_map *m, const double *cum, const pp_rollout_state *st, int64_t n,
                      int32_t c, pp_rollout_traffic *tr) {
  for (int64_t r = 0; r < n; r++) {
    for (int j = 0; j < c; j++) {
      tr->car_v0[r * c + j] = st->car_speed[r * c + j];
      tr->car_acc[r * c + j] = 0.0;
    }
    refstate rs;
    init_reference(m, st->ego_x[r], st->ego_y[r], &rs);
    ego_lane_state(m, cum, &rs, st->ego_x[r], st->ego_y[r], &tr->ego_lanes[r], &tr->ego_s[r * 3]);
  }
}

static double reduce_delta(double sc, double sf, double lam) {
  double d = sc - sf;
  if (d < 0)
    d += lam;
  else if (d >= lam)
    d -= lam;
  return d;
}

/* One tick of the simulator under the IDM model: state and traffic are stepped in place, given
 * the tick's plans (the ego's speed before the tick is st->ego_speed_mph on entry). */
void ppo_sim_advance_idm(ppo_map *m, const double *cum, pp_rollout_state *st,
                         pp_rollout_traffic *tr, int64_t n, int32_t c, uint64_t seed, int64_t first,
                         int32_t consume_k, const pp_plans *pl) {
  const size_t nc = (size_t)n * (size_t)c;
  int32_t *lane0 = (int32_t *)malloc((nc ? nc : 1) * sizeof(int32_t));
  double *s0 = (double *)malloc((nc ? nc : 1) * sizeof(double));
  double *v0 = (double *)malloc((nc ? nc : 1) * sizeof(double));
  double *mph0 = (double *)malloc((size_t)n * sizeof(double));
  int32_t *wp0 = (int32_t *)malloc((nc ? nc : 1) * sizeof(int32_t));
  double *u0 = (double *)malloc((nc ? nc : 1) * sizeof(double));
  /* the state before the tick */
  for (int64_t r = 0; r < n; r++) mph0[r] = st->ego_speed_mph[r];
  for (size_t q = 0; q < nc; q++) {
    const int L = st->car_lane[q], w = st->car_wp[q];
    lane0[q] = L;
    wp0[q] = w;
    u0[q] = st->car_ratio[q];
    s0[q] = cum[L * (m->n + 1) + w] + st->car_ratio[q] * lane_length(m, w, L);
    v0[q] = st->car_speed[q];
  }
  /* the ego, the kept path, the respawns (and a constant-speed advance of the other cars, which
   * is replaced below) */
  ppo_sim_advance(m, st, n, c, seed, first, consume_k, pl);
  for (int64_t r = 0; r < n; r++) {
    const int np = pl->n_points[r];
    const int k = consume_k < np ? consume_k : np;
    const double dt = 0.02 * (k > 0 ? k : 1);
    for (int j = 0; j < c; j++) {
      const int64_t q = r * c + j;
      const int m_lane = pl->car_lane[q];
      const double m_s = pl->car_s[q];
      if (m_lane < 0 || m_s < -100.0 || m_s > 300.0) { /* respawned by ppo_sim_advance */
        tr->car_v0[q] = st->car_speed[q];
        tr->car_acc[q] = 0.0;
        continue;
      }
      const int lane = lane0[q];
      const double sf = s0[q], lam = cum[lane * (m->n + 1) + m->n], half = lam / 2;
      int has = 0;
      double best = 0.0, vl = 0.0;
      for (int i = 0; i < c; i++) {
        if (lane0[r * c + i] != lane) continue;
        const double d = reduce_delta(s0[r * c + i], sf, lam);
        if (((d > 0 && d < half) || (d == 0 && i > j)) && (!has || d < best)) {
          has = 1;
          best = d;
          vl = v0[r * c + i];
        }
      }
      if ((tr->ego_lanes[r] >> lane) & 1) {
        const double d = reduce_delta(tr->ego_s[r * 3 + lane], sf, lam);
        if (((d > 0 && d < half) || d == 0) && (!has || d < best)) {
          has = 1;
          best = d;
          vl = mph0[r] / 2.237;
        }
      }
      const double v = v0[q];
      const double q1 = v / tr->car_v0[q], q2 = q1 * q1;
      double inter = 0.0;
      if (has) {
        double gap = best - PP_INC_CAR_HALF_LEN;
        if (gap < PP_TRF_GAP_FLOOR) gap = PP_TRF_GAP_FLOOR;
        double dyn = v * PP_TRF_HEADWAY + v * (v - vl) / (2.0 * sqrt(PP_TRF_ACC * PP_TRF_DEC));
        if (dyn < 0.0) dyn = 0.0;
        const double z = (PP_TRF_MIN_GAP + dyn) / gap;
        inter = z * z;
      }
      double acc = PP_TRF_ACC * (1.0 - q2 * q2 - inter);
      if (acc < -PP_TRF_MAX_DEC) acc = -PP_TRF_MAX_DEC;
      if (acc > PP_TRF_ACC) acc = PP_TRF_ACC;
      double v1 = v + acc * dt;
      if (v1 < 0) v1 = 0;
      const double ds = (v + v1) * 0.5 * dt;
      int w = wp0[q];
      double u = u0[q];
      u += ds / lane_length(m, w, lane);
      for (int guard = 0; guard < 64 && u >= 1; guard++) {
        const double left = (u - 1) * lane_length(m, w, lane);
        w = w + 1 == m->n ? 0 : w + 1;
        u = left / lane_length(m, w, lane);
      }
      st->car_wp[q] = w;
      st->car_ratio[q] = u;
      st->car_speed[q] = v1;
      tr->car_acc[q] = acc;
    }
    /* the ego's lane state at the tick's last driven point, for the next tick: the monitor's
     * lateral reference (the closest of rows ref_wp-3 .. ref_wp+3, then its completion) */
    const double px = st->ego_x[r], py = st->ego_y[r];
    const vec2 p = {px, py};
    const int rw = pl->ref_wp[r];
    int closest = rw - 3;
    vec2 w0 = wp_ref(m, closest);
    double bd = sq(w0.x - p.x) + sq(w0.y - p.y);
    for (int w = rw - 2; w <= rw + 3; w++) {
      const vec2 ww = wp_ref(m, w);
      const double d = sq(ww.x - p.x) + sq(ww.y - p.y);
      if (d < bd) {
        closest = w;
        bd = d;
      }
    }
    refstate rs;
    finish_reference(m, p, closest, &rs);
    ego_lane_state(m, cum, &rs, px, py, &tr->ego_lanes[r], &tr->ego_s[r * 3]);
  }
  free(lane0);
  free(s0);
  free(v0);
  free(mph0);
  free(wp0);
  free(u0);
}
