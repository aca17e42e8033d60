/* restart_oracle.c — TEST INFRASTRUCTURE.  CPU restatement of the episode restarts of the
 * closed-loop rollouts, specified in include/pp.h (pp_rollouts_set_restart), for the parity tests
 * (tests/test_restarts*.py, which compile it with the oracle's flags: -O2 -ffp-contract=off).
 *
 * It is built on the oracle and on the restatements of the monitor and the IDM model:
 * traffic_oracle.c includes incident_oracle.c, which includes the whole of oracle/pp_oracle.c,
 * so a restart resets the monitor's and the traffic model's own state and the ego's lane state
 * comes from the oracle's init_reference / lane_match.  The draw is pp_rollouts_create's, written
 * out again from pp.h.  Only + - * / and sqrt, and one atan2 for the yaw, as the host takes it.
 */
#include "traffic_oracle.c"

uint64_t ppo_rst_key(uint64_t seed, int64_t rollout, int64_t e) {
  const uint64_t k0 = sim_mix64(sim_mix64(seed ^ 0x1417ull) ^ ((uint64_t)rollout * 0xD1B54A32D192ED03ull));
  return e == 0 ? k0 : sim_mix64(k0 + (uint64_t)e * 0xA0761D6478BD642Full);
}

/* Rollout r of `st` drawn from `key`: the ego at rest on a lane centre (a cold start, no kept
 * path), c cars within [-100, 300] m. */
void ppo_rst_draw(const ppo_map *m, uint64_t key, int32_t c, pp_rollout_state *st, int64_t r) {
  uint64_t ctr = 0;
#define UNI() sim_u01(sim_mix64(key + (ctr++) * 0x9E3779B97F4A7C15ull))
  int w = (int)(UNI() * m->n);
  if (w >= m->n) w = m->n - 1;
  const double u = UNI();
  int lane = (int)(UNI() * 3);
  if (lane > 2) lane = 2;
  const vec2 a = wp_center(m, w - 1, lane), b = wp_center(m, w, lane);
  const double l = lane_length(m, w, lane);
  const double vx = 1.0 * ((b.x - a.x) / l), vy = 1.0 * ((b.y - a.y) / l);
  st->ego_x[r] = a.x + (b.x - a.x) * u;
  st->ego_y[r] = a.y + (b.y - a.y) * u;
  st->ego_yaw_deg[r] = atan2(vy, vx) * 180 / M_PI;
  st->ego_speed_mph[r] = 0.0;
  st->path_n[r] = 0;
  for (int i = 0; i < PP_PATH_LEN; i++) {
    if (st->path_x) st->path_x[r * PP_PATH_LEN + i] = 0.0;
    if (st->path_y) st->path_y[r * PP_PATH_LEN + i] = 0.0;
  }
  st->target_lane[r] = lane;
  for (int j = 0; j < c; j++) {
    int cl = (int)(UNI() * 3);
    if (cl > 2) cl = 2;
    const double ds = -100.0 + 400.0 * UNI();
    const double sp = 17.88 + 8.94 * UNI();
    int ww = w;
    double uu = u;
    sim_walk(m, &ww, &uu, cl, ds);
    st->car_lane[r * c + j] = cl;
    st->car_wp[r * c + j] = ww;
    st->car_ratio[r * c + j] = uu;
    st->car_speed[r * c + j] = sp;
  }
#undef UNI
}

/* Restart state: the monitor's counts and distance_m after the last tick, and the record. */
typedef struct ppo_rst_state {
  int32_t *count0; /* [R][PP_INC_KINDS] */
  double *dist0;   /* [R] */
  pp_rollout_restarts rec;
} ppo_rst_state;

/* The end of a tick with the mode on: `st`, the monitor `ms` and (under IDM, else NULL) the
 * traffic state `tr` are the state after the tick (st->tick already counted); every rollout in
 * which a bit of `mask` fired restarts. */
void ppo_rst_step(ppo_map *m, const double *cum, pp_rollout_state *st, ppo_mon_state *ms,
                  pp_rollout_traffic *tr, int64_t n, int32_t c, uint64_t seed, int64_t first,
                  uint32_t mask, ppo_rst_state *rs) {
  const pp_rollout_incidents *q = &ms->rec;
  const pp_rollout_restarts *o = &rs->rec;
  for (int64_t r = 0; r < n; r++) {
    uint32_t fired = 0;
    for (int kind = 0; kind < PP_INC_KINDS; kind++) {
      if (q->count[r * PP_INC_KINDS + kind] != rs->count0[r * PP_INC_KINDS + kind]) fired |= 1u << kind;
      rs->count0[r * PP_INC_KINDS + kind] = q->count[r * PP_INC_KINDS + kind];
    }
    double d = q->distance_m[r];
    if (!isfinite(d)) fired |= 1u << PP_REC_NONFINITE;
    const uint32_t hit = fired & mask;
    if (!hit) {
      rs->dist0[r] = d;
      continue;
    }
    int bit = 0;
    while (!((hit >> bit) & 1u)) bit++;
    if (!isfinite(d)) {
      d = rs->dist0[r];
      q->distance_m[r] = d;
    }
    const double ended = d - o->episode_m[r];
    o->ended_m[r] += ended;
    if (ended >= PP_RST_RUBRIC_M) o->ended_lap[r] += 1;
    o->by_bit[r * (PP_INC_KINDS + 1) + bit] += 1;
    o->episodes[r] += 1;
    o->episode_tick[r] = st->tick;
    o->episode_m[r] = d;
    rs->dist0[r] = d;
    ppo_rst_draw(m, ppo_rst_key(seed, first + r, o->episodes[r]), c, st, r);
    double *ring = ms->ring + r * PP_INC_HISTORY * 2;
    ring[0] = st->ego_x[r];
    ring[1] = st->ego_y[r];
    ms->pts[r] = 0;
    ms->active[r] = 0;
    ms->off_pts[r] = 0;
    q->clean_m[r] = 0;
    if (tr) {
      for (int j = 0; j < c; j++) {
        tr->car_v0[r * c + j] = st->car_speed[r * c + j];
        tr->car_acc[r * c + j] = 0.0;
      }
      refstate ref;
      init_reference(m, st->ego_x[r], st->ego_y[r], &ref);
      ego_lane_state(m, cum, &ref, st->ego_x[r], st->ego_y[r], &tr->ego_lanes[r], &tr->ego_s[r * 3]);
    }
  }
}
