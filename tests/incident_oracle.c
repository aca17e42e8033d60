/* incident_oracle.c — TEST INFRASTRUCTURE.  CPU restatement of the incident monitor of the
 * closed-loop rollouts, specified in include/pp.h (pp_rollout_incidents), for the parity tests
 * (tests/test_incidents*.py, which compile it with the oracle's flags: -O2 -ffp-contract=off).
 *
 * It is built on the oracle itself: the whole of oracle/pp_oracle.c is included below, so the
 * lateral check runs the oracle's own lane_match, wp_ref / wp_center and lane_length.  Only the
 * second half of init_reference_waypoint (src/main.cpp:157-196) is restated here, because the
 * monitor completes a reference point found in a window of the map (ref_wp +- 3) and the oracle
 * has that half only inline in its full-map search.  Only + - * / and sqrt.
 */
#include "../oracle/pp_oracle.c"

/* src/main.cpp:157-196, the second half of init_reference_waypoint (the same statements as
 * init_reference in pp_oracle.c), given the closest reference point */
static void finish_reference(const ppo_map *m, vec2 p, int closest, refstate *rs) {
  double rnom, snom, rdenom, d2[2];
  for (int k = 0; k < 2; k++)
    d2[k] = d2_pt_seg(p, wp_ref(m, closest + k - 1), wp_ref(m, closest + k), &rnom, &rdenom, &snom);
  if (d2[1] < d2[0]) {
    closest++;
  } else if (d2[1] == d2[0]) {
    const double *a = wp_row(m, closest - 1), *b = wp_row(m, closest);
    double ax = (a[8] + b[8]) / 2, ay = (a[9] + b[9]) / 2;
    double dpx = p.x - b[0], dpy = p.y - b[1];
    double dotp = ax * dpx + ay * dpy;
    if (dotp > 0) closest++;
  }
  rs->wp = closest;
  for (int lane = 0; lane < 3; lane++) {
    d2_pt_seg(p, wp_center(m, closest - 1, lane), wp_center(m, closest, lane), &rnom, &rdenom, &snom);
    rs->ratio[lane] = rnom / rdenom;
  }
}

/* position and unit lane tangent of a car at (lane, w, u) */
static void sim_car_pose(const ppo_map *m, int lane, int w, double u, double *x, double *y,
                         double *tx, double *ty) {
  const vec2 a = wp_center(m, w - 1, lane), b = wp_center(m, w, lane);
  const double l = lane_length(m, w, lane);
  *x = a.x + (b.x - a.x) * u;
  *y = a.y + (b.y - a.y) * u;
  *tx = (b.x - a.x) / l;
  *ty = (b.y - a.y) / l;
}

/* ==========================================================================
 * Incident monitor of the rollouts, specified in include/pp.h (pp_rollout_incidents) and
 * restated here for the parity tests.  The caller owns the state; ppo_sim_monitor steps it by
 * one tick given that tick's frames and plans and the car states before and after the tick.
 * ========================================================================== */
typedef struct ppo_mon_state {
  double *ring;     /* [R][PP_INC_HISTORY][2]: driven point D_j in row j % PP_INC_HISTORY */
  int64_t *pts;     /* [R] index i of the ego's current point D_i */
  uint32_t *active; /* [R] bit per kind: its condition held at the last evaluation */
  int32_t *off_pts; /* [R] driven points off the lane centre in a row */
  pp_rollout_incidents rec;
} ppo_mon_state;

/* D_0 = the initial ego pose, an empty record */
void ppo_sim_monitor_init(ppo_mon_state *s, int64_t n, const double *ego_x, const double *ego_y) {
  const pp_rollout_incidents *q = &s->rec;
  memset(s->ring, 0, (size_t)n * PP_INC_HISTORY * 2 * sizeof(double));
  for (int64_t r = 0; r < n; r++) {
    s->ring[r * PP_INC_HISTORY * 2] = ego_x[r];
    s->ring[r * PP_INC_HISTORY * 2 + 1] = ego_y[r];
    s->pts[r] = 0;
    s->active[r] = 0;
    s->off_pts[r] = 0;
    for (int k = 0; k < PP_INC_KINDS; k++) q->count[r * PP_INC_KINDS + k] = 0;
    q->first_tick[r] = -1;
    q->first_kind[r] = -1;
    q->distance_m[r] = q->clean_m[r] = q->best_clean_m[r] = 0;
    q->max_speed[r] = q->max_acc[r] = q->max_jerk[r] = 0;
  }
}

static void mon_count(const pp_rollout_incidents *q, int64_t r, int kind, int64_t t) {
  q->count[r * PP_INC_KINDS + kind] += 1;
  if (kind == PP_INC_COLLISION_REAR) return;
  if (q->first_tick[r] < 0) {
    q->first_tick[r] = t;
    q->first_kind[r] = kind;
  } else if (q->first_tick[r] == t && kind < q->first_kind[r]) {
    q->first_kind[r] = kind;
  }
}

/* 0 = no overlap, 1 = overlap with the car ahead of the ego along its lane, 2 = any other */
static int mon_overlap(double cx, double cy, double tx, double ty, double ex, double ey) {
  const double dx = cx - ex, dy = cy - ey;
  const double along = dx * tx + dy * ty;
  const double across = dx * ty - dy * tx;
  if (!(fabs(along) < PP_INC_CAR_HALF_LEN && fabs(across) < PP_INC_CAR_HALF_WIDTH)) return 0;
  return along > 0 ? 1 : 2;
}

void ppo_sim_monitor(ppo_map *m, ppo_mon_state *s, int64_t n, int32_t c, int32_t consume_k,
                     const pp_frames *fr, const pp_plans *pl, const pp_rollout_state *before,
                     const pp_rollout_state *after) {
  const int H = PP_INC_HISTORY;
  const pp_rollout_incidents *q = &s->rec;
  const int64_t t = before->tick;
  for (int64_t r = 0; r < n; r++) {
    const int np = pl->n_points[r];
    const int k = consume_k < np ? consume_k : np;
    const double *nx = pl->next_x + r * PP_PATH_LEN, *ny = pl->next_y + r * PP_PATH_LEN;
    double *ring = s->ring + r * H * 2;
    double px = fr->ego_x[r], py = fr->ego_y[r];
    if (k > 0) {
      /* the driven points */
      int64_t i = s->pts[r];
      for (int j = 0; j < k; j++) {
        const double x = nx[j], y = ny[j];
        i++;
        const int slot = (int)(i % H);
#define BACK(b) (ring + ((slot - (b) + H) % H) * 2)
        const double sx = x - px, sy = y - py;
        const double step = sqrt(sx * sx + sy * sy);
        q->distance_m[r] += step;
        q->clean_m[r] += step;
        if (q->clean_m[r] > q->best_clean_m[r]) q->best_clean_m[r] = q->clean_m[r];
        unsigned cond = 0;
        if (i >= 10) {
          const double *d10 = BACK(10);
          const double vx = (x - d10[0]) / 0.2, vy = (y - d10[1]) / 0.2;
          const double v = sqrt(vx * vx + vy * vy);
          if (v > q->max_speed[r]) q->max_speed[r] = v;
          if (v > PP_INC_MAX_SPEED) cond |= 1u << PP_INC_OVER_SPEED;
          if (i >= 20) {
            const double *d20 = BACK(20);
            const double wx = (d10[0] - d20[0]) / 0.2, wy = (d10[1] - d20[1]) / 0.2;
            const double ax = (vx - wx) / 0.2, ay = (vy - wy) / 0.2;
            const double a = sqrt(ax * ax + ay * ay);
            if (a > q->max_acc[r]) q->max_acc[r] = a;
            if (a > PP_INC_MAX_ACC) cond |= 1u << PP_INC_OVER_ACC;
            if (i >= H) {
              const double *d50 = BACK(50), *d60 = BACK(60), *d70 = BACK(70);
              const double v50x = (d50[0] - d60[0]) / 0.2, v50y = (d50[1] - d60[1]) / 0.2;
              const double v60x = (d60[0] - d70[0]) / 0.2, v60y = (d60[1] - d70[1]) / 0.2;
              const double a50x = (v50x - v60x) / 0.2, a50y = (v50y - v60y) / 0.2;
              const double jx = (ax - a50x) / 1.0, jy = (ay - a50y) / 1.0;
              const double jn = sqrt(jx * jx + jy * jy);
              if (jn > q->max_jerk[r]) q->max_jerk[r] = jn;
              if (jn > PP_INC_MAX_JERK) cond |= 1u << PP_INC_OVER_JERK;
            }
          }
        }
#undef BACK
        ring[slot * 2] = x; /* D_{i-70} had this row and has been read */
        ring[slot * 2 + 1] = y;
        const unsigned rise = cond & ~s->active[r];
        s->active[r] = (s->active[r] & ~((1u << PP_INC_OVER_SPEED) | (1u << PP_INC_OVER_ACC) |
                                         (1u << PP_INC_OVER_JERK))) | cond;
        for (int kind = PP_INC_OVER_SPEED; kind <= PP_INC_OVER_JERK; kind++)
          if ((rise >> kind) & 1u) mon_count(q, r, kind, t);
        if (rise) q->clean_m[r] = 0;
        px = x;
        py = y;
      }
      s->pts[r] = i;
      /* the lateral position of P: reference from the plan's ref_wp +- 3, then lane matching */
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
      double ms = 0, md = 0;
      int lane = 0, mwp = 0;
      const int ok = lane_match(m, &rs, px, py, &ms, &md, &lane, &mwp);
      const int off_centre = !ok || fabs(md - lane_center_offset(lane)) > PP_INC_LANE_TOL;
      if (!off_centre)
        s->off_pts[r] = 0;
      else if (s->off_pts[r] < (1 << 30))
        s->off_pts[r] += k;
      unsigned cond = 0;
      if (s->off_pts[r] > PP_INC_OUT_POINTS) cond |= 1u << PP_INC_OUT_OF_LANE;
      if (!ok || md < PP_INC_ROAD_MIN_D || md > PP_INC_ROAD_MAX_D) cond |= 1u << PP_INC_OFF_ROAD;
      const unsigned rise = cond & ~s->active[r];
      s->active[r] = (s->active[r] & ~((1u << PP_INC_OUT_OF_LANE) | (1u << PP_INC_OFF_ROAD))) | cond;
      for (int kind = PP_INC_OUT_OF_LANE; kind <= PP_INC_OFF_ROAD; kind++)
        if ((rise >> kind) & 1u) mon_count(q, r, kind, t);
      if (rise) q->clean_m[r] = 0;
    }
    /* collisions: overlaps that begin at this tick */
    unsigned began = 0;
    for (int j = 0; j < c; j++) {
      const int64_t qq = r * c + j;
      double x0, y0, tx0, ty0, x1, y1, tx1, ty1;
      sim_car_pose(m, before->car_lane[qq], before->car_wp[qq], before->car_ratio[qq], &x0, &y0,
                   &tx0, &ty0);
      sim_car_pose(m, after->car_lane[qq], after->car_wp[qq], after->car_ratio[qq], &x1, &y1, &tx1,
                   &ty1);
      const int was = mon_overlap(x0, y0, tx0, ty0, fr->ego_x[r], fr->ego_y[r]);
      const int now = mon_overlap(x1, y1, tx1, ty1, px, py);
      if (now && !was) began |= (unsigned)now;
    }
    if (began & 1u) {
      mon_count(q, r, PP_INC_COLLISION_FRONT, t);
      q->clean_m[r] = 0;
    }
    if (began & 2u) mon_count(q, r, PP_INC_COLLISION_REAR, t);
  }
}

