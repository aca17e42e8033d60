/* pp_oracle.c — TEST INFRASTRUCTURE.  CPU restatement (plain C99) of the
 * planning step of Fable3/CarND-Path-Planning-Project, used ONLY as the
 * checker for the CUDA path (tests/, __graft_entry__.smoke(), bench.py's
 * cpu_baseline / reference arm).  The product (carnd-path-planning-project_b200/)
 * never includes, links or calls this file.
 *
 * Parity status: PINNED.  Every function below is checked bit-for-bit against
 * the reference's own code compiled into oracle/_ref/libppref.so
 * (tests/test_oracle_vs_reference.py), against the seed known-answer values of
 * SURVEY Appendix B, against the lane-centre arrays the reference's author
 * pasted into DrawLines.ipynb, and against golden vectors generated from the
 * reference harness (tests/golden/).
 *
 * Each function cites the reference lines (relative to /root/reference/) it
 * follows.  Floating point: IEEE double, no contraction (-ffp-contract=off),
 * operation order exactly as the reference writes it.
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "../include/pp.h"

#define EPS 1e-5 /* src/main.cpp:24 EPSILON */

/* tunables, src/main.cpp:30,39-49: the reference's literals.  Every planning function takes
 * the tunables as a pp_config; the ppo_* entry points without the _cfg suffix plan with these. */
static const pp_config default_cfg = {
    5,    /* relaxed_acc */
    4,    /* min_relaxed_acc_while_braking */
    8,    /* maximum_acc */
    22.2, /* max_speed */
    4.5,  /* car_length */
    2,    /* safety_distance */
    10,   /* keep_distance */
    0.5,  /* keep_distance_leeway */
    0,    /* test_fast_lane_change */
    0,
};

typedef struct {
  double x, y;
} vec2;

typedef struct ppo_map {
  int n;
  double *t; /* n rows of PP_MAP_STRIDE doubles, layout of include/pp.h */
} ppo_map;

/* per-frame state the reference keeps on the Map object, src/main.cpp:132-133 */
typedef struct {
  int wp;
  double ratio[3];
} refstate;

static double sq(double v) { return v * v; }

/* src/helpers.h:38-40 distance() */
static double dist4(double x1, double y1, double x2, double y2) {
  return sqrt((x2 - x1) * (x2 - x1) + (y2 - y1) * (y2 - y1));
}

/* src/helpers.h:171-173 Point::length */
static double len2(double x, double y) { return sqrt(x * x + y * y); }

/* src/helpers.h:183-186 */
static double d2_pt_pt(vec2 p, vec2 a) { return (p.x - a.x) * (p.x - a.x) + (p.y - a.y) * (p.y - a.y); }

/* src/helpers.h:188-249 distancesq_pt_seg.
 * Quirks kept: clamp to A only when rnom < -1; clamped cases report rnom = 0 /
 * rnom = rdenom exactly; a degenerate segment returns dist(A,B) = 0. */
static double d2_pt_seg(vec2 p, vec2 a, vec2 b, double *rnom_o, double *rdenom_o, double *snom_o) {
  *rnom_o = 0;
  *rdenom_o = 1;
  *snom_o = 0;
  if (a.x == b.x && a.y == b.y) return d2_pt_pt(a, b);
  const double rdenom = d2_pt_pt(a, b);
  const double pdx = p.x - a.x, dx = b.x - a.x;
  const double pdy = p.y - a.y, dy = b.y - a.y;
  const double r1 = pdx * dx;
  const double r2 = pdy * dy;
  const double rnom = r1 + r2;
  *rdenom_o = rdenom;
  const double s1 = pdx * dy;
  const double s2 = pdy * dx;
  const double snom = s1 - s2;
  *snom_o = snom;
  if (rnom < -1) {
    *rnom_o = 0;
    return d2_pt_pt(p, a);
  }
  if (rnom > rdenom) {
    *rnom_o = rdenom;
    return d2_pt_pt(p, b);
  }
  *rnom_o = rnom;
  return snom * snom / rdenom;
}

/* src/main.cpp:134-137 get_waypoint: (idx + size) % size in size_t arithmetic */
static const double *wp_row(const ppo_map *m, int idx) {
  size_t k = ((size_t)idx + (size_t)m->n) % (size_t)m->n;
  return m->t + k * PP_MAP_STRIDE;
}
static vec2 wp_ref(const ppo_map *m, int idx) {
  const double *r = wp_row(m, idx);
  vec2 v = {r[0], r[1]};
  return v;
}
static vec2 wp_center(const ppo_map *m, int idx, int lane) {
  const double *r = wp_row(m, idx);
  vec2 v = {r[2 + 2 * lane], r[3 + 2 * lane]};
  return v;
}
/* src/main.cpp:84-88 */
static double lane_center_offset(int lane) {
  double lane_width = 4.0;
  return lane_width * (lane + 0.5);
}
/* src/main.cpp:138-142 get_lane_length (recomputed on demand, as the reference does) */
static double lane_length(const ppo_map *m, int wp, int lane) {
  vec2 a = wp_center(m, wp, lane), b = wp_center(m, wp - 1, lane);
  return len2(a.x - b.x, a.y - b.y);
}

/* src/main.cpp:89-131 Map::Init */
static ppo_map *map_init(const double *wx, const double *wy, int n) {
  if (n < 2) return NULL;
  ppo_map *m = (ppo_map *)calloc(1, sizeof *m);
  m->n = n;
  m->t = (double *)calloc((size_t)n * PP_MAP_STRIDE, sizeof(double));
  for (int i = 0; i < n; i++) {
    m->t[i * PP_MAP_STRIDE + 0] = wx[i];
    m->t[i * PP_MAP_STRIDE + 1] = wy[i];
  }
  for (int i = 0; i < n; i++) { /* :101-109 unit normal of segment (i-1 -> i) */
    double *w = m->t + (size_t)i * PP_MAP_STRIDE;
    vec2 pr = wp_ref(m, i - 1);
    double dx = w[0] - pr.x, dy = w[1] - pr.y;
    double dl = len2(dx, dy);
    w[8] = dy / dl;
    w[9] = -dx / dl;
  }
  for (int i = 0; i < n; i++) { /* :111-130 centre lines from averaged normals */
    double *w = m->t + (size_t)i * PP_MAP_STRIDE;
    const double *nx_row = wp_row(m, i + 1);
    double nx = (w[8] + nx_row[8]) / 2;
    double ny = (w[9] + nx_row[9]) / 2;
    double ang_n = atan2(w[9], w[8]);
    double ang_avg = atan2(ny, nx);
    double cos_alpha = cos(ang_avg - ang_n);
    nx /= cos_alpha;
    ny /= cos_alpha;
    for (int r = 0; r < 3; r++) {
      double off = lane_center_offset(r);
      w[2 + 2 * r] = w[0] + nx * off;
      w[3 + 2 * r] = w[1] + ny * off;
    }
  }
  for (int i = 0; i < n; i++)
    for (int l = 0; l < 3; l++) m->t[(size_t)i * PP_MAP_STRIDE + 10 + l] = lane_length(m, i, l);
  return m;
}

/* src/main.cpp:143-197 init_reference_waypoint */
static void init_reference(const ppo_map *m, double x, double y, refstate *rs) {
  int closest = 0;
  vec2 p = {x, y};
  vec2 r0 = wp_ref(m, 0);
  double best = sq(r0.x - p.x) + sq(r0.y - p.y);
  for (int i = 1; i < m->n; i++) {
    vec2 r = wp_ref(m, i);
    double d = sq(r.x - p.x) + sq(r.y - p.y);
    if (d < best) {
      closest = i;
      best = d;
    }
  }
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

/* src/main.cpp:199-275 lane_matching (lane_mask = all) */
static int lane_match(const ppo_map *m, const refstate *rs, double x, double y, double *out_s,
                      double *out_d, int *out_lane, int *out_wp) {
  int dir = 0, stop = 0, cur = rs->wp, found = 0;
  vec2 p = {x, y};
  double sum_s[3] = {0, 0, 0}, s_ratio[3];
  for (int i = 0; i < 3; i++) s_ratio[i] = rs->ratio[i];
  double best = 1000 * 1000;
  for (;;) {
    double rnom, snom, rdenom;
    int improved = 0;
    for (int lane = 0; lane < 3; lane++) {
      double d2 = d2_pt_seg(p, wp_center(m, cur - 1, lane), wp_center(m, cur, lane), &rnom, &rdenom, &snom);
      if (d2 < best) {
        best = d2;
        improved = 1;
        found = 1;
        double from_start = rnom / rdenom;
        double r_mod = from_start - s_ratio[lane];
        double seg = lane_length(m, cur, lane);
        *out_s = sum_s[lane] + seg * r_mod;
        double d = sqrt(d2);
        if (snom < 0) d = -d;
        *out_d = d + lane_center_offset(lane);
        *out_lane = lane;
        if (out_wp) *out_wp = cur;
      }
      if (rnom == 0) {
        if (dir == 1) stop = 1;
        dir = -1;
      } else if (rnom == rdenom) {
        if (dir == -1) stop = 1;
        dir = 1;
      } else {
        stop = 1;
      }
    }
    if (!improved || stop) break;
    if (dir > 0) {
      for (int lane = 0; lane < 3; lane++) {
        sum_s[lane] += (1 - s_ratio[lane]) * lane_length(m, cur, lane);
        s_ratio[lane] = 0;
      }
      cur++;
    } else {
      for (int lane = 0; lane < 3; lane++) {
        sum_s[lane] -= s_ratio[lane] * lane_length(m, cur, lane);
        s_ratio[lane] = 1;
      }
      cur--;
    }
  }
  return found;
}

/* src/main.cpp:277-328 get_lane_pos */
static vec2 lane_pos(const ppo_map *m, const refstate *rs, double s, int lane, int *out_wp,
                     double *out_dist) {
  double ratio = rs->ratio[lane];
  int wp = rs->wp;
  vec2 nxt, prv;
  double dest = 0;
  for (;;) {
    nxt = wp_center(m, wp, lane);
    prv = wp_center(m, wp - 1, lane);
    double wl = len2(nxt.x - prv.x, nxt.y - prv.y);
    /* NOT in the reference: with a NaN or infinite s (a NaN pose) neither branch below ever
     * breaks and the reference spins forever; with a huge finite s (a telemetry speed of 1e200)
     * subtracting a segment length no longer changes s, or takes 1e15 steps.  Both this
     * restatement and the CUDA path leave the loop with dest = s when |s| exceeds 10,000 km, so a
     * poisoned frame yields garbage points instead of a hang. */
    if (!(fabs(s) <= 1e7)) {
      dest = s;
      *out_dist = s;
      break;
    }
    if (s > 0) {
      double rem = wl * (1 - ratio);
      if (s <= rem) {
        dest = 1 - (rem - s) / wl;
        *out_dist = rem - s;
        break;
      }
      s -= rem;
      ratio = 0;
      wp++;
    } else {
      double rem = wl * ratio;
      if (-s <= rem) {
        dest = (rem + s) / wl;
        *out_dist = wl * (1 - ratio) - s;
        break;
      }
      s += rem;
      ratio = 1;
      wp--;
    }
  }
  vec2 r;
  r.x = nxt.x * dest + prv.x * (1 - dest);
  r.y = nxt.y * dest + prv.y * (1 - dest);
  *out_wp = wp;
  return r;
}

/* src/main.cpp:330-358 project_speed */
static void project_speed(const ppo_map *m, double vx, double vy, int next_wp, double *vs, double *vd) {
  vec2 a = wp_ref(m, next_wp), b = wp_ref(m, next_wp - 1);
  vec2 w = {a.x - b.x, a.y - b.y};
  double vl = len2(vx, vy);
  if (vl < EPS) {
    *vs = vl;
    *vd = 0;
    return;
  }
  double wl = len2(w.x, w.y);
  w.x *= vl / wl;
  w.y *= vl / wl;
  double sign = 1.0;
  if (w.x * vx + w.y * vy < 0) {
    vx *= -1;
    vy *= -1;
    sign = -1;
  }
  double rnom, rdenom, snom;
  vec2 v = {vx, vy}, o = {0, 0};
  d2_pt_seg(v, o, w, &rnom, &rdenom, &snom);
  *vs = (rnom / rdenom) * vl * sign;
  *vd = (snom / rdenom) * vl * sign;
}

/* the reference's Car (src/main.cpp:51-71), the fields the planner reads */
typedef struct {
  int id, lane;
  double vx, vy, s, d, vs, vd;
} car_t;

/* src/main.cpp:364-485 LaneChangePlanner::calculate_target_lane.
 * cars[] must be in ascending id order (std::map iteration order). */
static int choose_lane(const pp_config *cfg, const car_t *cars, int nc, int ego_lane,
                       int target_lane, double ego_s, double ego_vs, double dt0, uint32_t *flags) {
  const double max_speed = cfg->max_speed, car_length = cfg->car_length;
  const double safety_distance = cfg->safety_distance, relaxed_acc = cfg->relaxed_acc;
  double lane_speed[3], next_s[3];
  int open[3];
  for (int i = 0; i < 3; i++) {
    lane_speed[i] = max_speed;
    next_s[i] = 1000;
    open[i] = 1;
  }
  for (int c = 0; c < nc; c++) {
    const car_t *o = &cars[c];
    int lane = o->lane;
    double s = o->s + o->vs * dt0;
    if (s > ego_s) {
      if (s < next_s[lane]) {
        next_s[lane] = s;
        double far = 200;
        if (s - ego_s < far) {
          double cut = 100;
          int speed = (int)o->vs; /* :394 int truncation */
          if (speed > max_speed) speed = (int)max_speed;
          if (s - ego_s > cut) speed = (int)(speed + (max_speed - speed) * (s - ego_s - cut) / (far - cut));
          lane_speed[lane] = speed;
        }
      }
    }
    double extra = 2;
    if (target_lane == lane) extra = 0;
    double min_dist = car_length + safety_distance + extra;
    if (fabs(ego_s - s) < min_dist) {
      open[lane] = 0;
      *flags |= PP_F_CLOSED_RANGE;
    }
    if (s > ego_s && o->vs < ego_vs) {
      double gap = s - ego_s - car_length - safety_distance - extra;
      double dv = ego_vs - o->vs;
      double t = dv / relaxed_acc;
      double need = ego_vs * t - dv / 2 * t;
      if (gap < need) {
        open[lane] = 0;
        *flags |= PP_F_CLOSED_AHEAD;
      }
    }
    if (s < ego_s && o->vs > ego_vs && s + 50 > ego_s) {
      double gap = ego_s - s - car_length - safety_distance - extra;
      double dv = o->vs - ego_vs;
      double t = dv / relaxed_acc;
      if (target_lane == ego_lane) t += 2;
      double need = dv * t;
      if (gap < need) {
        open[lane] = 0;
        *flags |= PP_F_CLOSED_BEHIND;
      }
    }
  }
  int best_lane = ego_lane;
  double best = 0;
  for (int lane = 0; lane < 3; lane++) {
    if (lane != ego_lane && !open[lane]) continue;
    double q = lane_speed[lane] / max_speed;
    double speed_score = (1.0 < q) ? 1.0 : q; /* std::min(q, 1.0) */
    double distance_score = 1 - fabs((double)(target_lane - lane)) / 2;
    double fr = next_s[lane] / 100;
    double free_score = (fr < 1.0) ? fr : 1.0; /* std::min(1.0, fr) */
    if (cfg->test_fast_lane_change) distance_score = 0;
    double total = speed_score + distance_score / 2 + free_score;
    if (total > best) {
      best = total;
      best_lane = lane;
    }
  }
  if (abs(ego_lane - best_lane) > 1) {
    int nl = best_lane > ego_lane ? ego_lane + 1 : ego_lane - 1;
    target_lane = open[nl] ? nl : ego_lane;
  } else {
    target_lane = best_lane;
  }
  return target_lane;
}

/* src/main.cpp:488-548 SpeedController */
typedef struct {
  double start, target, time, shift;
} speedctl;

static void sc_init(const pp_config *cfg, speedctl *c, double ego_speed) {
  c->shift = 0;
  c->start = ego_speed;
  c->target = cfg->max_speed;
  c->time = fabs(ego_speed - cfg->max_speed) / cfg->relaxed_acc;
}
static double sc_speed(const speedctl *c, double t) {
  t -= c->shift;
  if (t < 0) t = 0;
  if (t > c->time) return c->target;
  return c->start + (c->target - c->start) * t / c->time;
}
static double dmax(double a, double b) { return (a < b) ? b : a; } /* std::max(a,b) */
static double dmin(double a, double b) { return (b < a) ? b : a; } /* std::min(a,b) */

static void sc_limit(speedctl *c, double new_speed, double new_time) {
  double tm = dmax(c->time, 0.02);
  double ntm = dmax(new_time, 0.02);
  double grade = (c->target - c->start) / tm;
  double ngrade = (new_speed - c->start) / ntm;
  if (ngrade < grade) {
    c->target = new_speed;
    c->time = new_time;
  }
}
static void sc_override(speedctl *c, double t, double speed) {
  if (t > c->time) return;
  if (fabs(c->target - c->start) < EPS) return;
  double mod_t = c->time * (speed - c->start) / (c->target - c->start);
  c->shift = t - mod_t;
}

/* src/main.cpp:1052-1151 LimitSpeed (one fresh instance per call, as in the glue) */
static void limit_speed(const pp_config *cfg, double car_vx, double car_vy, double next_s,
                        double ego_s, double ego_speed, double ego_acc, int in_lane,
                        double *t_speed, double *t_time, uint32_t *flags) {
  const double relaxed_acc = cfg->relaxed_acc, maximum_acc = cfg->maximum_acc;
  const double max_speed = cfg->max_speed, car_length = cfg->car_length;
  const double safety_distance = cfg->safety_distance, keep_distance = cfg->keep_distance;
  double target_speed = max_speed;
  double target_time = fabs(ego_speed - max_speed) / relaxed_acc;
  int can_accelerate = 1;
  double gap = next_s - ego_s - car_length;
  if (gap < 0) {
    *flags |= PP_F_COLLISION;
    gap = 0;
  }
  double car_speed = sqrt(car_vx * car_vx + car_vy * car_vy);
  if (ego_speed > car_speed) {
    double acc = relaxed_acc;
    if (ego_acc < 0) acc = cfg->min_relaxed_acc_while_braking;
    double dv = ego_speed - car_speed;
    double dt = dv / acc;
    double dd = ego_speed * dt - dv / 2 * dt;
    double max_dist = gap - safety_distance;
    if (dd > max_dist) {
      target_speed = car_speed;
      target_time = max_dist / (ego_speed - dv / 2);
      if (target_time < EPS || dv / target_time > maximum_acc) {
        *flags |= PP_F_MAXBRAKE;
        target_time = dv / maximum_acc;
      } else {
        *flags |= PP_F_BRAKE;
      }
      can_accelerate = 0;
    }
  }
  if (can_accelerate && in_lane) {
    double excess = ego_s + car_length + keep_distance - next_s;
    double t_opt = dmin(1.0, fabs(excess) / 1.0);
    if (ego_s + car_length + keep_distance > next_s) {
      target_speed = car_speed - excess / t_opt;
      target_time = t_opt;
      { /* maximize_acc(ego_speed, relaxed_acc) :1059-1067 */
        double mt = fabs(target_speed - ego_speed) / relaxed_acc;
        if (target_time < mt) target_time = mt;
      }
      *flags |= PP_F_ADJUST;
    } else if (ego_s + car_length + keep_distance + cfg->keep_distance_leeway > next_s) {
      target_speed = car_speed;
      target_time = 1.0;
      {
        double mt = fabs(target_speed - ego_speed) / relaxed_acc;
        if (target_time < mt) target_time = mt;
      }
      *flags |= PP_F_KEEP;
    }
  }
  *t_speed = target_speed;
  *t_time = target_time;
}

/* src/spline.h:284-373 set_points (natural boundaries, :100-105) with the
 * banded LU of :187-250 (reciprocal row pre-scaling); SURVEY Appendix A. */
#define MAXK 16
typedef struct {
  int n;
  double x[MAXK], y[MAXK], a[MAXK], b[MAXK], c[MAXK], b0, c0;
} spline_t;

static void spline_fit(spline_t *sp, const double *x, const double *y, int n) {
  double lo[MAXK], di[MAXK], up[MAXK], rhs[MAXK], sd[MAXK], z[MAXK];
  sp->n = n;
  for (int i = 0; i < n; i++) {
    sp->x[i] = x[i];
    sp->y[i] = y[i];
    lo[i] = di[i] = up[i] = 0;
  }
  for (int i = 1; i < n - 1; i++) { /* :302-307 */
    lo[i] = 1.0 / 3.0 * (x[i] - x[i - 1]);
    di[i] = 2.0 / 3.0 * (x[i + 1] - x[i - 1]);
    up[i] = 1.0 / 3.0 * (x[i + 1] - x[i]);
    rhs[i] = (y[i + 1] - y[i]) / (x[i + 1] - x[i]) - (y[i] - y[i - 1]) / (x[i] - x[i - 1]);
  }
  di[0] = 2.0; /* :311-313 */
  up[0] = 0.0;
  rhs[0] = 0.0;
  di[n - 1] = 2.0; /* :325-327 */
  lo[n - 1] = 0.0;
  rhs[n - 1] = 0.0;
  for (int i = 0; i < n; i++) { /* :195-204 */
    sd[i] = 1.0 / di[i];
    if (i > 0) lo[i] *= sd[i];
    di[i] *= sd[i];
    if (i < n - 1) up[i] *= sd[i];
    di[i] = 1.0;
  }
  for (int k = 0; k < n - 1; k++) { /* :207-219 */
    int i = k + 1;
    double f = -lo[i] / di[k];
    lo[i] = -f;
    di[i] = di[i] + f * up[k];
  }
  for (int i = 0; i < n; i++) { /* :222-235 l_solve */
    double sum = 0;
    if (i > 0) sum += lo[i] * z[i - 1];
    z[i] = (rhs[i] * sd[i]) - sum;
  }
  for (int i = n - 1; i >= 0; i--) { /* :237-250 r_solve */
    double sum = 0;
    if (i < n - 1) sum += up[i] * sp->b[i + 1];
    sp->b[i] = (z[i] - sum) / di[i];
  }
  for (int i = 0; i < n - 1; i++) { /* :345-349 */
    sp->a[i] = 1.0 / 3.0 * (sp->b[i + 1] - sp->b[i]) / (x[i + 1] - x[i]);
    sp->c[i] = (y[i + 1] - y[i]) / (x[i + 1] - x[i]) -
               1.0 / 3.0 * (2.0 * sp->b[i] + sp->b[i + 1]) * (x[i + 1] - x[i]);
  }
  sp->b0 = sp->b[0]; /* :362-372 */
  sp->c0 = sp->c[0];
  double h = x[n - 1] - x[n - 2];
  sp->a[n - 1] = 0.0;
  sp->c[n - 1] = 3.0 * sp->a[n - 2] * h * h + 2.0 * sp->b[n - 2] * h + sp->c[n - 2];
}

/* src/spline.h:375-396 operator() */
static double spline_eval(const spline_t *sp, double x) {
  int n = sp->n, pos = 0;
  { /* std::lower_bound: first knot not less than x (binary search, same probes) */
    int len = n;
    while (len > 0) {
      int half = len >> 1;
      if (sp->x[pos + half] < x) {
        pos = pos + half + 1;
        len = len - half - 1;
      } else {
        len = half;
      }
    }
  }
  int idx = pos - 1 > 0 ? pos - 1 : 0;
  double h = x - sp->x[idx];
  if (x < sp->x[0]) return (sp->b0 * h + sp->c0) * h + sp->y[0];
  if (x > sp->x[n - 1]) return (sp->b[n - 1] * h + sp->c[n - 1]) * h + sp->y[n - 1];
  return ((sp->a[idx] * h + sp->b[idx]) * h + sp->c[idx]) * h + sp->y[idx];
}

/* src/main.cpp:565-1049 TrajectoryBuilder::build.  prev has nprev (0 or 10)
 * points.  Returns the number of points written to ox/oy. */
static int build_trajectory(const ppo_map *m, const pp_config *cfg, const refstate *rs,
                            const vec2 *prev, int nprev, double ego_x, double ego_y, double yaw_deg,
                            int target_lane, double ego_d, double ego_vd, speedctl *sc, double *ox,
                            double *oy, uint32_t *flags) {
  const double PI = M_PI;
  const double maximum_acc = cfg->maximum_acc;
  int np = 0;
  for (int i = 0; i < nprev; i++) {
    ox[np] = prev[i].x;
    oy[np] = prev[i].y;
    np++;
  }
  double pos_x, pos_y, angle;
  if (nprev == 0) { /* :584-588 */
    pos_x = ego_x;
    pos_y = ego_y;
    angle = yaw_deg * PI / 180;
  } else {
    pos_x = prev[nprev - 1].x;
    pos_y = prev[nprev - 1].y;
    if (nprev == 1) {
      angle = yaw_deg * PI / 180;
    } else {
      double x2 = prev[nprev - 2].x, y2 = prev[nprev - 2].y;
      double vx = pos_x - x2, vy = pos_y - y2;
      if (vx * vx + vy * vy < EPS)
        angle = yaw_deg * PI / 180;
      else
        angle = atan2(pos_y - y2, pos_x - x2);
    }
  }
  /* control points: start + up to 5 lane points (:638-768) */
  vec2 cp[6];
  int ncp = 0;
  double total = 0;
  cp[ncp].x = pos_x;
  cp[ncp].y = pos_y;
  ncp++;
  double min_cp_dist = dmax(sc->start * 1, 5.0);
  double start_s = 0;
  {
    double d_diff = lane_center_offset(target_lane) - ego_d;
    double d_acc = 4;
    int slow = 0;
    double lst = 2.0;
    if ((ego_vd < 0) == (d_diff < 0)) {
      double dmaxd = ego_vd * ego_vd / d_acc / 2;
      if (dmaxd > fabs(d_diff)) { /* abs(double) at :665 resolves to std::abs(double) */
        slow = 1;
        lst = fabs(ego_vd) / d_acc;
      }
    }
    if (!slow) {
      double rel = ego_vd;
      if (d_diff < 0) rel *= -1;
      double ad = fabs(d_diff);
      double peak = sqrt(ad * d_acc + rel * rel / 2);
      lst = (peak * 2 - rel) / d_acc;
      if (lst < 0) *flags |= PP_F_LANE_SWITCH_NEG;
    }
    double dist = sc->start * lst;
    if (dist < 10.0) dist = 10.0;
    if (dist > 50) dist = 50;
    start_s = dist;
  }
  for (int i = 0; i < 5; i++) {
    int nw;
    double wd;
    vec2 pt = lane_pos(m, rs, start_s, target_lane, &nw, &wd);
    total += dist4(cp[ncp - 1].x, cp[ncp - 1].y, pt.x, pt.y);
    cp[ncp++] = pt;
    if (total > 50 && ncp > 2) break;
    start_s += min_cp_dist;
  }
  /* into the local frame (:786-831) */
  double ca = cos(-angle), sa = sin(-angle);
  double cx = pos_x, cy = pos_y;
  for (int i = 0; i < ncp; i++) {
    double px = cp[i].x - cx, py = cp[i].y - cy;
    cp[i].x = px * ca - py * sa;
    cp[i].y = px * sa + py * ca;
  }
  double kx[MAXK], ky[MAXK];
  int nk = 0;
  for (int i = 0; i < nprev - 1; i++) {
    double px = prev[i].x - cx, py = prev[i].y - cy;
    kx[nk] = px * ca - py * sa;
    ky[nk] = px * sa + py * ca;
    nk++;
  }
  int min_count = nk;
  pos_x = 0;
  pos_y = 0;
  double tangle = angle;
  ca = cos(tangle);
  sa = sin(tangle);
  for (int i = 0; i < ncp; i++) {
    kx[nk] = cp[i].x;
    ky[nk] = cp[i].y;
    nk++;
  }
  for (int i = 1; i < nk; i++) { /* :833-843 */
    if (kx[i] <= kx[i - 1]) {
      *flags |= PP_F_SPLINE_INPUT_ERR;
      nk = i;
      break;
    }
  }
  double t = 0.02;
  if (nk < 3 || nk <= min_count || fabs(ego_d) > 20) { /* :848-901 fallback */
    *flags |= PP_F_FALLBACK;
    double speed = sc_speed(sc, t);
    double cur = 0;
    int nxt = 1;
    while (np < 50 && nxt < ncp) {
      double step = speed / 50;
      double dx = cp[nxt].x - pos_x, dy = cp[nxt].y - pos_y;
      double cd = len2(dx, dy);
      if (cd < 5) {
        nxt++;
        continue;
      }
      t += 0.02;
      double want = atan2(dy, dx);
      double diff = fmod(want - cur + 3 * PI, 2 * PI) - PI;
      double max_acceleration = 4;
      double min_radius = dmax(10.0, speed * speed / max_acceleration);
      double rps = speed / min_radius;
      double max_step = rps / 50;
      if (fabs(diff) > max_step) {
        if (diff > 0)
          cur += max_step;
        else
          cur -= max_step;
      } else {
        cur += diff;
      }
      pos_x += cos(cur) * step;
      pos_y += sin(cur) * step;
      ox[np] = (pos_x * ca - pos_y * sa) + cx;
      oy[np] = (pos_x * sa + pos_y * ca) + cy;
      np++;
    }
    return np;
  }
  spline_t sp;
  spline_fit(&sp, kx, ky, nk); /* :904 */
  double arg = 0, prev_speed = sc->start, prev_angle = 0;
  while (arg < 50) { /* :911-1040 */
    double speed = sc_speed(sc, t);
    double step = speed / 50;
    double y = spline_eval(&sp, arg + step);
    double x = arg + step;
    double dist = dist4(pos_x, pos_y, x, y);
    if (dist + EPS < step) *flags |= PP_F_SPLINE_WARNING;
    double acc = fabs(speed - prev_speed) * 50;
    double ang = atan2(y - pos_y, x - pos_x);
    double diff = fmod(ang - prev_angle + 3 * PI, 2 * PI) - PI;
    double cen = speed * 50 * fabs(diff);
    if (acc + cen > maximum_acc) {
      if (speed > prev_speed) {
        double nacc = maximum_acc - cen;
        if (nacc < 0) {
          *flags |= PP_F_ACCT_HIGH;
          nacc = 0;
        }
        double nspeed = prev_speed + nacc / 50; /* inner "speed > prev_speed" is always true here */
        *flags |= PP_F_ACC_OVERRIDE;
        sc_override(sc, t, nspeed);
        speed = nspeed;
        sc->time += 0.02;
        step = speed / 50;
        acc = nacc;
      }
      if (acc + cen > maximum_acc) {
        double ncen = maximum_acc - acc;
        if (ncen < 0) {
          *flags |= PP_F_ACCN_HIGH;
          ncen = 0;
        }
        double ndiff = ncen / speed / 50;
        if (diff < 0) ndiff *= -1;
        double rot = ndiff - diff;
        *flags |= PP_F_CURV_ADJUST;
        double tx = (pos_x * ca - pos_y * sa) + cx;
        double ty = (pos_x * sa + pos_y * ca) + cy;
        double vx = cx - tx, vy = cy - ty;
        double rx = vx * cos(rot) - vy * sin(rot);
        double ry = vx * sin(rot) + vy * cos(rot);
        cx = tx + rx;
        cy = ty + ry;
        tangle += rot;
        ca = cos(tangle);
        sa = sin(tangle);
        double qx = (pos_x * ca - pos_y * sa) + cx;
        double qy = (pos_x * sa + pos_y * ca) + cy;
        if ((tx - qx) * (tx - qx) + (ty - qy) * (ty - qy) > EPS) *flags |= PP_F_TRANSFORM_ERR;
      }
    }
    t += 0.02;
    prev_speed = speed;
    prev_angle = ang;
    double sstep = (x - pos_x) * step / dist;
    pos_y += (y - pos_y) * step / dist;
    arg += sstep;
    pos_x += sstep;
    ox[np] = (pos_x * ca - pos_y * sa) + cx;
    oy[np] = (pos_x * sa + pos_y * ca) + cy;
    np++;
    if (np >= 50) break;
  }
  return np;
}

/* One frame: glue of main::onMessage, src/main.cpp:1254-1457. */
static void plan_frame(const ppo_map *m, const pp_config *cfg, const pp_frames *in,
                       const pp_plans *out, int64_t f) {
  const int K = PP_PREV_KEEP;
  uint32_t flags = 0;
  double ex = in->ego_x[f], ey = in->ego_y[f];
  double speed = in->ego_speed_mph[f];
  speed /= 2.237;
  double acc = 0, dt0 = 0, svx = 0, svy = 0;
  int target_lane = in->target_lane_in[f];
  vec2 prev[PP_PREV_KEEP];
  int nprev = 0;
  if (in->prev_n[f] >= K) { /* :1261-1282 */
    nprev = K;
    for (int i = 0; i < K; i++) {
      prev[i].x = in->prev_x[f * K + i];
      prev[i].y = in->prev_y[f * K + i];
    }
    double v2 = len2(prev[K - 2].x - prev[K - 3].x, prev[K - 2].y - prev[K - 3].y);
    svx = prev[K - 1].x - prev[K - 2].x;
    svy = prev[K - 1].y - prev[K - 2].y;
    double v3 = len2(svx, svy);
    acc = (v3 - v2) * 50;
    speed = v3 * 50;
    svx *= 50;
    svy *= 50;
    ex = prev[K - 1].x;
    ey = prev[K - 1].y;
    dt0 = K / 50.0;
  } else {
    flags |= PP_F_COLD_START;
  }
  refstate rs;
  init_reference(m, ex, ey, &rs); /* :1299 */
  int elane = 0;
  double es = 0, ed = 0;
  if (!lane_match(m, &rs, ex, ey, &es, &ed, &elane, NULL)) { /* :1302-1307 */
    flags |= PP_F_EGO_MATCH_FAIL;
    es = ed = 0;
    elane = 0;
  }
  double evs, evd;
  project_speed(m, svx, svy, rs.wp, &evs, &evd); /* :1313 */
  if (acc > cfg->maximum_acc) acc = cfg->maximum_acc;
  if (acc < -cfg->maximum_acc) acc = -cfg->maximum_acc;

  /* sensor fusion (:1325-1350), kept in ascending id order like std::map */
  car_t cars[PP_MAX_CARS];
  int nc = 0;
  const int mc = in->max_cars;
  const int ncar = in->n_cars[f];
  for (int j = 0; j < ncar; j++) {
    car_t c;
    c.id = in->car_id[f * mc + j];
    double cx = in->car_x[f * mc + j], cy = in->car_y[f * mc + j];
    c.vx = in->car_vx[f * mc + j];
    c.vy = in->car_vy[f * mc + j];
    c.s = c.d = c.vs = c.vd = 0;
    c.lane = 0;
    int nwp = 0, ok;
    const int frozen_lane = in->car_frozen_lane ? in->car_frozen_lane[f * mc + j] : -1;
    if (frozen_lane >= 0) {
      /* a car held over from an earlier message (pp_frames::car_frozen_*): the Frenet values of
       * its last sighting, never matched and never dropped; car_vx / car_vy still feed LimitSpeed */
      ok = 1;
      c.lane = frozen_lane;
      c.s = in->car_frozen_s[f * mc + j];
      c.d = in->car_frozen_d[f * mc + j];
      c.vs = in->car_frozen_vs[f * mc + j];
      c.vd = in->car_frozen_vd[f * mc + j];
    } else {
      ok = lane_match(m, &rs, cx, cy, &c.s, &c.d, &c.lane, &nwp);
      if (ok) project_speed(m, c.vx, c.vy, nwp, &c.vs, &c.vd);
    }
    if (out->car_lane) out->car_lane[f * mc + j] = ok ? c.lane : -1;
    if (out->car_next_wp) out->car_next_wp[f * mc + j] = ok ? nwp : 0;
    if (out->car_s) out->car_s[f * mc + j] = ok ? c.s : 0;
    if (out->car_d) out->car_d[f * mc + j] = ok ? c.d : 0;
    if (out->car_vs) out->car_vs[f * mc + j] = ok ? c.vs : 0;
    if (out->car_vd) out->car_vd[f * mc + j] = ok ? c.vd : 0;
    /* position of this id in the ordered set */
    int pos = 0;
    while (pos < nc && cars[pos].id < c.id) pos++;
    int exists = pos < nc && cars[pos].id == c.id;
    if (!ok) {
      flags |= PP_F_CAR_DROPPED;
      if (exists) { /* erase */
        for (int k = pos; k < nc - 1; k++) cars[k] = cars[k + 1];
        nc--;
      }
      continue;
    }
    if (!exists) {
      for (int k = nc; k > pos; k--) cars[k] = cars[k - 1];
      nc++;
    }
    cars[pos] = c;
  }

  target_lane = choose_lane(cfg, cars, nc, elane, target_lane, es, evs, dt0, &flags); /* :1355 */
  if (target_lane != elane) { /* :1358-1369 */
    double dtl = lane_center_offset(target_lane);
    double diff = fabs(evd * 1.0 + ed - dtl);
    if (diff > 6.0) {
      flags |= PP_F_VETO;
      target_lane = elane;
    }
  }
  int nid = -1, nid_tl = -1, nidx = -1, nidx_tl = -1; /* :1383-1411 */
  double ns = 0, ns_tl = 0;
  double dtl = lane_center_offset(target_lane);
  for (int c = 0; c < nc; c++) {
    double s0 = cars[c].s + cars[c].vs * dt0;
    double d0 = cars[c].d + cars[c].vd * dt0;
    if (s0 > es && fabs(d0 - ed) < 3) {
      if (nid == -1 || ns > s0) {
        nid = cars[c].id;
        nidx = c;
        ns = s0;
      }
    }
    if (s0 >= es - cfg->car_length - cfg->safety_distance && fabs(d0 - dtl) < 3) {
      if (nid_tl == -1 || ns_tl > s0) {
        nid_tl = cars[c].id;
        nidx_tl = c;
        ns_tl = s0;
      }
    }
  }
  if (nid_tl == nid) nid_tl = -1;

  speedctl sc;
  sc_init(cfg, &sc, speed); /* :1422 */
  if (nid != -1) {
    double ts, tt;
    limit_speed(cfg, cars[nidx].vx, cars[nidx].vy, ns, es, speed, acc, 1, &ts, &tt, &flags);
    sc_limit(&sc, ts, tt);
  }
  if (nid_tl != -1) {
    double ts, tt;
    limit_speed(cfg, cars[nidx_tl].vx, cars[nidx_tl].vy, ns_tl, es, speed, acc, 0, &ts, &tt,
                &flags);
    sc_limit(&sc, ts, tt);
  }
  if (out->target_speed) out->target_speed[f] = sc.target;
  if (out->target_time) out->target_time[f] = sc.time;

  int np = build_trajectory(m, cfg, &rs, prev, nprev, ex, ey, in->ego_yaw_deg[f], target_lane, ed,
                            evd, &sc, out->next_x + f * PP_PATH_LEN, out->next_y + f * PP_PATH_LEN,
                            &flags);
  out->n_points[f] = np;
  out->ego_lane[f] = elane;
  out->ref_wp[f] = rs.wp;
  out->target_lane[f] = target_lane;
  if (out->flags) out->flags[f] = flags;
  if (out->ego_s) out->ego_s[f] = es;
  if (out->ego_d) out->ego_d[f] = ed;
  if (out->ego_vs) out->ego_vs[f] = evs;
  if (out->ego_vd) out->ego_vd[f] = evd;
  if (out->ego_speed) out->ego_speed[f] = speed;
  if (out->ego_acc) out->ego_acc[f] = acc;
  if (out->next_car_id) out->next_car_id[f] = nid;
  if (out->next_car_in_target_lane) out->next_car_in_target_lane[f] = nid_tl;
}

/* ------------------------------------------------------------------ exports */

uint32_t ppo_observable_flags(void) { return (1u << PP_NUM_FLAGS) - 1; }

ppo_map *ppo_map_create(const double *wx, const double *wy, int n) { return map_init(wx, wy, n); }

/* CSV as src/main.cpp:1171-1191: x,y read as double, the rest ignored. */
ppo_map *ppo_map_create_from_csv(const char *path) {
  FILE *fp = fopen(path, "r");
  if (!fp) return NULL;
  int cap = 256, n = 0;
  double *xs = (double *)malloc(cap * sizeof(double)), *ys = (double *)malloc(cap * sizeof(double));
  char line[512];
  while (fgets(line, sizeof line, fp)) {
    char *e1, *e2;
    double x = strtod(line, &e1);
    if (e1 == line) continue;
    double y = strtod(e1, &e2);
    if (n == cap) {
      cap *= 2;
      xs = (double *)realloc(xs, cap * sizeof(double));
      ys = (double *)realloc(ys, cap * sizeof(double));
    }
    xs[n] = x;
    ys[n] = y;
    n++;
  }
  fclose(fp);
  ppo_map *m = map_init(xs, ys, n);
  free(xs);
  free(ys);
  return m;
}
void ppo_map_destroy(ppo_map *m) {
  if (m) {
    free(m->t);
    free(m);
  }
}
int ppo_map_num_waypoints(ppo_map *m) { return m->n; }
void ppo_map_table(ppo_map *m, double *out) { memcpy(out, m->t, (size_t)m->n * PP_MAP_STRIDE * sizeof(double)); }

typedef struct {
  const ppo_map *m;
  const pp_config *cfg;
  const pp_frames *in;
  const pp_plans *out;
  int64_t lo, hi;
} span_t;
static void *span_main(void *arg) {
  span_t *sp = (span_t *)arg;
  for (int64_t f = sp->lo; f < sp->hi; f++) plan_frame(sp->m, sp->cfg, sp->in, sp->out, f);
  return NULL;
}

/* Plan n frames with `threads` host threads (contiguous spans; the map is
 * read-only here, per-frame reference state lives on the stack). */
int ppo_plan_frames_cfg(ppo_map *m, const pp_config *cfg, const pp_frames *in, const pp_plans *out,
                        int64_t n, int threads, int want_flags) {
  (void)want_flags;
  if (!m || !cfg || !in || !out) return PP_E_ARG;
  if (threads < 1) threads = 1;
  if (threads > 1024) threads = 1024;
  if (threads == 1) {
    span_t one = {m, cfg, in, out, 0, n};
    span_main(&one);
    return PP_OK;
  }
  pthread_t *tid = (pthread_t *)calloc((size_t)threads, sizeof *tid);
  span_t *sp = (span_t *)calloc((size_t)threads, sizeof *sp);
  int64_t per = (n + threads - 1) / threads;
  int started = 0;
  for (int t = 0; t < threads; t++) {
    int64_t lo = t * per, hi = lo + per < n ? lo + per : n;
    if (lo >= hi) break;
    span_t s1 = {m, cfg, in, out, lo, hi};
    sp[t] = s1;
    pthread_create(&tid[t], NULL, span_main, &sp[t]);
    started++;
  }
  for (int t = 0; t < started; t++) pthread_join(tid[t], NULL);
  free(tid);
  free(sp);
  return PP_OK;
}
int ppo_plan_frames(ppo_map *m, const pp_frames *in, const pp_plans *out, int64_t n, int threads,
                    int want_flags) {
  return ppo_plan_frames_cfg(m, &default_cfg, in, out, n, threads, want_flags);
}

void ppo_distancesq_pt_seg(const double *px, const double *py, const double *ax, const double *ay,
                           const double *bx, const double *by, double *d2, double *rnom,
                           double *rdenom, double *snom, int64_t n) {
  for (int64_t i = 0; i < n; i++) {
    vec2 p = {px[i], py[i]}, a = {ax[i], ay[i]}, b = {bx[i], by[i]};
    d2[i] = d2_pt_seg(p, a, b, &rnom[i], &rdenom[i], &snom[i]);
  }
}

void ppo_init_reference_waypoint(ppo_map *m, const double *x, const double *y, int32_t *ref_wp,
                                 double *ratio, int64_t n) {
  for (int64_t i = 0; i < n; i++) {
    refstate rs;
    init_reference(m, x[i], y[i], &rs);
    ref_wp[i] = rs.wp;
    for (int l = 0; l < 3; l++) ratio[i * 3 + l] = rs.ratio[l];
  }
}

void ppo_lane_matching(ppo_map *m, const double *rx, const double *ry, const double *x,
                       const double *y, const double *vx, const double *vy, int32_t *ok,
                       int32_t *lane, int32_t *next_wp, double *s, double *d, double *vs,
                       double *vd, int64_t n) {
  for (int64_t i = 0; i < n; i++) {
    refstate rs;
    init_reference(m, rx[i], ry[i], &rs);
    int ln = 0, nwp = 0;
    double ss = 0, dd = 0, a = 0, b = 0;
    int good = lane_match(m, &rs, x[i], y[i], &ss, &dd, &ln, &nwp);
    if (good) project_speed(m, vx[i], vy[i], nwp, &a, &b);
    ok[i] = good;
    lane[i] = good ? ln : -1;
    next_wp[i] = good ? nwp : 0;
    s[i] = good ? ss : 0;
    d[i] = good ? dd : 0;
    vs[i] = good ? a : 0;
    vd[i] = good ? b : 0;
  }
}

void ppo_get_lane_pos(ppo_map *m, const double *rx, const double *ry, const double *s,
                      const int32_t *lane, double *ox, double *oy, int32_t *owp, double *odist,
                      int64_t n) {
  for (int64_t i = 0; i < n; i++) {
    refstate rs;
    init_reference(m, rx[i], ry[i], &rs);
    int wp = 0;
    double dist = 0;
    vec2 p = lane_pos(m, &rs, s[i], lane[i], &wp, &dist);
    ox[i] = p.x;
    oy[i] = p.y;
    owp[i] = wp;
    odist[i] = dist;
  }
}

void ppo_spline(const double *kx, const double *ky, int32_t nk, const double *q, int32_t nq,
                double *out, int64_t ns) {
  for (int64_t i = 0; i < ns; i++) {
    spline_t sp;
    spline_fit(&sp, kx + i * nk, ky + i * nk, nk);
    for (int j = 0; j < nq; j++) out[i * nq + j] = spline_eval(&sp, q[i * nq + j]);
  }
}

/* ---- Udacity starter helpers, src/helpers.h:43-155 (never called by the
 * reference planner; part of its API surface). ---- */
static int closest_waypoint(double x, double y, const double *mx, const double *my, int n) {
  double best = 100000;
  int arg = 0;
  for (int i = 0; i < n; i++) {
    double d = dist4(x, y, mx[i], my[i]);
    if (d < best) {
      best = d;
      arg = i;
    }
  }
  return arg;
}
static int next_waypoint(double x, double y, double theta, const double *mx, const double *my, int n) {
  int c = closest_waypoint(x, y, mx, my, n);
  double heading = atan2((my[c] - y), (mx[c] - x));
  double angle = fabs(theta - heading);
  angle = dmin(2 * M_PI - angle, angle);
  if (angle > M_PI / 2) {
    ++c;
    if (c == n) c = 0;
  }
  return c;
}
static void get_frenet(double x, double y, double theta, const double *mx, const double *my, int n,
                       double *os, double *od) {
  int nw = next_waypoint(x, y, theta, mx, my, n);
  int pw = nw - 1;
  if (nw == 0) pw = n - 1;
  double n_x = mx[nw] - mx[pw], n_y = my[nw] - my[pw];
  double x_x = x - mx[pw], x_y = y - my[pw];
  double proj_norm = (x_x * n_x + x_y * n_y) / (n_x * n_x + n_y * n_y);
  double proj_x = proj_norm * n_x, proj_y = proj_norm * n_y;
  double fd = dist4(x_x, x_y, proj_x, proj_y);
  double center_x = 1000 - mx[pw], center_y = 2000 - my[pw];
  double c2p = dist4(center_x, center_y, x_x, x_y);
  double c2r = dist4(center_x, center_y, proj_x, proj_y);
  if (c2p <= c2r) fd *= -1;
  double fs = 0;
  for (int i = 0; i < pw; ++i) fs += dist4(mx[i], my[i], mx[i + 1], my[i + 1]);
  fs += dist4(0, 0, proj_x, proj_y);
  *os = fs;
  *od = fd;
}
/* Defined only for maps_s[0] < s (the reference indexes maps_*[-1] otherwise, SURVEY a21). */
static void get_xy(double s, double d, const double *ms, const double *mx, const double *my, int n,
                   double *ox, double *oy) {
  int pw = -1;
  while (s > ms[pw + 1] && (pw < (int)(n - 1))) ++pw;
  int w2 = (pw + 1) % n;
  double heading = atan2((my[w2] - my[pw]), (mx[w2] - mx[pw]));
  double seg_s = (s - ms[pw]);
  double seg_x = mx[pw] + seg_s * cos(heading);
  double seg_y = my[pw] + seg_s * sin(heading);
  double perp = heading - M_PI / 2;
  *ox = seg_x + d * cos(perp);
  *oy = seg_y + d * sin(perp);
}

void ppo_closest_waypoint(const double *x, const double *y, const double *mx, const double *my,
                          int32_t nwp, int32_t *out, int64_t n) {
  for (int64_t i = 0; i < n; i++) out[i] = closest_waypoint(x[i], y[i], mx, my, nwp);
}
void ppo_next_waypoint(const double *x, const double *y, const double *th, const double *mx,
                       const double *my, int32_t nwp, int32_t *out, int64_t n) {
  for (int64_t i = 0; i < n; i++) out[i] = next_waypoint(x[i], y[i], th[i], mx, my, nwp);
}
void ppo_get_frenet(const double *x, const double *y, const double *th, const double *mx,
                    const double *my, int32_t nwp, double *os, double *od, int64_t n) {
  for (int64_t i = 0; i < n; i++) get_frenet(x[i], y[i], th[i], mx, my, nwp, &os[i], &od[i]);
}
void ppo_get_xy(const double *s, const double *d, const double *ms, const double *mx,
                const double *my, int32_t nwp, double *ox, double *oy, int64_t n) {
  for (int64_t i = 0; i < n; i++) get_xy(s[i], d[i], ms, mx, my, nwp, &ox[i], &oy[i]);
}

void ppo_lane_change_cfg(const pp_config *cfg, const int32_t *car_id, const double *car_s,
                         const double *car_vs, const int32_t *car_lane, int32_t nc,
                         const int32_t *ego_lane, const int32_t *target_lane, const double *ego_s,
                         const double *ego_vs, const double *dt0, int32_t *out, int64_t n) {
  for (int64_t i = 0; i < n; i++) {
    car_t cars[PP_MAX_CARS];
    int k = 0;
    for (int j = 0; j < nc; j++) {
      if (car_lane[i * nc + j] < 0) continue;
      car_t c;
      memset(&c, 0, sizeof c);
      c.id = car_id[i * nc + j];
      c.s = car_s[i * nc + j];
      c.vs = car_vs[i * nc + j];
      c.lane = car_lane[i * nc + j];
      int pos = 0;
      while (pos < k && cars[pos].id < c.id) pos++;
      if (!(pos < k && cars[pos].id == c.id)) {
        for (int q = k; q > pos; q--) cars[q] = cars[q - 1];
        k++;
      }
      cars[pos] = c;
    }
    uint32_t fl = 0;
    out[i] = choose_lane(cfg, cars, k, ego_lane[i], target_lane[i], ego_s[i], ego_vs[i], dt0[i], &fl);
  }
}
void ppo_lane_change(const int32_t *car_id, const double *car_s, const double *car_vs,
                     const int32_t *car_lane, int32_t nc, const int32_t *ego_lane,
                     const int32_t *target_lane, const double *ego_s, const double *ego_vs,
                     const double *dt0, int32_t *out, int64_t n) {
  ppo_lane_change_cfg(&default_cfg, car_id, car_s, car_vs, car_lane, nc, ego_lane, target_lane,
                      ego_s, ego_vs, dt0, out, n);
}

void ppo_limit_speed_cfg(const pp_config *cfg, const double *car_vx, const double *car_vy,
                         const double *next_s, const double *ego_s, const double *ego_speed,
                         const double *ego_acc, const int32_t *in_lane, double *ls_speed,
                         double *ls_time, double *sc_speed_o, double *sc_time, uint32_t *flags,
                         int64_t n) {
  for (int64_t i = 0; i < n; i++) {
    uint32_t fl = 0;
    limit_speed(cfg, car_vx[i], car_vy[i], next_s[i], ego_s[i], ego_speed[i], ego_acc[i],
                in_lane[i], &ls_speed[i], &ls_time[i], &fl);
    speedctl sc;
    sc_init(cfg, &sc, ego_speed[i]);
    sc_limit(&sc, ls_speed[i], ls_time[i]);
    sc_speed_o[i] = sc.target;
    sc_time[i] = sc.time;
    flags[i] = fl & (PP_F_COLLISION | PP_F_BRAKE | PP_F_MAXBRAKE | PP_F_ADJUST | PP_F_KEEP);
  }
}
void ppo_limit_speed(const double *car_vx, const double *car_vy, const double *next_s,
                     const double *ego_s, const double *ego_speed, const double *ego_acc,
                     const int32_t *in_lane, double *ls_speed, double *ls_time, double *sc_speed_o,
                     double *sc_time, uint32_t *flags, int64_t n) {
  ppo_limit_speed_cfg(&default_cfg, car_vx, car_vy, next_s, ego_s, ego_speed, ego_acc, in_lane,
                      ls_speed, ls_time, sc_speed_o, sc_time, flags, n);
}

/* TrajectoryBuilder::build on explicit inputs (the reference point is the last
 * kept previous point, or the telemetry pose on a cold start). */
void ppo_trajectory_build_cfg(ppo_map *m, const pp_config *cfg, const int32_t *prev_n,
                              const double *prev_x, const double *prev_y, const double *ego_x,
                              const double *ego_y, const double *yaw, const int32_t *target_lane,
                              const double *ego_d, const double *ego_vd, const double *sc_start,
                              const double *sc_target, const double *sc_time, double *out_x,
                              double *out_y, int32_t *out_n, uint32_t *out_flags, int64_t n) {
  const int K = PP_PREV_KEEP;
  for (int64_t i = 0; i < n; i++) {
    vec2 prev[PP_PREV_KEEP];
    int nprev = prev_n[i] >= K ? K : 0;
    for (int k = 0; k < K; k++) {
      prev[k].x = prev_x[i * K + k];
      prev[k].y = prev_y[i * K + k];
    }
    double rx = nprev ? prev[K - 1].x : ego_x[i], ry = nprev ? prev[K - 1].y : ego_y[i];
    refstate rs;
    init_reference(m, rx, ry, &rs);
    speedctl sc;
    sc.shift = 0;
    sc.start = sc_start[i];
    sc.target = sc_target[i];
    sc.time = sc_time[i];
    uint32_t fl = 0;
    out_n[i] = build_trajectory(m, cfg, &rs, prev, nprev, rx, ry, yaw[i], target_lane[i], ego_d[i],
                                ego_vd[i], &sc, out_x + i * PP_PATH_LEN, out_y + i * PP_PATH_LEN, &fl);
    out_flags[i] = fl;
  }
}
void ppo_trajectory_build(ppo_map *m, const int32_t *prev_n, const double *prev_x,
                          const double *prev_y, const double *ego_x, const double *ego_y,
                          const double *yaw, const int32_t *target_lane, const double *ego_d,
                          const double *ego_vd, const double *sc_start, const double *sc_target,
                          const double *sc_time, double *out_x, double *out_y, int32_t *out_n,
                          uint32_t *out_flags, int64_t n) {
  ppo_trajectory_build_cfg(m, &default_cfg, prev_n, prev_x, prev_y, ego_x, ego_y, yaw, target_lane,
                           ego_d, ego_vd, sc_start, sc_target, sc_time, out_x, out_y, out_n,
                           out_flags, n);
}

/* ==========================================================================
 * Simulator model of the closed-loop rollouts (BASELINE config 3).  NOT part of
 * the reference (the reference was validated against the Udacity simulator
 * binary, README.md:12-17): the model is specified in include/pp.h
 * (pp_rollouts) and restated here independently of the CUDA code so that the
 * tests can check the device state tick by tick, bit for bit.  Only + - * /
 * and sqrt are used.
 * ========================================================================== */
static uint64_t sim_mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
static double sim_u01(uint64_t v) { return (double)(v >> 11) * (1.0 / 9007199254740992.0); }

static void sim_walk(const ppo_map *m, int *w, double *u, int lane, double ds) {
  for (int guard = 0; guard < 4 * m->n; guard++) {
    const double l = lane_length(m, *w, lane);
    if (ds >= 0) {
      const double rem = l * (1 - *u);
      if (ds <= rem) {
        *u += ds / l;
        break;
      }
      ds -= rem;
      *u = 0;
      (*w)++;
    } else {
      const double rem = l * *u;
      if (-ds <= rem) {
        *u += ds / l;
        break;
      }
      ds += rem;
      *u = 1;
      (*w)--;
    }
  }
  *w %= m->n;
  if (*w < 0) *w += m->n;
}

/* frame <- state */
void ppo_sim_frames(ppo_map *m, const pp_rollout_state *st, int64_t n, int32_t c,
                    const pp_frames *fr) {
  for (int64_t r = 0; r < n; r++) {
    ((double *)fr->ego_x)[r] = st->ego_x[r];
    ((double *)fr->ego_y)[r] = st->ego_y[r];
    ((double *)fr->ego_yaw_deg)[r] = st->ego_yaw_deg[r];
    ((double *)fr->ego_speed_mph)[r] = st->ego_speed_mph[r];
    const int pn = st->path_n[r];
    ((int32_t *)fr->prev_n)[r] = pn;
    for (int i = 0; i < PP_PREV_KEEP; i++) {
      ((double *)fr->prev_x)[r * PP_PREV_KEEP + i] = i < pn ? st->path_x[r * PP_PATH_LEN + i] : 0.0;
      ((double *)fr->prev_y)[r * PP_PREV_KEEP + i] = i < pn ? st->path_y[r * PP_PATH_LEN + i] : 0.0;
    }
    ((int32_t *)fr->target_lane_in)[r] = st->target_lane[r];
    ((int32_t *)fr->n_cars)[r] = c;
    for (int j = 0; j < c; j++) {
      const int64_t k = r * c + j;
      const int lane = st->car_lane[k], w = st->car_wp[k];
      const vec2 a = wp_center(m, w - 1, lane), b = wp_center(m, w, lane);
      const double l = lane_length(m, w, lane);
      const double u = st->car_ratio[k], v = st->car_speed[k];
      const double tx = (b.x - a.x) / l, ty = (b.y - a.y) / l;
      ((int32_t *)fr->car_id)[k] = j;
      ((double *)fr->car_x)[k] = a.x + (b.x - a.x) * u;
      ((double *)fr->car_y)[k] = a.y + (b.y - a.y) * u;
      ((double *)fr->car_vx)[k] = v * tx;
      ((double *)fr->car_vy)[k] = v * ty;
    }
  }
}

/* state <- simulator step(plan) */
void ppo_sim_advance(ppo_map *m, pp_rollout_state *st, int64_t n, int32_t c, uint64_t seed,
                     int64_t first, int32_t consume_k, const pp_plans *pl) {
  const double tick_s = 0.02;
  for (int64_t r = 0; r < n; r++) {
    const int np = pl->n_points[r];
    const int k = consume_k < np ? consume_k : np;
    const double *nx = pl->next_x + r * PP_PATH_LEN, *ny = pl->next_y + r * PP_PATH_LEN;
    if (k > 0) {
      const double ox = st->ego_x[r], oy = st->ego_y[r];
      const double qx = nx[k - 1], qy = ny[k - 1];
      const double d = sqrt((qx - ox) * (qx - ox) + (qy - oy) * (qy - oy));
      st->ego_x[r] = qx;
      st->ego_y[r] = qy;
      st->ego_speed_mph[r] = d / (tick_s * k) * 2.237;
    }
    for (int i = 0; i < PP_PATH_LEN; i++) {
      st->path_x[r * PP_PATH_LEN + i] = i + k < np ? nx[i + k] : 0.0;
      st->path_y[r * PP_PATH_LEN + i] = i + k < np ? ny[i + k] : 0.0;
    }
    st->path_n[r] = np - k;
    st->target_lane[r] = pl->target_lane[r];
    const double dt = tick_s * (k > 0 ? k : 1);
    const int ref_wp = pl->ref_wp[r];
    for (int j = 0; j < c; j++) {
      const int64_t q = r * c + j;
      int lane = st->car_lane[q], w = st->car_wp[q];
      double u = st->car_ratio[q], v = st->car_speed[q];
      const int m_lane = pl->car_lane[q];
      const double m_s = pl->car_s[q];
      if (m_lane < 0 || m_s < -100.0 || m_s > 300.0) {
        const uint64_t key =
            sim_mix64(sim_mix64(seed ^ 0x5157ull) ^ ((uint64_t)(first + r) * 0xD1B54A32D192ED03ull));
        const uint64_t h =
            sim_mix64(key ^ ((uint64_t)st->tick * 0x9E3779B97F4A7C15ull) ^ ((uint64_t)j << 48));
        const double u1 = sim_u01(sim_mix64(h + 1)), u2 = sim_u01(sim_mix64(h + 2)),
                     u3 = sim_u01(sim_mix64(h + 3));
        const double ds = (m_lane >= 0 && m_s < -100.0) ? 200.0 + 100.0 * u1 : -(60.0 + 40.0 * u1);
        lane = (int)(3.0 * u2);
        if (lane > 2) lane = 2;
        v = 17.88 + 8.94 * u3;
        w = ref_wp;
        u = 0.5;
        sim_walk(m, &w, &u, lane, ds);
      } else {
        u += (v * dt) / lane_length(m, w, lane);
        for (int guard = 0; guard < 64 && u >= 1; guard++) {
          const double left = (u - 1) * lane_length(m, w, lane);
          w = w + 1 == m->n ? 0 : w + 1;
          u = left / lane_length(m, w, lane);
        }
      }
      st->car_lane[q] = lane;
      st->car_wp[q] = w;
      st->car_ratio[q] = u;
      st->car_speed[q] = v;
    }
  }
  st->tick++;
}
