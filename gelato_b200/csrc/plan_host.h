/* plan_host.h -- host-side helpers shared by the CUDA library and the test
 * emulator: PlanView scalar fields from a GelatoPlanDesc, the node / row lists
 * and the block tables of the two kernels, and the test grid of the mesh error
 * estimate. */
#ifndef GELATO_B200_PLAN_HOST_H_
#define GELATO_B200_PLAN_HOST_H_

#include <algorithm>
#include <cmath>
#include <vector>

#include "jobs.h"
#include "mesh_error.h"

/* fills every non-pointer field of the view; pointer fields are left untouched */
static inline void planview_scalars(const GelatoPlanDesc* d, PlanView& v) {
  const int S = d->n_sections, N = d->n_nodes, M = N + S;
  v.S = S; v.N = N; v.M = M;
  v.n_vars = M + 3 * M + 3 * M + 4 * M + 2 * N + S + 1;
  v.n_rows = d->n_rows;
  v.n_vals = d->n_vals;
  v.payload_mode = d->payload_mode;
  v.off_pos = M; v.off_vel = 4 * M; v.off_quat = 7 * M; v.off_u = 11 * M; v.off_t = 11 * M + 2 * N;
  v.un.mass = d->unit_mass; v.un.pos = d->unit_pos; v.un.vel = d->unit_vel; v.un.u = d->unit_u;
  v.un.t = d->unit_t; v.un.dx = d->dx;
  v.n_wind = d->n_wind; v.n_ca = d->n_ca;
  v.n_lin = d->n_lin; v.n_aero = d->n_aero; v.n_evt = d->n_evt;
}

/* Bounds of every index table of a plan description; returns NULL or what is wrong.  The kernels trust
 * these tables, so a description that fails here is refused before anything is uploaded. */
static inline const char* validate_desc(const GelatoPlanDesc* d) {
  if (!d) return "null description";
  const long long S = d->n_sections, N = d->n_nodes, M = N + S;
  if (S <= 0 || N <= 0) return "empty problem";
  if (!(d->dx > 0.0)) return "dx must be positive";
  if (d->n_rows <= 0 || d->n_vals < 0) return "bad n_rows / n_vals";
  if (!d->sec_i32 || !d->sec_i64 || !d->sec_f64 || !d->d_pool || !d->tau_pool) return "missing section tables";
  if (!d->vals_template && d->n_vals > 0) return "missing vals_template";
  if (d->n_wind < 2 || !d->wind || d->n_ca < 2 || !d->ca) return "wind / CA tables need at least two rows";
  const long long n_vars = 11 * M + 2 * N + S + 1;
  long long nodes = 0;
  for (long long s = 0; s < S; s++) {
    const int32_t* si = d->sec_i32 + s * GS_I32_COLS;
    const long long n = si[GS_N];
    if (n < 1) return "a section has no nodes";
    if (si[GS_UA] != nodes) return "sections must tile the control rows in order";
    if (si[GS_XA] < 0 || si[GS_XA] + n + 1 > M) return "state rows of a section out of range";
    if (si[GS_D_OFF] < 0 || si[GS_D_OFF] + n * (n + 1) > d->d_pool_len) return "D block outside the pool";
    if (si[GS_TAU_OFF] < 0 || si[GS_TAU_OFF] + n > d->tau_pool_len) return "tau outside the pool";
    for (int c = GS_R_MASS; c <= GS_R_QUAT; c++)
      if (si[c] < 1 || si[c] >= d->n_rows) return "residual row offset of a section out of range";
    nodes += n;
  }
  if (nodes != N) return "section node counts do not add up to n_nodes";
  if (d->n_lin < 0 || d->n_aero < 0 || d->n_evt < 0) return "negative table length";
  for (long long k = 0; k < d->n_lin; k++) {
    const int32_t* li = d->lin_i32 + k * GL_I32_COLS;
    if (li[GL_ROW] < 1 || li[GL_ROW] >= d->n_rows) return "linear row out of range";
    if (li[GL_IDX_PLUS] < -1 || li[GL_IDX_PLUS] >= n_vars || li[GL_IDX_MINUS] < -1 || li[GL_IDX_MINUS] >= n_vars)
      return "linear row reads outside x";
  }
  for (long long k = 0; k < d->n_aero; k++) {
    const int32_t* ai = d->aero_i32 + k * GA_I32_COLS;
    if (ai[GA_KIND] < 0 || ai[GA_KIND] > 2) return "unknown aero kind";
    if (ai[GA_SECTION] < 0 || ai[GA_SECTION] >= S) return "aero job section out of range";
    const long long n = d->sec_i32[ai[GA_SECTION] * GS_I32_COLS + GS_N];
    if (ai[GA_NK] < 1 || ai[GA_NK] > n + 1) return "aero job has more rows than its section has state nodes";
    if (ai[GA_ROW0] < 1 || ai[GA_ROW0] + ai[GA_NK] > d->n_rows) return "aero rows out of range";
  }
  for (long long k = 0; k < d->n_evt; k++) {
    const int32_t* ei = d->evt_i32 + k * GE_I32_COLS;
    if (ei[GE_TYPE] < GE_LLH || ei[GE_TYPE] >= GE_N_TYPES) return "unknown event job type";
    if (ei[GE_SROW] < 0 || ei[GE_SROW] >= M) return "event job state row out of range";
    if (ei[GE_TIDX] < -1 || ei[GE_TIDX] > S) return "event job time index out of range";
    if (ei[GE_ROW] < 1 || ei[GE_ROW] + ei[GE_NROW] > d->n_rows || ei[GE_NROW] < 1 || ei[GE_NROW] > 3)
      return "event job rows out of range";
    if (ei[GE_TYPE] == GE_USER_ORBIT) {
      for (int r = 0; r < ei[GE_NROW]; r++)
        if (((ei[GE_COMP] >> (8 * r)) & 0xff) >= GEQ_N) return "unknown quantity code of a user built-in";
    } else if (ei[GE_COMP] < 0 || ei[GE_COMP] > 2) {
      return "event job component out of range";
    }
    for (int c = 0; c < 7; c++)
      if (ei[GE_RC0 + c] < 0) return "negative residue count of an event job";
  }
  /* every Jacobian slot offset the kernel writes through, with the extent of its block, inside [0, n_vals) */
  const long long nv = d->n_vals;
#define GELATO_RANGE(off, len) ((off) >= 0 && (long long)(off) + (long long)(len) <= nv)
  for (long long s = 0; s < S; s++) {
    const int32_t* si = d->sec_i32 + s * GS_I32_COLS;
    const int64_t* sj = d->sec_i64 + s * GS_I64_COLS;
    const long long n = si[GS_N];
    const int fl = si[GS_FLAGS];
    if (!GELATO_RANGE(sj[GS_JP_VEL], 3 * n) || !GELATO_RANGE(sj[GS_JP_T], 6 * n) || !GELATO_RANGE(sj[GS_JV_MASS], 3 * n) ||
        !GELATO_RANGE(sj[GS_JV_POS], 9 * n) || !GELATO_RANGE(sj[GS_JV_QUAT], 12 * n) || !GELATO_RANGE(sj[GS_JV_T], 6 * n))
      return "a section's Jacobian block offset is outside vals";
    if ((fl & GSF_AIR_FD) && !GELATO_RANGE(sj[GS_JV_VEL], 9 * n * (n + 1))) return "a section's velocity block is outside vals";
    if (!(fl & GSF_HOLD) && (!GELATO_RANGE(sj[GS_JQ_QUAT], 16 * n * (n + 1)) || !GELATO_RANGE(sj[GS_JQ_U], 8 * n) ||
                             !GELATO_RANGE(sj[GS_JQ_T], 8 * n)))
      return "a section's quaternion block is outside vals";
  }
  for (long long k = 0; k < d->n_aero; k++) {
    const int32_t* ai = d->aero_i32 + k * GA_I32_COLS;
    const int64_t* aj = d->aero_i64 + k * GA_I64_COLS;
    const long long nk = ai[GA_NK];
    if (!GELATO_RANGE(aj[GA_J_POS], 3 * nk) || !GELATO_RANGE(aj[GA_J_VEL], 3 * nk) || !GELATO_RANGE(aj[GA_J_T], 2 * nk) ||
        (ai[GA_KIND] != 1 && !GELATO_RANGE(aj[GA_J_QUAT], 4 * nk)))
      return "an aero job's Jacobian block is outside vals";
  }
  for (long long k = 0; k < d->n_evt; k++) {
    const int32_t* ei = d->evt_i32 + k * GE_I32_COLS;
    const int64_t* ej = d->evt_i64 + k * GE_I64_COLS;
    const int type = ei[GE_TYPE];
    bool ok;
    if (type == GE_TERM) ok = GELATO_RANGE(ej[GE_J_POS], 3 * ei[GE_NROW]) && GELATO_RANGE(ej[GE_J_VEL], 3 * ei[GE_NROW]);
    else if (type >= GE_USER_ORBIT) ok = GELATO_RANGE(ej[GE_J_POS], GE_USER_AUX * ei[GE_NROW]);
    else ok = GELATO_RANGE(ej[GE_J_POS], 3) && GELATO_RANGE(ej[GE_J_T], 1) && (type != GE_IIP || GELATO_RANGE(ej[GE_J_VEL], 3));
    if (!ok) return "an event job's Jacobian block is outside vals";
  }
#undef GELATO_RANGE
  return nullptr;
}

struct HostTables {
  /* BT_COLS ints per block.  jac_blocks: the n_jac_main dynamics / aero / event blocks (heavy and light roles
   * interleaved), then the linear-row blocks of a pair evaluation; jac_heavy / jac_light: the same blocks by
   * role group (measurements).  res_blocks: the residual kernel's. */
  std::vector<int32_t> jac_blocks, jac_heavy, jac_light, res_blocks;
  int n_jac_main = 0;
  int vac_first = 0, n_vac = 0; /* vacuum nodes [vac_first, vac_first + n_vac) of jac_rec: one thread per node */
  std::vector<NodeRec> node_rec;               /* [N] natural order */
  std::vector<NodeRec> jac_rec;                /* [N] air-FD nodes, then vacuum nodes, then fallback nodes */
  std::vector<AeroRec> aero_rows;              /* one per aero constraint row */
};

/* Packed output of the Jacobian kernel: the INDEPENDENT x-dependent values of one scenario, contiguous per
 * section / job, n_pack of them (15 % fewer than the x-dependent COO slots, and no scattered stores):
 *   per section   eqcon_dyn_pos/velocity 1 (all 3n entries are equal) | eqcon_dyn_pos/t 3n (the tf half is the
 *                 negated to half) | eqcon_dyn_vel: mass 3n, position 9n, velocity node-diagonal [9][n] (air),
 *                 quaternion 12n, t 6n (air) or 3n (vacuum: tf = -to) | eqcon_dyn_quat (free attitude):
 *                 node-diagonal [4n][4], u 8n, t 4n (tf = -to)
 *   per aero job  position 3nk | velocity 3nk | quaternion 4nk (not for max-q) | t 2nk
 *   per event job as in COO order
 * `full_slot` (ascending) lists every x-dependent COO slot, `src` / `sgn` say which packed value it holds and
 * with what sign:  vals[full_slot[i]] = sgn[i] * packed[src[i]]. */
struct PackedLayout {
  std::vector<int64_t> sec_pk, aero_pk, evt_pk;
  long long n_pack = 0;
  std::vector<int64_t> full_slot, src;
  std::vector<double> sgn;
};

static inline void build_packed_layout(const GelatoPlanDesc* d, PackedLayout& L) {
  const int S = d->n_sections;
  L.sec_pk.assign((size_t)S * GS_I64_COLS, -1);
  L.aero_pk.assign((size_t)d->n_aero * GA_I64_COLS, -1);
  L.evt_pk.assign((size_t)d->n_evt * GE_I64_COLS, -1);
  struct Ent { int64_t full, src; double sgn; };
  std::vector<Ent> ents;
  long long c = 0;
  auto direct = [&](int64_t full0, long long len) { /* len COO slots in a row = len packed values */
    const long long at = c;
    for (long long i = 0; i < len; i++) ents.push_back({full0 + i, at + i, 1.0});
    c += len;
    return at;
  };
  auto mirrored = [&](int64_t full0, long long half) { /* [half values][their negations] */
    const long long at = c;
    for (long long i = 0; i < half; i++) {
      ents.push_back({full0 + i, at + i, 1.0});
      ents.push_back({full0 + half + i, at + i, -1.0});
    }
    c += half;
    return at;
  };
  for (int s = 0; s < S; s++) {
    const int32_t* si = d->sec_i32 + (size_t)s * GS_I32_COLS;
    const int64_t* sj = d->sec_i64 + (size_t)s * GS_I64_COLS;
    int64_t* pk = L.sec_pk.data() + (size_t)s * GS_I64_COLS;
    const long long n = si[GS_N];
    const int fl = si[GS_FLAGS];
    pk[GS_JP_VEL] = c;
    for (long long i = 0; i < 3 * n; i++) ents.push_back({sj[GS_JP_VEL] + i, c, 1.0});
    c += 1;
    pk[GS_JP_T] = mirrored(sj[GS_JP_T], 3 * n);
    pk[GS_JV_MASS] = direct(sj[GS_JV_MASS], 3 * n);
    pk[GS_JV_POS] = direct(sj[GS_JV_POS], 9 * n);
    if (fl & GSF_AIR_FD) {
      pk[GS_JV_VEL] = c;
      for (long long b = 0; b < 9; b++)
        for (long long j = 0; j < n; j++)
          ents.push_back({sj[GS_JV_VEL] + b * n * (n + 1) + j * (n + 1) + (j + 1), c + b * n + j, 1.0});
      c += 9 * n;
    }
    pk[GS_JV_QUAT] = direct(sj[GS_JV_QUAT], 12 * n);
    pk[GS_JV_T] = (fl & GSF_AIR_FD) ? direct(sj[GS_JV_T], 6 * n) : mirrored(sj[GS_JV_T], 3 * n);
    if (!(fl & GSF_HOLD)) {
      pk[GS_JQ_QUAT] = c;
      for (long long j = 0; j < n; j++)
        for (long long a = 0; a < 4; a++)
          for (long long kk = 0; kk < 4; kk++)
            ents.push_back({sj[GS_JQ_QUAT] + (4 * j + a) * (4 * (n + 1)) + 4 * (j + 1) + kk, c + (4 * j + a) * 4 + kk, 1.0});
      c += 16 * n;
      pk[GS_JQ_U] = direct(sj[GS_JQ_U], 8 * n);
      pk[GS_JQ_T] = mirrored(sj[GS_JQ_T], 4 * n);
    }
  }
  for (int k = 0; k < d->n_aero; k++) {
    const int32_t* ai = d->aero_i32 + (size_t)k * GA_I32_COLS;
    const int64_t* aj = d->aero_i64 + (size_t)k * GA_I64_COLS;
    int64_t* pk = L.aero_pk.data() + (size_t)k * GA_I64_COLS;
    const long long nk = ai[GA_NK];
    pk[GA_J_POS] = direct(aj[GA_J_POS], 3 * nk);
    pk[GA_J_VEL] = direct(aj[GA_J_VEL], 3 * nk);
    if (ai[GA_KIND] != 1) pk[GA_J_QUAT] = direct(aj[GA_J_QUAT], 4 * nk);
    pk[GA_J_T] = direct(aj[GA_J_T], 2 * nk);
  }
  for (int k = 0; k < d->n_evt; k++) {
    const int32_t* ei = d->evt_i32 + (size_t)k * GE_I32_COLS;
    const int64_t* ej = d->evt_i64 + (size_t)k * GE_I64_COLS;
    int64_t* pk = L.evt_pk.data() + (size_t)k * GE_I64_COLS;
    const int type = ei[GE_TYPE];
    if (type == GE_TERM) {
      pk[GE_J_POS] = direct(ej[GE_J_POS], 3 * ei[GE_NROW]);
      pk[GE_J_VEL] = direct(ej[GE_J_VEL], 3 * ei[GE_NROW]);
    } else if (type >= GE_USER_ORBIT) {
      pk[GE_J_POS] = direct(ej[GE_J_POS], (long long)GE_USER_AUX * ei[GE_NROW]);
    } else {
      pk[GE_J_POS] = direct(ej[GE_J_POS], 3);
      if (type == GE_IIP) pk[GE_J_VEL] = direct(ej[GE_J_VEL], 3);
      pk[GE_J_T] = direct(ej[GE_J_T], 1);
    }
  }
  L.n_pack = c;
  std::sort(ents.begin(), ents.end(), [](const Ent& a, const Ent& b) { return a.full < b.full; });
  L.full_slot.resize(ents.size());
  L.src.resize(ents.size());
  L.sgn.resize(ents.size());
  for (size_t i = 0; i < ents.size(); i++) {
    L.full_slot[i] = ents[i].full;
    L.src[i] = ents[i].src;
    L.sgn[i] = ents[i].sgn;
  }
}

static inline void push_block(std::vector<int32_t>& t, int role, int job, int start, int count) {
  t.push_back(role);
  t.push_back(job);
  t.push_back(start);
  t.push_back(count);
}
static inline void push_chunks(std::vector<int32_t>& t, int role, int first, int total, int per_block) {
  for (int a = 0; a < total; a += per_block) push_block(t, role, 0, first + a, std::min(per_block, total - a));
}

static inline void build_host_tables(const GelatoPlanDesc* d, HostTables& h) {
  const int S = d->n_sections, N = d->n_nodes;
  h.node_rec.assign(N, NodeRec());
  std::vector<int32_t> air, vac, gen;
  for (int s = 0; s < S; s++) {
    const int32_t* si = d->sec_i32 + s * GS_I32_COLS;
    const int flags = si[GS_FLAGS];
    for (int j = 0; j < si[GS_N]; j++) {
      const int g = si[GS_UA] + j;
      NodeRec& q = h.node_rec[g];
      q.sec = s; q.j = j; q.row = si[GS_XA] + 1 + j; q.ua = si[GS_UA];
      q.n = si[GS_N]; q.flags = flags; q.d_off = si[GS_D_OFF]; q.tau_off = si[GS_TAU_OFF];
      if (flags & GSF_AIR_FD) air.push_back(g);
      else if (!(flags & GSF_AIR)) vac.push_back(g);
      else gen.push_back(g);
    }
  }
  for (const std::vector<int32_t>* list : {&air, &vac, &gen})
    for (int32_t g : *list) h.jac_rec.push_back(h.node_rec[g]);
  for (int k = 0; k < d->n_aero; k++) {
    const int32_t* ai = d->aero_i32 + k * GA_I32_COLS;
    const int32_t* si = d->sec_i32 + ai[GA_SECTION] * GS_I32_COLS;
    for (int r = 0; r < ai[GA_NK]; r++) {
      AeroRec q;
      q.job = k; q.r = r; q.sec = ai[GA_SECTION]; q.row = si[GS_XA] + r;
      q.kind = ai[GA_KIND]; q.nk = ai[GA_NK]; q.tau_off = si[GS_TAU_OFF]; q.row0 = ai[GA_ROW0];
      h.aero_rows.push_back(q);
    }
  }
  const int n_aero_rows = (int)h.aero_rows.size();

  /* Jacobian blocks: the heavy roles' (air dynamics, aero rows) and the light roles' (vacuum dynamics, fallback,
   * event rows; vacuum dynamics nodes are not blocks at all: k_jacobian_noair, one thread per node) interleaved evenly, so that the blocks resident on an SM at one time mix FP64-issue-bound and
   * latency-bound work (separate kernels on separate streams ran one after the other: the first fills every SM;
   * profiles/r02a_ab_probe.txt); then the linear-row blocks, which only a pair evaluation launches */
  std::vector<int32_t> heavy, light;
  push_chunks(heavy, BR_DYN_AIR, 0, (int)air.size(), GD_NODES);
  push_chunks(heavy, BR_AERO, 0, n_aero_rows, GJ_NODES);
  push_chunks(light, BR_DYN_GEN, (int)(air.size() + vac.size()), (int)gen.size(), GG_NODES);
  push_chunks(light, BR_EVT, 0, d->n_evt, GJ_EVT);
  h.jac_heavy = heavy;
  h.jac_light = light;
  h.vac_first = (int)air.size(); /* vacuum nodes: one thread each, kernel k_jacobian_noair */
  h.n_vac = (int)vac.size();
  std::vector<int32_t>& jb = h.jac_blocks;
  const long long nh = (long long)heavy.size() / BT_COLS, nl = (long long)light.size() / BT_COLS;
  for (long long ih = 0, il = 0; ih < nh || il < nl;) {
    /* next from the list that is behind its share */
    const bool take_heavy = il >= nl || (ih < nh && ih * nl <= il * nh);
    const std::vector<int32_t>& src = take_heavy ? heavy : light;
    const long long k = take_heavy ? ih++ : il++;
    jb.insert(jb.end(), src.begin() + k * BT_COLS, src.begin() + (k + 1) * BT_COLS);
  }
  h.n_jac_main = (int)(jb.size() / BT_COLS);
  push_chunks(jb, BR_LIN, 0, d->n_lin, GJ_THREADS);

  std::vector<int32_t>& rb = h.res_blocks;
  push_chunks(rb, BR_DYN, 0, N, GR_NODES);
  push_chunks(rb, BR_AERO, 0, n_aero_rows, GR_THREADS);
  push_chunks(rb, BR_EVT, 0, d->n_evt, GR_THREADS);
  push_chunks(rb, BR_LIN, 0, d->n_lin, GR_THREADS);
}

/* The test grid of the mesh error estimate (include/gelato_b200.h: GelatoMeshGridDesc) over S sections of n[i] LGR
 * nodes: its sections and the list of its test points.  Returns NULL or why the grid is refused.  The kernels trust
 * the grid, so one that fails here is not uploaded. */
static inline const char* build_mesh_grid(const GelatoMeshGridDesc* g, const int32_t* n, int S, std::vector<MeshSec>& secs,
                                          std::vector<MeshPt>& pts) {
  secs.assign(S, MeshSec());
  pts.clear();
  for (int i = 0; i < S; i++) {
    const long long m = g->m[i], ni = n[i], off = g->off[i];
    if (m < 1) return "every section needs at least one test point";
    if (off < 0 || off > g->pool_len || m > (g->pool_len - off) / (m + 2 * ni + 2))
      return "a section's tables lie outside the pool";
    if ((long long)pts.size() + m > 0x7fffffffLL / MESH_PT) return "too many test points";
    secs[i].m = (int32_t)m;
    secs[i].pt0 = (int32_t)pts.size();
    secs[i].off = off;
    for (int l = 0; l < m; l++) pts.push_back(MeshPt{i, l});
  }
  for (int64_t k = 0; k < g->pool_len; k++)
    if (!std::isfinite(g->pool[k])) return "the table pool holds a value that is not finite";
  return nullptr;
}

#endif
