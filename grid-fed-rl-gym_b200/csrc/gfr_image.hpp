// gfr_image.hpp - host-side check of a gfr_feeder_desc and its packing into the "image" the
// kernels read (ints first, then doubles; offsets recorded in gfr::Layout).
//
// An image is built for one (solver, lanes) pair.  Everything a lane touches in the hot loops is laid
// out by SCHEDULE POSITION p = row * lanes + lane (row = one elimination step, leaf -> root order being
// rows nrows-1 .. 0): the per-position record (bus, parent, flags, pool slot, child list), the branch
// and diagonal admittances, the flat-start factors.  A lane therefore reads consecutive 16-byte units
// next to its neighbours', with no index chain (the position is known before anything is loaded).
// The sweep keeps its compact per-bus arrays (position = bus index there).
#pragma once
#include <algorithm>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/gfr_b200.h"
#include "gfr_device.cuh"

namespace gfr {

struct ImageBuilder {
  std::vector<int32_t> ints;
  std::vector<double> dbls;
  int add_i(const int32_t* p, int count) {
    while (ints.size() % 4) ints.push_back(0);            // every int array starts 16-byte aligned
    int off = (int)ints.size();
    if (count > 0) ints.insert(ints.end(), p, p + count);
    return off;
  }
  int add_d(const double* p, int count) {
    if (dbls.size() % 2) dbls.push_back(0.0);             // every double array starts 16-byte aligned
    int off = (int)dbls.size();
    if (count > 0) dbls.insert(dbls.end(), p, p + count);
    return off;
  }
};

struct FeederImage {
  Layout lay{};
  bool has_pv = false;
  bool root_is_slack = false;
  int center_depth = 0;            // levels of the tree rooted at its center (ceil(diameter / 2) + 1), uncapped
  int lanes = 0, solver = 0;
  int n_reg_edges = 0;             // branches whose hand-off stays in registers (Newton)
  std::vector<unsigned char> img;
  std::vector<double> load_pq;     // [2L] static active / reactive power (observation)
};

// A deep copy of a description (the library builds images for other lane counts after the caller's
// arrays are gone).
struct DescCopy {
  gfr_feeder_desc d{};
  std::vector<std::vector<int32_t>> iv;
  std::vector<std::vector<double>> dv;
  const int32_t* keep_i(const int32_t* p, size_t c) {
    if (!p) return nullptr;
    iv.emplace_back(p, p + c);
    if (iv.back().empty()) iv.back().push_back(0);
    return iv.back().data();
  }
  const double* keep_d(const double* p, size_t c) {
    if (!p) return nullptr;
    dv.emplace_back(p, p + c);
    if (dv.back().empty()) dv.back().push_back(0.0);
    return dv.back().data();
  }
  void assign(const gfr_feeder_desc* s) {
    d = *s;
    const size_t n = s->n_bus > 0 ? s->n_bus : 0, nl = s->n_levels > 0 ? s->n_levels : 0, L = s->n_load > 0 ? s->n_load : 0,
                 G = s->n_gen > 0 ? s->n_gen : 0, Bt = s->n_bat > 0 ? s->n_bat : 0;
    iv.reserve(32); dv.reserve(32);                       // the inner vectors must not move once pointed at
    d.order = keep_i(s->order, n); d.parent = keep_i(s->parent, n); d.level_ptr = keep_i(s->level_ptr, nl + 1);
    d.child_ptr = keep_i(s->child_ptr, n + 1); d.child_idx = keep_i(s->child_idx, n ? n - 1 : 0);
    d.lane_of = keep_i(s->lane_of, n); d.bus_type = keep_i(s->bus_type, n);
    d.vm_set = keep_d(s->vm_set, n); d.g = keep_d(s->g, n); d.b = keep_d(s->b, n); d.gdiag = keep_d(s->gdiag, n);
    d.bdiag = keep_d(s->bdiag, n); d.r = keep_d(s->r, n); d.x = keep_d(s->x, n); d.line_of = keep_i(s->line_of, n);
    d.from_is_parent = keep_i(s->from_is_parent, n); d.rating = keep_d(s->rating, n);
    d.load_bus = keep_i(s->load_bus, L); d.load_base = keep_d(s->load_base, L); d.load_p = keep_d(s->load_p, L);
    d.load_q = keep_d(s->load_q, L); d.gen_type = keep_i(s->gen_type, G); d.gen_bus = keep_i(s->gen_bus, G);
    d.gen_cap = keep_d(s->gen_cap, G); d.gen_p0 = keep_d(s->gen_p0, G); d.gen_p1 = keep_d(s->gen_p1, G);
    d.gen_p2 = keep_d(s->gen_p2, G); d.bat_bus = keep_i(s->bat_bus, Bt); d.bat_cap = keep_d(s->bat_cap, Bt);
    d.bat_rating = keep_d(s->bat_rating, Bt); d.bat_eff = keep_d(s->bat_eff, Bt); d.bat_soc0 = keep_d(s->bat_soc0, Bt);
    d.load_profile = keep_d(s->load_profile, 24);
    const size_t t = s->n_tie > 0 ? s->n_tie : 0;
    d.tie_line = keep_i(s->tie_line, t); d.tie_from = keep_i(s->tie_from, t); d.tie_to = keep_i(s->tie_to, t);
    d.tie_r = keep_d(s->tie_r, t); d.tie_x = keep_d(s->tie_x, t); d.tie_rating = keep_d(s->tie_rating, t);
    d.tie_zinv = keep_d(s->tie_zinv, 2 * t * t);
  }
};

// structure checks of a description: root at k = 0, parents before children, one slack bus, child lists
inline std::string check_feeder_desc(const gfr_feeder_desc* d) {
  const int n = d->n_bus, nl = d->n_levels, L = d->n_load, G = d->n_gen, Bt = d->n_bat;
  if (n < 1 || nl < 1 || L < 0 || G < 0 || Bt < 0) return "bad feeder dimensions";
  if (n > 65535) return "more than 65535 buses";
  if (!(d->s_base > 0.0)) return "s_base must be > 0";
  if (!d->order || !d->parent || !d->level_ptr || !d->child_ptr || (n > 1 && !d->child_idx) || !d->bus_type || !d->vm_set || !d->g ||
      !d->b || !d->gdiag || !d->bdiag || !d->r || !d->x || !d->line_of || !d->from_is_parent ||
      !d->rating || !d->load_profile)
    return "missing topology array";
  if ((L && (!d->load_bus || !d->load_base || !d->load_p || !d->load_q)) ||
      (G && (!d->gen_type || !d->gen_bus || !d->gen_cap || !d->gen_p0 || !d->gen_p1 || !d->gen_p2)) ||
      (Bt && (!d->bat_bus || !d->bat_cap || !d->bat_rating || !d->bat_eff || !d->bat_soc0)))
    return "missing component array";
  if (d->parent[0] != -1) return "k = 0 must be the root (parent -1)";
  if (d->level_ptr[0] != 0 || d->level_ptr[nl] != n) return "level_ptr must span [0, n]";
  if (d->level_ptr[1] != 1) return "level 0 must hold the root only";
  const int nt = d->n_tie;
  if (nt < 0 || nt > 4095) return "n_tie out of range";
  if (nt && (!d->tie_line || !d->tie_from || !d->tie_to || !d->tie_r || !d->tie_x || !d->tie_rating || !d->tie_zinv))
    return "missing tie array";
  const int m_all = n - 1 + nt;
  std::vector<int32_t> seen_ref(n, 0), seen_line(m_all > 0 ? m_all : 0, 0), seen_child(n, 0);
  std::vector<int> level(n, 0);
  for (int l = 0; l < nl; ++l) {
    if (d->level_ptr[l + 1] <= d->level_ptr[l]) return "empty level";
    for (int k = d->level_ptr[l]; k < d->level_ptr[l + 1]; ++k) level[k] = l;
  }
  int n_slack = 0;
  if (d->child_ptr[0] != 0 || d->child_ptr[n] != n - 1) return "child_ptr must span [0, n-1]";
  for (int k = 0; k < n; ++k) {
    if (d->order[k] < 0 || d->order[k] >= n || seen_ref[d->order[k]]++) return "order is not a permutation";
    if (d->child_ptr[k + 1] < d->child_ptr[k]) return "child_ptr must be non-decreasing";
    if (d->bus_type[k] != GFR_BUS_SLACK && d->bus_type[k] != GFR_BUS_PV && d->bus_type[k] != GFR_BUS_PQ)
      return "unknown bus_type";
    n_slack += d->bus_type[k] == GFR_BUS_SLACK;
    for (int q = d->child_ptr[k]; q < d->child_ptr[k + 1]; ++q) {
      const int c = d->child_idx[q];
      if (c <= k || c >= n || d->parent[c] != k || seen_child[c]++) return "child_idx does not match parent";
    }
    if (k > 0) {
      const int p = d->parent[k];
      if (p < 0 || p >= k) return "parent must precede its child in level order";
      if (level[p] >= level[k]) return "a bus must sit in a later level than its parent";
      const int li = d->line_of[k];
      if (li < 0 || li >= m_all || seen_line[li]++) return "line_of is not a permutation of the lines";
      if (!(d->g[k] == d->g[k]) || !(d->b[k] == d->b[k]) || (d->g[k] == 0.0 && d->b[k] == 0.0))
        return "branch with zero / NaN admittance";
    }
  }
  for (int k = 1; k < n; ++k) if (!seen_child[k]) return "child_idx does not list every bus";
  for (int i = 0; i < nt; ++i) {
    const int li = d->tie_line[i];
    if (li < 0 || li >= m_all || seen_line[li]++) return "tie_line and line_of do not partition the lines";
    if (d->tie_from[i] < 0 || d->tie_from[i] >= n || d->tie_to[i] < 0 || d->tie_to[i] >= n || d->tie_from[i] == d->tie_to[i])
      return "tie end out of range";
    if (!(d->tie_r[i] == d->tie_r[i]) || !(d->tie_x[i] == d->tie_x[i]) || (d->tie_r[i] == 0.0 && d->tie_x[i] == 0.0))
      return "tie with zero / NaN impedance";
  }
  if (n_slack != 1) return "exactly one slack bus is required";
  for (int l = 0; l < L; ++l) if (d->load_bus[l] < 0 || d->load_bus[l] >= n) return "load_bus out of range";
  for (int g = 0; g < G; ++g) {
    if (d->gen_bus[g] < 0 || d->gen_bus[g] >= n) return "gen_bus out of range";
    if (d->gen_type[g] != GFR_GEN_SOLAR && d->gen_type[g] != GFR_GEN_WIND) return "unknown gen_type";
  }
  for (int b = 0; b < Bt; ++b) if (d->bat_bus[b] < 0 || d->bat_bus[b] >= n) return "bat_bus out of range";
  if (d->n_pool < 0 || d->n_pool > n) return "n_pool must be in [0, n]";
  return std::string();
}

// The elimination schedule on `lanes` lanes: row and lane of every bus.  The description's levels are
// the rows and its lane_of the lanes whenever they fit (every level at most `lanes` wide, lanes
// distinct inside a level); otherwise levels are cut into rows of `lanes` buses in index order.
struct Schedule {
  int nrows = 0;
  bool as_described = false;               // rows == the description's levels
  std::vector<int> row, lane;              // per bus
};
inline Schedule make_schedule(const gfr_feeder_desc* d, int lanes) {
  const int n = d->n_bus, nl = d->n_levels;
  Schedule s;
  s.row.assign(n, 0); s.lane.assign(n, 0);
  bool fits = true;
  for (int l = 0; l < nl && fits; ++l) {
    const int k0 = d->level_ptr[l], k1 = d->level_ptr[l + 1];
    if (k1 - k0 > lanes) { fits = false; break; }
    if (d->lane_of) {
      unsigned long long seen[4] = {0, 0, 0, 0};
      for (int k = k0; k < k1; ++k) {
        const int ln = d->lane_of[k];
        if (ln < 0 || ln >= lanes || (seen[ln >> 6] >> (ln & 63) & 1ull)) { fits = false; break; }
        seen[ln >> 6] |= 1ull << (ln & 63);
      }
    }
  }
  if (fits) {
    s.as_described = true;
    s.nrows = nl;
    for (int l = 0; l < nl; ++l)
      for (int k = d->level_ptr[l]; k < d->level_ptr[l + 1]; ++k) {
        s.row[k] = l;
        s.lane[k] = d->lane_of ? d->lane_of[k] : k - d->level_ptr[l];
      }
    return s;
  }
  int r = 0;
  for (int l = 0; l < nl; ++l) {
    const int k0 = d->level_ptr[l], k1 = d->level_ptr[l + 1];
    for (int k = k0; k < k1; ++k) { s.row[k] = r + (k - k0) / lanes; s.lane[k] = (k - k0) % lanes; }
    r += (k1 - k0 + lanes - 1) / lanes;
  }
  s.nrows = r;
  return s;
}

// returns an empty string on success, the complaint otherwise
// flat_start_factors: include the factorisation of the flat-start Jacobian (96 B per position)
inline std::string build_feeder_image(const gfr_feeder_desc* d, int lanes, int solver, FeederImage* out,
                                      bool flat_start_factors = true) {
  {
    std::string complaint = check_feeder_desc(d);
    if (!complaint.empty()) return complaint;
  }
  if (lanes < 1 || lanes > 256) return "lanes out of range";
  const bool newton = solver == GFR_SOLVER_NEWTON;
  const int n = d->n_bus, nl = d->n_levels, L = d->n_load, G = d->n_gen, Bt = d->n_bat, nt = d->n_tie;
  if (newton && nt)
    return "the feeder has loop-closing lines: the tree-ordered Newton-Raphson takes radial feeders "
           "(GFR_SOLVER_SWEEP restores the loops by compensation)";
  FeederImage* f = out;
  f->lanes = lanes; f->solver = solver; f->n_reg_edges = 0; f->has_pv = false;
  {
    // depth of the tree rooted at its center: the longest path (in edges) is found leaf -> root from the two
    // deepest subtrees of every bus (children come after their parent in level order)
    std::vector<int> h(n, 0);
    int diam = 0;
    for (int k = n - 1; k > 0; --k) {
      const int p = d->parent[k];
      diam = std::max(diam, h[p] + h[k] + 1);
      h[p] = std::max(h[p], h[k] + 1);
    }
    f->center_depth = (diam + 1) / 2 + 1;
  }
  Layout& lay = f->lay;
  lay = Layout{};
  lay.n = n; lay.nl = nl; lay.L = L; lay.G = G; lay.Bt = Bt; lay.A = Bt + G; lay.m = n - 1 + nt; lay.n_tie = nt;
  lay.D = 2 * n + 2 * lay.m + 1 + 2 * L + G + 2 * Bt;
  lay.n_src = L + G + Bt; lay.R = R_BAT + 2 * Bt; lay.n_noise = 4 + L;
  lay.s_base = d->s_base;
  lay.inv_s_base = 1.0 / d->s_base;
  double lp = 0.0;
  for (int l = 0; l < L; ++l) lp = lp + d->load_p[l];   // sequential, as grid_env.py:744
  lay.load_p_sum = lp;

  // ---- schedule positions: Newton = (row, lane); sweep = the bus index itself
  Schedule sch;
  std::vector<int> pos(n);
  if (newton) {
    sch = make_schedule(d, lanes);
    for (int k = 0; k < n; ++k) pos[k] = sch.row[k] * lanes + sch.lane[k];
    lay.nrows = sch.nrows;
    lay.P = sch.nrows * lanes;
    if (lay.P > 65535) return "more than 65535 schedule positions";
  } else {
    for (int k = 0; k < n; ++k) pos[k] = k;
    lay.nrows = nl;
    lay.P = n;
  }
  const int P = lay.P;
  std::vector<int> bus_at(P, -1);
  for (int k = 0; k < n; ++k) bus_at[pos[k]] = k;

  std::vector<int32_t> flags(n), rank(n), rankp(n), bol(lay.m > 0 ? lay.m : 0);
  for (int i = 0; i < nt; ++i) bol[d->tie_line[i]] = -1 - i;          // a tie: its index, negated
  for (int k = 0; k < n; ++k) {
    int fl = FL_VALID;
    if (d->bus_type[k] == GFR_BUS_PQ) fl |= FL_PQ;
    else fl |= FL_FIXED_VM;
    if (d->bus_type[k] != GFR_BUS_SLACK) fl |= FL_THETA;
    if (d->bus_type[k] == GFR_BUS_PV) f->has_pv = true;
    if (d->from_is_parent[k]) fl |= FL_FROM_IS_PARENT;
    flags[k] = fl;
    rank[d->order[k]] = k;
    rankp[d->order[k]] = pos[k];
    if (k > 0) bol[d->line_of[k]] = pos[k];
  }
  // the slack bus and the path from it to the root of the elimination tree (sweep)
  {
    int ks = 0;
    for (int k = 0; k < n; ++k) if (d->bus_type[k] == GFR_BUS_SLACK) ks = k;
    lay.k_slack = ks;
    for (int k = ks; k > 0; k = d->parent[k]) flags[k] |= FL_SLACK_PATH;
  }
  // ---- register hand-off (Newton): a bus eliminated right after one of its children on the same lane
  //      takes that child's Schur terms from registers, and hands its correction back the same way
  std::vector<int> heir(n, -1);
  if (newton) {
    for (int k = 1; k < n; ++k) {
      const int p = d->parent[k];
      if (sch.row[k] == sch.row[p] + 1 && sch.lane[k] == sch.lane[p] && heir[p] < 0) {
        heir[p] = k;
        flags[p] |= FL_C_REG;
        flags[k] |= FL_P_REG;
        ++f->n_reg_edges;
      }
    }
    flags[0] |= FL_P_REG;               // the root has no parent: its "correction from above" is the zero its lane starts with
  }
  // ---- sibling chains (Newton): the children handed over through shared memory ("pool children") are summed
  //      along chains instead of by their parent alone.  Taken in elimination order (rows nrows-1 .. 0), each
  //      pool child ABSORBS the partial sum of one sibling eliminated in a strictly earlier row - it adds that
  //      sibling's slot to its own hand-off and writes the sum into its own slot - and the heir absorbs one more
  //      into the hand-off it passes in registers.  Siblings of one row run in parallel and cannot chain; each
  //      starts or continues its own chain.  The parent gathers only the chain TAILS nobody absorbed: at most as
  //      many as it has pool children in one row, instead of all of them on one lane.
  //      Groups of fewer than CHAIN_MIN_LANES lanes run without chains: every pool child is a tail of its own.
  std::vector<int> absorb(n, -1), reader_row(n, -1);       // the sibling whose partial a bus absorbs; row its slot is read in
  std::vector<std::vector<int>> tails(n);                  // per bus: the chain tails it gathers, in summation order
  if (newton) {
    std::vector<int> kids;
    for (int k = 0; k < n; ++k) {
      kids.clear();
      for (int q = d->child_ptr[k]; q < d->child_ptr[k + 1]; ++q)
        if (d->child_idx[q] != heir[k]) kids.push_back(d->child_idx[q]);
      if (lanes < CHAIN_MIN_LANES) {
        tails[k] = kids;
        for (int c : kids) reader_row[c] = sch.row[k];
        continue;
      }
      std::stable_sort(kids.begin(), kids.end(), [&](int a, int b) { return sch.row[a] > sch.row[b]; });
      std::vector<int>& open = tails[k];                   // chain tails so far, oldest first
      for (size_t i = 0; i < kids.size();) {
        const int r = sch.row[kids[i]];
        size_t j = i;
        size_t avail = open.size();                        // tails of earlier rows: the ones open before this row
        std::vector<int> started;
        for (; j < kids.size() && sch.row[kids[j]] == r; ++j) {
          const int c = kids[j];
          if (avail > 0) {
            absorb[c] = open.front();
            reader_row[open.front()] = r;
            open.erase(open.begin());
            --avail;
          }
          started.push_back(c);
        }
        open.insert(open.end(), started.begin(), started.end());
        i = j;
      }
      // the heir (row of k + 1, the last row before k's) absorbs the oldest tail unless that one shares its row
      if (heir[k] >= 0 && !open.empty() && sch.row[open.front()] > sch.row[heir[k]]) {
        absorb[heir[k]] = open.front();
        reader_row[open.front()] = sch.row[heir[k]];
        open.erase(open.begin());
      }
      for (int c : open) reader_row[c] = sch.row[k];
    }
  }
  // ---- pool plan (Newton): a slot for every bus whose hand-off goes through shared memory, held from its own
  //      row up to the row that reads it (the next link of its chain, or its parent).  Slots are handed out row by
  //      row; a slot read (released) in one row is reused by LATER rows only, so the group barrier that ends a row
  //      orders every read before the next write.
  std::vector<int32_t> pool_slot(n, 0);
  lay.n_pool = 1;
  if (newton) {
    std::vector<std::vector<int>> by_row(sch.nrows), read_in(sch.nrows);
    for (int k = 0; k < n; ++k) {
      by_row[sch.row[k]].push_back(k);
      if (reader_row[k] >= 0) read_in[reader_row[k]].push_back(k);
    }
    std::vector<int> free_slots;
    int np = 0;
    for (int r = sch.nrows - 1; r >= 0; --r) {
      for (int k : by_row[r]) {
        if (flags[k] & FL_P_REG) continue;            // handed over in registers (or the root)
        if (!free_slots.empty()) {
          auto it = std::min_element(free_slots.begin(), free_slots.end());
          pool_slot[k] = *it;
          free_slots.erase(it);
        } else {
          pool_slot[k] = np++;
        }
      }
      for (int k : read_in[r]) free_slots.push_back(pool_slot[k]);
    }
    lay.n_pool = std::max(np, 1);
  }
  // ---- correction plan (Newton, back-substitution, root -> leaf): a bus with pool children writes its correction
  //      once, into a slot every such child reads in its own row.  The slot is held from the parent's row to the
  //      last of those children's rows, and reused from the row after that on.  This pass writes nothing else
  //      into the pool, and group barriers separate it from the leaf -> root passes.
  std::vector<int32_t> kids_x_slot(n, -1), x_slot(n, 0);
  if (newton) {
    std::vector<int> last_read(n, -1);
    for (int k = 1; k < n; ++k)
      if (k != heir[d->parent[k]]) last_read[d->parent[k]] = std::max(last_read[d->parent[k]], sch.row[k]);
    std::vector<std::vector<int>> by_row(sch.nrows), freed_after(sch.nrows);
    for (int k = 0; k < n; ++k)
      if (last_read[k] >= 0) { by_row[sch.row[k]].push_back(k); freed_after[last_read[k]].push_back(k); }
    std::vector<int> free_slots;
    int np = 0;
    for (int r = 0; r < sch.nrows; ++r) {
      if (r > 0)
        for (int k : freed_after[r - 1]) free_slots.push_back(kids_x_slot[k]);
      for (int k : by_row[r]) {
        if (!free_slots.empty()) {
          auto it = std::min_element(free_slots.begin(), free_slots.end());
          kids_x_slot[k] = *it;
          free_slots.erase(it);
        } else {
          kids_x_slot[k] = np++;
        }
      }
    }
    for (int k = 1; k < n; ++k)
      if (k != heir[d->parent[k]]) x_slot[k] = kids_x_slot[d->parent[k]];
    lay.n_pool = std::max(lay.n_pool, np);
    if (d->n_pool > lay.n_pool) lay.n_pool = d->n_pool;      // the caller asks for more (padding experiments)
    if (lay.n_pool > FL_POOL_MASK) return "more than 4095 pool slots";
  }

  ImageBuilder ib;
  // ---- per-position records + tail lists (the slots of the chain tails a bus gathers, in the order every pass
  //      sums them in: after the heir's hand-off)
  std::vector<int32_t> sched(4 * (size_t)P, 0), child_slot;
  std::vector<int32_t> topo(4 * (size_t)n);
  for (int p = 0; p < P; ++p) {
    const int k = bus_at[p];
    if (k < 0) continue;
    const int kp = k > 0 ? d->parent[k] : 0;
    const int begin = (int)child_slot.size();
    for (int c : tails[k]) child_slot.push_back(pool_slot[c]);
    const int n_tails = (int)tails[k].size();
    if (n_tails > 65535) return "more than 65535 chain tails on one bus";
    sched[4 * p + 0] = (int32_t)((uint32_t)k | ((uint32_t)kp << 16));
    if (begin > REC_LIST_MASK) return "child lists too long";
    sched[4 * p + 1] = (int32_t)((uint32_t)begin | ((uint32_t)(kids_x_slot[k] + 1) << REC_KIDX_SHIFT));
    sched[4 * p + 2] = (int32_t)((uint32_t)flags[k] | ((uint32_t)pool_slot[k] << FL_POOL_SHIFT) | ((uint32_t)x_slot[k] << FL_XSLOT_SHIFT));
    sched[4 * p + 3] = (int32_t)((uint32_t)n_tails | ((uint32_t)(absorb[k] >= 0 ? pool_slot[absorb[k]] + 1 : 0) << 16));
  }
  for (int k = 0; k < n; ++k) {
    topo[4 * k + 0] = k > 0 ? d->parent[k] : 0;
    topo[4 * k + 1] = d->child_ptr[k];
    topo[4 * k + 2] = d->child_ptr[k + 1];
    topo[4 * k + 3] = flags[k];
  }
  lay.o_sched = ib.add_i(sched.data(), 4 * P);
  // injection sources per POSITION: loads, then generators, then batteries (reference accumulation order)
  std::vector<int32_t> inj_ptr(P + 1, 0), inj_idx(lay.n_src);
  {
    std::vector<int> cnt(P, 0);
    for (int l = 0; l < L; ++l) cnt[pos[d->load_bus[l]]]++;
    for (int g = 0; g < G; ++g) cnt[pos[d->gen_bus[g]]]++;
    for (int b = 0; b < Bt; ++b) cnt[pos[d->bat_bus[b]]]++;
    for (int p = 0; p < P; ++p) inj_ptr[p + 1] = inj_ptr[p] + cnt[p];
    std::vector<int> fill(inj_ptr.begin(), inj_ptr.end() - 1);
    for (int l = 0; l < L; ++l) inj_idx[fill[pos[d->load_bus[l]]]++] = l;
    for (int g = 0; g < G; ++g) inj_idx[fill[pos[d->gen_bus[g]]]++] = L + g;
    for (int b = 0; b < Bt; ++b) inj_idx[fill[pos[d->bat_bus[b]]]++] = L + G + b;
  }
  lay.o_rank = ib.add_i(rank.data(), n);
  lay.o_rankp = newton ? ib.add_i(rankp.data(), n) : lay.o_rank;
  lay.o_branch_of_line = ib.add_i(bol.data(), lay.m);
  lay.o_inj_ptr = ib.add_i(inj_ptr.data(), P + 1);
  lay.o_inj_idx = ib.add_i(inj_idx.data(), lay.n_src);
  lay.o_gen_type = ib.add_i(d->gen_type, G);
  lay.o_child_ent = lay.o_child_slot = lay.o_topo = lay.o_child_idx = -1;
  lay.o_kids = -1;
  lay.o_rowrec = -1; lay.sw_rows = 0;
  if (newton) {
    lay.o_child_slot = ib.add_i(child_slot.data(), (int)child_slot.size());
    if (lanes >= GFR_WIDE_GROUP_MIN_LANES) {
      // CTA-wide groups: the first 8 chain tails' slots of every position, 16 bits each, in list order
      std::vector<int32_t> kids(4 * (size_t)P, 0);
      for (int p = 0; p < P; ++p) {
        const uint32_t begin = (uint32_t)sched[4 * p + 1] & (uint32_t)REC_LIST_MASK;
        const uint32_t nt = (uint32_t)sched[4 * p + 3] & 0xffffu;
        for (uint32_t j = 0; j < nt && j < 8; ++j) {
          const uint32_t slot = (uint32_t)child_slot[begin + j];
          kids[4 * p + (j >> 1)] = (int32_t)((uint32_t)kids[4 * p + (j >> 1)] | (slot << (16 * (j & 1))));
        }
      }
      lay.o_kids = ib.add_i(kids.data(), 4 * P);
    }
  } else {
    lay.o_topo = ib.add_i(topo.data(), 4 * n);
    lay.o_child_idx = ib.add_i(d->child_idx, n - 1);
    if (lanes > 1) {
      // several lanes: the levels cut into rows of at most `lanes` buses, one record per (row, lane)
      const Schedule sw = make_schedule(d, lanes);
      std::vector<int32_t> rowrec(4 * (size_t)sw.nrows * lanes, 0);
      for (int k = 0; k < n; ++k) {
        int32_t* r = &rowrec[4 * ((size_t)sw.row[k] * lanes + sw.lane[k])];
        r[0] = (int32_t)((uint32_t)k | ((uint32_t)(k > 0 ? d->parent[k] : 0) << 16));
        r[1] = d->child_ptr[k];
        r[2] = d->child_ptr[k + 1];
        r[3] = flags[k];
      }
      lay.sw_rows = sw.nrows;
      lay.o_rowrec = ib.add_i(rowrec.data(), (int)rowrec.size());
    }
  }
  lay.o_tie_ends = lay.o_tie_ptr = lay.o_tie_inc = lay.o_tie_y = lay.o_tie_z = lay.o_tie_rating = lay.o_tie_zinv = -1;
  if (nt) {
    // tie ends (from, to) as ef indices, and per bus the ties that meet it: entry = tie << 1 | (1 if the bus is the to-end)
    std::vector<int32_t> ends(2 * (size_t)nt), tptr(n + 1, 0), tinc(2 * (size_t)nt);
    std::vector<int> cnt(n, 0);
    for (int i = 0; i < nt; ++i) { ends[2 * i] = d->tie_from[i]; ends[2 * i + 1] = d->tie_to[i]; cnt[d->tie_from[i]]++; cnt[d->tie_to[i]]++; }
    for (int k = 0; k < n; ++k) tptr[k + 1] = tptr[k] + cnt[k];
    std::vector<int> fill(tptr.begin(), tptr.end() - 1);
    for (int i = 0; i < nt; ++i) { tinc[fill[d->tie_from[i]]++] = i << 1; tinc[fill[d->tie_to[i]]++] = (i << 1) | 1; }
    lay.o_tie_ends = ib.add_i(ends.data(), 2 * nt);
    lay.o_tie_ptr = ib.add_i(tptr.data(), n + 1);
    lay.o_tie_inc = ib.add_i(tinc.data(), 2 * nt);
  }
  const int n_int_padded = ((int)ib.ints.size() + 3) / 4 * 4;      // keep the doubles 16-byte aligned
  const int dbase = n_int_padded / 2;
  // paired arrays by position (one 128-bit load each): branch (g, b), diagonal (Re, Im Y_kk), branch (r, x)
  std::vector<double> gb(2 * (size_t)P, 0.0), gbd(2 * (size_t)P, 0.0), rx(2 * (size_t)P, 0.0), rating(P, 0.0), vm_set(P, 1.0);
  for (int k = 0; k < n; ++k) {
    const int p = pos[k];
    gb[2 * p] = k > 0 ? d->g[k] : 0.0; gb[2 * p + 1] = k > 0 ? d->b[k] : 0.0;   // the root has no branch
    gbd[2 * p] = d->gdiag[k]; gbd[2 * p + 1] = d->bdiag[k];
    rx[2 * p] = d->r[k]; rx[2 * p + 1] = d->x[k];
    rating[p] = d->rating[k];
    vm_set[p] = d->vm_set[k];
  }
  lay.o_gb = dbase + ib.add_d(gb.data(), 2 * P);
  lay.o_gbd = lay.o_rx = lay.o_f0 = -1;
  if (newton) lay.o_gbd = dbase + ib.add_d(gbd.data(), 2 * P);
  else lay.o_rx = dbase + ib.add_d(rx.data(), 2 * P);
  // Factorisation of the flat-start Jacobian (the first Newton iteration of every instance):
  // the same leaf -> root block elimination the kernel runs, done once here.
  if (newton) {
    std::vector<double> f0(12 * (size_t)P, 0.0), C(4 * (size_t)n, 0.0);
    bool ok = flat_start_factors;
    for (int k = n - 1; k >= 0 && ok; --k) {           // children have larger indices: done before their parent
      const bool th = d->bus_type[k] != GFR_BUS_SLACK, pq = d->bus_type[k] == GFR_BUS_PQ;
      const double vk = pq ? 1.0 : d->vm_set[k];
      auto vm = [&](int j) { return d->bus_type[j] == GFR_BUS_PQ ? 1.0 : d->vm_set[j]; };
      const double v2 = vk * vk;
      double Pc = d->gdiag[k] * v2, Qc = -d->bdiag[k] * v2;
      if (k > 0) { const double a = vk * vm(d->parent[k]); Pc += -d->g[k] * a; Qc += d->b[k] * a; }
      for (int q = d->child_ptr[k]; q < d->child_ptr[k + 1]; ++q) {
        const int c = d->child_idx[q];
        const double a = vk * vm(c);
        Pc += -d->g[c] * a; Qc += d->b[c] * a;
      }
      double d00 = -Qc - d->bdiag[k] * v2, d01 = Pc + d->gdiag[k] * v2, d10 = Pc - d->gdiag[k] * v2,
             d11 = Qc - d->bdiag[k] * v2;
      for (int q = d->child_ptr[k]; q < d->child_ptr[k + 1]; ++q) {
        const double* cc = &C[4 * (size_t)d->child_idx[q]];
        d00 -= cc[0]; d01 -= cc[1]; d10 -= cc[2]; d11 -= cc[3];
      }
      const double a = k > 0 ? vk * vm(d->parent[k]) : 0.0;
      const double gk = k > 0 ? d->g[k] : 0.0, bk = k > 0 ? d->b[k] : 0.0;
      const double ga = -gk * a, al = bk * a, gl = -gk * a, ll = bk * a;      // sin = 0 at a flat start
      double u00 = al, u01 = ga, u10 = -ga, u11 = al;
      if (!th) { d00 = 1.0; d01 = 0.0; u00 = u01 = 0.0; }
      if (!pq) { d10 = 0.0; d11 = 1.0; u10 = u11 = 0.0; }
      const double det = d00 * d11 - d01 * d10;
      if (det == 0.0 || !(det == det)) { ok = false; break; }
      const double inv = 1.0 / det;
      const double i00 = d11 * inv, i01 = -d01 * inv, i10 = -d10 * inv, i11 = d00 * inv;
      const double m00 = i00 * u00 + i01 * u10, m01 = i00 * u01 + i01 * u11,
                   m10 = i10 * u00 + i11 * u10, m11 = i10 * u01 + i11 * u11;
      // six 16-byte fields per position, field-major (field f of position p at f0[2 * (f * P + p)]): the lanes
      // of a row read consecutive 16-byte units
      const int p = pos[k];
      auto put = [&](int fld, double a0, double a1) {
        f0[2 * ((size_t)fld * P + p)] = a0; f0[2 * ((size_t)fld * P + p) + 1] = a1;
      };
      put(0, i00, i01); put(1, i10, i11);
      put(2, m00, m01); put(3, m10, m11);
      put(4, ll, gl);
      put(5, Pc, Qc);                                  // calculated injections of the flat profile
      double* cc = &C[4 * (size_t)k];
      cc[0] = ll * m00 + gl * m10; cc[1] = ll * m01 + gl * m11;
      cc[2] = -gl * m00 + ll * m10; cc[3] = -gl * m01 + ll * m11;
    }
    lay.o_f0 = ok ? dbase + ib.add_d(f0.data(), 12 * P) : -1;     // singular at the flat start: no shortcut
  }
  if (nt) {
    std::vector<double> ty(2 * (size_t)nt), tz(2 * (size_t)nt);
    for (int i = 0; i < nt; ++i) {
      const double r = d->tie_r[i], x = d->tie_x[i], z2 = r * r + x * x;
      ty[2 * i] = r / z2; ty[2 * i + 1] = -x / z2;            // y = 1 / (r + jx), as power_flow.py:62
      tz[2 * i] = r; tz[2 * i + 1] = x;
    }
    lay.o_tie_y = dbase + ib.add_d(ty.data(), 2 * nt);
    lay.o_tie_z = dbase + ib.add_d(tz.data(), 2 * nt);
    lay.o_tie_zinv = dbase + ib.add_d(d->tie_zinv, 2 * nt * nt);
    lay.o_tie_rating = dbase + ib.add_d(d->tie_rating, nt);
  }
  lay.o_rating = dbase + ib.add_d(rating.data(), P);
  lay.o_vm_set = dbase + ib.add_d(vm_set.data(), P);
  lay.o_load_base = dbase + ib.add_d(d->load_base, L);
  lay.o_gen_cap = dbase + ib.add_d(d->gen_cap, G);
  lay.o_gen_p0 = dbase + ib.add_d(d->gen_p0, G);
  lay.o_gen_p1 = dbase + ib.add_d(d->gen_p1, G);
  lay.o_gen_p2 = dbase + ib.add_d(d->gen_p2, G);
  lay.o_bat_cap = dbase + ib.add_d(d->bat_cap, Bt);
  lay.o_bat_rating = dbase + ib.add_d(d->bat_rating, Bt);
  lay.o_bat_eff = dbase + ib.add_d(d->bat_eff, Bt);
  lay.o_profile = dbase + ib.add_d(d->load_profile, 24);
  const size_t img_bytes = ((size_t)n_int_padded * 4 + ib.dbls.size() * 8 + 15) / 16 * 16;
  lay.img_bytes = (int)img_bytes;
  std::vector<unsigned char> img(img_bytes, 0);
  std::memcpy(img.data(), ib.ints.data(), ib.ints.size() * 4);
  std::memcpy(img.data() + (size_t)n_int_padded * 4, ib.dbls.data(), ib.dbls.size() * 8);

  std::vector<double> load_pq(2 * (size_t)L + 1, 0.0);
  for (int l = 0; l < L; ++l) { load_pq[2 * l] = d->load_p[l]; load_pq[2 * l + 1] = d->load_q[l]; }

  f->root_is_slack = d->bus_type[0] == GFR_BUS_SLACK;
  f->img.swap(img);
  f->load_pq.swap(load_pq);
  return std::string();
}

}  // namespace gfr
