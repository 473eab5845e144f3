// kino_search.h -- KinoAstar::plan (front_end/src/kino_astar.cpp:67-236; helpers front_end/include/front_end/kino_astar.h:177-291) over
// the UnevenMap occupancy grids, written once for the host (csrc/kino_astar.cpp: one search per thread) and the device
// (csrc/ualm_front_end.cu: one search per warp).  Templated on the trigonometry (TrigLibm / TrigDet, csrc/dubins.h).
//
// Behaviour kept from the reference, because every one of these decides which path comes out:
//   * hybrid-state grid: cell = (x, y) of the map and a yaw bin of kino_astar/yaw_resolution (NOT the map's) -- kino_astar.h:190-194;
//   * the motion primitives are built by the same floating-point running sums (kino_astar.cpp:128-136);
//   * a node whose cost improves while OPEN is rewritten in place and NOT re-sorted in the queue (kino_astar.cpp:213-224).  OPEN is
//     the std::priority_queue of the reference restated: Heap below is libstdc++'s stl_heap.h (__push_heap, pop_heap ->
//     __adjust_heap -> __push_heap) over node indices compared through the nodes' current f_score, so equal-f ties, stale orderings
//     and NaN-cost nodes resolve exactly as there;
//   * the goal test is "within oneshot_range and the Dubins one-shot is collision free", tried on the node at the top of the queue
//     before it is popped (kino_astar.cpp:107-121); the result is start .. node, then the one-shot samples (kino_astar.h:268-291);
//   * the node pool holds X * Y nodes (kino_astar.h:177-185); the insert that fills it ends the search without a path.
// The expanded-node map (std::unordered_map in the reference) is an open-addressing table: only find / insert are observable.
//
// Float -> int conversions go through floor_to_int: x86-64's cvttsd2si, what the reference's (int)std::floor compiles to, returns
// INT_MIN for NaN and out-of-range values, and the v = 0 steering primitives produce NaN states whose key (INT_MIN, INT_MIN, INT_MIN)
// decides which later primitives are skipped.  CUDA's conversion returns 0 for NaN and saturates, so both sides use the helper.
#pragma once
#include <limits.h>
#include <math.h>
#include <stdint.h>

#include "dubins.h"
#include "ualm.h"

namespace ualm_kino {

// (int)floor(x) as x86-64 computes it: INT_MIN when x is NaN or floor(x) is outside int's range
UALM_KHD int floor_to_int(double x)
{
    const double f = floor(x);
    return (f >= -2147483648.0 && f < 2147483648.0) ? (int)f : INT_MIN;
}

// the smallest non-negative value congruent to c modulo n (n > 0): what `while (c > n - 1) c -= n; while (c < 0) c += n;` ends with.
// Written in closed form because a NaN state reaches it with c = INT_MIN + w: 33 M iterations of the loop
UALM_KHD int wrap_index(int c, int n)
{
    const int r = c % n;
    return r < 0 ? r + n : r;
}

struct MapView {
    ualm_map_geom_t g;
    const float *cells;
    const double *cells64;
    const uint8_t *occ3, *occ2;
    double xy_inv, yaw_inv;

    // uneven_map.h:411-417
    UALM_KHD void posToIndex(const double p[3], int id[3]) const
    {
        id[0] = floor_to_int((p[0] - g.origin[0]) * xy_inv);
        id[1] = floor_to_int((p[1] - g.origin[1]) * xy_inv);
        id[2] = floor_to_int((p[2] - g.origin[2]) * yaw_inv);
    }
    // uneven_map.h:437-454
    UALM_KHD bool inMap(const double p[3]) const
    {
        for (int k = 0; k < 3; k++) if (p[k] < g.origin[k] + 1e-4) return false;
        for (int k = 0; k < 3; k++) if (p[k] > g.max_boundary[k] - 1e-4) return false;
        return true;
    }
    // uneven_map.h:456-471
    UALM_KHD bool inMapIdx(const int id[3]) const
    {
        if (id[0] < 0 || id[1] < 0 || id[2] < 0) return false;
        return !(id[0] > g.voxel_num[0] - 1 || id[1] > g.voxel_num[1] - 1 || id[2] > g.voxel_num[2] - 1);
    }
    UALM_KHD size_t addr(int x, int y, int w) const { return (size_t)x * g.voxel_num[1] * g.voxel_num[2] + (size_t)y * g.voxel_num[2] + w; }
    // uneven_map.h:473-488
    UALM_KHD int occupancy(const double p[3]) const
    {
        int id[3];
        posToIndex(p, id);
        if (!inMapIdx(id)) return -1;
        return (int)occ3[addr(id[0], id[1], id[2])];
    }
    // uneven_map.h:490-500
    UALM_KHD int occupancyXY(const double p[3]) const
    {
        int id[3];
        posToIndex(p, id);
        if (!inMapIdx(id)) return -1;
        return (int)occ2[(size_t)id[0] * g.voxel_num[1] + id[1]];
    }
    UALM_KHD double sigma_at(int x, int y, int w) const
    {
        const size_t a = addr(x, y, w);
        return cells64 ? cells64[4 * a + 1] : (double)cells[4 * a + 1];
    }
    // UnevenMap::getTerrainSig = the sigma component of getTerrain's trilinear blend (uneven_map.h:154-201, 389-396).  A NaN state
    // passes inMap (every comparison is false) and lands here: idx = INT_MIN, x / y clamp to 0, the yaw index wraps, the result is NaN
    template <class T> UALM_KHD double terrainSig(const double pos[3]) const
    {
        if (!inMap(pos)) return 0.0;
        double pm[3] = {pos[0] - 0.5 * g.xy_resolution, pos[1] - 0.5 * g.xy_resolution, pos[2] - 0.5 * g.yaw_resolution};
        while (pm[2] < -M_PI) pm[2] += 2 * M_PI;       // normSO2, uneven_map.cpp:64-71 (pos is in the map: at most one turn)
        while (pm[2] > M_PI) pm[2] -= 2 * M_PI;
        int idx[3];
        posToIndex(pm, idx);
        const double ip[3] = {(idx[0] + 0.5) * g.xy_resolution + g.origin[0], (idx[1] + 0.5) * g.xy_resolution + g.origin[1],
                              (idx[2] + 0.5) * g.yaw_resolution + g.origin[2]};
        double diff[3] = {(pos[0] - ip[0]) * xy_inv, (pos[1] - ip[1]) * xy_inv, 0.0};
        diff[2] = T::atan2(T::sin(pos[2] - ip[2]), T::cos(pos[2] - ip[2])) * yaw_inv;
        double v[2][2][2];
        for (int x = 0; x < 2; x++)
            for (int y = 0; y < 2; y++)
                for (int w = 0; w < 2; w++) {
                    int c[3] = {idx[0] + x, idx[1] + y, idx[2] + w};
                    c[0] = c[0] < g.voxel_num[0] - 1 ? c[0] : g.voxel_num[0] - 1;       // boundIndex, uneven_map.h:398-409
                    c[0] = c[0] > 0 ? c[0] : 0;
                    c[1] = c[1] < g.voxel_num[1] - 1 ? c[1] : g.voxel_num[1] - 1;
                    c[1] = c[1] > 0 ? c[1] : 0;
                    c[2] = wrap_index(c[2], g.voxel_num[2]);
                    v[x][y][w] = sigma_at(c[0], c[1], c[2]);
                }
        const double v00 = v[0][0][0] * (1 - diff[0]) + v[1][0][0] * diff[0];
        const double v01 = v[0][0][1] * (1 - diff[0]) + v[1][0][1] * diff[0];
        const double v10 = v[0][1][0] * (1 - diff[0]) + v[1][1][0] * diff[0];
        const double v11 = v[0][1][1] * (1 - diff[0]) + v[1][1][1] * diff[0];
        const double v0 = v00 * (1 - diff[1]) + v10 * diff[1];
        const double v1 = v01 * (1 - diff[1]) + v11 * diff[1];
        return v0 * (1 - diff[2]) + v1 * diff[2];
    }
};

// false when the map is incomplete
inline bool view_of(const ualm_astar_map_t *m, MapView &v)
{
    if (!m || !m->geom || (!m->cells && !m->cells64) || !m->occ3 || !m->occ2) return false;
    v.g = *m->geom; v.cells = m->cells; v.cells64 = m->cells64; v.occ3 = m->occ3; v.occ2 = m->occ2;
    v.xy_inv = 1.0 / m->geom->xy_resolution; v.yaw_inv = 1.0 / m->geom->yaw_resolution;
    return true;
}

enum : char { ST_CLOSE = 'a', ST_OPEN = 'b', ST_NOT_EXPAND = 'c' };
struct Node {
    int index[3];
    double state[3];
    double input[2];
    double g_score, f_score;
    char node_state;
    int parent;        // pool index, -1 for the start
};

// kino_astar.h:196-207.  |a| <= pi + one primitive's turn for every state the search makes
UALM_KHD double norm_angle(double a)
{
    while (a > M_PI) a -= 6.283185307179586;
    while (a < -M_PI) a += 6.283185307179586;
    return a;
}
// kino_astar.h:220-244
template <class T> UALM_KHD void state_transit(const ualm_astar_params_t &p, const double s0[3], double s1[3], const double in[2], double dt)
{
    const double v = in[0], delta = in[1];
    const double s = v * dt;
    const double y = s * T::tan(delta) / p.wheel_base;
    if (fabs(delta) > 1e-4) {
        const double r = s / y;
        s1[0] = s0[0] + r * (T::sin(s0[2] + y) - T::sin(s0[2]));
        s1[1] = s0[1] - r * (T::cos(s0[2] + y) - T::cos(s0[2]));
        s1[2] = s0[2] + y;
        s1[2] = norm_angle(s1[2]);
    } else {
        s1[0] = s0[0] + s * T::cos(s0[2]);
        s1[1] = s0[1] + s * T::sin(s0[2]);
        s1[2] = s0[2];
    }
}

// the expansion inputs (v, steer) of kino_astar.cpp:128-136, by the same running sums; returns their number (at most `cap` written)
UALM_KHD int build_inputs(const ualm_astar_params_t &p, double *inputs, int cap)
{
    int n = 0;
    for (double v = 0; v <= p.max_vel + 1e-3; v += 0.5 * p.max_vel)
        for (double steer = -p.max_steer; steer <= p.max_steer + 1e-3; steer += 0.5 * p.max_steer) {
            if (n < cap) { inputs[2 * n] = v; inputs[2 * n + 1] = steer; }
            n++;
        }
    return n;
}

// libstdc++'s binary heap (bits/stl_heap.h) over node indices with the comparator ByF(a, b) = a.f_score > b.f_score: the top is the
// node with the smallest f among those the (possibly stale) order puts there, exactly as std::priority_queue<Node*, ..., ByF>
struct Heap {
    int *h;
    int n;
    UALM_KHD static bool byf(const Node *pool, int a, int b) { return pool[a].f_score > pool[b].f_score; }
    UALM_KHD void push_hole(const Node *pool, int hole, int top, int value)        // std::__push_heap
    {
        int parent = (hole - 1) / 2;
        while (hole > top && byf(pool, h[parent], value)) {
            h[hole] = h[parent];
            hole = parent;
            parent = (hole - 1) / 2;
        }
        h[hole] = value;
    }
    UALM_KHD void push(const Node *pool, int value)                                // push_back + std::push_heap
    {
        h[n] = value;
        n++;
        push_hole(pool, n - 1, 0, h[n - 1]);
    }
    UALM_KHD void pop(const Node *pool)                                            // std::pop_heap + pop_back
    {
        if (n > 1) {
            const int len = n - 1;                   // __pop_heap(first, last - 1, last - 1)
            const int value = h[len];
            h[len] = h[0];
            int hole = 0, second = 0;                // std::__adjust_heap(first, 0, len, value)
            while (second < (len - 1) / 2) {
                second = 2 * (second + 1);
                if (byf(pool, h[second], h[second - 1])) second--;
                h[hole] = h[second];
                hole = second;
            }
            if ((len & 1) == 0 && second == (len - 2) / 2) {
                second = 2 * (second + 1);
                h[hole] = h[second - 1];
                hole = second - 1;
            }
            push_hole(pool, hole, 0, value);
        }
        n--;
    }
};

// open addressing, linear probing, keys (x, y, yaw bin) read back from the nodes; capacity a power of two >= 2 x the pool
struct Table {
    int *slot;        // node index or -1
    unsigned mask;
    UALM_KHD static unsigned hash(const int k[3])
    {
        return ((unsigned)k[0] * 73856093u) ^ ((unsigned)k[1] * 19349663u) ^ ((unsigned)k[2] * 83492791u);
    }
    UALM_KHD int find(const Node *pool, const int k[3]) const
    {
        for (unsigned i = hash(k) & mask;; i = (i + 1) & mask) {        // the table is never more than half full
            const int s = slot[i];
            if (s < 0) return -1;
            if (pool[s].index[0] == k[0] && pool[s].index[1] == k[1] && pool[s].index[2] == k[2]) return s;
        }
    }
    UALM_KHD void insert(const Node *pool, int node)       // only called after find returned -1
    {
        unsigned i = hash(pool[node].index) & mask;
        while (slot[i] >= 0) i = (i + 1) & mask;
        slot[i] = node;
    }
};
inline unsigned table_capacity(long long pool_size)
{
    unsigned c = 1;
    while ((long long)c < 2 * pool_size) c <<= 1;
    return c;
}

// one primitive applied to the current node: everything that does not depend on the expanded-node map
struct Prim {
    double state[3];
    double input[2];
    double g, f;
    int id[3];
    int ok;            // in the map and collision free
};

// the result of a search
enum { KS_SEARCHING = 0, KS_FOUND = 1, KS_NO_PATH = 2, KS_POOL_FULL = 3, KS_SHOT_OVERFLOW = 4 };

template <class T> struct Search {
    MapView map;
    ualm_astar_params_t p;
    double yaw_inv;
    double rho;                       // the one-shot's turning radius
    Node *pool;
    int pool_size;
    Heap open;
    Table closed;                     // expanded_nodes
    int use_node_num, iter_num;

    UALM_KHD void state_to_index(const double s[3], int id[3]) const    // kino_astar.h:190-194
    {
        map.posToIndex(s, id);
        id[2] = floor_to_int((norm_angle(s[2]) + M_PI) * yaw_inv);
    }
    UALM_KHD double heu(const double a[3], const double b[3]) const     // kino_astar.h:215-218
    {
        const double tie_breaker = 1.0 + 1.0 / 10000;
        const double dx = a[0] - b[0], dy = a[1] - b[1];
        return tie_breaker * sqrt(dx * dx + dy * dy);
    }
    UALM_KHD bool near_goal(const Node &n, const double goal[3]) const
    {
        const double ex = n.state[0] - goal[0], ey = n.state[1] - goal[1];
        return sqrt(ex * ex + ey * ey) < p.oneshot_range;
    }

    // kino_astar.cpp:85-104: the entry checks and the start node; false when start or goal is occupied
    UALM_KHD bool begin(const double start[3], const double goal[3])
    {
        open.n = 0;
        use_node_num = 0; iter_num = 0;
        if (map.occupancy(start) == 1) return false;
        if (map.occupancyXY(goal) == 1) return false;
        Node &cur = pool[0];
        cur.parent = -1;
        cur.state[0] = start[0]; cur.state[1] = start[1]; cur.state[2] = norm_angle(start[2]);
        state_to_index(cur.state, cur.index);
        cur.g_score = 0.0;
        cur.input[0] = 0.0; cur.input[1] = 0.0;
        cur.f_score = p.lambda_heu * heu(cur.state, goal);
        cur.node_state = ST_OPEN;
        open.push(pool, 0);
        use_node_num += 1;
        closed.insert(pool, 0);
        return true;
    }

    // kino_astar.h:246-258: the Dubins curve from the node to the goal, sampled at l = 0, ci, ci + ci, ... (a running sum, as there)
    // while l <= its length.  Samples [k0, k1) of at most `cap`, every `stride`-th from k0 (a lane's share); returns the number of
    // samples of the whole curve
    UALM_KHD int shot_samples(const double s1[3], const double goal[3], double *out, int cap, int k0, int stride, bool *hit) const
    {
        const ualm_dubins::Path path = ualm_dubins::shortest<T>(s1, goal, rho);
        const double len = rho * path.length();
        int k = 0;
        for (double l = 0.0; l <= len; l += p.collision_interval, k++) {
            if (k >= cap) return k + 1;                                // cannot be stored: reported as an overflow
            if (k < k0 || (k - k0) % stride) continue;
            ualm_dubins::interpolate<T>(s1, path, rho, l / len, out + 3 * k);
            if (map.occupancyXY(out + 3 * k) == 1) *hit = true;
        }
        return k;
    }

    // kino_astar.cpp:128-205 for one input: the child state, its collision test (times t = ct, ct + ct, ... <= T: a running sum) and costs
    UALM_KHD void primitive(const Node &cur, const double input[2], const double goal[3], Prim &o) const
    {
        o.input[0] = input[0]; o.input[1] = input[1];
        o.ok = 0;
        state_transit<T>(p, cur.state, o.state, input, p.time_interval);
        if (!map.inMap(o.state)) return;
        state_to_index(o.state, o.id);
        const double arc = input[0] * p.time_interval;
        const double temp_ct = p.collision_interval / arc * p.time_interval;
        for (double t = temp_ct; t <= p.time_interval + 1e-3; t += temp_ct) {       // v = 0: temp_ct = inf, no sample
            double xt[3];
            state_transit<T>(p, cur.state, xt, input, t);
            if (map.occupancyXY(xt) == 1) return;
        }
        double g = 0.0;
        g += p.weight_r2 * arc;
        g += p.weight_so2 * fabs(input[1]) * arc;
        g += p.weight_v_change * fabs(input[0] - cur.input[0]);
        g += p.weight_delta_change * fabs(input[1] - cur.input[1]);
        g += p.weight_sigma * map.terrainSig<T>(o.state);
        g += cur.g_score;
        o.g = g;
        o.f = g + p.lambda_heu * heu(o.state, goal);
        o.ok = 1;
    }

    // kino_astar.cpp:176-224 for one primitive of node `cur`, in primitive order: skip if CLOSE, insert + push, or rewrite in place.
    // Returns false when this insert filled the pool ("run out of memory.")
    UALM_KHD bool apply(int cur, const Prim &o)
    {
        if (!o.ok) return true;
        int pro = closed.find(pool, o.id);
        if (pro >= 0 && pool[pro].node_state == ST_CLOSE) return true;
        if (pro < 0) {
            pro = use_node_num;
            Node &n = pool[pro];
            n.index[0] = o.id[0]; n.index[1] = o.id[1]; n.index[2] = o.id[2];
            n.state[0] = o.state[0]; n.state[1] = o.state[1]; n.state[2] = o.state[2];
            n.f_score = o.f; n.g_score = o.g;
            n.input[0] = o.input[0]; n.input[1] = o.input[1];
            n.parent = cur;
            n.node_state = ST_OPEN;
            open.push(pool, pro);
            closed.insert(pool, pro);
            use_node_num++;
            if (use_node_num == pool_size) return false;
        } else if (pool[pro].node_state == ST_OPEN) {
            if (o.g < pool[pro].g_score) {
                Node &n = pool[pro];
                n.index[0] = o.id[0]; n.index[1] = o.id[1]; n.index[2] = o.id[2];
                n.state[0] = o.state[0]; n.state[1] = o.state[1]; n.state[2] = o.state[2];
                n.f_score = o.f; n.g_score = o.g;
                n.input[0] = o.input[0]; n.input[1] = o.input[1];
                n.parent = cur;
            }
        }
        return true;
    }

    // retrievePath (kino_astar.h:268-291): the number of nodes from the start to `node`
    UALM_KHD int chain_length(int node) const
    {
        int n = 0;
        for (int k = node; k >= 0 && n <= pool_size; k = pool[k].parent) n++;
        return n;
    }
    // ... and the polyline: those nodes' states from the start, then the one-shot samples
    UALM_KHD void retrieve(int node, int chain, const double *shot, int nshot, double *out) const
    {
        int k = node;
        for (int i = chain - 1; i >= 0; i--, k = pool[k].parent)
            for (int c = 0; c < 3; c++) out[3 * i + c] = pool[k].state[c];
        for (int i = 0; i < 3 * nshot; i++) out[3 * chain + i] = shot[i];
    }

    // KinoAstar::plan (kino_astar.cpp:67-236), one thread.  inputs: build_inputs' list (nin entries); shot: room for shot_cap samples.
    // Returns a KS_* status; on KS_FOUND *node is the node the one-shot left from and *nshot the number of its samples in `shot`
    UALM_KHD int plan(const double start[3], const double goal[3], const double *inputs, int nin, double *shot, int shot_cap, int *node, int *nshot)
    {
        if (!begin(start, goal)) return KS_NO_PATH;
        // every pass closes one node and at most pool_size nodes exist: the loop ends after at most pool_size passes
        for (int pass = 0; open.n > 0 && pass <= pool_size; pass++) {
            const int cur = open.h[0];
            if (near_goal(pool[cur], goal)) {
                bool hit = false;
                const int ns = shot_samples(pool[cur].state, goal, shot, shot_cap, 0, 1, &hit);
                if (ns > shot_cap) return KS_SHOT_OVERFLOW;
                if (!hit) { *node = cur; *nshot = ns; return KS_FOUND; }
            }
            open.pop(pool);
            pool[cur].node_state = ST_CLOSE;
            iter_num += 1;
            for (int i = 0; i < nin; i++) {
                Prim o;
                primitive(pool[cur], inputs + 2 * i, goal, o);
                if (!apply(cur, o)) return KS_POOL_FULL;
            }
        }
        return KS_NO_PATH;
    }
};

// the one-shot's samples fit in floor((6 pi rho + oneshot_range) / collision_interval) + 3: every Dubins word is at most 6 pi rho
// longer than the distance, which is below oneshot_range when the one-shot is tried
inline int shot_capacity(const ualm_astar_params_t &p, double rho)
{
    const double n = floor((6.0 * M_PI * rho + p.oneshot_range) / p.collision_interval) + 3.0;
    return n < 1e7 ? (int)n : -1;
}

}  // namespace ualm_kino
