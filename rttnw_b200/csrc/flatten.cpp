// flatten.cpp — scene description -> flat records, transform chains and SAH BVHs.
//
// What the reference does per ray (src/math/hittable.rs): List::hit scans every top-level
// item (:153-163), wrappers Translate/YRotate re-express the ray (:599-605, :686-697) and
// BvhTree::hit recurses through Arc<dyn Hittable> (:355-368). Here the same tree is turned,
// once, into:
//   * leaf records (sphere / moving sphere / rectangle / box; a Cube is one box item for the
//     traversal plus its six rectangles, in the order of Cube::new :560-569, for the hit record),
//   * one transform chain per distinct wrapper path (outermost op first),
//   * ONE BVH over the world, in world space (a wrapped primitive carries the index of its chain
//     and world bounds; its f64 test pushes the ray through the chain), and one per general
//     ConstantMedium boundary; the media themselves are a short list with world bounds that
//     every ray checks before it traverses (device_types.h, DMedium).
// Bounds are geometrically correct rotated bounds — NOT YRotate::new's (:654-672, SURVEY Q15),
// which the reference never uses for culling either.
#include "flatten.hpp"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>

namespace rtx {

void Aabb::reset() {
    for (int i = 0; i < 3; ++i) { lo[i] = INFINITY; hi[i] = -INFINITY; }
}
void Aabb::grow(const Aabb& o) {
    for (int i = 0; i < 3; ++i) { lo[i] = std::fmin(lo[i], o.lo[i]); hi[i] = std::fmax(hi[i], o.hi[i]); }
}
void Aabb::grow_point(const double p[3]) {
    for (int i = 0; i < 3; ++i) { lo[i] = std::fmin(lo[i], p[i]); hi[i] = std::fmax(hi[i], p[i]); }
}
double Aabb::half_area() const {
    double dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
    if (!(dx >= 0) || !(dy >= 0) || !(dz >= 0)) return 0.0;
    return dx * dy + dy * dz + dz * dx;
}

BvhPolicy BvhPolicy::from_env() {
    BvhPolicy p;
    if (const char* v = std::getenv("RTX_BVH_LEAF")) p.max_leaf = std::min(kBvhMaxLeafLimit, std::max(1, std::atoi(v)));
    if (const char* v = std::getenv("RTX_BVH_CPRIM")) p.cost_prim = std::max(0.1, std::atof(v));
    return p;
}

namespace {

struct Item {
    Record rec;
    Aabb box;
    bool solo() const { return false; }  // (no record kind needs a leaf of its own any more)
};

float round_down(double v) {
    float f = (float)v;
    if ((double)f > v) f = std::nextafterf(f, -INFINITY);
    return f;
}
float round_up(double v) {
    float f = (float)v;
    if ((double)f < v) f = std::nextafterf(f, INFINITY);
    return f;
}

// ---------------------------------------------------------------------------
// Binned-SAH BVH over a set of items; appends nodes and (reordered) records.
// ---------------------------------------------------------------------------
struct BvhBuilder {
    std::vector<BvhNode>& nodes;
    std::vector<Record>& records;
    std::vector<Item>& items;
    static constexpr int kBins = kBvhBins;
    const BvhPolicy pol = BvhPolicy::from_env();

    struct Tmp {
        Aabb box;
        int left = -1, right = -1;
        int first = 0, count = 0;
        int32_t leaf_code = 0;  // set by emit_leaf (leaf codes are negative)
    };
    std::vector<Tmp> tmp;
    // what the builder touches per primitive, packed and partitioned in place (the Items are 144 bytes apart)
    struct Prim {
        double lo[3], hi[3], c[3];
        int idx;
        bool solo;
    };
    std::vector<Prim> prims;

    BvhBuilder(std::vector<BvhNode>& n, std::vector<Record>& r, std::vector<Item>& it) : nodes(n), records(r), items(it) {}

    int build_range(int lo, int hi) {
        Tmp t;
        t.box.reset();
        Aabb cbox;
        cbox.reset();
        bool any_solo = false;
        for (int i = lo; i < hi; ++i) {
            const Prim& p = prims[(size_t)i];
            for (int a = 0; a < 3; ++a) {
                t.box.lo[a] = std::fmin(t.box.lo[a], p.lo[a]); t.box.hi[a] = std::fmax(t.box.hi[a], p.hi[a]);
                cbox.lo[a] = std::fmin(cbox.lo[a], p.c[a]); cbox.hi[a] = std::fmax(cbox.hi[a], p.c[a]);
            }
            any_solo = any_solo || p.solo;
        }
        t.first = lo;
        t.count = hi - lo;
        int n = hi - lo;
        int self = (int)tmp.size();
        tmp.push_back(t);
        if (n <= 1) return self;

        // one pass fills the bins of all three axes (small nodes — most of them — get as many bins as primitives)
        const int nb = std::min(kBins, std::max(2, n));
        Aabb bin_box[3][kBins];
        int bin_n[3][kBins];
        double scale[3];
        for (int a = 0; a < 3; ++a) {
            scale[a] = cbox.hi[a] > cbox.lo[a] ? nb / (cbox.hi[a] - cbox.lo[a]) : 0.0;
            for (int b = 0; b < nb; ++b) { bin_box[a][b].reset(); bin_n[a][b] = 0; }
        }
        for (int i = lo; i < hi; ++i) {
            const Prim& p = prims[(size_t)i];
            for (int a = 0; a < 3; ++a) {
                if (scale[a] == 0.0) continue;
                int b = std::min(nb - 1, std::max(0, (int)((p.c[a] - cbox.lo[a]) * scale[a])));
                Aabb& bb = bin_box[a][b];
                for (int k = 0; k < 3; ++k) { bb.lo[k] = std::fmin(bb.lo[k], p.lo[k]); bb.hi[k] = std::fmax(bb.hi[k], p.hi[k]); }
                bin_n[a][b]++;
            }
        }
        double best_cost = INFINITY;
        int best_axis = -1, best_split = -1;
        for (int axis = 0; axis < 3; ++axis) {
            if (scale[axis] == 0.0) continue;
            double right_area[kBins];
            int right_n[kBins];
            Aabb acc;
            acc.reset();
            int cnt = 0;
            for (int b = nb - 1; b >= 1; --b) {
                acc.grow(bin_box[axis][b]);
                cnt += bin_n[axis][b];
                right_area[b] = acc.half_area();
                right_n[b] = cnt;
            }
            acc.reset();
            cnt = 0;
            for (int b = 0; b < nb - 1; ++b) {
                acc.grow(bin_box[axis][b]);
                cnt += bin_n[axis][b];
                if (cnt == 0 || right_n[b + 1] == 0) continue;
                double cost = acc.half_area() * cnt + right_area[b + 1] * right_n[b + 1];
                if (cost < best_cost) { best_cost = cost; best_axis = axis; best_split = b; }
            }
        }
        double area = t.box.half_area();
        bool make_leaf = false;
        if (any_solo) {
            make_leaf = false;  // the traversal switches space on these: one per leaf
        } else if (best_axis < 0) {
            make_leaf = n <= pol.max_leaf;  // all centroids coincide
        } else if (n <= pol.max_leaf) {
            double split_cost = pol.cost_traverse + (area > 0 ? best_cost / area : 0.0) * pol.cost_prim;
            make_leaf = n * pol.cost_prim <= split_cost;
        }
        if (make_leaf) return self;

        int mid;
        if (best_axis < 0) {
            mid = lo + n / 2;  // degenerate: split the index range
        } else {
            const double cmin = cbox.lo[best_axis], sc = scale[best_axis];
            auto it = std::partition(prims.begin() + lo, prims.begin() + hi, [&](const Prim& p) {
                int b = std::min(nb - 1, std::max(0, (int)((p.c[best_axis] - cmin) * sc)));
                return b <= best_split;
            });
            mid = (int)(it - prims.begin());
            if (mid == lo || mid == hi) mid = lo + n / 2;
        }
        int l = build_range(lo, mid);
        int r = build_range(mid, hi);
        tmp[(size_t)self].left = l;
        tmp[(size_t)self].right = r;
        return self;
    }

    static void set_child_box(BvhNode& n, int which, const Aabb& b) {
        float lo[3], hi[3];
        for (int i = 0; i < 3; ++i) { lo[i] = round_down(b.lo[i]); hi[i] = round_up(b.hi[i]); }
        if (which == 0) {
            n.c0x[0] = lo[0]; n.c0x[1] = hi[0]; n.c0y[0] = lo[1]; n.c0y[1] = hi[1]; n.c0z[0] = lo[2]; n.c0z[1] = hi[2];
        } else {
            n.c1x[0] = lo[0]; n.c1x[1] = hi[0]; n.c1y[0] = lo[1]; n.c1y[1] = hi[1]; n.c1z[0] = lo[2]; n.c1z[1] = hi[2];
        }
    }
    static void set_child_empty(BvhNode& n, int which) {
        Aabb e;
        for (int i = 0; i < 3; ++i) { e.lo[i] = FLT_MAX; e.hi[i] = -FLT_MAX; }
        set_child_box(n, which, e);
        (which == 0 ? n.child0 : n.child1) = kEmptyChild;
    }
    int32_t emit_leaf(Tmp& t) {
        int32_t first = (int32_t)records.size();
        for (int i = 0; i < t.count; ++i) records.push_back(items[(size_t)prims[(size_t)(t.first + i)].idx].rec);
        t.leaf_code = ~((first << 4) | t.count);
        return t.leaf_code;
    }
    int depth = 0;  // inner nodes on the longest root-to-leaf path (set by build)
    int32_t emit(int ti, int level = 1) {  // ti is an inner tmp node
        depth = std::max(depth, level);
        int32_t idx = (int32_t)nodes.size();
        nodes.push_back(BvhNode{});
        int kids[2] = {tmp[(size_t)ti].left, tmp[(size_t)ti].right};
        for (int k = 0; k < 2; ++k) {
            const bool leaf = tmp[(size_t)kids[k]].left < 0;
            int32_t ref = leaf ? emit_leaf(tmp[(size_t)kids[k]]) : emit(kids[k], level + 1);
            BvhNode& n = nodes[(size_t)idx];
            set_child_box(n, k, tmp[(size_t)kids[k]].box);
            (k == 0 ? n.child0 : n.child1) = ref;
        }
        return idx;
    }
    // The same tree with every other level collapsed: a 4-wide node is TWO consecutive BvhNode entries (128 bytes,
    // even index), its up to four children the grandchildren of the binary node (a child that is a leaf stays a
    // child). Child references are leaf codes (the binary tree's: the records are shared) or the index of the first
    // entry of another wide node. Call after emit(). Returns that index; wide_depth counts wide levels.
    int wide_depth = 0;
    int32_t emit_wide(int ti, int level = 1) {
        wide_depth = std::max(wide_depth, level);
        int kids[4], nk = 0;
        const int two[2] = {tmp[(size_t)ti].left, tmp[(size_t)ti].right};
        for (int k = 0; k < 2; ++k) {
            const Tmp& c = tmp[(size_t)two[k]];
            if (c.left < 0) {
                kids[nk++] = two[k];
            } else {
                kids[nk++] = c.left;
                kids[nk++] = c.right;
            }
        }
        if (nodes.size() & 1) {  // 128-byte alignment of the pair: an unreferenced filler entry
            nodes.push_back(BvhNode{});
            set_child_empty(nodes.back(), 0);
            set_child_empty(nodes.back(), 1);
        }
        const int32_t idx = (int32_t)nodes.size();
        nodes.push_back(BvhNode{});
        nodes.push_back(BvhNode{});
        for (int j = 0; j < 4; ++j) {
            if (j >= nk) {
                set_child_empty(nodes[(size_t)idx + (size_t)(j >> 1)], j & 1);
                continue;
            }
            const bool leaf = tmp[(size_t)kids[j]].left < 0;
            const int32_t ref = leaf ? tmp[(size_t)kids[j]].leaf_code : emit_wide(kids[j], level + 1);
            BvhNode& n = nodes[(size_t)idx + (size_t)(j >> 1)];
            set_child_box(n, j & 1, tmp[(size_t)kids[j]].box);
            ((j & 1) == 0 ? n.child0 : n.child1) = ref;
        }
        return idx;
    }
    int root_tmp = -1;  // the root of the last build() when it is an inner node
    // Returns the root node index; `bounds` gets the f64 bounds of everything.
    int32_t build(Aabb& bounds) {
        bounds.reset();
        depth = 1;
        for (const auto& it : items) bounds.grow(it.box);
        prims.resize(items.size());
        tmp.reserve(2 * items.size() + 1);
        for (size_t i = 0; i < items.size(); ++i) {
            Prim& p = prims[i];
            const Aabb& b = items[i].box;
            for (int a = 0; a < 3; ++a) { p.lo[a] = b.lo[a]; p.hi[a] = b.hi[a]; p.c[a] = 0.5 * (b.lo[a] + b.hi[a]); }
            p.idx = (int)i;
            p.solo = items[i].solo();
        }
        if (items.empty()) {
            int32_t idx = (int32_t)nodes.size();
            nodes.push_back(BvhNode{});
            set_child_empty(nodes[(size_t)idx], 0);
            set_child_empty(nodes[(size_t)idx], 1);
            return idx;
        }
        int root = build_range(0, (int)items.size());
        if (tmp[(size_t)root].left < 0) {  // the whole set is one leaf
            int32_t idx = (int32_t)nodes.size();
            nodes.push_back(BvhNode{});
            int32_t ref = emit_leaf(tmp[(size_t)root]);
            set_child_box(nodes[(size_t)idx], 0, tmp[(size_t)root].box);
            nodes[(size_t)idx].child0 = ref;
            set_child_empty(nodes[(size_t)idx], 1);
            return idx;
        }
        root_tmp = root;
        return emit(root);
    }
};

// ---------------------------------------------------------------------------
// Tree walk
// ---------------------------------------------------------------------------
// One closest-hit query space: the world, or the boundary of a ConstantMedium. Every primitive in
// it carries the index of its wrapper chain and WORLD-space bounds, so one BVH serves the whole
// space and the traversal never switches coordinate systems (the f64 test of a wrapped primitive
// pushes the ray through the chain first).
struct World {
    bool is_boundary = false;
    std::vector<Item> items;
    std::vector<Item> media;
};

struct Flattener {
    const rtx_scene_desc& d;
    FlatScene& out;
    std::string& err;
    std::vector<int> first_id;   // per node: first primitive id handed out, -1 = not visited
    std::vector<int> medium_ord; // per MEDIUM node
    std::map<std::vector<int>, int32_t> chain_of_path;  // wrapper path (node indices) -> chain index
    int next_prim = 0, next_medium = 0;
    double t_a = 0, t_b = 1;  // time interval moving-sphere bounds must cover
    bool defer_world = false;
    bool wide_copy = false;  // also emit the 4-wide copy of the world BVH

    Flattener(const rtx_scene_desc& desc, FlatScene& o, std::string& e) : d(desc), out(o), err(e) {}

    bool fail(const std::string& m) { err = m; return false; }

    // object -> world: undo the chain, innermost op first
    static void to_world(const std::vector<XformOp>& chain, double p[3]) {
        for (size_t i = chain.size(); i-- > 0;) {
            const XformOp& op = chain[i];
            if (op.kind == XF_TRANSLATE) {
                p[0] += op.v[0]; p[1] += op.v[1]; p[2] += op.v[2];
            } else {
                double s = op.v[0], c = op.v[1];
                double x = c * p[0] + s * p[2];
                double z = -s * p[0] + c * p[2];
                p[0] = x; p[2] = z;
            }
        }
    }
    // World bounds of an object-space box under `chain`: the geometrically correct rotated bounds, NOT
    // YRotate::new's (hittable.rs:654-672, Q15), padded for the rounding of the rotation arithmetic.
    static Aabb world_box(const Aabb& ob, const std::vector<XformOp>& chain) {
        if (chain.empty()) return ob;
        Aabb wb;
        wb.reset();
        for (int corner = 0; corner < 8; ++corner) {
            double p[3] = {(corner & 1) ? ob.hi[0] : ob.lo[0], (corner & 2) ? ob.hi[1] : ob.lo[1], (corner & 4) ? ob.hi[2] : ob.lo[2]};
            to_world(chain, p);
            wb.grow_point(p);
        }
        for (int i = 0; i < 3; ++i) {
            double pad = 1e-12 * std::fmax(1.0, std::fmax(std::fabs(wb.lo[i]), std::fabs(wb.hi[i])));
            wb.lo[i] -= pad; wb.hi[i] += pad;
        }
        return wb;
    }
    static Aabb world_sphere_box(const double c[3], double r, const std::vector<XformOp>& chain) {
        double w[3] = {c[0], c[1], c[2]};
        to_world(chain, w);  // a sphere is rotation invariant: move the centre
        Aabb b;
        for (int i = 0; i < 3; ++i) {
            double pad = chain.empty() ? 0.0 : 1e-12 * std::fmax(1.0, std::fabs(w[i]) + std::fabs(r));
            b.lo[i] = w[i] - std::fabs(r) - pad; b.hi[i] = w[i] + std::fabs(r) + pad;
        }
        return b;
    }

    // Registers a wrapper path: its ops (for the way out) and their composition (for the way in).
    int32_t chain_index(const std::vector<int>& path, const std::vector<XformOp>& chain) {
        if (chain.empty()) return 0;
        auto it = chain_of_path.find(path);
        if (it != chain_of_path.end()) return it->second;
        DChain c;
        std::memset(&c, 0, sizeof(c));
        c.cs = 1.0;
        c.begin = (int32_t)out.xforms.size();
        c.len = (int32_t)chain.size();
        for (const auto& op : chain) {  // outermost first, the order the wrappers see the ray
            out.xforms.push_back(op);
            if (op.kind == XF_TRANSLATE) {
                c.tx -= op.v[0]; c.ty -= op.v[1]; c.tz -= op.v[2];
            } else {
                double s = op.v[0], k = op.v[1];
                double cs = k * c.cs - s * c.sn, sn = s * c.cs + k * c.sn;
                double tx = k * c.tx - s * c.tz, tz = s * c.tx + k * c.tz;
                c.cs = cs; c.sn = sn; c.tx = tx; c.tz = tz;
            }
        }
        out.chains.push_back(c);
        int32_t idx = (int32_t)out.chains.size() - 1;
        chain_of_path.emplace(path, idx);
        return idx;
    }

    // Rectangle record in its own space + its object-space bounds (Rectangle::bounding_box pads k by 1e-4,
    // hittable.rs:532-546; ranges may be given reversed)
    static Record rect_record(int plane, double a0, double a1, double b0, double b1, double k, int material, int prim_id, int32_t chain, Aabb& ob) {
        Record r;
        std::memset(&r, 0, sizeof(r));
        r.type = REC_RECT_XY + plane;
        r.a = material;
        r.b = prim_id;
        r.c = chain;
        r.d[0] = a0; r.d[1] = a1; r.d[2] = b0; r.d[3] = b1; r.d[4] = k;
        static const int ax0[3] = {0, 0, 1}, ax1[3] = {1, 2, 2}, axk[3] = {2, 1, 0};
        ob.lo[ax0[plane]] = std::fmin(a0, a1); ob.hi[ax0[plane]] = std::fmax(a0, a1);
        ob.lo[ax1[plane]] = std::fmin(b0, b1); ob.hi[ax1[plane]] = std::fmax(b0, b1);
        ob.lo[axk[plane]] = k - 0.0001; ob.hi[axk[plane]] = k + 0.0001;
        return r;
    }

    bool check_material(int m) { return m >= 0 && m < d.n_materials; }

    bool collect(int ni, std::vector<int>& path, std::vector<XformOp>& chain, World& w, int depth) {
        if (ni < 0 || ni >= d.n_nodes) return fail("node index out of range");
        if (depth > 256) return fail("scene tree deeper than 256 (cycle?)");
        const rtx_node& n = d.nodes[ni];
        const double* f = n.f;
        switch (n.kind) {
            case RTX_NODE_SPHERE: {
                if (!check_material(n.material)) return fail("sphere: bad material index");
                if (first_id[(size_t)ni] < 0) first_id[(size_t)ni] = next_prim++;
                Item it;
                std::memset(&it.rec, 0, sizeof(it.rec));
                it.rec.type = REC_SPHERE; it.rec.a = n.material; it.rec.b = first_id[(size_t)ni];
                it.rec.c = chain_index(path, chain);
                for (int i = 0; i < 4; ++i) it.rec.d[i] = f[i];
                it.box = world_sphere_box(f, f[3], chain);
                w.items.push_back(it);
                return true;
            }
            case RTX_NODE_MOVING_SPHERE: {
                if (!check_material(n.material)) return fail("moving sphere: bad material index");
                if (first_id[(size_t)ni] < 0) first_id[(size_t)ni] = next_prim++;
                Item it;
                std::memset(&it.rec, 0, sizeof(it.rec));
                it.rec.type = REC_MSPHERE; it.rec.a = n.material; it.rec.b = first_id[(size_t)ni];
                it.rec.c = chain_index(path, chain);
                double r = f[6], t0 = f[7], t1 = f[8];
                for (int i = 0; i < 3; ++i) { it.rec.d[i] = f[i]; it.rec.d[3 + i] = f[3 + i] - f[i]; }
                it.rec.d[6] = r; it.rec.d[7] = t0; it.rec.d[8] = 1.0 / (t1 - t0);
                // MovingSphere::bounding_box (hittable.rs:233-244) over the shutter interval
                it.box.reset();
                const double ts[2] = {t_a, t_b};
                for (double t : ts) {
                    double c[3];
                    for (int i = 0; i < 3; ++i) c[i] = f[i] + ((t - t0) / (t1 - t0)) * (f[3 + i] - f[i]);
                    it.box.grow(world_sphere_box(c, r, chain));
                }
                w.items.push_back(it);
                return true;
            }
            case RTX_NODE_RECT_XY:
            case RTX_NODE_RECT_XZ:
            case RTX_NODE_RECT_YZ: {
                if (!check_material(n.material)) return fail("rectangle: bad material index");
                if (first_id[(size_t)ni] < 0) first_id[(size_t)ni] = next_prim++;
                Item it;
                Aabb ob;
                it.rec = rect_record(n.kind - RTX_NODE_RECT_XY, f[0], f[1], f[2], f[3], f[4], n.material, first_id[(size_t)ni],
                                     chain_index(path, chain), ob);
                it.box = world_box(ob, chain);
                w.items.push_back(it);
                return true;
            }
            case RTX_NODE_CUBE: {
                if (!check_material(n.material)) return fail("cube: bad material index");
                if (first_id[(size_t)ni] < 0) { first_id[(size_t)ni] = next_prim; next_prim += 6; }
                int id = first_id[(size_t)ni];
                int32_t ch = chain_index(path, chain);
                // Cube::new, hittable.rs:560-569 with Plane::points :451-479: six rectangles, in this order
                Aabb ob[6];
                Record rr[6] = {rect_record(0, f[0], f[3], f[1], f[4], f[2], n.material, id + 0, ch, ob[0]),
                                rect_record(0, f[0], f[3], f[1], f[4], f[5], n.material, id + 1, ch, ob[1]),
                                rect_record(1, f[0], f[3], f[2], f[5], f[1], n.material, id + 2, ch, ob[2]),
                                rect_record(1, f[0], f[3], f[2], f[5], f[4], n.material, id + 3, ch, ob[3]),
                                rect_record(2, f[1], f[4], f[2], f[5], f[0], n.material, id + 4, ch, ob[4]),
                                rect_record(2, f[1], f[4], f[2], f[5], f[3], n.material, id + 5, ch, ob[5])};
                if (f[0] < f[3] && f[1] < f[4] && f[2] < f[5]) {
                    // A proper box: ONE traversal item. A line meets the six rectangles exactly where it enters
                    // and where it leaves the box, so the closest rectangle hit in [t_min, t_max] is the entry
                    // face, or the exit face when the ray starts inside — one f64 slab computation (REC_BOX).
                    // The six rectangle records stay (outside every leaf) for the hit record of the face.
                    Item it;
                    std::memset(&it.rec, 0, sizeof(it.rec));
                    it.rec.type = REC_BOX;
                    it.rec.a = (int32_t)out.records.size();
                    it.rec.b = id;
                    it.rec.c = ch;
                    for (int k = 0; k < 6; ++k) { out.records.push_back(rr[k]); it.rec.d[k] = f[k]; }
                    Aabb cb;
                    for (int k = 0; k < 3; ++k) { cb.lo[k] = f[k] - 0.0001; cb.hi[k] = f[3 + k] + 0.0001; }
                    it.box = world_box(cb, chain);
                    w.items.push_back(it);
                } else {  // degenerate or reversed extents: keep the reference's six rectangles as they are
                    for (int k = 0; k < 6; ++k) {
                        Item it;
                        it.rec = rr[k];
                        it.box = world_box(ob[k], chain);
                        w.items.push_back(it);
                    }
                }
                return true;
            }
            case RTX_NODE_LIST:
            case RTX_NODE_BVH: {
                if (n.n_children < 0 || n.child < 0 || n.child + n.n_children > d.n_children) return fail("list: bad children range");
                for (int c = 0; c < n.n_children; ++c)
                    if (!collect(d.children[n.child + c], path, chain, w, depth + 1)) return false;
                return true;
            }
            case RTX_NODE_TRANSLATE:
            case RTX_NODE_ROTATE_Y: {
                XformOp op;
                std::memset(&op, 0, sizeof(op));
                if (n.kind == RTX_NODE_TRANSLATE) {
                    op.kind = XF_TRANSLATE;
                    op.v[0] = f[0]; op.v[1] = f[1]; op.v[2] = f[2];
                } else {
                    op.kind = XF_ROTATE_Y;
                    const double PI = 3.14159265358979323846;
                    double radians = f[0] * (PI / 180.0);  // f64::to_radians, hittable.rs:641-643
                    op.v[0] = std::sin(radians);
                    op.v[1] = std::cos(radians);
                }
                if (chain.size() >= 16) return fail("more than 16 nested translate/rotate_y wrappers");
                path.push_back(ni);
                chain.push_back(op);
                bool ok = collect(n.child, path, chain, w, depth + 1);
                path.pop_back();
                chain.pop_back();
                return ok;
            }
            case RTX_NODE_MEDIUM: {
                if (w.is_boundary) return fail("ConstantMedium inside a ConstantMedium boundary is not supported");
                if (n.material < 0 || n.material >= d.n_textures) return fail("medium: bad phase texture index");
                if (!(f[0] != 0.0)) return fail("medium: density must be non-zero");
                World bw;
                bw.is_boundary = true;
                if (!collect(n.child, path, chain, bw, depth + 1)) return false;
                if (first_id[(size_t)ni] < 0) {
                    first_id[(size_t)ni] = next_prim++;
                    medium_ord[(size_t)ni] = next_medium++;
                }
                Aabb bounds;
                Item it;
                std::memset(&it.rec, 0, sizeof(it.rec));
                const Item* only = bw.items.size() == 1 ? &bw.items[0] : nullptr;
                int32_t root = -1;
                if (only && only->rec.type == REC_SPHERE && only->rec.c == 0) {
                    // The common case (scenes.rs:282-301): the boundary is one untransformed Sphere. Its two
                    // boundary.hit() calls (hittable.rs:745-752) then reduce to the two roots of one quadratic.
                    for (int i = 0; i < 4; ++i) it.rec.d[4 + i] = only->rec.d[i];
                    bounds = only->box;
                } else if (only && only->rec.type == REC_BOX) {
                    // The other shipped case (scenes.rs:213-233): one Cube, possibly under Translate / YRotate
                    // wrappers — entry and exit of one f64 slab computation in the cube's own space.
                    root = -2 - only->rec.c;
                    for (int i = 0; i < 6; ++i) it.rec.d[4 + i] = only->rec.d[i];
                    bounds = only->box;
                    // the boundary's six face records are never looked at (a medium hit has its own record): drop them
                    if ((size_t)only->rec.a + 6 == out.records.size()) out.records.resize((size_t)only->rec.a);
                } else {
                    root = build_world(bw, bounds);
                }
                it.rec.type = REC_MEDIUM;
                it.rec.a = n.material;
                it.rec.b = first_id[(size_t)ni];
                it.rec.c = root;
                it.rec.d[0] = -1.0 / f[0];  // ConstantMedium::new, hittable.rs:731-735
                it.rec.d[1] = (double)medium_ord[(size_t)ni];
                it.rec.d[2] = (double)chain_index(path, chain);
                it.box = bounds;
                w.media.push_back(it);
                return true;
            }
            default:
                return fail("unknown node kind");
        }
    }

    // Stack entries a traversal can need: the sentinel + one deferred sibling per level of the BVH.
    int32_t build_world(World& w, Aabb& bounds, bool defer = false) {
        int32_t root = -1;
        if (defer && w.items.size() >= 2) {
            // the device builder (lbvh.cuh) makes this BVH: hand over the records in item order and their boxes
            out.world_deferred = true;
            out.world_first_record = (int32_t)out.records.size();
            out.world_count = (int32_t)w.items.size();
            out.world_boxes.reserve(6 * w.items.size());
            bounds.reset();
            for (const auto& it : w.items) {
                out.records.push_back(it.rec);
                for (int i = 0; i < 3; ++i) out.world_boxes.push_back(round_down(it.box.lo[i]));
                for (int i = 0; i < 3; ++i) out.world_boxes.push_back(round_up(it.box.hi[i]));
                bounds.grow(it.box);
            }
        } else {
            BvhBuilder b(out.nodes, out.records, w.items);
            const size_t first_node = out.nodes.size();
            root = b.build(bounds);
            out.max_stack = std::max(out.max_stack, 1 + b.depth + 1);
            if (!w.is_boundary) {
                out.world_first_node = (int32_t)first_node;
                out.world_node_count = (int32_t)(out.nodes.size() - first_node);
                out.world_depth = b.depth;
            }
            if (wide_copy && !w.is_boundary && b.root_tmp >= 0) {  // the 4-wide copy of the world BVH (opt-in traversal, RTX_BVH_WIDE)
                const int32_t wide = b.emit_wide(b.root_tmp);
                if (1 + 3 * b.wide_depth + 1 <= kTraversalStack) out.wide_root = wide;  // up to three siblings deferred per level
            }
        }
        // media: records outside every BVH + a bounds list (only the main world has any)
        for (auto& m : w.media) {
            DMedium dm;
            std::memset(&dm, 0, sizeof(dm));
            for (int i = 0; i < 3; ++i) { dm.lo[i] = round_down(m.box.lo[i]); dm.hi[i] = round_up(m.box.hi[i]); }
            dm.record = (int32_t)out.records.size();
            dm.ordinal = (int32_t)m.rec.d[1];
            {
                float lb = (float)std::fabs(m.rec.d[0]);  // |-1 / density|
                if ((double)lb > std::fabs(m.rec.d[0])) lb = std::nextafterf(lb, 0.f);
                dm.inv_density_lb = lb;
            }
            out.records.push_back(m.rec);
            out.media.push_back(dm);
            bounds.grow(m.box);
        }
        return root;
    }

    bool run() {
        if (!d.nodes || d.n_nodes <= 0) return fail("scene has no nodes");
        if (d.root < 0 || d.root >= d.n_nodes) return fail("root index out of range");
        {
            DChain identity;
            std::memset(&identity, 0, sizeof(identity));
            identity.cs = 1.0;
            out.chains.push_back(identity);
        }
        first_id.assign((size_t)d.n_nodes, -1);
        medium_ord.assign((size_t)d.n_nodes, -1);
        t_a = std::fmin(0.0, d.camera.open_time);
        t_b = std::fmax(1.0, d.camera.close_time);
        // materials / textures / perlin tables in device precision
        out.materials.resize((size_t)d.n_materials);
        for (int i = 0; i < d.n_materials; ++i) {
            const rtx_material& m = d.materials[i];
            DMaterial& o = out.materials[(size_t)i];
            std::memset(&o, 0, sizeof(o));
            if (m.kind < RTX_MAT_LAMBERTIAN || m.kind > RTX_MAT_ISOTROPIC) return fail("unknown material kind");
            bool needs_tex = m.kind == RTX_MAT_LAMBERTIAN || m.kind == RTX_MAT_DIFFUSE_LIGHT || m.kind == RTX_MAT_ISOTROPIC;
            if (needs_tex && (m.texture < 0 || m.texture >= d.n_textures)) return fail("material: bad texture index");
            o.kind = m.kind;
            o.texture = m.texture;
            for (int c = 0; c < 3; ++c) o.albedo[c] = (float)m.albedo[c];
            o.param = (float)(m.kind == RTX_MAT_METAL ? std::fmin(m.param, 1.0) : m.param);  // material.rs:126-131
        }
        out.textures.resize((size_t)d.n_textures);
        for (int i = 0; i < d.n_textures; ++i) {
            const rtx_texture& t = d.textures[i];
            DTexture& o = out.textures[(size_t)i];
            std::memset(&o, 0, sizeof(o));
            o.kind = t.kind; o.a = t.a; o.b = t.b;
            for (int c = 0; c < 4; ++c) o.f[c] = (float)t.f[c];
            switch (t.kind) {
                case RTX_TEX_SOLID: break;
                case RTX_TEX_CHECKER:
                    if (t.a < 0 || t.a >= d.n_textures || t.b < 0 || t.b >= d.n_textures) return fail("checker: bad child texture");
                    break;
                case RTX_TEX_NOISE:
                    if (t.a < 0 || t.a >= d.n_perlins) return fail("noise: bad perlin index");
                    break;
                case RTX_TEX_IMAGE:
                    if (t.a < 0 || t.a >= d.n_images) return fail("image texture: bad image index");
                    break;
                default: return fail("unknown texture kind");
            }
        }
        // _pad = 1 when evaluating the texture needs the surface (u, v): images, and checkers over them
        for (int pass = 0; pass < 8; ++pass)
            for (int i = 0; i < d.n_textures; ++i) {
                DTexture& o = out.textures[(size_t)i];
                if (o.kind == RTX_TEX_IMAGE) o._pad = 1;
                if (o.kind == RTX_TEX_CHECKER) o._pad = out.textures[(size_t)o.a]._pad | out.textures[(size_t)o.b]._pad;
            }
        out.perlins.resize((size_t)d.n_perlins);
        for (int i = 0; i < d.n_perlins; ++i) {
            const rtx_perlin& p = d.perlins[i];
            DPerlin& o = out.perlins[(size_t)i];
            for (int k = 0; k < 256; ++k) {
                o.ranvec[k][0] = (float)p.ranvec[k][0]; o.ranvec[k][1] = (float)p.ranvec[k][1];
                o.ranvec[k][2] = (float)p.ranvec[k][2]; o.ranvec[k][3] = 0.f;
                o.perm[0][k] = (uint8_t)(p.perm_x[k] & 255); o.perm[1][k] = (uint8_t)(p.perm_y[k] & 255);
                o.perm[2][k] = (uint8_t)(p.perm_z[k] & 255);
            }
        }
        World w;
        std::vector<int> path;
        std::vector<XformOp> chain;
        if (!collect(d.root, path, chain, w, 0)) return false;
        out.world_root = build_world(w, out.world_bounds, defer_world);
        if (out.max_stack > kTraversalStack) return fail("BVH deeper than the device traversal stack");
        out.n_media = (int32_t)out.media.size();
        out.n_prims = next_prim;
        camera_view(d.camera, d.background, out.camera);
        return true;
    }
};

}  // namespace

bool flatten_scene(const rtx_scene_desc& desc, FlatScene& out, std::string& err, bool defer_world_bvh, bool wide_copy) {
    out = FlatScene();
    Flattener f(desc, out, err);
    f.defer_world = defer_world_bvh;
    f.wide_copy = wide_copy;
    return f.run();
}

// Camera::new, src/math/camera.rs:32-61, evaluated once on the host in f64.
void camera_view(const rtx_camera& d, const double background[3], CameraView& o) {
    const double PI = 3.14159265358979323846;
    auto sub = [](const double a[3], const double b[3], double r[3]) { for (int i = 0; i < 3; ++i) r[i] = a[i] - b[i]; };
    auto cross = [](const double a[3], const double b[3], double r[3]) {  // vec3.rs:82-88
        r[0] = a[1] * b[2] - a[2] * b[1];
        r[1] = -(a[0] * b[2] - a[2] * b[0]);
        r[2] = a[0] * b[1] - a[1] * b[0];
    };
    auto unit = [](double v[3]) {
        double k = 1.0 / std::sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);
        for (int i = 0; i < 3; ++i) v[i] *= k;
    };
    o.lens_radius = d.aperture / 2.0;
    double theta = d.vertical_fov * PI / 180.0;
    double half_height = std::tan(theta / 2.0);
    double half_width = d.aspect_ratio * half_height;
    double w[3], u[3], v[3];
    sub(d.lookfrom, d.lookat, w);
    unit(w);
    cross(d.view_up, w, u);
    unit(u);
    cross(w, u, v);
    for (int i = 0; i < 3; ++i) {
        o.origin[i] = d.lookfrom[i];
        o.u[i] = u[i]; o.v[i] = v[i];
        o.lower_left[i] = d.lookfrom[i] - half_width * d.focus_distance * u[i] - half_height * d.focus_distance * v[i] -
                          d.focus_distance * w[i];
        o.horizontal[i] = 2.0 * half_width * d.focus_distance * u[i];
        o.vertical[i] = 2.0 * half_height * d.focus_distance * v[i];
        o.background[i] = (float)background[i];
    }
    o.time0 = d.open_time;
    o.time1 = d.close_time;
}

// ---------------------------------------------------------------------------
// Invariant checker (host logic tests): every BVH reachable from the world root
// (and from medium records) must contain its records, in world space.
// ---------------------------------------------------------------------------
namespace {
struct Checker {
    const FlatScene& fs;
    std::string& err;
    std::vector<int> node_seen, rec_seen;
    std::vector<int> leaf_rec = {}, wide_rec = {};  // records found in leaves of the binary trees / of the 4-wide world tree
    bool fail(const std::string& m) { err = m; return false; }

    static bool inside(const float lo[3], const float hi[3], const Aabb& b) {
        for (int i = 0; i < 3; ++i)
            if (!((double)lo[i] <= b.lo[i] && (double)hi[i] >= b.hi[i])) return false;
        return true;
    }
    // object -> world through the record's chain (composition of its ops; cs/sn/t map world -> object)
    void to_world_point(int32_t chain, double p[3]) const {
        if (chain == 0) return;
        const DChain& c = fs.chains[(size_t)chain];
        for (int k = c.len - 1; k >= 0; --k) {
            const XformOp& op = fs.xforms[(size_t)(c.begin + k)];
            if (op.kind == XF_TRANSLATE) {
                p[0] += op.v[0]; p[1] += op.v[1]; p[2] += op.v[2];
            } else {
                double sn = op.v[0], cs = op.v[1];
                double x = cs * p[0] + sn * p[2], z = -sn * p[0] + cs * p[2];
                p[0] = x; p[2] = z;
            }
        }
    }
    // WORLD-space points the leaf box of a record must contain (its object-space extreme points, moved out)
    bool record_box(const Record& r, Aabb& b) {
        b.reset();
        if (r.c < 0 || r.c >= (int32_t)fs.chains.size()) return false;
        static const int ax0[3] = {0, 0, 1}, ax1[3] = {1, 2, 2}, axk[3] = {2, 1, 0};
        Aabb ob;
        ob.reset();
        switch (r.type) {
            case REC_SPHERE:
            case REC_MSPHERE: {  // a moving sphere at its own t0 (a point the bounds must contain when t0 is in the shutter)
                double c[3] = {r.d[0], r.d[1], r.d[2]};
                double rad = std::fabs(r.type == REC_SPHERE ? r.d[3] : r.d[6]);
                to_world_point(r.c, c);
                for (int i = 0; i < 3; ++i) { b.lo[i] = c[i] - rad; b.hi[i] = c[i] + rad; }
                return true;
            }
            case REC_RECT_XY: case REC_RECT_XZ: case REC_RECT_YZ: {
                int p = r.type - REC_RECT_XY;
                ob.lo[ax0[p]] = std::fmin(r.d[0], r.d[1]); ob.hi[ax0[p]] = std::fmax(r.d[0], r.d[1]);
                ob.lo[ax1[p]] = std::fmin(r.d[2], r.d[3]); ob.hi[ax1[p]] = std::fmax(r.d[2], r.d[3]);
                ob.lo[axk[p]] = r.d[4]; ob.hi[axk[p]] = r.d[4];
                break;
            }
            case REC_BOX:
                for (int i = 0; i < 3; ++i) { ob.lo[i] = r.d[i]; ob.hi[i] = r.d[3 + i]; }
                break;
            default: return false;
        }
        for (int corner = 0; corner < 8; ++corner) {
            double p[3] = {(corner & 1) ? ob.hi[0] : ob.lo[0], (corner & 2) ? ob.hi[1] : ob.lo[1], (corner & 4) ? ob.hi[2] : ob.lo[2]};
            to_world_point(r.c, p);
            b.grow_point(p);
        }
        return true;
    }
    // returns the union of the float boxes of the subtree through `bounds_lo/hi`
    bool walk(int32_t ni, int depth, int& n_records) {
        if (ni < 0 || ni >= (int32_t)fs.nodes.size()) return fail("node index out of range");
        if (depth > 128) return fail("BVH deeper than 128");
        if (node_seen[(size_t)ni]++) return fail("node reachable twice");
        const BvhNode& n = fs.nodes[(size_t)ni];
        for (int k = 0; k < 2; ++k) {
            int32_t ref = k == 0 ? n.child0 : n.child1;
            float lo[3] = {k == 0 ? n.c0x[0] : n.c1x[0], k == 0 ? n.c0y[0] : n.c1y[0], k == 0 ? n.c0z[0] : n.c1z[0]};
            float hi[3] = {k == 0 ? n.c0x[1] : n.c1x[1], k == 0 ? n.c0y[1] : n.c1y[1], k == 0 ? n.c0z[1] : n.c1z[1]};
            if (ref >= 0) {
                // child inner node: both of ITS child boxes must lie inside this box
                const BvhNode& c = fs.nodes[(size_t)ref];
                const float* cl[2][3] = {{&c.c0x[0], &c.c0y[0], &c.c0z[0]}, {&c.c1x[0], &c.c1y[0], &c.c1z[0]}};
                const float* ch[2][3] = {{&c.c0x[1], &c.c0y[1], &c.c0z[1]}, {&c.c1x[1], &c.c1y[1], &c.c1z[1]}};
                for (int j = 0; j < 2; ++j) {
                    if ((j == 0 ? c.child0 : c.child1) == kEmptyChild) continue;
                    for (int i = 0; i < 3; ++i)
                        if (!(*cl[j][i] >= lo[i] && *ch[j][i] <= hi[i])) return fail("child box not inside parent box");
                }
                if (!walk(ref, depth + 1, n_records)) return false;
            } else {
                int32_t v = ~ref;
                int first = v >> 4, count = v & 15;
                if (count > kBvhMaxLeafLimit && count != 0) return fail("leaf larger than the maximum");
                if (first < 0 || first + count > (int)fs.records.size()) return fail("leaf range out of bounds");
                for (int i = 0; i < count; ++i) {
                    const Record& r = fs.records[(size_t)(first + i)];
                    if (rec_seen[(size_t)(first + i)]++) return fail("record reachable twice");
                    if (!leaf_rec.empty()) leaf_rec[(size_t)(first + i)]++;
                    n_records++;
                    Aabb b;
                    if (record_box(r, b)) {
                        if (!inside(lo, hi, b)) return fail("record not inside its leaf box");
                        if (r.type == REC_BOX) {  // its six face records live outside every leaf
                            if (r.a < 0 || r.a + 6 > (int32_t)fs.records.size()) return fail("box face records out of range");
                            for (int k = 0; k < 6; ++k) {
                                const Record& fr = fs.records[(size_t)(r.a + k)];
                                if (fr.type < REC_RECT_XY || fr.type > REC_RECT_YZ || fr.c != r.c) return fail("box face record is not a rectangle of the box");
                                if (rec_seen[(size_t)(r.a + k)]++) return fail("box face record referenced twice");
                            }
                        }
                    } else {
                        return fail("unknown record type");
                    }
                }
            }
        }
        return true;
    }
    // The 4-wide copy of the world BVH: node `ni` is the pair of entries ni, ni + 1. Every child box must hold what is
    // below it; the leaves are the binary tree's leaf codes.
    bool walk_wide(int32_t ni, int depth) {
        if (ni < 0 || ni + 1 >= (int32_t)fs.nodes.size() || (ni & 1)) return fail("wide node index out of range or odd");
        if (depth > 64) return fail("wide BVH deeper than 64");
        if (node_seen[(size_t)ni]++ || node_seen[(size_t)ni + 1]++) return fail("wide node reachable twice");
        for (int j = 0; j < 4; ++j) {
            const BvhNode& n = fs.nodes[(size_t)ni + (size_t)(j >> 1)];
            const int k = j & 1;
            const int32_t ref = k == 0 ? n.child0 : n.child1;
            float lo[3] = {k == 0 ? n.c0x[0] : n.c1x[0], k == 0 ? n.c0y[0] : n.c1y[0], k == 0 ? n.c0z[0] : n.c1z[0]};
            float hi[3] = {k == 0 ? n.c0x[1] : n.c1x[1], k == 0 ? n.c0y[1] : n.c1y[1], k == 0 ? n.c0z[1] : n.c1z[1]};
            if (ref >= 0) {
                if (ref + 1 >= (int32_t)fs.nodes.size()) return fail("wide child out of range");
                for (int q = 0; q < 4; ++q) {
                    const BvhNode& c = fs.nodes[(size_t)ref + (size_t)(q >> 1)];
                    if (((q & 1) == 0 ? c.child0 : c.child1) == kEmptyChild) continue;
                    const float clo[3] = {(q & 1) == 0 ? c.c0x[0] : c.c1x[0], (q & 1) == 0 ? c.c0y[0] : c.c1y[0], (q & 1) == 0 ? c.c0z[0] : c.c1z[0]};
                    const float chi[3] = {(q & 1) == 0 ? c.c0x[1] : c.c1x[1], (q & 1) == 0 ? c.c0y[1] : c.c1y[1], (q & 1) == 0 ? c.c0z[1] : c.c1z[1]};
                    for (int i = 0; i < 3; ++i)
                        if (!(clo[i] >= lo[i] && chi[i] <= hi[i])) return fail("wide child box not inside its parent box");
                }
                if (!walk_wide(ref, depth + 1)) return false;
            } else {
                const int32_t v = ~ref;
                const int first = v >> 4, count = v & 15;
                if (first < 0 || first + count > (int)fs.records.size()) return fail("wide leaf range out of bounds");
                for (int i = 0; i < count; ++i) {
                    Aabb b;
                    if (!record_box(fs.records[(size_t)(first + i)], b)) return fail("unknown record type in a wide leaf");
                    if (!inside(lo, hi, b)) return fail("record not inside its wide leaf box");
                    wide_rec[(size_t)(first + i)]++;
                }
            }
        }
        return true;
    }
};
}  // namespace

bool check_flat_scene(const FlatScene& fs, std::string& err) {
    Checker c{fs, err, std::vector<int>(fs.nodes.size(), 0), std::vector<int>(fs.records.size(), 0)};
    int n = 0;
    c.leaf_rec.assign(fs.records.size(), 0);
    if (!c.walk(fs.world_root, 0, n)) return false;
    if (fs.wide_root >= 0) {  // the 4-wide copy reaches exactly the records of the world's leaves, once each
        c.wide_rec.assign(fs.records.size(), 0);
        if (!c.walk_wide(fs.wide_root, 0)) return false;
        if (c.wide_rec != c.leaf_rec) { err = "the 4-wide BVH does not reach the same records as the binary one"; return false; }
    }
    c.leaf_rec.clear();  // (boundary BVHs below have no wide copy)
    for (const DMedium& m : fs.media) {  // media: listed, not in a BVH; their boundary BVHs are walked here
        if (m.record < 0 || m.record >= (int32_t)fs.records.size()) { err = "medium record out of range"; return false; }
        const Record& r = fs.records[(size_t)m.record];
        if (r.type != REC_MEDIUM) { err = "media list entry is not a medium record"; return false; }
        if (c.rec_seen[(size_t)m.record]++) { err = "medium record listed twice"; return false; }
        if (r.a < 0 || r.a >= (int)fs.textures.size()) { err = "medium texture out of range"; return false; }
        int sub = 0;
        if (r.c >= 0 && !c.walk(r.c, 0, sub)) return false;  // -1: analytic sphere boundary
    }
    if (fs.max_stack > kTraversalStack) { err = "BVH too deep for the traversal stack"; return false; }
    for (size_t i = 0; i < fs.records.size(); ++i)
        if (c.rec_seen[i] != 1) { err = "record not reachable from the world root"; return false; }
    for (size_t i = 0; i < fs.nodes.size(); ++i) {
        const BvhNode& nd = fs.nodes[i];
        const bool filler = nd.child0 == kEmptyChild && nd.child1 == kEmptyChild && fs.wide_root >= 0;  // alignment entries of the wide copy
        if (c.node_seen[i] != 1 && !(filler && c.node_seen[i] == 0)) { err = "node not reachable from the world root"; return false; }
    }
    return true;
}

}  // namespace rtx
