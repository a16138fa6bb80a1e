// capi_host.cpp — plain-C entry points over the C++ host mirror, for bindings and tests
// (ctypes in tests/host_lib.py).  The element / edge records have the layout of the records in
// oracle/ref_driver.cpp, so the same fixture drives the reference build and this library.
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <limits>
#include <optional>
#include <memory>
#include <stdexcept>
#include <unordered_map>
#include <vector>

#include <gcs/b200/canvas_transform.hpp>
#include <gcs/b200/leaf_batch.hpp>
#include <gcs/b200/sketch_program.hpp>
#include <gcs/decomposition/top_down/stree_top_down_strategy.hpp>
#include <gcs/model/constraints.hpp>
#include <gcs/model/elements.hpp>
#include <gcs/model/gcs_data_structures.hpp>
#include <gcs/orchestration/geometric_constraint_system.hpp>

#include "solving/bottom_up/merge3_batched.hpp"
#include "solving/bottom_up/merge3_ppp_batched.hpp"
#include "solving/bottom_up/merge3_solver_common.hpp"
#include "solving/component_solver.hpp"
#include "solving/equations/newton_raphson.hpp"

using Eigen::Vector2d;

extern "C" {

typedef struct gcs_host_element {
    int32_t type;      // 0 = Point, 1 = Line
    int32_t is_set;    // in: already solved (pos valid); out: Element::isElementSet() afterwards
    double canvas[4];  // point: x,y ; line: x1,y1,x2,y2
    double pos[4];     // solver-space position, same layout
} gcs_host_element;

typedef struct gcs_host_edge {
    int32_t a, b;  // element indices
    int32_t type;  // 0 = Distance, 1 = Angle, 2 = virtual edge (no constraint)
    int32_t flip;  // AngleConstraint::flipOrientation
    double value;  // distance, or angle in radians
} gcs_host_edge;

}  // extern "C"

namespace {

thread_local char g_msg[512] = "";

std::shared_ptr<Gcs::Element> makeElement(const gcs_host_element& e)
{
    std::shared_ptr<Gcs::Element> el;
    if (e.type == 0) {
        el = std::make_shared<Gcs::Element>(Gcs::Point(Vector2d(e.canvas[0], e.canvas[1])));
        if (e.is_set) el->updateElementPosition(Vector2d(e.pos[0], e.pos[1]));
    } else {
        el = std::make_shared<Gcs::Element>(Gcs::Line(Vector2d(e.canvas[0], e.canvas[1]), Vector2d(e.canvas[2], e.canvas[3])));
        if (e.is_set) el->updateElementPosition(Vector2d(e.pos[0], e.pos[1]), Vector2d(e.pos[2], e.pos[3]));
    }
    // tests: GCS_HOST_SERIAL_STRIDE = k leaves k element serial numbers unused after every element,
    // which takes the leaf scheduler off its dense per-element tables (leaf_batch.cpp, SlotIndex)
    if (const char* stride = std::getenv("GCS_HOST_SERIAL_STRIDE")) Gcs::Element::skipSerials(std::strtoull(stride, nullptr, 10));
    return el;
}

void readBack(const Gcs::Element& el, gcs_host_element& e)
{
    e.is_set = el.isElementSet() ? 1 : 0;
    if (e.type == 0) {
        const auto& p = el.getElement<Gcs::Point>();
        e.pos[0] = p.position.x(), e.pos[1] = p.position.y();
    } else {
        const auto& l = el.getElement<Gcs::Line>();
        e.pos[0] = l.p1.x(), e.pos[1] = l.p1.y(), e.pos[2] = l.p2.x(), e.pos[3] = l.p2.y();
    }
}

// one leaf graph over (a subset of) shared elements; `local[i]` = index into `elems` of node i
// `made` (may be null) receives the constraints of the real edges, in edge order
Gcs::ConstraintGraph makeLeaf(const std::vector<std::shared_ptr<Gcs::Element>>& elems, const int32_t* local, int n_local,
    const gcs_host_edge* edges, int n_edges, std::vector<std::shared_ptr<Gcs::Constraint>>* made = nullptr)
{
    Gcs::ConstraintGraph g;
    std::vector<Gcs::ConstraintGraph::NodeIdType> nodes;
    std::vector<int> globalOf;
    for (int i = 0; i < n_local; ++i) {
        const auto node = g.getGraph().addNode();
        g.addElement(node, elems[static_cast<std::size_t>(local[i])]);
        nodes.push_back(node);
        globalOf.push_back(local[i]);
    }
    auto nodeOf = [&](int global) {
        for (std::size_t i = 0; i < globalOf.size(); ++i)
            if (globalOf[i] == global) return nodes[i];
        throw std::runtime_error("edge endpoint is not an element of the leaf");
    };
    for (int k = 0; k < n_edges; ++k) {
        const auto& ed = edges[k];
        if (ed.type == 2) {
            g.addVirtualEdge(nodeOf(ed.a), nodeOf(ed.b));
            continue;
        }
        const auto eid = g.getGraph().addEdge(nodeOf(ed.a), nodeOf(ed.b)).value();
        auto con = ed.type == 0 ? std::make_shared<Gcs::Constraint>(Gcs::DistanceConstraint(ed.value))
                                : std::make_shared<Gcs::Constraint>(Gcs::AngleConstraint(ed.value, ed.flip != 0));
        if (made) made->push_back(con);
        g.addConstraint(eid, std::move(con));
    }
    return g;
}

// A whole sketch as one graph over new elements; `made` (may be null) receives the constraints of
// the real edges, in edge order.
Gcs::ConstraintGraph makeSketch(std::vector<std::shared_ptr<Gcs::Element>>& elems, int n_el, const gcs_host_element* el, int n_edges,
    const gcs_host_edge* edges, std::vector<std::shared_ptr<Gcs::Constraint>>* made = nullptr)
{
    Gcs::ConstraintGraph g;
    std::vector<Gcs::ConstraintGraph::NodeIdType> nodes;
    elems.reserve(static_cast<std::size_t>(n_el));
    for (int i = 0; i < n_el; ++i) {
        elems.push_back(makeElement(el[i]));
        nodes.push_back(g.getGraph().addNode());
        g.addElement(nodes.back(), elems.back());
    }
    for (int k = 0; k < n_edges; ++k) {
        const auto& ed = edges[k];
        const auto a = nodes.at(static_cast<std::size_t>(ed.a)), b = nodes.at(static_cast<std::size_t>(ed.b));
        if (ed.type == 2) {
            g.addVirtualEdge(a, b);
            continue;
        }
        const auto eid = g.getGraph().addEdge(a, b).value();
        auto con = ed.type == 0 ? std::make_shared<Gcs::Constraint>(Gcs::DistanceConstraint(ed.value))
                                : std::make_shared<Gcs::Constraint>(Gcs::AngleConstraint(ed.value, ed.flip != 0));
        if (made) made->push_back(con);
        g.addConstraint(eid, std::move(con));
    }
    return g;
}

int fail(const std::exception& ex)
{
    std::snprintf(g_msg, sizeof(g_msg), "%s", ex.what());
    return -1;
}

}  // namespace

extern "C" {

GCS_API const char* gcs_host_last_error(void) { return g_msg; }

// Self-check of ConstraintGraph::triangleDigest (the per-leaf summary the scheduler plans from):
// it must follow every change made to the graph, through the class or through getGraph(), and
// copies of elements must be new objects to the scheduler.  Returns 0, or the number of the
// first check that failed.
GCS_API int gcs_host_selftest_digest(void)
{
    using namespace Gcs;
    try {
        ConstraintGraph g;
        std::vector<std::shared_ptr<Element>> el;
        std::vector<ConstraintGraph::NodeIdType> nd;
        for (int i = 0; i < 3; ++i) {
            el.push_back(std::make_shared<Element>(Point(Vector2d(i, 2 * i))));
            nd.push_back(g.getGraph().addNode());
            if (g.triangleDigest().simple) return 1;  // fewer than three elements
            g.addElement(nd.back(), el.back());
        }
        const TriangleDigest* d = &g.triangleDigest();
        if (!d->simple || d->edgeCount != 0 || d->element[0] != el[0].get() || d->element[2] != el[2].get()) return 2;
        const auto e01 = g.getGraph().addEdge(nd[0], nd[1]).value();  // behind the class's back
        d = &g.triangleDigest();
        if (!d->simple || d->edgeCount != 1 || d->constraint[0] != nullptr) return 3;
        auto c01 = std::make_shared<Constraint>(DistanceConstraint(3.0));
        g.addConstraint(e01, c01);
        d = &g.triangleDigest();
        if (!d->simple || d->constraint[0] != c01.get() || d->constraint[1] || d->constraint[2]) return 4;
        const auto v12 = g.addVirtualEdge(nd[1], nd[2]);
        d = &g.triangleDigest();
        if (!d->simple || d->edgeCount != 2 || d->constraint[2] != nullptr) return 5;
        const auto e02 = g.getGraph().addEdge(nd[0], nd[2]).value();
        auto c02 = std::make_shared<Constraint>(AngleConstraint(0.5, true));
        g.addConstraint(e02, c02);
        d = &g.triangleDigest();
        if (!d->simple || d->edgeCount != 3 || d->constraint[1] != c02.get()) return 6;
        ConstraintGraph copy = g;  // a copy shares elements and constraints, and answers for itself afterwards
        g.removeVirtualEdge(v12);
        if (g.triangleDigest().edgeCount != 2 || copy.triangleDigest().edgeCount != 3) return 7;
        const auto p01 = copy.getGraph().addEdge(nd[0], nd[1]).value();  // a second edge on one pair: not simple any more
        if (copy.triangleDigest().simple) return 8;
        copy.removeConstraintEdge(p01);
        if (!copy.triangleDigest().simple) return 9;
        g.removeConstraintEdge(e01);
        d = &g.triangleDigest();
        if (!d->simple || d->edgeCount != 1 || d->constraint[0] || d->constraint[1] != c02.get()) return 10;
        g.removeElement(nd[2]);
        if (g.triangleDigest().simple) return 11;
        // element serial numbers: unique per object, ascending, untouched by assignment
        Element a(Point(Vector2d(1, 2))), b(a);
        if (a.serial() == b.serial() || b.serial() < a.serial()) return 12;
        const auto sb = b.serial();
        b = *el[1];
        if (b.serial() != sb || !b.isElementType<Point>()) return 13;
        Element::skipSerials(1000);
        Element c(Line(Vector2d(0, 0), Vector2d(1, 1)));
        if (c.serial() < sb + 1000) return 14;
        return 0;
    } catch (const std::exception& ex) {
        fail(ex);
        return -1;
    }
}

// Kernel class of the host mirror's launches (Gcs::B200::setKernelVariant); returns the previous one.
GCS_API int gcs_host_set_variant(int variant) { return Gcs::B200::setKernelVariant(variant); }

// A 3-element leaf through classifyAndSolve (batch of one on the device).
// Returns SolveStatus (0 Success, 1 Unsupported, 2 Failed) or -1 on an exception.
GCS_API int gcs_host_component_solve(int n_el, gcs_host_element* el, int n_edges, const gcs_host_edge* edges)
{
    try {
        std::vector<std::shared_ptr<Gcs::Element>> elems;
        std::vector<int32_t> local;
        for (int i = 0; i < n_el; ++i) elems.push_back(makeElement(el[i])), local.push_back(i);
        Gcs::ConstraintGraph g = makeLeaf(elems, local.data(), n_el, edges, n_edges);
        const Gcs::SolveResult r = Gcs::classifyAndSolve(g);
        for (int i = 0; i < n_el; ++i) readBack(*elems[static_cast<std::size_t>(i)], el[i]);
        return static_cast<int>(r.status);
    } catch (const std::exception& ex) {
        return fail(ex);
    } catch (...) {
        std::snprintf(g_msg, sizeof(g_msg), "unknown exception");
        return -1;
    }
}

// Packer only (no device): classify the leaf, assign roles, place anchors, and return the batch
// row the kernel would receive plus the index of the element that receives the result.
// Returns the SolverId (0 = unsupported) or -1 on an exception.
GCS_API int gcs_host_component_pack(int n_el, gcs_host_element* el, int n_edges, const gcs_host_edge* edges, int32_t* kind,
    double in[GCS_MAX_IN_COLS], uint8_t* code, int32_t* target)
{
    try {
        std::vector<std::shared_ptr<Gcs::Element>> elems;
        std::vector<int32_t> local;
        for (int i = 0; i < n_el; ++i) elems.push_back(makeElement(el[i])), local.push_back(i);
        Gcs::ConstraintGraph g = makeLeaf(elems, local.data(), n_el, edges, n_edges);
        const Gcs::B200::SolverId id = Gcs::B200::classify(g);
        *kind = 0, *target = -1;
        if (id == Gcs::B200::SolverId::None) return 0;
        const Gcs::B200::PackedLeaf row = Gcs::B200::pack(id, g);
        *kind = row.kind;
        *code = row.code;
        for (int c = 0; c < GCS_MAX_IN_COLS; ++c) in[c] = row.in[c];
        for (int i = 0; i < n_el; ++i) {
            if (elems[static_cast<std::size_t>(i)].get() == row.target) *target = i;
            readBack(*elems[static_cast<std::size_t>(i)], el[i]);
        }
        return static_cast<int>(id);
    } catch (const std::exception& ex) {
        return fail(ex);
    } catch (...) {
        std::snprintf(g_msg, sizeof(g_msg), "unknown exception");
        return -1;
    }
}

// Many leaves over shared elements (what DeficitStreeBasedTopDownStrategy::solveGcs receives).
//   leaf_elems   [3 * n_leaves] element indices, node order of each leaf
//   edge_offsets [n_leaves + 1] range of each leaf's edges in `edges` (a, b = element indices)
//   mode 0: the reference's loop, one classifyAndSolve per leaf (a launch per leaf)
//        1: DeficitStreeBasedTopDownStrategy::solveGcs (dependency waves, a launch per kind per wave)
//        2: plan only (no device): solver + wave per leaf
//   status/level/solver [n_leaves] (may be NULL); stats[0] = waves, stats[1] = launches, stats[2] = solved, stats[3] = microseconds spent planning
// Returns 0, or -1 after an exception (elements solved before it are still written back).
GCS_API int gcs_host_leaves_solve(int n_el, gcs_host_element* el, int n_leaves, const int32_t* leaf_elems,
    const int32_t* edge_offsets, const gcs_host_edge* edges, int mode, int32_t* status, int32_t* level, int32_t* solver,
    int64_t* stats)
{
    std::vector<std::shared_ptr<Gcs::Element>> elems;
    int rc = 0;
    try {
        for (int i = 0; i < n_el; ++i) elems.push_back(makeElement(el[i]));
        std::vector<Gcs::ConstraintGraph> leaves;
        for (int l = 0; l < n_leaves; ++l)
            leaves.push_back(makeLeaf(elems, leaf_elems + 3 * l, 3, edges + edge_offsets[l], edge_offsets[l + 1] - edge_offsets[l]));
        if (stats) stats[0] = stats[1] = stats[2] = stats[3] = 0;
        if (mode == 0) {
            for (int l = 0; l < n_leaves; ++l) {
                const Gcs::B200::SolverId id = Gcs::B200::classify(leaves[static_cast<std::size_t>(l)]);
                if (solver) solver[l] = static_cast<int32_t>(id);
                const Gcs::SolveResult r = Gcs::classifyAndSolve(leaves[static_cast<std::size_t>(l)]);
                if (status) status[l] = static_cast<int32_t>(r.status);
                if (level) level[l] = l;
                if (stats && r.status == Gcs::SolveStatus::Success) ++stats[1], ++stats[2];
            }
        } else {
            Gcs::B200::BatchReport rep;
            if (mode == 1) {
                Gcs::DeficitStreeBasedTopDownStrategy strategy;
                try {
                    strategy.solveGcs(leaves);
                    rep = strategy.lastReport();
                } catch (const std::exception& ex) {
                    rc = fail(ex);
                    rep = Gcs::B200::planLeaves(leaves);  // not reached by the solved prefix; reporting only
                }
            } else {
                rep = Gcs::B200::planLeaves(leaves);
            }
            for (int l = 0; l < n_leaves; ++l) {
                const auto i = static_cast<std::size_t>(l);
                if (status) status[l] = static_cast<int32_t>(rep.status[i]);
                if (level) level[l] = rep.level[i];
                if (solver) solver[l] = static_cast<int32_t>(rep.solver[i]);
            }
            if (stats) stats[0] = static_cast<int64_t>(rep.waves), stats[1] = static_cast<int64_t>(rep.launches), stats[2] = static_cast<int64_t>(rep.solved), stats[3] = static_cast<int64_t>(rep.planSeconds * 1e6);
        }
    } catch (const std::exception& ex) {
        rc = fail(ex);
    } catch (...) {
        std::snprintf(g_msg, sizeof(g_msg), "unknown exception");
        rc = -1;
    }
    for (std::size_t i = 0; i < elems.size(); ++i) readBack(*elems[i], el[i]);
    return rc;
}

// Equations::solve2D through the mirror.  pair: 1 P2P+P2P (6 params: x0,y0,d, x0,y0,d);
// 2 SDD+unit (dx,dy,s1,s2); 3 P2P+P2L (x0,y0,d, xa,ya,xb,yb,d,L); 4 P2L+P2L (2 x (xa,ya,xb,yb,d,L));
// 5 angle+unit (fdx,fdy,L,cosA).  guesses: 4 doubles (g0x,g0y,g1x,g1y) or NULL for the defaults.
GCS_API int gcs_host_solve2d(int pair, const double* p, const double* guesses, double* cand4, int32_t* iters2, int32_t* conv2)
{
    namespace Eq = Gcs::Equations;
    try {
        std::array<Vector2d, 2> gs = Eq::DEFAULT_SPATIAL_GUESSES;
        if (guesses) gs = { Vector2d(guesses[0], guesses[1]), Vector2d(guesses[2], guesses[3]) };
        Eq::Solve2DInfo info;
        std::array<Vector2d, 2> r;
        switch (pair) {
        case 1: r = Eq::solve2D(Eq::pointToPointDistance(p[0], p[1], p[2]), Eq::pointToPointDistance(p[3], p[4], p[5]), gs, &info); break;
        case 2: r = Eq::solve2D(Eq::lineNormalSignedDistanceDiff(p[0], p[1], p[2], p[3]), Eq::unitNormalConstraint(), gs, &info); break;
        case 3: r = Eq::solve2D(Eq::pointToPointDistance(p[0], p[1], p[2]), Eq::pointToLineDistance(p[3], p[4], p[5], p[6], p[7], p[8]), gs, &info); break;
        case 4: r = Eq::solve2D(Eq::pointToLineDistance(p[0], p[1], p[2], p[3], p[4], p[5]), Eq::pointToLineDistance(p[6], p[7], p[8], p[9], p[10], p[11]), gs, &info); break;
        case 5: r = Eq::solve2D(Eq::lineNormalAngleConstraint(p[0], p[1], p[2], p[3]), Eq::unitNormalConstraint(), gs, &info); break;
        default: std::snprintf(g_msg, sizeof(g_msg), "unknown equation pair %d", pair); return -1;
        }
        cand4[0] = r[0].x(), cand4[1] = r[0].y(), cand4[2] = r[1].x(), cand4[3] = r[1].y();
        for (int s = 0; s < 2; ++s) {
            if (iters2) iters2[s] = info.iterations[s];
            if (conv2) conv2[s] = info.converged[s] ? 1 : 0;
        }
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// GeometricConstraintSystem with the top-down strategy on a whole sketch: constrainedness check,
// decomposition (a 3-element sketch is its own leaf - BASELINE config 1; larger Henneberg-style
// sketches go through the degree-2 peeling of gcs/b200/peel_decomposition.hpp - config 4), then
// the batched solveGcs.  stats (may be NULL): [0] leaves, [1] waves, [2] launches, [3] solved,
// [4] microseconds in check + decomposition, [5] microseconds in solveGcs, of which [6] planning
// (symbolic classification + wave levels), [7] packing, [8] device calls, [9] write-back, [10] launches that
// went over several devices (GCS_HOST_DEVICES).  stats holds 12 values.
GCS_API int gcs_host_system_solve_ex(int n_el, gcs_host_element* el, int n_edges, const gcs_host_edge* edges, int64_t* stats)
{
    try {
        std::vector<std::shared_ptr<Gcs::Element>> elems;
        Gcs::ConstraintGraph g = makeSketch(elems, n_el, el, n_edges, edges);
        // the three steps of GeometricConstraintSystem::solveGeometricConstraintSystem, timed apart
        auto strategy = std::make_unique<Gcs::DeficitStreeBasedTopDownStrategy>();
        Gcs::DeficitStreeBasedTopDownStrategy* st = strategy.get();
        // GCS_HOST_DEVICES = n: every wave over the first n devices of gcs_b200_init (bench / tests)
        if (const char* e = std::getenv("GCS_HOST_DEVICES")) {
            const char* m = std::getenv("GCS_HOST_MIN_ROWS");
            st->setDeviceCount(std::atoi(e), m ? static_cast<std::size_t>(std::atoll(m)) : 16384);
        }
        const auto t0 = std::chrono::steady_clock::now();
        if (st->checkConstraintGraphConstrainedness(g) != Gcs::Constrainedness::WELL_CONSTRAINED && !st->resolve(g))
            throw std::runtime_error("Gcs is not well-constrained, current algorithms do not support such inputs");
        auto leaves = st->decomposeConstraintGraph(g);
        const auto t1 = std::chrono::steady_clock::now();
        st->solveGcs(leaves);
        const auto t2 = std::chrono::steady_clock::now();
        if (stats) {
            const auto& rep = st->lastReport();
            stats[0] = static_cast<int64_t>(rep.leaves), stats[1] = static_cast<int64_t>(rep.waves);
            stats[2] = static_cast<int64_t>(rep.launches), stats[3] = static_cast<int64_t>(rep.solved);
            stats[4] = std::chrono::duration_cast<std::chrono::microseconds>(t1 - t0).count();
            stats[5] = std::chrono::duration_cast<std::chrono::microseconds>(t2 - t1).count();
            stats[6] = static_cast<int64_t>(rep.planSeconds * 1e6), stats[7] = static_cast<int64_t>(rep.packSeconds * 1e6);
            stats[8] = static_cast<int64_t>(rep.deviceSeconds * 1e6), stats[9] = static_cast<int64_t>(rep.applySeconds * 1e6);
            stats[10] = static_cast<int64_t>(rep.shardedLaunches);
        }
        for (int i = 0; i < n_el; ++i) readBack(*elems[static_cast<std::size_t>(i)], el[i]);
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

GCS_API int gcs_host_system_solve(int n_el, gcs_host_element* el, int n_edges, const gcs_host_edge* edges)
{
    // through the class itself (the timed variant above repeats its three calls)
    if (n_el == 3) {
        try {
            std::vector<std::shared_ptr<Gcs::Element>> elems;
            std::vector<int32_t> local;
            for (int i = 0; i < n_el; ++i) elems.push_back(makeElement(el[i])), local.push_back(i);
            Gcs::ConstraintGraph g = makeLeaf(elems, local.data(), n_el, edges, n_edges);
            Gcs::GeometricConstraintSystem sys(std::make_unique<Gcs::DeficitStreeBasedTopDownStrategy>());
            sys.solveGeometricConstraintSystem(g);
            for (int i = 0; i < n_el; ++i) readBack(*elems[static_cast<std::size_t>(i)], el[i]);
            return 0;
        } catch (const std::exception& ex) {
            return fail(ex);
        }
    }
    return gcs_host_system_solve_ex(n_el, el, n_edges, edges, nullptr);
}

// Decomposition only (no device): leaf count and, per leaf, its three element indices in node
// order (leaf_elems, 3 per leaf, capacity given in leaves) - for tests.  Returns the number of
// leaves or -1.
GCS_API int gcs_host_decompose(int n_el, const gcs_host_element* el, int n_edges, const gcs_host_edge* edges, int32_t* leaf_elems,
    int32_t* leaf_virtual, int32_t* leaf_real, int capacity)
{
    try {
        std::vector<std::shared_ptr<Gcs::Element>> elems;
        Gcs::ConstraintGraph g;
        std::vector<Gcs::ConstraintGraph::NodeIdType> nodes;
        std::unordered_map<const Gcs::Element*, int32_t> indexOf;
        for (int i = 0; i < n_el; ++i) {
            elems.push_back(makeElement(el[i]));
            indexOf[elems.back().get()] = i;
            nodes.push_back(g.getGraph().addNode());
            g.addElement(nodes.back(), elems.back());
        }
        for (int k = 0; k < n_edges; ++k) {
            const auto& ed = edges[k];
            const auto a = nodes.at(static_cast<std::size_t>(ed.a)), b = nodes.at(static_cast<std::size_t>(ed.b));
            if (ed.type == 2) {
                g.addVirtualEdge(a, b);
                continue;
            }
            const auto eid = g.getGraph().addEdge(a, b).value();
            if (ed.type == 0)
                g.addConstraint(eid, std::make_shared<Gcs::Constraint>(Gcs::DistanceConstraint(ed.value)));
            else
                g.addConstraint(eid, std::make_shared<Gcs::Constraint>(Gcs::AngleConstraint(ed.value, ed.flip != 0)));
        }
        Gcs::DeficitStreeBasedTopDownStrategy st;
        const auto t0 = std::chrono::steady_clock::now();
        const auto leaves = st.decomposeConstraintGraph(g);
        if (std::getenv("GCS_HOST_TRACE"))
            std::fprintf(stderr, "[host] decomposeConstraintGraph: %.1f ms for %zu leaves\n",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(), leaves.size());
        int l = 0;
        for (const auto& leaf : leaves) {
            if (l >= capacity) break;
            int k = 0;
            for (const auto& [node, e] : leaf.getElementMap()) leaf_elems[3 * l + k++] = indexOf.at(e.get());
            leaf_virtual[l] = static_cast<int32_t>(leaf.getVirtualEdges().size());
            leaf_real[l] = static_cast<int32_t>(leaf.getConstraintMap().size());
            ++l;
        }
        return static_cast<int>(leaves.size());
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// ---- bottom-up Merge3 numeric helpers (solving/bottom_up/merge3_solver_common.hpp) ----
// kase 1: point from two fixed points   rows of 12: fixedA(2) fixedB(2) distA distB canvasA(2) canvasB(2) canvasFree(2) -> 2
//      2: line from two fixed points    rows of 14: fixedA(2) fixedB(2) distA distB canvasA(2) canvasB(2) canvasFreeLine(4) -> 4
//      3: point from point and line     rows of 16: fixedPoint(2) fixedLine(4) distP distL canvasPoint(2) canvasLine(4) canvasFree(2) -> 2
//      4: point from two lines          rows of 20: lineA(4) lineB(4) distA distB canvasA(4) canvasB(4) canvasFree(2) -> 2
// mode 0: pack only (no device): packed[i][13] + code[i] = the kernel row, ok[i] = 0 where the
//         reference answers nullopt without numerics;
//      1: all rows as ONE Merge3Batch (one launch); 2: row by row through the single-call functions.
// stats (may be NULL): [0] launches.  Returns 0 or -1 after an exception.
GCS_API int gcs_host_m3_solve(int kase, int64_t n, const double* rows, double* out, uint8_t* ok, int mode, double* packed,
    uint8_t* code, int64_t* stats)
{
    namespace Bu = Gcs::Solvers::BottomUp;
    auto v2 = [](const double* p) { return Vector2d(p[0], p[1]); };
    auto ln = [&](const double* p) { return Bu::LinePose { v2(p), v2(p + 2) }; };
    static const int width[5] = { 0, 12, 14, 16, 20 }, nout[5] = { 0, 2, 4, 2, 2 };
    try {
        if (kase < 1 || kase > 4) throw std::invalid_argument("unknown Merge3 case");
        const int w = width[kase], no = nout[kase];
        auto add = [&](Gcs::B200::Merge3Batch& b, const double* r) {
            switch (kase) {
            case 1: return b.addFreePointFromFixedPoints(v2(r), v2(r + 2), r[4], r[5], v2(r + 6), v2(r + 8), v2(r + 10));
            case 2: return b.addFreeLineFromFixedPoints(v2(r), v2(r + 2), r[4], r[5], v2(r + 6), v2(r + 8), ln(r + 10));
            case 3: return b.addFreePointFromFixedPointAndLine(v2(r), ln(r + 2), r[6], r[7], v2(r + 8), ln(r + 10), v2(r + 14));
            default: return b.addFreePointFromFixedLines(ln(r), ln(r + 4), r[8], r[9], ln(r + 10), ln(r + 14), v2(r + 18));
            }
        };
        auto store = [&](int64_t i, const std::optional<Vector2d>& p, const std::optional<Bu::LinePose>& l) {
            ok[i] = (no == 2) ? p.has_value() : l.has_value();
            for (int c = 0; c < no; ++c) out[no * i + c] = std::numeric_limits<double>::quiet_NaN();
            if (no == 2 && p) out[2 * i] = p->x(), out[2 * i + 1] = p->y();
            if (no == 4 && l) out[4 * i] = l->p1.x(), out[4 * i + 1] = l->p1.y(), out[4 * i + 2] = l->p2.x(), out[4 * i + 3] = l->p2.y();
        };
        if (stats) stats[0] = 0;
        if (mode == 2) {
            for (int64_t i = 0; i < n; ++i) {
                const double* r = rows + w * i;
                switch (kase) {
                case 1: store(i, Bu::solveFreePointFromFixedPoints(v2(r), v2(r + 2), r[4], r[5], v2(r + 6), v2(r + 8), v2(r + 10)), {}); break;
                case 2: store(i, {}, Bu::solveFreeLineFromFixedPoints(v2(r), v2(r + 2), r[4], r[5], v2(r + 6), v2(r + 8), ln(r + 10))); break;
                case 3: store(i, Bu::solveFreePointFromFixedPointAndLine(v2(r), ln(r + 2), r[6], r[7], v2(r + 8), ln(r + 10), v2(r + 14)), {}); break;
                default: store(i, Bu::solveFreePointFromFixedLines(ln(r), ln(r + 4), r[8], r[9], ln(r + 10), ln(r + 14), v2(r + 18)), {}); break;
                }
                if (stats) ++stats[0];
            }
            return 0;
        }
        Gcs::B200::Merge3Batch batch;
        std::vector<Gcs::B200::Merge3Batch::Handle> h;
        for (int64_t i = 0; i < n; ++i) h.push_back(add(batch, rows + w * i));
        if (mode == 0) {
            for (int64_t i = 0; i < n; ++i) {
                const int kind = batch.kindOf(h[static_cast<std::size_t>(i)]);
                ok[i] = kind != 0;
                for (int c = 0; c < GCS_MAX_IN_COLS; ++c) packed[GCS_MAX_IN_COLS * i + c] = 0.0;
                code[i] = 0;
                if (kind == 0) continue;
                const auto& kb = batch.rows(kind);
                const std::size_t row = batch.rowOf(h[static_cast<std::size_t>(i)]);
                for (int c = 0; c < gcs_b200_kind_in_cols(kind); ++c) packed[GCS_MAX_IN_COLS * i + c] = kb.column(c)[row];
                code[i] = kb.codes()[row];
            }
            return 0;
        }
        batch.solve();
        if (stats) stats[0] = static_cast<int64_t>(batch.launches());
        for (int64_t i = 0; i < n; ++i) {
            if (no == 2)
                store(i, batch.point(h[static_cast<std::size_t>(i)]), {});
            else
                store(i, {}, batch.line(h[static_cast<std::size_t>(i)]));
        }
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// estimateRigidTransform on npts point pairs; out6 = R00 R01 R10 R11 tx ty.  Returns 1, 0 (nullopt) or -1.
GCS_API int gcs_host_m3_rigid_transform(int npts, const double* src, const double* dst, double* out6)
{
    try {
        std::vector<Vector2d> s, t;
        for (int i = 0; i < npts; ++i) s.emplace_back(src[2 * i], src[2 * i + 1]), t.emplace_back(dst[2 * i], dst[2 * i + 1]);
        const auto tr = Gcs::Solvers::BottomUp::estimateRigidTransform(s, t);
        if (!tr) return 0;
        out6[0] = tr->rotation(0, 0), out6[1] = tr->rotation(0, 1), out6[2] = tr->rotation(1, 0), out6[3] = tr->rotation(1, 1);
        out6[4] = tr->translation.x(), out6[5] = tr->translation.y();
        return 1;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// scoreMergedPose over a graph of n_el elements (type 0 point / 1 line; canvas4 and pose4: x,y or
// x1,y1,x2,y2); in_pose[i] != 0 puts element i into the merged pose, inserted in index order.
GCS_API double gcs_host_m3_score(int n_el, const int32_t* type, const double* canvas4, const double* pose4, const uint8_t* in_pose)
{
    namespace Bu = Gcs::Solvers::BottomUp;
    Gcs::ConstraintGraph g;
    Bu::ClusterPose merged;
    for (int i = 0; i < n_el; ++i) {
        const double* c = canvas4 + 4 * i;
        const double* p = pose4 + 4 * i;
        const auto node = g.getGraph().addNode();
        if (type[i] == 0)
            g.addElement(node, std::make_shared<Gcs::Element>(Gcs::Point(Vector2d(c[0], c[1]))));
        else
            g.addElement(node, std::make_shared<Gcs::Element>(Gcs::Line(Vector2d(c[0], c[1]), Vector2d(c[2], c[3]))));
        if (!in_pose[i]) continue;
        if (type[i] == 0)
            merged.emplace(node, Bu::PointPose { Vector2d(p[0], p[1]) });
        else
            merged.emplace(node, Bu::LinePose { Vector2d(p[0], p[1]), Vector2d(p[2], p[3]) });
    }
    return Bu::scoreMergedPose(g, merged);
}

// Gcs::B200::solveMerge3Ppp (solving/bottom_up/merge3_ppp_batched.hpp) on three child clusters of one
// sketch: the batched form of the reference's Merge3PppSolver::solve enumeration loop.  Same flat
// layout as the reference-side test driver: elements i = 0..n_el-1 (type 0 point / 1 line, canvas4),
// cluster c = 0..2 holds counts[c] elements (ids / pose4 concatenated, in insertion order).
// Returns the size of the merged pose (0: no candidate; -1: error), out_ids ascending; stats[3] =
// candidates solved, candidates scored, kernel launches; *score = the winning score.
GCS_API int gcs_host_m3_merge(int which, int n_el, const int32_t* type, const double* canvas4, const int32_t* counts, const int32_t* ids,
    const double* pose4, int32_t* out_ids, double* out_pose4, double* score, int64_t* stats);

GCS_API int gcs_host_m3_ppp_merge(int n_el, const int32_t* type, const double* canvas4, const int32_t* counts, const int32_t* ids,
    const double* pose4, int32_t* out_ids, double* out_pose4, double* score, int64_t* stats)
{
    return gcs_host_m3_merge(0, n_el, type, canvas4, counts, ids, pose4, out_ids, out_pose4, score, stats);
}

// The same for every Merge3 case (solving/bottom_up/merge3_batched.hpp): which = 0 PPP, 1 PLL, 2 LPP,
// 3 LLP enumeration loop, 4 the rigid fallback, 5 the whole merge node (the reference's case order);
// stats[4] = candidates solved, candidates scored, kernel launches, case that produced the pose
// (Merge3Case; which itself unless which = 5).  Returns the size of the merged pose (0: none; -1: error).
GCS_API int gcs_host_m3_merge(int which, int n_el, const int32_t* type, const double* canvas4, const int32_t* counts, const int32_t* ids,
    const double* pose4, int32_t* out_ids, double* out_pose4, double* score, int64_t* stats)
{
    namespace Bu = Gcs::Solvers::BottomUp;
    try {
        Gcs::ConstraintGraph g;
        std::vector<Gcs::ConstraintGraph::NodeIdType> nodes;
        for (int i = 0; i < n_el; ++i) {
            const double* c = canvas4 + 4 * i;
            nodes.push_back(g.getGraph().addNode());
            if (type[i] == 0)
                g.addElement(nodes.back(), std::make_shared<Gcs::Element>(Gcs::Point(Vector2d(c[0], c[1]))));
            else
                g.addElement(nodes.back(), std::make_shared<Gcs::Element>(Gcs::Line(Vector2d(c[0], c[1]), Vector2d(c[2], c[3]))));
        }
        Bu::ClusterPose pose[3];
        int at = 0;
        for (int c = 0; c < 3; ++c)
            for (int k = 0; k < counts[c]; ++k, ++at) {
                const double* p = pose4 + 4 * at;
                const auto node = nodes.at(static_cast<std::size_t>(ids[at]));
                if (type[ids[at]] == 0)
                    pose[c].emplace(node, Bu::PointPose { Vector2d(p[0], p[1]) });
                else
                    pose[c].emplace(node, Bu::LinePose { Vector2d(p[0], p[1]), Vector2d(p[2], p[3]) });
            }
        const Gcs::B200::Merge3Children children { &pose[0], &pose[1], &pose[2] };
        std::optional<Bu::ClusterPose> merged;
        int64_t st[4] = { 0, 0, 0, which };
        double best = 0.0;
        if (which == 0) {
            Gcs::B200::Merge3PppReport rep;
            merged = Gcs::B200::solveMerge3Ppp(g, children, 0, &rep);
            st[0] = static_cast<int64_t>(rep.candidates), st[1] = static_cast<int64_t>(rep.scored), st[2] = static_cast<int64_t>(rep.launches);
            best = rep.bestScore;
        } else if (which >= 1 && which <= 3) {
            Gcs::B200::Merge3Report rep;
            merged = which == 1 ? Gcs::B200::solveMerge3Pll(g, children, 0, &rep)
                : which == 2    ? Gcs::B200::solveMerge3Lpp(g, children, 0, &rep)
                                : Gcs::B200::solveMerge3Llp(g, children, 0, &rep);
            st[0] = static_cast<int64_t>(rep.candidates), st[1] = static_cast<int64_t>(rep.scored), st[2] = static_cast<int64_t>(rep.launches);
            best = rep.bestScore;
        } else if (which == 4) {
            merged = Gcs::B200::solveMerge3Fallback(children);
        } else if (which == 5) {
            Gcs::B200::Merge3NodeReport rep;
            merged = Gcs::B200::solveMerge3Node(g, children, 0, &rep);
            st[0] = static_cast<int64_t>(rep.candidates), st[1] = static_cast<int64_t>(rep.scored), st[2] = static_cast<int64_t>(rep.launches);
            st[3] = static_cast<int64_t>(rep.solvedBy);
            best = rep.bestScore;
        } else {
            throw std::invalid_argument("gcs_host_m3_merge: which must be 0..5");
        }
        if (stats) stats[0] = st[0], stats[1] = st[1], stats[2] = st[2];
        if (stats && which != 0) stats[3] = st[3];  // the PPP entry point keeps its three-word layout
        if (score) *score = best;
        if (!merged) return 0;
        int n = 0;
        for (int i = 0; i < n_el; ++i) {
            const auto it = merged->find(nodes[static_cast<std::size_t>(i)]);
            if (it == merged->end()) continue;
            out_ids[n] = i;
            double* o = out_pose4 + 4 * n;
            o[0] = o[1] = o[2] = o[3] = 0.0;
            if (const auto* pp = std::get_if<Bu::PointPose>(&it->second))
                o[0] = pp->position.x(), o[1] = pp->position.y();
            else {
                const auto& l = std::get<Bu::LinePose>(it->second);
                o[0] = l.p1.x(), o[1] = l.p1.y(), o[2] = l.p2.x(), o[3] = l.p2.y();
            }
            ++n;
        }
        return n;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// A level of merge nodes through ONE batch (Gcs::B200::solveMerge3Level).  Node k has n_el[k] elements; type /
// canvas4 / out_ids / out_pose4 are concatenated over the nodes (n_el[k] slots each), counts holds 3 entries per
// node, ids / pose4 the nodes' cluster members one node after the other.  out_n[k] = size of node k's merged pose
// (0: none), solved_by[k] = Merge3Case; stats[3] = nodes, candidates solved, kernel launches.  Returns 0 or -1.
GCS_API int gcs_host_m3_level(int n_nodes, const int32_t* n_el, const int32_t* type, const double* canvas4, const int32_t* counts,
    const int32_t* ids, const double* pose4, int32_t* out_n, int32_t* out_ids, double* out_pose4, int32_t* solved_by, int64_t* stats)
{
    namespace Bu = Gcs::Solvers::BottomUp;
    try {
        struct Node {
            Gcs::ConstraintGraph g;
            std::vector<Gcs::ConstraintGraph::NodeIdType> nodes;
            Bu::ClusterPose pose[3];
        };
        std::vector<std::unique_ptr<Node>> built;
        std::vector<Gcs::B200::Merge3NodeInput> inputs;
        std::size_t el0 = 0, at = 0;
        for (int k = 0; k < n_nodes; ++k) {
            auto nd = std::make_unique<Node>();
            for (int i = 0; i < n_el[k]; ++i) {
                const double* c = canvas4 + 4 * (el0 + static_cast<std::size_t>(i));
                nd->nodes.push_back(nd->g.getGraph().addNode());
                if (type[el0 + static_cast<std::size_t>(i)] == 0)
                    nd->g.addElement(nd->nodes.back(), std::make_shared<Gcs::Element>(Gcs::Point(Vector2d(c[0], c[1]))));
                else
                    nd->g.addElement(nd->nodes.back(), std::make_shared<Gcs::Element>(Gcs::Line(Vector2d(c[0], c[1]), Vector2d(c[2], c[3]))));
            }
            for (int c = 0; c < 3; ++c)
                for (int j = 0; j < counts[3 * k + c]; ++j, ++at) {
                    const double* p = pose4 + 4 * at;
                    const auto local = static_cast<std::size_t>(ids[at]);
                    const auto node = nd->nodes.at(local);
                    if (type[el0 + local] == 0)
                        nd->pose[c].emplace(node, Bu::PointPose { Vector2d(p[0], p[1]) });
                    else
                        nd->pose[c].emplace(node, Bu::LinePose { Vector2d(p[0], p[1]), Vector2d(p[2], p[3]) });
                }
            inputs.push_back({ &nd->g, { &nd->pose[0], &nd->pose[1], &nd->pose[2] } });
            built.push_back(std::move(nd));
            el0 += static_cast<std::size_t>(n_el[k]);
        }
        std::vector<Gcs::B200::Merge3NodeReport> reports;
        Gcs::B200::Merge3LevelReport level;
        const auto merged = Gcs::B200::solveMerge3Level(inputs, 0, &reports, &level);
        if (stats) stats[0] = static_cast<int64_t>(level.nodes), stats[1] = static_cast<int64_t>(level.candidates), stats[2] = static_cast<int64_t>(level.launches);
        el0 = 0;
        for (int k = 0; k < n_nodes; ++k) {
            int n = 0;
            if (solved_by) solved_by[k] = static_cast<int32_t>(reports[static_cast<std::size_t>(k)].solvedBy);
            if (merged[static_cast<std::size_t>(k)]) {
                const auto& m = *merged[static_cast<std::size_t>(k)];
                for (int i = 0; i < n_el[k]; ++i) {
                    const auto it = m.find(built[static_cast<std::size_t>(k)]->nodes[static_cast<std::size_t>(i)]);
                    if (it == m.end()) continue;
                    out_ids[el0 + static_cast<std::size_t>(n)] = i;
                    double* o = out_pose4 + 4 * (el0 + static_cast<std::size_t>(n));
                    o[0] = o[1] = o[2] = o[3] = 0.0;
                    if (const auto* pp = std::get_if<Bu::PointPose>(&it->second))
                        o[0] = pp->position.x(), o[1] = pp->position.y();
                    else {
                        const auto& l = std::get<Bu::LinePose>(it->second);
                        o[0] = l.p1.x(), o[1] = l.p1.y(), o[2] = l.p2.x(), o[3] = l.p2.y();
                    }
                    ++n;
                }
            }
            out_n[k] = n;
            el0 += static_cast<std::size_t>(n_el[k]);
        }
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// The step after the solve (gcs/b200/canvas_transform.hpp): elements with is_set != 0 carry solver
// positions in pos; on return canvas holds the transformed sketch.  Returns 0 or -1.
GCS_API int gcs_host_canvas_transform(int n_el, gcs_host_element* el)
{
    try {
        std::vector<std::shared_ptr<Gcs::Element>> elems;
        Gcs::ConstraintGraph g;
        for (int i = 0; i < n_el; ++i) {
            elems.push_back(makeElement(el[i]));
            g.addElement(g.getGraph().addNode(), elems.back());
        }
        Gcs::B200::applySolverToCanvasTransform(g);
        for (int i = 0; i < n_el; ++i) {
            const auto& e = *elems[static_cast<std::size_t>(i)];
            if (el[i].type == 0) {
                const auto& p = e.getElement<Gcs::Point>();
                el[i].canvas[0] = p.canvasPosition.x(), el[i].canvas[1] = p.canvasPosition.y();
            } else {
                const auto& l = e.getElement<Gcs::Line>();
                el[i].canvas[0] = l.canvasP1.x(), el[i].canvas[1] = l.canvasP1.y();
                el[i].canvas[2] = l.canvasP2.x(), el[i].canvas[3] = l.canvasP2.y();
            }
        }
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}


// ---- sketch programs (gcs/b200/sketch_program.hpp) ----
// A handle holds the sketch's elements and constraints and the program compiled from them.  Values
// are indexed by the order of the real (non-virtual) edges in `edges`.
struct gcs_host_program {
    std::vector<std::shared_ptr<Gcs::Element>> elems;
    std::vector<std::shared_ptr<Gcs::Constraint>> cons;
    std::unique_ptr<Gcs::B200::SketchProgram> prog;
};

// Check, decompose and compile a whole sketch (no device).  Returns 0 or -1.
GCS_API int gcs_host_program_create(int n_el, const gcs_host_element* el, int n_edges, const gcs_host_edge* edges, gcs_host_program** out)
{
    try {
        auto h = std::make_unique<gcs_host_program>();
        Gcs::ConstraintGraph g = makeSketch(h->elems, n_el, el, n_edges, edges, &h->cons);
        Gcs::DeficitStreeBasedTopDownStrategy st;
        if (st.checkConstraintGraphConstrainedness(g) != Gcs::Constrainedness::WELL_CONSTRAINED && !st.resolve(g))
            throw std::runtime_error("Gcs is not well-constrained, current algorithms do not support such inputs");
        const auto leaves = st.decomposeConstraintGraph(g);
        h->prog = std::make_unique<Gcs::B200::SketchProgram>(Gcs::B200::SketchProgram::compile(leaves, h->elems, h->cons));
        *out = h.release();
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// Compile a given leaf list (the records of gcs_host_leaves_solve; no device).  Returns 0 or -1.
GCS_API int gcs_host_program_create_leaves(int n_el, const gcs_host_element* el, int n_leaves, const int32_t* leaf_elems,
    const int32_t* edge_offsets, const gcs_host_edge* edges, gcs_host_program** out)
{
    try {
        auto h = std::make_unique<gcs_host_program>();
        for (int i = 0; i < n_el; ++i) h->elems.push_back(makeElement(el[i]));
        std::vector<Gcs::ConstraintGraph> leaves;
        for (int l = 0; l < n_leaves; ++l)
            leaves.push_back(makeLeaf(h->elems, leaf_elems + 3 * l, 3, edges + edge_offsets[l], edge_offsets[l + 1] - edge_offsets[l], &h->cons));
        h->prog = std::make_unique<Gcs::B200::SketchProgram>(Gcs::B200::SketchProgram::compile(leaves, h->elems, h->cons));
        *out = h.release();
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// counts[6] = waves, rows, slots, values, leaves, unsupported leaves.  Every other array may be NULL:
// offsets [waves * 5 + 1] (rows of wave w, kind k: offsets[5w + k-1] .. offsets[5w + k]); per row
// solver, leaf, elems [3] (slots of roles a, b, c), values [3] (value slots of v0..v2, -1 = none), code;
// per slot solved_after (solved flag after a run); per leaf solver and level (-1 = not run).
GCS_API int gcs_host_program_describe(const gcs_host_program* h, int64_t* counts, int64_t* offsets, int32_t* row_solver, int64_t* row_leaf,
    int32_t* row_elems, int32_t* row_values, uint8_t* row_code, uint8_t* solved_after, int32_t* leaf_solver, int32_t* leaf_level)
{
    const auto& p = *h->prog;
    const auto& rows = p.rows();
    const auto& rep = p.report();
    if (counts) {
        counts[0] = static_cast<int64_t>(p.waves()), counts[1] = static_cast<int64_t>(rows.size());
        counts[2] = static_cast<int64_t>(p.nSlots()), counts[3] = static_cast<int64_t>(p.nValues());
        counts[4] = static_cast<int64_t>(rep.leaves), counts[5] = static_cast<int64_t>(rep.unsupported);
    }
    if (offsets) std::memcpy(offsets, p.offsets().data(), p.offsets().size() * sizeof(int64_t));
    for (std::size_t r = 0; r < rows.size(); ++r) {
        if (row_solver) row_solver[r] = rows[r].solver;
        if (row_leaf) row_leaf[r] = p.rowLeaf()[r];
        if (row_code) row_code[r] = static_cast<uint8_t>(rows[r].code);
        for (int q = 0; q < 3; ++q) {
            if (row_elems) row_elems[3 * r + static_cast<std::size_t>(q)] = rows[r].elem[q];
            if (row_values) row_values[3 * r + static_cast<std::size_t>(q)] = rows[r].value[q];
        }
    }
    if (solved_after) std::memcpy(solved_after, p.solvedAfter().data(), p.solvedAfter().size());
    for (std::size_t l = 0; l < rep.leaves; ++l) {
        if (leaf_solver) leaf_solver[l] = static_cast<int32_t>(rep.solver[l]);
        if (leaf_level) leaf_level[l] = rep.level[l];
    }
    return 0;
}

// The descriptor of the compiled program (gcs_b200_program_desc), pointing into the program's own
// tables: valid while the handle lives.  Returns 0.
GCS_API int gcs_host_program_desc(const gcs_host_program* h, gcs_b200_program_desc* out)
{
    *out = h->prog->desc();
    return 0;
}

static void programStats(const gcs_host_program* h, const Gcs::B200::ProgramRunStats& st, int n_devices, int64_t* stats)
{
    if (!stats) return;
    stats[0] = st.launches, stats[1] = static_cast<int64_t>(h->prog->compileSeconds() * 1e6);
    stats[2] = static_cast<int64_t>(st.uploadMs * 1e3), stats[3] = static_cast<int64_t>(st.deviceMs * 1e3);
    stats[4] = static_cast<int64_t>(st.downloadMs * 1e3), stats[5] = static_cast<int64_t>(st.seconds * 1e6);
    stats[6] = n_devices;
}

// K instances: values [K][n_values] (angles in radians), positions out [K][n_slots][4], nonconverged
// [K] (may be NULL).  stats (may be NULL) holds 7 values: launches, compile us, upload us, device us,
// download us (device time), run us (host clock), devices used.  Returns 0 or -1.
GCS_API int gcs_host_program_run(gcs_host_program* h, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int n_devices, int64_t* stats)
{
    try {
        programStats(h, h->prog->run(values, K, positions, nonconverged, n_devices), n_devices, stats);
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// The same with the derivatives along T directions (SketchProgram::runTangents): dvalues [K][n_values][T]
// (radians for angles), dpositions out [K][n_slots][4][T].  Returns 0 or -1.
GCS_API int gcs_host_program_run_tangents(gcs_host_program* h, int64_t K, const double* values, int T, const double* dvalues,
    double* positions, double* dpositions, uint32_t* nonconverged, int n_devices, int64_t* stats)
{
    try {
        programStats(h, h->prog->runTangents(values, K, dvalues, T, positions, dpositions, nonconverged, n_devices), n_devices, stats);
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// run(), recording what gcs_host_program_adjoints needs (SketchProgram::record).  Returns 0 or -1.
GCS_API int gcs_host_program_run_recorded(gcs_host_program* h, int64_t K, const double* values, double* positions, uint32_t* nonconverged,
    int n_devices, int64_t* stats)
{
    try {
        programStats(h, h->prog->record(values, K, positions, nonconverged, n_devices), n_devices, stats);
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// Reverse mode over the last recorded run (SketchProgram::adjoints): adj_positions [K][n_slots][4][T],
// adj_values out [K][n_values][T] (radians for angles); stats as gcs_host_program_run (devices: those of
// the recorded run).  Returns 0 or -1.
GCS_API int gcs_host_program_adjoints(gcs_host_program* h, int T, const double* adj_positions, double* adj_values, int64_t* stats)
{
    try {
        const Gcs::B200::ProgramRunStats st = h->prog->adjoints(adj_positions, T, adj_values);
        programStats(h, st, h->prog->recordedDevices(), stats);
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

// The edit loop: values (may be NULL: keep the current ones) become the constraints' values, then
// SketchProgram::solve(); el receives every element's solved flag and position.  Returns 0 or -1.
GCS_API int gcs_host_program_solve(gcs_host_program* h, const double* values, gcs_host_element* el)
{
    try {
        if (values)
            for (std::size_t v = 0; v < h->cons.size(); ++v) {
                if (auto* d = h->cons[v]->getConstraintAs<Gcs::DistanceConstraint>()) d->distance = values[v];
                if (auto* a = h->cons[v]->getConstraintAs<Gcs::AngleConstraint>()) a->angle = values[v];
            }
        h->prog->solve();
        for (std::size_t i = 0; i < h->elems.size(); ++i) readBack(*h->elems[i], el[i]);
        return 0;
    } catch (const std::exception& ex) {
        return fail(ex);
    }
}

GCS_API void gcs_host_program_destroy(gcs_host_program* h) { delete h; }

}  // extern "C"
