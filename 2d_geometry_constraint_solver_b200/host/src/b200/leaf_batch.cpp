// leaf_batch.cpp — classification, role assignment, packing, write-back and the batched leaf
// scheduler behind the reference-shaped solver entry points (see gcs/b200/leaf_batch.hpp).
//
// What each piece restates (all paths relative to src/constraint_solver/src/solving/):
//   matches()      the eight predicates           solvers/point_point_solvers.cpp:14-24, :87-95
//                                                 solvers/point_line_solvers.cpp:114-133, :261-289,
//                                                 :405-443, :547-575
//                                                 solvers/line_angle_solvers.cpp:169-185, :377-415
//   classify()     first-match dispatch order     component_solver.hpp:31-66
//   assignRoles()  ascending-NodeId role loops    point_point_solvers.cpp:28-45, :110-123, ...
//   packNumeric()  anchoring, signed distances, canvas normals, canvas-side signs: everything
//                  the reference's solve() does before and around solve2D that is not a function
//                  of the Newton candidates.  The candidate-dependent rest runs in the kernels.
// Numerics on this side are plain IEEE doubles evaluated in the reference's order (one rounding
// per operation; the host build uses -ffp-contract=off like the reference's baseline x86-64 build).
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <mutex>
#include <cstring>
#include <cmath>
#include <exception>
#include <memory>
#include <stdexcept>
#include <unordered_map>
#include <unordered_set>

#include <gcs/b200/leaf_batch.hpp>
#include <gcs/model/constraints.hpp>
#include <gcs/model/elements.hpp>

#include "plan.hpp"
#include "solving/solvers/heuristics.hpp"

namespace Gcs::B200 {

using Eigen::Vector2d;
using NodeId = ConstraintGraph::NodeIdType;
using detail::CanvasRow;
using detail::ColdFacts;
using detail::Plan;
using detail::Roles;
using detail::makePlan;

namespace {

bool querySet(const SetQuery& q, const Element* e) { return q ? q(e) : e->isElementSet(); }

int sign3(double x) { return (x > 0) - (x < 0); }            // heuristics.hpp:54 (three-valued)
double signOf(double x) { return (x > 0.0) ? 1.0 : -1.0; }   // point_line_solvers.cpp:195 (zero -> -1)

struct Census {
    int points = 0, lines = 0;
    int solved = 0, solvedPoints = 0, unsolvedPoints = 0, solvedLines = 0, unsolvedLines = 0;
};

Census census(const ConstraintGraph& g, const SetQuery& q)
{
    Census c;
    for (const auto& [node, e] : g.getElementMap()) {
        const bool set = querySet(q, e.get());
        c.solved += set ? 1 : 0;
        if (e->isElementType<Point>()) {
            ++c.points;
            ++(set ? c.solvedPoints : c.unsolvedPoints);
        } else if (e->isElementType<Line>()) {
            ++c.lines;
            ++(set ? c.solvedLines : c.unsolvedLines);
        }
    }
    return c;
}

struct ConstraintCensus {
    int total = 0, distance = 0, angle = 0;
};

bool matchesCountsOn(SolverId id, int edgeCount, const Census& c, const ConstraintCensus& k);  // below, with the predicates

ConstraintCensus constraintCensus(const ConstraintGraph& g)
{
    // the constraint map holds real constraints only: virtual edges carry none
    ConstraintCensus c;
    for (const auto& [edge, k] : g.getConstraintMap()) {
        if (g.isVirtualEdge(edge)) continue;
        ++c.total;
        if (k->isConstraintType<DistanceConstraint>())
            ++c.distance;
        else if (k->isConstraintType<AngleConstraint>())
            ++c.angle;
    }
    return c;
}

double valueBetween(const ConstraintGraph& g, NodeId s, NodeId t, const Constraint*& con, bool* flip = nullptr)
{
    // getConstraintBetweenNodes throws std::bad_expected_access for a missing / virtual edge,
    // getConstraintValue().value() for a constraint without a value - as in the reference
    const auto k = g.getConstraintBetweenNodes(s, t);
    con = k.get();
    if (flip) {
        const auto* ang = k->getConstraintAs<AngleConstraint>();
        *flip = ang != nullptr && ang->flipOrientation;  // line_angle_solvers.cpp:322-326
    }
    return k->getConstraintValue().value();
}

Roles assignRoles(SolverId id, const ConstraintGraph& g, const SetQuery& q)
{
    Roles r;
    r.id = id;
    NodeId na {}, nb {}, nc {};
    bool haveA = false;
    const auto& map = g.getElementMap();
    switch (id) {
    case SolverId::ZeroFixedPointsTriangle: {  // point_point_solvers.cpp:28-45
        int i = 0;
        for (const auto& [node, e] : map) {
            if (i == 0) r.a = e.get(), na = node;
            if (i == 1) r.b = e.get(), nb = node;
            if (i == 2) r.c = e.get(), nc = node;
            ++i;
        }
        r.v0 = valueBetween(g, na, nb, r.k[0]);
        r.v1 = valueBetween(g, na, nc, r.k[1]);
        r.v2 = valueBetween(g, nb, nc, r.k[2]);
        break;
    }
    case SolverId::ZeroFixedPPLTriangle:  // point_line_solvers.cpp:148-161
    case SolverId::TwoFixedPointsLine: {  // point_line_solvers.cpp:304-317
        for (const auto& [node, e] : map) {
            if (e->isElementType<Line>()) {
                r.c = e.get(), nc = node;
            } else if (e->isElementType<Point>()) {
                if (!haveA)
                    r.a = e.get(), na = node, haveA = true;
                else
                    r.b = e.get(), nb = node;
            }
        }
        if (id == SolverId::ZeroFixedPPLTriangle) r.v0 = valueBetween(g, na, nb, r.k[0]);
        r.v1 = valueBetween(g, na, nc, r.k[1]);
        r.v2 = valueBetween(g, nb, nc, r.k[2]);
        break;
    }
    case SolverId::ZeroFixedLLPAngleTriangle: {  // line_angle_solvers.cpp:202-215
        for (const auto& [node, e] : map) {
            if (e->isElementType<Point>()) {
                r.b = e.get(), nb = node;
            } else if (e->isElementType<Line>()) {
                if (!haveA)
                    r.a = e.get(), na = node, haveA = true;
                else
                    r.c = e.get(), nc = node;
            }
        }
        r.v0 = valueBetween(g, na, nc, r.k[0], &r.flip);
        r.v1 = valueBetween(g, nb, na, r.k[1]);
        r.v2 = valueBetween(g, nb, nc, r.k[2]);
        break;
    }
    case SolverId::TwoFixedPointsDistance: {  // point_point_solvers.cpp:110-123
        for (const auto& [node, e] : map) {
            if (querySet(q, e.get())) {
                if (!haveA)
                    r.a = e.get(), na = node, haveA = true;
                else
                    r.b = e.get(), nb = node;
            } else {
                r.c = e.get(), nc = node;
            }
        }
        if (!r.c)
            throw std::logic_error("TwoFixedPointsDistanceSolver: all three points are already solved; the reference "
                                   "dereferences a null free point here (point_point_solvers.cpp:89, :110-127)");
        r.v1 = valueBetween(g, na, nc, r.k[1]);
        r.v2 = valueBetween(g, nb, nc, r.k[2]);
        break;
    }
    case SolverId::FixedPointAndLineFreePoint: {  // point_line_solvers.cpp:458-471
        for (const auto& [node, e] : map) {
            if (e->isElementType<Line>()) {
                r.b = e.get(), nb = node;
            } else if (e->isElementType<Point>()) {
                if (querySet(q, e.get()))
                    r.a = e.get(), na = node;
                else
                    r.c = e.get(), nc = node;
            }
        }
        r.v1 = valueBetween(g, na, nc, r.k[1]);
        r.v2 = valueBetween(g, nb, nc, r.k[2]);
        break;
    }
    case SolverId::TwoFixedLinesFreePoint: {  // point_line_solvers.cpp:590-603
        for (const auto& [node, e] : map) {
            if (e->isElementType<Point>()) {
                r.c = e.get(), nc = node;
            } else if (e->isElementType<Line>()) {
                if (!haveA)
                    r.a = e.get(), na = node, haveA = true;
                else
                    r.b = e.get(), nb = node;
            }
        }
        r.v1 = valueBetween(g, na, nc, r.k[1]);
        r.v2 = valueBetween(g, nb, nc, r.k[2]);
        break;
    }
    case SolverId::FixedLineAndPointFreeLine: {  // line_angle_solvers.cpp:432-445
        for (const auto& [node, e] : map) {
            if (e->isElementType<Point>()) {
                r.b = e.get(), nb = node;
            } else if (e->isElementType<Line>()) {
                if (querySet(q, e.get()))
                    r.a = e.get(), na = node;
                else
                    r.c = e.get(), nc = node;
            }
        }
        r.v0 = valueBetween(g, na, nc, r.k[0], &r.flip);
        r.v2 = valueBetween(g, nb, nc, r.k[2]);
        break;
    }
    case SolverId::None: break;
    }
    return r;
}

bool zeroFixed(SolverId id)
{
    return id == SolverId::ZeroFixedPointsTriangle || id == SolverId::ZeroFixedPPLTriangle
        || id == SolverId::ZeroFixedLLPAngleTriangle;
}

Footprint footprintOf(const Roles& r)
{
    Footprint f;
    if (r.id == SolverId::None) return f;
    if (zeroFixed(r.id)) {
        f.writes = { r.a, r.b, r.c };
        f.nWrites = 3;
    } else {
        f.writes[0] = r.c;
        f.nWrites = 1;
        f.reads = { r.a, r.b, nullptr };
        f.nReads = 2;
    }
    return f;
}

// canvas unit normal of a line: (-dir.y / len, dir.x / len), two separate divisions
// (point_line_solvers.cpp:213-216, line_angle_solvers.cpp:300-305)
void canvasNormal(const Line& l, double& nx, double& ny, double& len)
{
    const Vector2d dir = l.canvasP2 - l.canvasP1;
    len = dir.norm();
    nx = -dir.y() / len;
    ny = dir.x() / len;
}

}  // namespace

// Canvas half of pack(): orientation code, canvas-side signs and canvas constants of a row.
CanvasRow detail::packCanvas(const Roles& r)
{
    CanvasRow cv;
    double* cst = cv.cst;
    switch (r.id) {
    case SolverId::ZeroFixedPointsTriangle:
    case SolverId::TwoFixedPointsDistance: {
        // point_point_solvers.cpp:48-71 / :136-151
        const double ori = Solvers::triangleOrientation(r.a->getElement<Point>().canvasPosition,
            r.b->getElement<Point>().canvasPosition, r.c->getElement<Point>().canvasPosition);
        cv.code = GCS_MAKE_CODE(sign3(ori), 0, 0);
        break;
    }
    case SolverId::ZeroFixedPPLTriangle:
    case SolverId::TwoFixedPointsLine: {
        // point_line_solvers.cpp:179-219 / :335-364
        const auto& ln = r.c->getElement<Line>();
        const double c1 = Solvers::signedDistanceToLine(r.a->getElement<Point>().canvasPosition, ln.canvasP1, ln.canvasP2);
        const double c2 = Solvers::signedDistanceToLine(r.b->getElement<Point>().canvasPosition, ln.canvasP1, ln.canvasP2);
        cv.sign[1] = signOf(c1), cv.sign[2] = signOf(c2);
        canvasNormal(ln, cst[0], cst[1], cst[2]);
        cv.code = GCS_MAKE_CODE(sign3(c1), sign3(c2), 0);
        break;
    }
    case SolverId::FixedPointAndLineFreePoint: {
        // point_line_solvers.cpp:485-529
        const auto& fp = r.a->getElement<Point>();
        const auto& ln = r.b->getElement<Line>();
        const auto& fr = r.c->getElement<Point>();
        const double cs = Solvers::signedDistanceToLine(fr.canvasPosition, ln.canvasP1, ln.canvasP2);
        cv.sign[2] = signOf(cs);
        cst[0] = fr.canvasPosition.x(), cst[1] = fr.canvasPosition.y();
        const Vector2d canvasFoot = Solvers::perpendicularFoot(fp.canvasPosition, ln.canvasP1, ln.canvasP2);
        const double ori = Solvers::triangleOrientation(fp.canvasPosition, canvasFoot, fr.canvasPosition);
        const int flags = (std::abs(ori) < GCS_COLLINEAR_EPSILON) ? GCS_CODE_COLLINEAR : 0;  // heuristics.hpp:209-217
        cv.code = GCS_MAKE_CODE(sign3(ori), 0, flags);
        break;
    }
    case SolverId::TwoFixedLinesFreePoint: {
        // point_line_solvers.cpp:617-682
        const auto& l1 = r.a->getElement<Line>();
        const auto& l2 = r.b->getElement<Line>();
        const auto& fr = r.c->getElement<Point>();
        const double c1 = Solvers::signedDistanceToLine(fr.canvasPosition, l1.canvasP1, l1.canvasP2);
        const double c2 = Solvers::signedDistanceToLine(fr.canvasPosition, l2.canvasP1, l2.canvasP2);
        cv.sign[1] = signOf(c1), cv.sign[2] = signOf(c2);
        cst[0] = fr.canvasPosition.x(), cst[1] = fr.canvasPosition.y();
        const auto ci = Solvers::lineLineIntersection(l1.canvasP1, l1.canvasP2, l2.canvasP1, l2.canvasP2);
        if (!ci) {
            cv.code = GCS_MAKE_CODE(0, 0, GCS_CODE_CANVAS_PARALLEL);
        } else {
            const Vector2d canvasDir = (l1.canvasP2 - l1.canvasP1).normalized();
            const Vector2d canvasRef = *ci + canvasDir;
            const double ori = Solvers::triangleOrientation(*ci, canvasRef, fr.canvasPosition);
            const int flags = (std::abs(ori) < GCS_COLLINEAR_EPSILON) ? GCS_CODE_COLLINEAR : 0;
            cv.code = GCS_MAKE_CODE(sign3(ori), 0, flags);
        }
        break;
    }
    case SolverId::ZeroFixedLLPAngleTriangle:
    case SolverId::FixedLineAndPointFreeLine: {
        // line_angle_solvers.cpp:245-361 / :474-557
        const auto& fixed = r.a->getElement<Line>();
        const auto& pt = r.b->getElement<Point>();
        const auto& fr = r.c->getElement<Line>();
        const Vector2d canvasFixed = fixed.canvasP2 - fixed.canvasP1;
        canvasNormal(fr, cst[0], cst[1], cst[4]);
        cst[2] = canvasFixed.x(), cst[3] = canvasFixed.y();
        Vector2d canvasFree = fr.canvasP2 - fr.canvasP1;
        if (r.flip) canvasFree = -canvasFree;
        const double cross = (canvasFixed.x() * canvasFree.y()) - (canvasFixed.y() * canvasFree.x());  // heuristics.hpp:310-312
        const double cs2 = Solvers::signedDistanceToLine(pt.canvasPosition, fr.canvasP1, fr.canvasP2);
        cv.sign[2] = signOf(cs2);
        if (r.id == SolverId::ZeroFixedLLPAngleTriangle) {
            // line1 anchored on the x axis, centred on the origin; the point above or below it
            const double len1 = canvasFixed.norm();
            const Vector2d a1 { -len1 / 2.0, 0.0 }, a2 { len1 / 2.0, 0.0 };
            const Vector2d anchorDir = a2 - a1;
            cst[5] = anchorDir.x(), cst[6] = anchorDir.y(), cst[7] = a1.x(), cst[8] = a2.x();
            cv.sign[1] = signOf(Solvers::signedDistanceToLine(pt.canvasPosition, fixed.canvasP1, fixed.canvasP2));
        }
        cv.code = GCS_MAKE_CODE(sign3(cross), 0, 0);
        break;
    }
    case SolverId::None: break;
    }
    return cv;
}

namespace {

// Numeric half of pack(): reads solved positions, places anchors, fills the batch row.  The
// sketch program's gather_row (csrc/sketch_program.cu) is the device's copy of this function.
PackedLeaf packNumeric(const Roles& r)
{
    const CanvasRow cv = detail::packCanvas(r);
    const double* cst = cv.cst;
    PackedLeaf p;
    p.solver = r.id;
    p.kind = kindOf(r.id);
    p.target = r.c;
    p.code = cv.code;
    double* in = p.in;
    switch (r.id) {
    case SolverId::ZeroFixedPointsTriangle:
    case SolverId::TwoFixedPointsDistance: {
        if (r.id == SolverId::ZeroFixedPointsTriangle) {
            r.a->updateElementPosition(Vector2d { 0.0, 0.0 });
            r.b->updateElementPosition(Vector2d { r.v0, 0.0 });
        }
        const auto& p1 = r.a->getElement<Point>();
        const auto& p2 = r.b->getElement<Point>();
        in[0] = p1.position.x(), in[1] = p1.position.y(), in[2] = r.v1;
        in[3] = p2.position.x(), in[4] = p2.position.y(), in[5] = r.v2;
        break;
    }
    case SolverId::ZeroFixedPPLTriangle:
    case SolverId::TwoFixedPointsLine: {
        if (r.id == SolverId::ZeroFixedPPLTriangle) {
            r.a->updateElementPosition(Vector2d { 0.0, 0.0 });
            r.b->updateElementPosition(Vector2d { r.v0, 0.0 });
        }
        const auto& p1 = r.a->getElement<Point>();
        const auto& p2 = r.b->getElement<Point>();
        in[0] = p1.position.x(), in[1] = p1.position.y();
        in[2] = p2.position.x(), in[3] = p2.position.y();
        in[4] = cv.sign[1] * r.v1;
        in[5] = cv.sign[2] * r.v2;
        in[6] = cst[0], in[7] = cst[1], in[8] = cst[2];
        break;
    }
    case SolverId::FixedPointAndLineFreePoint: {
        const auto& fp = r.a->getElement<Point>();
        const auto& ln = r.b->getElement<Line>();
        in[0] = fp.position.x(), in[1] = fp.position.y(), in[2] = r.v1;
        in[3] = ln.p1.x(), in[4] = ln.p1.y(), in[5] = ln.p2.x(), in[6] = ln.p2.y();
        in[7] = cv.sign[2] * r.v2;
        in[8] = cst[0], in[9] = cst[1];
        break;
    }
    case SolverId::TwoFixedLinesFreePoint: {
        const auto& l1 = r.a->getElement<Line>();
        const auto& l2 = r.b->getElement<Line>();
        in[0] = l1.p1.x(), in[1] = l1.p1.y(), in[2] = l1.p2.x(), in[3] = l1.p2.y(), in[4] = cv.sign[1] * r.v1;
        in[5] = l2.p1.x(), in[6] = l2.p1.y(), in[7] = l2.p2.x(), in[8] = l2.p2.y(), in[9] = cv.sign[2] * r.v2;
        in[10] = cst[0], in[11] = cst[1];
        break;
    }
    case SolverId::ZeroFixedLLPAngleTriangle: {
        r.a->updateElementPosition(Vector2d { cst[7], 0.0 }, Vector2d { cst[8], 0.0 });
        const Vector2d anchorPoint { 0.0, cv.sign[1] * r.v1 };
        r.b->updateElementPosition(anchorPoint);
        in[0] = cst[5], in[1] = cst[6];
        in[2] = std::cos(r.v0);
        in[3] = cst[0], in[4] = cst[1], in[12] = cst[4];
        in[5] = cst[2], in[6] = cst[3];
        in[7] = anchorPoint.x(), in[8] = anchorPoint.y();
        in[9] = cv.sign[2] * r.v2;
        in[10] = 0.0, in[11] = 0.0;  // second reference point: the origin (line_angle_solvers.cpp:353)
        break;
    }
    case SolverId::FixedLineAndPointFreeLine: {
        const auto& fl = r.a->getElement<Line>();
        const auto& pt = r.b->getElement<Point>();
        const Vector2d fd = fl.p2 - fl.p1;
        in[0] = fd.x(), in[1] = fd.y();
        in[2] = std::cos(r.v0);
        in[3] = cst[0], in[4] = cst[1], in[12] = cst[4];
        in[5] = cst[2], in[6] = cst[3];
        in[7] = pt.position.x(), in[8] = pt.position.y();
        in[9] = cv.sign[2] * r.v2;
        const Vector2d mid = fl.midpoint();
        in[10] = mid.x(), in[11] = mid.y();
        break;
    }
    case SolverId::None: break;
    }
    return p;
}

void solveBatchOnDevice(KindBatch& batch, int device)
{
    gcs_b200_batch d = batch.descriptor();
    const int rc = gcs_b200_solve_host(&d, device);
    if (rc != GCS_OK)
        throw std::runtime_error(std::string("gcs_b200_solve_host failed (") + std::to_string(rc) + "): " + gcs_b200_last_error()
            + " - the sub-problem solvers run on the CUDA path only");
    batch.applyAll();
}

// ---------------------------------------------------------------------------------------------
// The symbolic pass in two steps.
//  (A) per leaf, independent of every other leaf (hence over all host threads): the three
//      elements in ascending node id, their types, the constraint on each of the three node pairs
//      (kind, value, orientation flag; virtual and missing edges carry none), the counts the eight
//      predicates ask for.  This is where the graph containers are walked.
//  (B) one sequential sweep over those facts with the PREDICTED solved flags: the reference's
//      first-match dispatch (component_solver.hpp:31-66), its role loops, the read / write footprint
//      and the wave of every leaf.  No container is touched here; elements are numbered on first
//      sight through a tag kept in the Element itself.
// A leaf the facts cannot describe (not three nodes, a role whose constraint is missing, ...) goes
// through the general code (classify / assignRoles on the graph), which raises what the reference
// raises.
// ---------------------------------------------------------------------------------------------
//
// The facts of a leaf come in two parts.  What the sweep reads for every leaf is 32 bytes (element
// numbers, the kinds / counts of the leaf folded into a key, which elements are solved already,
// which node pairs carry a value); pointers and constraint values are only read again when the
// leaf's row is packed, on whatever thread packs it.
struct HotFacts {
    std::uint64_t serial[3];  // Element::serial(): what the sweep's per-element tables are indexed by
    std::uint32_t shapeKey;   // Shape::key(): what classification depends on besides the solved flags
    std::uint8_t setNow;      // bit 2 - k: element k is solved already
    std::uint8_t has;         // bit p: node pair p - (0,1), (0,2), (1,2) - has a constraint with a value
    std::uint8_t simple;      // 0: the general code decides (and raises what the reference raises)
    std::uint8_t pad;
};
}  // namespace
struct detail::ColdFacts {
    Element* e[3];
    double val[3];    // node pairs (0,1), (0,2), (1,2): value of the real constraint on the edge, if `has`
    const Constraint* con[3];  // ... and the constraint itself
    std::uint8_t flip;  // bit p: AngleConstraint::flipOrientation of pair p
};
namespace {

inline int pairIndex(int a, int b) { return a + b - 1; }  // {0,1} -> 0, {0,2} -> 1, {1,2} -> 2

// kinds and counts of a three-element leaf: everything the eight predicates ask besides the solved flags
struct Shape {
    bool isPoint[3] = {}, isLine[3] = {};
    int edgeCount = 0;                     // virtual edges included; at most three in a digest-described leaf
    int total = 0, distance = 0, angle = 0;  // constraintCensus()
    std::uint32_t key() const
    {
        std::uint32_t k = 0;
        for (int i = 0; i < 3; ++i) k = (k << 2) | (isPoint[i] ? 1u : isLine[i] ? 2u : 0u);
        k = (k << 2) | static_cast<std::uint32_t>(edgeCount & 3);
        k = (k << 2) | static_cast<std::uint32_t>(total & 3);
        k = (k << 2) | static_cast<std::uint32_t>(distance & 3);
        return (k << 2) | static_cast<std::uint32_t>(angle & 3);
    }
    static Shape ofKey(std::uint32_t k)
    {
        Shape s;
        s.angle = static_cast<int>(k & 3), k >>= 2;
        s.distance = static_cast<int>(k & 3), k >>= 2;
        s.total = static_cast<int>(k & 3), k >>= 2;
        s.edgeCount = static_cast<int>(k & 3), k >>= 2;
        for (int i = 2; i >= 0; --i) s.isPoint[i] = (k & 3) == 1, s.isLine[i] = (k & 3) == 2, k >>= 2;
        return s;
    }
};

// false: the leaf is not one the digest describes
bool gatherFacts(const ConstraintGraph& g, HotFacts& hot, ColdFacts& cold)
{
    hot = HotFacts {};
    // the graph's own digest: three elements in ascending node id, the constraint of each node pair
    // (ConstraintGraph::triangleDigest; the decomposition left it warm).  Flags, kinds and values are
    // read here, through the pointers: they may have changed since the digest was taken.
    const TriangleDigest& d = g.triangleDigest();
    if (!d.simple) return false;
    cold = ColdFacts {};
    Shape shape;
    for (int n = 0; n < 3; ++n) {
        Element* el = d.element[n];
        cold.e[n] = el;
        shape.isPoint[n] = el->isElementType<Point>();
        shape.isLine[n] = el->isElementType<Line>();
        if (el->isElementSet()) hot.setNow |= static_cast<std::uint8_t>(4 >> n);
        hot.serial[n] = el->serial();
    }
    shape.edgeCount = d.edgeCount;
    for (int p = 0; p < 3; ++p) {
        const Constraint* con = d.constraint[p];
        if (!con) continue;
        ++shape.total;  // constraintCensus(): every real constraint, with or without a value
        const auto* ang = con->getConstraintAs<AngleConstraint>();
        if (con->isConstraintType<DistanceConstraint>())
            ++shape.distance;
        else if (ang)
            ++shape.angle;
        const auto v = con->getConstraintValue();
        if (!v.has_value()) continue;
        hot.has |= static_cast<std::uint8_t>(1 << p);
        cold.val[p] = v.value();
        cold.con[p] = con;
        if (ang != nullptr && ang->flipOrientation) cold.flip |= static_cast<std::uint8_t>(1 << p);
    }
    hot.shapeKey = shape.key();
    hot.simple = 1;
    return true;
}

constexpr long long kFactsLookAhead = 12;

void prefetchFacts(const ConstraintGraph& g)
{
    const TriangleDigest& d = g.triangleDigest();
    if (!d.simple) return;
    for (int n = 0; n < 3; ++n) {
        // kind, solved flag and serial number sit behind the shape's coordinates
        const char* tail = reinterpret_cast<const char*>(d.element[n]) + sizeof(Element) - 1;
        __builtin_prefetch(tail);
        __builtin_prefetch(tail - 23);
    }
    for (int p = 0; p < 3; ++p)
        if (d.constraint[p]) __builtin_prefetch(d.constraint[p]);
}

// classify() on a shape: same counts, same order
SolverId classifyShape(const Shape& f, const bool set[3])
{
    Census c;
    for (int i = 0; i < 3; ++i) {
        c.solved += set[i] ? 1 : 0;
        if (f.isPoint[i]) {
            ++c.points;
            ++(set[i] ? c.solvedPoints : c.unsolvedPoints);
        } else if (f.isLine[i]) {
            ++c.lines;
            ++(set[i] ? c.solvedLines : c.unsolvedLines);
        }
    }
    static constexpr SolverId order[] = { SolverId::ZeroFixedPointsTriangle, SolverId::ZeroFixedPPLTriangle,
        SolverId::ZeroFixedLLPAngleTriangle, SolverId::TwoFixedPointsDistance, SolverId::TwoFixedPointsLine,
        SolverId::FixedPointAndLineFreePoint, SolverId::TwoFixedLinesFreePoint, SolverId::FixedLineAndPointFreeLine };
    const ConstraintCensus k { f.total, f.distance, f.angle };
    for (SolverId id : order)
        if (matchesCountsOn(id, f.edgeCount, c, k)) return id;
    return SolverId::None;
}

// assignRoles() on a shape: who plays which part (indices into the leaf's three elements).
// false when the shape is one the role loops do not fill.
bool roleIndices(SolverId id, const Shape& f, const bool set[3], int& ia, int& ib, int& ic)
{
    ia = ib = ic = -1;
    auto firstSecond = [&](auto pred, int& first, int& second) {  // "if (!haveA) a = e else b = e" over ascending ids
        for (int i = 0; i < 3; ++i)
            if (pred(i)) {
                if (first < 0)
                    first = i;
                else
                    second = i;
            }
    };
    auto last = [&](auto pred, int& slot) {
        for (int i = 0; i < 3; ++i)
            if (pred(i)) slot = i;
    };
    switch (id) {
    case SolverId::ZeroFixedPointsTriangle: ia = 0, ib = 1, ic = 2; break;
    case SolverId::ZeroFixedPPLTriangle:
    case SolverId::TwoFixedPointsLine:
        last([&](int i) { return f.isLine[i]; }, ic);
        firstSecond([&](int i) { return !f.isLine[i] && f.isPoint[i]; }, ia, ib);
        break;
    case SolverId::ZeroFixedLLPAngleTriangle:
        last([&](int i) { return f.isPoint[i]; }, ib);
        firstSecond([&](int i) { return !f.isPoint[i] && f.isLine[i]; }, ia, ic);
        break;
    case SolverId::TwoFixedPointsDistance:
        firstSecond([&](int i) { return set[i]; }, ia, ib);
        last([&](int i) { return !set[i]; }, ic);  // all three solved: ic stays -1, the general code raises the reference's failure
        break;
    case SolverId::FixedPointAndLineFreePoint:
        last([&](int i) { return f.isLine[i]; }, ib);
        last([&](int i) { return !f.isLine[i] && f.isPoint[i] && set[i]; }, ia);
        last([&](int i) { return !f.isLine[i] && f.isPoint[i] && !set[i]; }, ic);
        break;
    case SolverId::TwoFixedLinesFreePoint:
        last([&](int i) { return f.isPoint[i]; }, ic);
        firstSecond([&](int i) { return !f.isPoint[i] && f.isLine[i]; }, ia, ib);
        break;
    case SolverId::FixedLineAndPointFreeLine:
        last([&](int i) { return f.isPoint[i]; }, ib);
        last([&](int i) { return !f.isPoint[i] && f.isLine[i] && set[i]; }, ia);
        last([&](int i) { return !f.isPoint[i] && f.isLine[i] && !set[i]; }, ic);
        break;
    case SolverId::None: return false;
    }
    return ia >= 0 && ib >= 0 && ic >= 0 && ia != ib && ia != ic && ib != ic;
}

// Which constraint feeds which value of a solver: v0 / v1 / v2 of Roles, as node pairs of the roles
// (-1: the solver does not read that value).  The reference's solve() bodies, e.g.
// point_point_solvers.cpp:48-50, line_angle_solvers.cpp:322-333.
struct ValuePairs {
    int v0 = -1, v1 = -1, v2 = -1;  // pairIndex() of the two elements
    bool flipFromV0 = false;
};
ValuePairs valuePairs(SolverId id, int ia, int ib, int ic)
{
    auto pair = [](int a, int b) { return pairIndex(a < b ? a : b, a < b ? b : a); };
    ValuePairs v;
    switch (id) {
    case SolverId::ZeroFixedPointsTriangle:
    case SolverId::ZeroFixedPPLTriangle: v.v0 = pair(ia, ib), v.v1 = pair(ia, ic), v.v2 = pair(ib, ic); break;
    case SolverId::ZeroFixedLLPAngleTriangle: v.v0 = pair(ia, ic), v.flipFromV0 = true, v.v1 = pair(ib, ia), v.v2 = pair(ib, ic); break;
    case SolverId::TwoFixedPointsDistance:
    case SolverId::TwoFixedPointsLine:
    case SolverId::FixedPointAndLineFreePoint:
    case SolverId::TwoFixedLinesFreePoint: v.v1 = pair(ia, ic), v.v2 = pair(ib, ic); break;
    case SolverId::FixedLineAndPointFreeLine: v.v0 = pair(ia, ic), v.flipFromV0 = true, v.v2 = pair(ib, ic); break;
    case SolverId::None: break;
    }
    return v;
}

// What the sweep decides for a leaf from its shape and the predicted solved flags, remembered per
// distinct combination: a sketch has a handful of them.
struct Verdict {
    SolverId id = SolverId::None;
    std::int8_t ia = -1, ib = -1, ic = -1;
    bool roles = false;      // ia, ib, ic are valid
    std::uint8_t need = 0;   // bit p: node pair p must carry a value (else the general code raises the reference's exception)
};

Verdict decide(std::uint32_t shapeKey, unsigned setBits)
{
    const Shape shape = Shape::ofKey(shapeKey);
    const bool set[3] = { (setBits & 4) != 0, (setBits & 2) != 0, (setBits & 1) != 0 };
    Verdict v;
    v.id = classifyShape(shape, set);
    if (v.id == SolverId::None) return v;
    int ia, ib, ic;
    v.roles = roleIndices(v.id, shape, set, ia, ib, ic);
    v.ia = static_cast<std::int8_t>(ia), v.ib = static_cast<std::int8_t>(ib), v.ic = static_cast<std::int8_t>(ic);
    if (v.roles) {
        const ValuePairs vp = valuePairs(v.id, ia, ib, ic);
        for (int p : { vp.v0, vp.v1, vp.v2 })
            if (p >= 0) v.need |= static_cast<std::uint8_t>(1 << p);
    }
    return v;
}

class VerdictMemo {
public:
    const Verdict& get(std::uint32_t shapeKey, unsigned setBits)
    {
        const std::uint32_t key = (shapeKey << 3) | setBits;
        Entry& e = m_rows[(key * 2654435761u) >> 24];
        if (e.key != key) e.key = key, e.verdict = decide(shapeKey, setBits);
        return e.verdict;
    }

private:
    struct Entry {
        std::uint32_t key = ~0u;
        Verdict verdict;
    };
    Entry m_rows[256];
};

// The roles of a leaf the sweep decided from its facts: put together where the row is packed.
// code: ia | ib << 2 | ic << 4 (kRolesStored: the general code stored them in Plan::roles instead).
constexpr std::uint8_t kRolesStored = 0xff;
Roles rolesFromFacts(SolverId id, std::uint8_t code, const ColdFacts& f)
{
    const int ia = code & 3, ib = (code >> 2) & 3, ic = (code >> 4) & 3;
    const ValuePairs vp = valuePairs(id, ia, ib, ic);
    Roles r;
    r.id = id;
    r.a = f.e[ia], r.b = f.e[ib], r.c = f.e[ic];
    if (vp.v0 >= 0) r.v0 = f.val[vp.v0], r.k[0] = f.con[vp.v0];
    if (vp.v1 >= 0) r.v1 = f.val[vp.v1], r.k[1] = f.con[vp.v1];
    if (vp.v2 >= 0) r.v2 = f.val[vp.v2], r.k[2] = f.con[vp.v2];
    r.flip = vp.flipFromV0 && ((f.flip >> vp.v0) & 1) != 0;
    return r;
}

// Element serial -> index into the sweep's per-element tables.  The elements of one sketch were
// constructed together, so their serials fill a narrow range and the index is a subtraction; a
// plan over elements scattered through the life of the process falls back to a hash table.
struct SlotIndex {
    std::uint64_t lo = 0;
    bool direct = true;
    std::unordered_map<std::uint64_t, int> sparse;
    int of(std::uint64_t serial)
    {
        if (direct) return static_cast<int>(serial - lo);
        return sparse.try_emplace(serial, static_cast<int>(sparse.size())).first->second;
    }
};

// Working memory of a plan, kept by the thread between plans: a sketch is solved again and again
// while it is edited, and fresh memory for 1e5 leaves costs more in page faults (~3 ms) than the
// facts pass takes.  Buffers that have grown far beyond what the last plans needed are given back.
struct PlanScratch {
    template <typename T>
    struct Buffer {
        T* p = nullptr;
        std::size_t cap = 0;
        int idle = 0;  // plans in a row that used less than a quarter
        T* get(std::size_t n)
        {
            idle = (cap > 65536 && n < cap / 4) ? idle + 1 : 0;
            if (n > cap || idle >= 8) {
                std::free(p);
                cap = std::max<std::size_t>(n + n / 4, 64);
                p = static_cast<T*>(std::malloc(sizeof(T) * cap));
                if (!p) {
                    cap = 0;
                    throw std::bad_alloc();
                }
                idle = 0;
            }
            return p;
        }
        ~Buffer() { std::free(p); }
    };
    Buffer<HotFacts> hot;
    Buffer<ColdFacts> cold;
    Buffer<Roles> roles;
    Buffer<std::uint8_t> roleCode;
    std::vector<char> predicted;
    std::vector<int> lastWrite, lastRead;
};
thread_local PlanScratch t_planScratch;

}  // namespace

Roles detail::Plan::rolesOf(std::size_t i) const
{
    return roleCode[i] == kRolesStored ? roles[i] : rolesFromFacts(report.solver[i], roleCode[i], cold[i]);
}

Plan detail::makePlan(const std::vector<ConstraintGraph>& leaves)
{
    const auto t0 = std::chrono::steady_clock::now();
    Plan plan;
    const std::size_t n = leaves.size();
    plan.report.leaves = n;
    plan.report.level.assign(n, -1);
    plan.report.solver.assign(n, SolverId::None);
    // (per leaf a status; the one message there is - "no solver matches" - is put together by
    // BatchReport::result() when somebody asks)
    plan.report.status.assign(n, SolveStatus::Success);
    PlanScratch& scratch = t_planScratch;
    HotFacts* const hot = scratch.hot.get(n);
    ColdFacts* const cold = scratch.cold.get(n);
    Roles* const roles = scratch.roles.get(n);  // written for the few leaves the general code decides
    std::uint8_t* const roleCode = scratch.roleCode.get(n);
    plan.cold = cold, plan.roles = roles, plan.roleCode = roleCode;
    plan.stop = n;

    // (A) per-leaf facts, every host thread.  Nothing is written to but the facts: a pass that tags
    // the elements (an index claimed by compare-and-swap) spent its time moving their cache lines
    // from core to core and did not get faster with more threads.
    const auto tA = std::chrono::steady_clock::now();
    const long long nn = static_cast<long long>(n);
    unsigned long long lo = ~0ull, hi = 0;
#pragma omp parallel for schedule(static) reduction(min : lo) reduction(max : hi) if (nn > 2048)
    for (long long i = 0; i < nn; ++i) {
        HotFacts& h = hot[static_cast<std::size_t>(i)];
        bool simple = false;
        try {
            // the leaves lie one after the other, what they point to does not: ask for the elements
            // and constraints of a leaf a few iterations before they are read
            if (i + kFactsLookAhead < nn) prefetchFacts(leaves[static_cast<std::size_t>(i + kFactsLookAhead)]);
            simple = gatherFacts(leaves[static_cast<std::size_t>(i)], h, cold[static_cast<std::size_t>(i)]);
        } catch (...) {
            h = HotFacts {};  // not simple: the general code decides (and raises) in step (B)
        }
        if (simple) {
            for (int k = 0; k < 3; ++k) lo = std::min<unsigned long long>(lo, h.serial[k]), hi = std::max<unsigned long long>(hi, h.serial[k]);
        } else {
            for (const auto& [node, e] : leaves[static_cast<std::size_t>(i)].getElementMap())
                if (e) lo = std::min<unsigned long long>(lo, e->serial()), hi = std::max<unsigned long long>(hi, e->serial());
        }
    }

    // (B) the sequential sweep.  What the symbolic pass knows about an element (solved once the
    // leaves so far have run; wave of its last write / last read) lives in flat arrays indexed by
    // the element's serial number, so no table is searched and this loop touches no element at all
    // for the leaves step (A) could describe: 32 bytes read and 13 written per leaf.
    const auto tB = std::chrono::steady_clock::now();
    SlotIndex index;
    index.lo = lo;
    const std::uint64_t span = hi >= lo ? hi - lo + 1 : 0;
    index.direct = span <= 16 * static_cast<std::uint64_t>(n) + 65536;
    std::vector<char>& predicted = scratch.predicted;
    std::vector<int>&lastWrite = scratch.lastWrite, &lastRead = scratch.lastRead;
    predicted.assign(index.direct ? static_cast<std::size_t>(span) : 0, 0);
    lastWrite.assign(predicted.size(), -1), lastRead.assign(predicted.size(), -1);
    auto slotOfSerial = [&](std::uint64_t serial) {
        const int slot = index.of(serial);
        if (static_cast<std::size_t>(slot) >= predicted.size()) predicted.push_back(0), lastWrite.push_back(-1), lastRead.push_back(-1);
        return slot;
    };
    auto slotOfElement = [&](const Element* e) { return slotOfSerial(e->serial()); };
    VerdictMemo memo;
    int top = -1;
    for (std::size_t i = 0; i < n; ++i) {
        const HotFacts& h = hot[i];
        SolverId id = SolverId::None;
        bool haveRoles = false;
        int slot3[3] = { -1, -1, -1 };
        int rs[2], ws[3], nr = 0, nw = 0;  // read / write footprint as table indices
        if (h.simple) {
            for (int k = 0; k < 3; ++k) slot3[k] = slotOfSerial(h.serial[k]);
            const unsigned setBits = h.setNow | (predicted[static_cast<std::size_t>(slot3[0])] ? 4u : 0u)
                | (predicted[static_cast<std::size_t>(slot3[1])] ? 2u : 0u) | (predicted[static_cast<std::size_t>(slot3[2])] ? 1u : 0u);
            const Verdict& v = memo.get(h.shapeKey, setBits);
            id = v.id;
            if (v.roles && (v.need & ~h.has) == 0) {
                haveRoles = true;
                roleCode[i] = static_cast<std::uint8_t>(v.ia | (v.ib << 2) | (v.ic << 4));
                // footprintOf(): the zero-fixed shapes write all three elements, the others read a, b and write c
                if (zeroFixed(id)) {
                    ws[nw++] = slot3[v.ia], ws[nw++] = slot3[v.ib], ws[nw++] = slot3[v.ic];
                } else {
                    rs[nr++] = slot3[v.ia], rs[nr++] = slot3[v.ib];
                    ws[nw++] = slot3[v.ic];
                }
            }
        }
        if (!haveRoles && (!h.simple || id != SolverId::None)) {
            // the general code: same decisions on the graph itself, raising what the reference raises
            const SetQuery q = [&](const Element* e) {
                return e->isElementSet() || predicted[static_cast<std::size_t>(slotOfElement(e))] != 0;
            };
            id = classify(leaves[i], q);
            if (id != SolverId::None) {
                try {
                    roles[i] = assignRoles(id, leaves[i], q);
                } catch (...) {
                    plan.error = std::current_exception();
                    plan.stop = i;
                    break;
                }
                roleCode[i] = kRolesStored;
                const Roles& r = roles[i];
                if (zeroFixed(id)) {
                    ws[nw++] = slotOfElement(r.a), ws[nw++] = slotOfElement(r.b), ws[nw++] = slotOfElement(r.c);
                } else {
                    rs[nr++] = slotOfElement(r.a), rs[nr++] = slotOfElement(r.b);
                    ws[nw++] = slotOfElement(r.c);
                }
            }
        }
        plan.report.solver[i] = id;
        if (id == SolverId::None) {
            ++plan.report.unsupported;
            plan.report.status[i] = SolveStatus::Unsupported;
            continue;
        }
        int lvl = -1;
        for (int k = 0; k < nr; ++k) lvl = std::max(lvl, lastWrite[static_cast<std::size_t>(rs[k])]);
        for (int k = 0; k < nw; ++k) lvl = std::max({ lvl, lastWrite[static_cast<std::size_t>(ws[k])], lastRead[static_cast<std::size_t>(ws[k])] });
        ++lvl;
        plan.report.level[i] = lvl;
        top = std::max(top, lvl);
        for (int k = 0; k < nr; ++k) {
            int& rd = lastRead[static_cast<std::size_t>(rs[k])];
            rd = std::max(rd, lvl);
        }
        for (int k = 0; k < nw; ++k) {
            lastWrite[static_cast<std::size_t>(ws[k])] = lvl;
            predicted[static_cast<std::size_t>(ws[k])] = 1;
        }
        ++plan.report.solved;
    }
    for (std::size_t i = plan.stop; i < n; ++i) {
        plan.report.level[i] = -1;
        plan.report.status[i] = SolveStatus::Unsupported;
        plan.report.solver[i] = SolverId::None;
    }
    plan.report.waves = static_cast<std::size_t>(top + 1);
    if (std::getenv("GCS_HOST_TRACE"))
        std::fprintf(stderr, "[host] plan: set-up %.1f ms, facts %.1f ms, sweep %.1f ms, %zu leaves\n",
            std::chrono::duration<double>(tA - t0).count() * 1e3, std::chrono::duration<double>(tB - tA).count() * 1e3,
            std::chrono::duration<double>(std::chrono::steady_clock::now() - tB).count() * 1e3, n);
    return plan;
}


const char* solverName(SolverId id)
{
    switch (id) {
    case SolverId::ZeroFixedPointsTriangle: return "ZeroFixedPointsTriangleSolver";
    case SolverId::ZeroFixedPPLTriangle: return "ZeroFixedPPLTriangleSolver";
    case SolverId::ZeroFixedLLPAngleTriangle: return "ZeroFixedLLPAngleTriangleSolver";
    case SolverId::TwoFixedPointsDistance: return "TwoFixedPointsDistanceSolver";
    case SolverId::TwoFixedPointsLine: return "TwoFixedPointsLineSolver";
    case SolverId::FixedPointAndLineFreePoint: return "FixedPointAndLineFreePointSolver";
    case SolverId::TwoFixedLinesFreePoint: return "TwoFixedLinesFreePointSolver";
    case SolverId::FixedLineAndPointFreeLine: return "FixedLineAndPointFreeLineSolver";
    case SolverId::None: break;
    }
    return "None";
}

int kindOf(SolverId id)
{
    switch (id) {
    case SolverId::ZeroFixedPointsTriangle:
    case SolverId::TwoFixedPointsDistance: return GCS_KIND_PP;
    case SolverId::ZeroFixedPPLTriangle:
    case SolverId::TwoFixedPointsLine: return GCS_KIND_SDD;
    case SolverId::FixedPointAndLineFreePoint: return GCS_KIND_PPL;
    case SolverId::TwoFixedLinesFreePoint: return GCS_KIND_PLL;
    case SolverId::ZeroFixedLLPAngleTriangle:
    case SolverId::FixedLineAndPointFreeLine: return GCS_KIND_ANG;
    case SolverId::None: break;
    }
    return 0;
}

namespace {

// the eight matches() predicates on the counts of one leaf
bool matchesCountsOn(SolverId id, int edgeCount, const Census& c, const ConstraintCensus& k)
{
    const bool allDistance = k.distance == k.total;
    switch (id) {
    case SolverId::ZeroFixedPointsTriangle:
        return edgeCount == 3 && c.solved == 0 && c.points == 3 && allDistance;
    case SolverId::ZeroFixedPPLTriangle:
        return edgeCount == 3 && c.solved == 0 && c.points == 2 && c.lines == 1 && allDistance;
    case SolverId::ZeroFixedLLPAngleTriangle:
        return edgeCount == 3 && c.solved == 0 && c.points == 1 && c.lines == 2 && k.angle == 1 && k.distance == 2;
    case SolverId::TwoFixedPointsDistance:
        return c.solved >= 2 && c.points == 3 && allDistance;
    case SolverId::TwoFixedPointsLine:
        return c.solved >= 2 && c.points == 2 && c.lines == 1 && c.unsolvedPoints == 0 && c.solvedLines == 0 && allDistance;
    case SolverId::FixedPointAndLineFreePoint:
        return c.solved >= 2 && c.points == 2 && c.lines == 1 && c.solvedPoints == 1 && c.unsolvedPoints == 1
            && c.solvedLines == 1 && allDistance;
    case SolverId::TwoFixedLinesFreePoint:
        return c.solved >= 2 && c.points == 1 && c.lines == 2 && c.solvedPoints == 0 && c.unsolvedLines == 0 && allDistance;
    case SolverId::FixedLineAndPointFreeLine:
        return c.solved >= 2 && c.points == 1 && c.lines == 2 && c.solvedLines == 1 && c.unsolvedLines == 1
            && c.solvedPoints == 1 && k.angle == 1 && k.distance == 1;
    case SolverId::None: break;
    }
    return false;
}

bool matchesCounts(SolverId id, const ConstraintGraph& g, const Census& c, const ConstraintCensus& k)
{
    return matchesCountsOn(id, static_cast<int>(g.edgeCount()), c, k);
}

}  // namespace

bool matches(SolverId id, const ConstraintGraph& g, const SetQuery& q)
{
    if (g.nodeCount() != 3) return false;
    return matchesCounts(id, g, census(g, q), constraintCensus(g));
}

SolverId classify(const ConstraintGraph& g, const SetQuery& q)
{
    // component_solver.hpp:35-60: fully unsolved shapes first, then the partially solved ones
    static constexpr SolverId order[] = { SolverId::ZeroFixedPointsTriangle, SolverId::ZeroFixedPPLTriangle,
        SolverId::ZeroFixedLLPAngleTriangle, SolverId::TwoFixedPointsDistance, SolverId::TwoFixedPointsLine,
        SolverId::FixedPointAndLineFreePoint, SolverId::TwoFixedLinesFreePoint, SolverId::FixedLineAndPointFreeLine };
    if (g.nodeCount() != 3) return SolverId::None;
    const Census c = census(g, q);  // counted once: the predicates differ only in what they ask of the counts
    const ConstraintCensus k = constraintCensus(g);
    for (SolverId id : order)
        if (matchesCounts(id, g, c, k)) return id;
    return SolverId::None;
}

Footprint footprint(SolverId id, const ConstraintGraph& g, const SetQuery& q) { return footprintOf(assignRoles(id, g, q)); }

PackedLeaf pack(SolverId id, ConstraintGraph& g) { return packNumeric(assignRoles(id, g, {})); }

void apply(const PackedLeaf& leaf, const double out[GCS_MAX_OUT_COLS])
{
    if (!leaf.target) return;
    if (gcs_b200_kind_out_cols(leaf.kind) == 2)
        leaf.target->updateElementPosition(Vector2d { out[0], out[1] });
    else
        leaf.target->updateElementPosition(Vector2d { out[0], out[1] }, Vector2d { out[2], out[3] });
}

// ---- storage of a KindBatch ------------------------------------------------------------------
namespace {

struct Block {
    unsigned char* p = nullptr;
    std::size_t bytes = 0;
    bool pinned = false;
};

// Page-locking memory costs a system call and a driver call per block (hundreds of microseconds):
// blocks go back to this pool instead of to the system.  Never destroyed (freeing page-locked
// memory from a static destructor would run after the CUDA runtime has shut down).
struct BlockPool {
    std::mutex mu;
    std::vector<Block> idle;
    std::size_t idleBytes = 0;
};
BlockPool& pool()
{
    static BlockPool* p = new BlockPool;
    return *p;
}
constexpr std::size_t kPinFrom = 16 * 1024;            // smaller batches (single leaves, merge candidates) stay in ordinary memory
constexpr std::size_t kPoolBytes = std::size_t { 256 } << 20;
constexpr std::size_t kPoolBlocks = 32;

Block acquireBlock(std::size_t bytes)
{
    if (bytes >= kPinFrom) {
        BlockPool& bp = pool();
        std::lock_guard<std::mutex> lk(bp.mu);
        std::size_t best = bp.idle.size();
        for (std::size_t i = 0; i < bp.idle.size(); ++i)
            if (bp.idle[i].bytes >= bytes && bp.idle[i].bytes <= 4 * bytes && (best == bp.idle.size() || bp.idle[i].bytes < bp.idle[best].bytes))
                best = i;
        if (best != bp.idle.size()) {
            const Block b = bp.idle[best];
            bp.idle.erase(bp.idle.begin() + static_cast<std::ptrdiff_t>(best));
            bp.idleBytes -= b.bytes;
            return b;
        }
    }
    Block b;
    b.bytes = bytes;
    if (bytes >= kPinFrom) b.p = static_cast<unsigned char*>(gcs_b200_host_alloc(bytes));  // NULL without a device
    b.pinned = b.p != nullptr;
    if (!b.p) b.p = static_cast<unsigned char*>(std::aligned_alloc(256, (bytes + 255) / 256 * 256));
    if (!b.p) throw std::bad_alloc();
    return b;
}

void releaseBlock(const Block& b)
{
    if (!b.p) return;
    if (b.pinned) {
        BlockPool& bp = pool();
        std::lock_guard<std::mutex> lk(bp.mu);
        if (bp.idle.size() < kPoolBlocks && bp.idleBytes + b.bytes <= kPoolBytes) {
            bp.idle.push_back(b);
            bp.idleBytes += b.bytes;
            return;
        }
    }
    if (b.pinned)
        gcs_b200_host_free(b.p);
    else
        std::free(b.p);
}

}  // namespace

KindBatch::KindBatch(int kind) : m_kind(kind) {}

KindBatch::~KindBatch() { release(); }

KindBatch::KindBatch(KindBatch&& o) noexcept
    : m_kind(o.m_kind), m_nin(o.m_nin), m_nout(o.m_nout), m_size(o.m_size), m_cap(o.m_cap), m_bytes(o.m_bytes), m_slab(o.m_slab),
      m_pinned(o.m_pinned), m_target(std::move(o.m_target))
{
    o.m_slab = nullptr, o.m_cap = o.m_size = o.m_bytes = 0, o.m_pinned = false;
}

KindBatch& KindBatch::operator=(KindBatch&& o) noexcept
{
    if (this != &o) {
        release();
        m_kind = o.m_kind, m_nin = o.m_nin, m_nout = o.m_nout, m_size = o.m_size, m_cap = o.m_cap, m_bytes = o.m_bytes;
        m_slab = o.m_slab, m_pinned = o.m_pinned, m_target = std::move(o.m_target);
        o.m_slab = nullptr, o.m_cap = o.m_size = o.m_bytes = 0, o.m_pinned = false;
    }
    return *this;
}

void KindBatch::release()
{
    releaseBlock(Block { m_slab, m_bytes, m_pinned });
    m_slab = nullptr, m_cap = m_bytes = 0, m_pinned = false;
}

void KindBatch::clear()
{
    m_size = 0;
    m_target.clear();
}

// capacity for `rows` rows: a new block (columns of the old one copied over), 64-row granules so
// that every column starts on a 512-byte boundary
void KindBatch::grow(std::size_t rows)
{
    if (m_kind < 1 || m_kind > GCS_KIND_COUNT) throw std::invalid_argument("KindBatch: storage asked for before the kind is known");
    m_nin = gcs_b200_kind_in_cols(m_kind), m_nout = gcs_b200_kind_out_cols(m_kind);
    const std::size_t cap = (std::max<std::size_t>(rows, 64) + 63) / 64 * 64;
    const std::size_t ncol = static_cast<std::size_t>(m_nin + m_nout);
    const Block nb = acquireBlock(ncol * cap * sizeof(double) + cap);
    // a recycled block may be larger than asked for: the spacing follows what was asked, the rest is slack
    if (m_slab && m_size) {
        for (int c = 0; c < m_nin; ++c)
            std::memcpy(nb.p + static_cast<std::size_t>(c) * cap * sizeof(double), column(c), m_size * sizeof(double));
        std::memcpy(nb.p + ncol * cap * sizeof(double), codes(), m_size);
    }
    release();
    m_slab = nb.p, m_bytes = nb.bytes, m_pinned = nb.pinned, m_cap = cap;
}

void KindBatch::reserve(std::size_t rows)
{
    if (rows > m_cap) grow(rows);
}

void KindBatch::resize(std::size_t rows)
{
    reserve(rows);
    m_size = rows;
    m_target.assign(rows, nullptr);
}

void KindBatch::set(std::size_t row, const PackedLeaf& leaf)
{
    if (leaf.kind != m_kind) throw std::invalid_argument("KindBatch::set: leaf of another kind");
    double* cols = reinterpret_cast<double*>(m_slab);
    for (int c = 0; c < m_nin; ++c) cols[static_cast<std::size_t>(c) * m_cap + row] = leaf.in[c];
    m_slab[static_cast<std::size_t>(m_nin + m_nout) * m_cap * sizeof(double) + row] = leaf.code;
    m_target[row] = leaf.target;
}

void KindBatch::push(const PackedLeaf& leaf)
{
    if (m_kind == 0) m_kind = leaf.kind;
    if (leaf.kind != m_kind) throw std::invalid_argument("KindBatch::push: leaf of another kind");
    if (m_size == m_cap) grow(std::max<std::size_t>(2 * m_cap, 64));
    m_target.push_back(nullptr);
    set(m_size++, leaf);
}

namespace {
int& variantSetting()
{
    static int v = [] {
        const char* e = std::getenv("GCS_B200_HOST_VARIANT");
        return e ? std::atoi(e) : GCS_VARIANT_DEFAULT;
    }();
    return v;
}
}  // namespace

int kernelVariant() { return variantSetting(); }
int setKernelVariant(int variant)
{
    const int old = variantSetting();
    variantSetting() = variant;
    return old;
}

gcs_b200_batch KindBatch::descriptor()
{
    gcs_b200_batch d {};
    d.kind = m_kind;
    d.n_seeds = 2;  // Equations::solve2D runs exactly two guesses (newton_raphson.hpp:42-53)
    d.n = static_cast<std::int64_t>(m_size);
    d.mem = GCS_MEM_HOST;
    d.variant = variantSetting();
    if (m_size == 0) return d;
    for (int c = 0; c < m_nin; ++c) d.in[c] = column(c);
    d.code = codes();
    d.guesses = nullptr;
    for (int c = 0; c < m_nout; ++c) d.out[c] = const_cast<double*>(out(c));
    // candidates, iteration counts, flags and root indices stay on the device: nothing here reads them
    d.cand = nullptr, d.iters = nullptr, d.converged = nullptr, d.root_index = nullptr;
    return d;
}

void KindBatch::applyAll()
{
    // the rows of a batch write distinct elements (one wave of the scheduler, or the independent
    // candidates of a merge): every host thread
    const long long m = static_cast<long long>(m_size);
    PackedLeaf shape;
    shape.kind = m_kind;
#pragma omp parallel for schedule(static) firstprivate(shape) if (m > 1024)
    for (long long i = 0; i < m; ++i) {
        double o[GCS_MAX_OUT_COLS] = {};
        for (int c = 0; c < m_nout; ++c) o[c] = out(c)[static_cast<std::size_t>(i)];
        shape.target = m_target[static_cast<std::size_t>(i)];
        apply(shape, o);
    }
}

SolveResult solveSingle(SolverId id, ConstraintGraph& component, int device)
{
    if (id == SolverId::None) return SolveResult::unsupported("No solver matches this component configuration");
    KindBatch batch(kindOf(id));
    batch.push(pack(id, component));
    solveBatchOnDevice(batch, device);
    return SolveResult::success();  // every reference solver returns success() (e.g. point_point_solvers.cpp:163)
}

BatchReport planLeaves(const std::vector<ConstraintGraph>& leaves)
{
    const auto t0 = std::chrono::steady_clock::now();
    BatchReport rep = makePlan(leaves).report;
    rep.planSeconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return rep;
}

namespace {
BatchReport solveLeavesImpl(std::vector<ConstraintGraph>& leaves, int device, int nDevices, std::size_t minRowsPerDevice);
}

BatchReport solveLeaves(std::vector<ConstraintGraph>& leaves, int device) { return solveLeavesImpl(leaves, device, 1, 0); }

BatchReport solveLeavesOnDevices(std::vector<ConstraintGraph>& leaves, int nDevices, std::size_t minRowsPerDevice)
{
    return solveLeavesImpl(leaves, 0, nDevices < 1 ? 1 : nDevices, minRowsPerDevice);
}

namespace {
BatchReport solveLeavesImpl(std::vector<ConstraintGraph>& leaves, int device, int nDevices, std::size_t minRowsPerDevice)
{
    using Clock = std::chrono::steady_clock;
    auto since = [](Clock::time_point t) { return std::chrono::duration<double>(Clock::now() - t).count(); };
    if (const char* reps = std::getenv("GCS_HOST_PLAN_REPS"))  // measurement aid: the plan alone, repeated (GCS_HOST_TRACE prints its split)
        for (int k = std::atoi(reps); k > 0; --k) (void)makePlan(leaves);
    auto t0 = Clock::now();
    Plan plan = makePlan(leaves);
    BatchReport& rep = plan.report;
    rep.planSeconds = since(t0);
    // leaves of a wave, in input order
    std::vector<std::vector<std::size_t>> byWave(rep.waves);
    for (std::size_t i = 0; i < plan.stop; ++i)
        if (rep.level[i] >= 0) byWave[static_cast<std::size_t>(rep.level[i])].push_back(i);
    KindBatch batches[GCS_KIND_COUNT + 1];
    for (int k = 1; k <= GCS_KIND_COUNT; ++k) batches[k] = KindBatch(k);
    {  // one block per kind for the whole solve: the largest wave decides
        std::vector<std::array<std::size_t, GCS_KIND_COUNT + 1>> count(rep.waves);
        for (std::size_t i = 0; i < plan.stop; ++i)
            if (rep.level[i] >= 0) ++count[static_cast<std::size_t>(rep.level[i])][static_cast<std::size_t>(kindOf(rep.solver[i]))];
        for (int k = 1; k <= GCS_KIND_COUNT; ++k) {
            std::size_t most = 0;
            for (const auto& c : count) most = std::max(most, c[static_cast<std::size_t>(k)]);
            if (most) batches[k].reserve(most);
        }
    }
    std::vector<std::size_t> rowOf;
    for (const auto& wave : byWave) {
        t0 = Clock::now();
        // rows of the kind batches in input order
        std::size_t rowsOfKind[GCS_KIND_COUNT + 1] = {};
        rowOf.resize(wave.size());
        for (std::size_t j = 0; j < wave.size(); ++j) rowOf[j] = rowsOfKind[kindOf(rep.solver[wave[j]])]++;
        for (int k = 1; k <= GCS_KIND_COUNT; ++k) batches[k].resize(rowsOfKind[k]);
        // The leaves of a wave touch disjoint elements wherever one of them writes (that is what a
        // wave is: nobody reads or writes what another leaf of the wave writes - the anchors the
        // zero-fixed shapes place included), so their rows are packed on every host thread,
        // straight into the kind batches.
        const long long m = static_cast<long long>(wave.size());
        std::exception_ptr packError;
#pragma omp parallel for schedule(static) if (m > 1024)
        for (long long j = 0; j < m; ++j) {
            try {
                const PackedLeaf row = packNumeric(plan.rolesOf(wave[static_cast<std::size_t>(j)]));
                batches[row.kind].set(rowOf[static_cast<std::size_t>(j)], row);
            } catch (...) {
#pragma omp critical
                if (!packError) packError = std::current_exception();
            }
        }
        if (packError) std::rethrow_exception(packError);
        rep.packSeconds += since(t0);
        // The kind batches of a wave are independent jobs: all of them are queued (upload / kernel /
        // download pipelines on the library's streams) before any is waited for, then written back.
        t0 = Clock::now();
        auto failed = [&](const char* what, int rc) {
            gcs_b200_wait(device);  // leave nothing in flight behind the exception
            throw std::runtime_error(std::string(what) + " failed (" + std::to_string(rc) + "): " + gcs_b200_last_error()
                + " - the sub-problem solvers run on the CUDA path only");
        };
        int queued = 0;
        for (int k = 1; k <= GCS_KIND_COUNT; ++k) {
            if (batches[k].size() == 0) continue;
            gcs_b200_batch d = batches[k].descriptor();
            const bool shard = nDevices > 1 && batches[k].size() >= minRowsPerDevice * static_cast<std::size_t>(nDevices);
            if (shard) {
                const int rc = gcs_b200_solve_sharded(&d, nDevices);
                if (rc != GCS_OK) failed("gcs_b200_solve_sharded", rc);
                ++rep.shardedLaunches;
            } else {
                const int rc = gcs_b200_solve_host_async(&d, device);
                if (rc != GCS_OK) failed("gcs_b200_solve_host_async", rc);
                ++queued;
            }
            ++rep.launches;
            if (std::getenv("GCS_HOST_TRACE")) std::fprintf(stderr, "[host] wave launch kind %d rows %zu\n", k, batches[k].size());
        }
        if (queued) {
            const int rc = gcs_b200_wait(device);
            if (rc != GCS_OK) failed("gcs_b200_wait", rc);
        }
        rep.deviceSeconds += since(t0);
        if (std::getenv("GCS_HOST_TRACE")) std::fprintf(stderr, "[host] wave of %zu leaves: device calls %.1f us\n", wave.size(), since(t0) * 1e6);
        t0 = Clock::now();
        for (int k = 1; k <= GCS_KIND_COUNT; ++k)
            if (batches[k].size() != 0) batches[k].applyAll();
        rep.applySeconds += since(t0);
    }
    if (plan.error) std::rethrow_exception(plan.error);
    return rep;
}
}  // namespace

}  // namespace Gcs::B200
