// plan.hpp — the leaf scheduler's plan and the canvas half of a batch row, shared by the wave
// solver (leaf_batch.cpp) and the sketch-program compiler (sketch_program.cpp).  Internal header.
#pragma once

#include <cstddef>
#include <cstdint>
#include <exception>
#include <vector>

#include <gcs/b200/leaf_batch.hpp>
#include <gcs/model/constraints.hpp>

namespace Gcs::B200::detail {

// Who plays which part in a leaf, plus the constraint values the solver reads.  Filled without
// touching any position, so it can run ahead of the numeric solve (on predicted solved flags).
struct Roles {
    SolverId id = SolverId::None;
    // a, b: the two "known" elements in the solver's own naming order; c: the element solved for
    //  1 ZeroFixedPoints      a=P1 b=P2 c=P3            v0=d12 v1=d13 v2=d23
    //  2 ZeroFixedPPL         a=P1 b=P2 c=line          v0=d12 v1=d(P1,line) v2=d(P2,line)
    //  3 ZeroFixedLLPAngle    a=line1 b=point c=line2   v0=angle v1=d(P,line1) v2=d(P,line2)
    //  4 TwoFixedPointsDist   a=fixed1 b=fixed2 c=free  v1=d(f1,free) v2=d(f2,free)
    //  5 TwoFixedPointsLine   a=fixed1 b=fixed2 c=line  v1=d(f1,line) v2=d(f2,line)
    //  6 FixedPointAndLine    a=fixedPt b=line c=free   v1=d(fixedPt,free) v2=d(line,free)
    //  7 TwoFixedLines        a=line1 b=line2 c=free    v1=d(l1,free) v2=d(l2,free)
    //  8 FixedLineAndPoint    a=fixedLine b=point c=freeLine  v0=angle v2=d(point,freeLine)
    Element* a = nullptr;
    Element* b = nullptr;
    Element* c = nullptr;
    double v0 = 0.0, v1 = 0.0, v2 = 0.0;
    const Constraint* k[3] = {};  // the constraint behind v0, v1, v2 (null where the solver reads none)
    bool flip = false;  // AngleConstraint::flipOrientation of the line-line constraint
};

// The canvas half of a batch row: everything the packer derives from canvas positions alone.
// With the roles' constraint values and the solved positions it makes the row (packNumeric; on the
// device, the sketch program's gather kernel):
//   sign[v]  signOf(canvas side) factor of value v (1 where the value is not signed)
//   cst[]    1, 4     -
//            2, 5     0 gnx  1 gny  2 canvas_len            (canvas unit normal of the free line)
//            6, 7     0 cfx  1 cfy                          (canvas position of the free point)
//            3, 8     0 gnx  1 gny  2 cfdx  3 cfdy  4 canvas_len  (free line's normal, fixed line's direction)
//            3        5 fdx  6 fdy  7 x1  8 x2              (direction and x of the anchored line1: (x1, 0) - (x2, 0))
struct CanvasRow {
    std::uint8_t code = 0;
    double sign[3] = { 1.0, 1.0, 1.0 };
    double cst[9] = {};
};
CanvasRow packCanvas(const Roles& r);

struct ColdFacts;

struct Plan {
    BatchReport report;
    // per solved leaf: roleCode[i] says who plays which part among cold[i].e (the sweep decided from
    // the facts), or kRolesStored: the general code left the roles in roles[i].  All three live in
    // the thread's scratch memory: a plan is used up before the thread makes its next one.
    const ColdFacts* cold = nullptr;
    const std::uint8_t* roleCode = nullptr;
    const Roles* roles = nullptr;
    std::size_t stop = 0;              // leaves [0, stop) are solved; == leaves.size() when no leaf throws
    std::exception_ptr error;          // what the reference's loop would have thrown at leaf `stop`
    Roles rolesOf(std::size_t i) const;
};

// The symbolic pass: per leaf the solver the reference's loop would choose (on predicted solved
// flags), its roles and its wave.  No numerics, no device.
Plan makePlan(const std::vector<ConstraintGraph>& leaves);

}  // namespace Gcs::B200::detail
