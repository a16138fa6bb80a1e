// sketch_program.cpp — Gcs::B200::SketchProgram (gcs/b200/sketch_program.hpp): the plan of
// solveLeaves and the canvas half of its rows (plan.hpp, shared with leaf_batch.cpp) turned into the
// row records of gcs_b200_program_create.
#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstring>
#include <exception>
#include <stdexcept>
#include <string>
#include <thread>
#include <unordered_map>

#include <gcs/b200/sketch_program.hpp>
#include <gcs/model/elements.hpp>

#include "plan.hpp"

namespace Gcs::B200 {

namespace {

using Clock = std::chrono::steady_clock;

[[noreturn]] void cudaFailure(const char* what, int rc)
{
    throw std::runtime_error(std::string(what) + " failed (" + std::to_string(rc) + "): " + gcs_b200_last_error()
        + " - sketch programs run on the CUDA path only");
}

bool isZeroFixed(int solver) { return solver >= 1 && solver <= 3; }

// the devices K >= 1 instances split over: nDevices clamped to [1, devices present], at most K
int devicesFor(int nDevices, std::int64_t K)
{
    const int avail = gcs_b200_device_count();
    if (avail < 1) cudaFailure("gcs_b200_device_count", GCS_E_NO_DEVICE);
    return static_cast<int>(std::min<std::int64_t>(std::clamp(nDevices, 1, avail), K));
}

// K instances over devices 0 .. nDevices-1, one host thread per device: part(g, lo, hi, ms) runs
// instances [lo, hi) = [K*g/n, K*(g+1)/n) on device g through the C entry point `entry`, returns its
// code and fills ms[3].  A failed part throws, naming `entry`.  Returns the launches and the summed
// times; seconds are the caller's.
template <class Part>
ProgramRunStats fanOut(std::int64_t K, int nDevices, const char* entry, Part&& part)
{
    const std::int64_t launches0 = gcs_b200_launch_count();
    std::vector<int> rc(static_cast<std::size_t>(nDevices), GCS_OK);
    std::vector<std::array<float, 3>> ms(static_cast<std::size_t>(nDevices));
    auto one = [&](int g) {
        const std::size_t i = static_cast<std::size_t>(g);
        rc[i] = part(g, K * g / nDevices, K * (g + 1) / nDevices, ms[i].data());
    };
    if (nDevices == 1) {
        one(0);
    } else {
        std::vector<std::thread> threads;
        for (int g = 0; g < nDevices; ++g) threads.emplace_back(one, g);
        for (auto& t : threads) t.join();
    }
    for (int r : rc)
        if (r != GCS_OK) cudaFailure(entry, r);
    ProgramRunStats st;
    st.launches = gcs_b200_launch_count() - launches0;
    for (const auto& m : ms) st.uploadMs += m[0], st.deviceMs += m[1], st.downloadMs += m[2];
    return st;
}

}  // namespace

SketchProgram SketchProgram::compile(const std::vector<ConstraintGraph>& leaves, const std::vector<std::shared_ptr<Element>>& elements,
    const std::vector<std::shared_ptr<Constraint>>& constraints)
{
    const auto t0 = Clock::now();
    SketchProgram prog;
    const detail::Plan plan = detail::makePlan(leaves);
    if (plan.error) std::rethrow_exception(plan.error);
    prog.m_report = plan.report;
    prog.m_elements = elements;
    prog.m_constraints = constraints;

    std::unordered_map<const Element*, int> slotOf;
    const std::size_t nSlots = elements.size();
    prog.m_slotIsLine.assign(nSlots, 0);
    prog.m_solvedAfter.assign(nSlots, 0);
    prog.m_initial.assign(nSlots * 4, 0.0);
    for (std::size_t s = 0; s < nSlots; ++s) {
        const Element& e = *elements[s];
        slotOf.emplace(&e, static_cast<int>(s));
        double* p = prog.m_initial.data() + 4 * s;
        if (e.isElementType<Line>()) {
            const auto& l = e.getElement<Line>();
            prog.m_slotIsLine[s] = 1;
            p[0] = l.p1.x(), p[1] = l.p1.y(), p[2] = l.p2.x(), p[3] = l.p2.y();
        } else if (e.isElementType<Point>()) {
            const auto& pt = e.getElement<Point>();
            p[0] = pt.position.x(), p[1] = pt.position.y();
        }
        prog.m_solvedAfter[s] = e.isElementSet() ? 1 : 0;
    }
    std::unordered_map<const Constraint*, int> valueOf;
    for (std::size_t v = 0; v < constraints.size(); ++v) valueOf.emplace(constraints[v].get(), static_cast<int>(v));
    prog.m_valueIsAngle.assign(constraints.size(), 0);
    std::vector<std::uint8_t> usedAsDistance(constraints.size(), 0);

    // rows of (wave, kind) in input order
    const std::size_t waves = plan.report.waves;
    std::vector<std::vector<std::size_t>> segment(waves * GCS_KIND_COUNT);
    for (std::size_t i = 0; i < plan.stop; ++i)
        if (plan.report.level[i] >= 0)
            segment[static_cast<std::size_t>(plan.report.level[i]) * GCS_KIND_COUNT + static_cast<std::size_t>(kindOf(plan.report.solver[i]) - 1)].push_back(i);
    prog.m_offsets.assign(1, 0);
    for (const auto& seg : segment) {
        for (std::size_t i : seg) {
            const detail::Roles r = plan.rolesOf(i);
            const detail::CanvasRow cv = detail::packCanvas(r);
            gcs_b200_program_row row {};
            row.solver = static_cast<std::int32_t>(r.id);
            const Element* role[3] = { r.a, r.b, r.c };
            for (int q = 0; q < 3; ++q) {
                const auto it = slotOf.find(role[q]);
                if (it == slotOf.end()) throw std::invalid_argument("SketchProgram::compile: leaf " + std::to_string(i) + " holds an element that is not in the element list");
                row.elem[q] = it->second;
                row.value[q] = -1;
                if (!r.k[q]) continue;
                const auto vt = valueOf.find(r.k[q]);
                if (vt == valueOf.end()) throw std::invalid_argument("SketchProgram::compile: leaf " + std::to_string(i) + " reads a constraint that is not in the constraint list");
                row.value[q] = vt->second;
                const bool cosine = q == 0 && (r.id == SolverId::ZeroFixedLLPAngleTriangle || r.id == SolverId::FixedLineAndPointFreeLine);
                (cosine ? prog.m_valueIsAngle : usedAsDistance)[static_cast<std::size_t>(vt->second)] = 1;
            }
            row.code = cv.code;
            for (int q = 0; q < 3; ++q) row.sign[q] = cv.sign[q];
            std::memcpy(row.canvas, cv.cst, sizeof(row.canvas));
            prog.m_solvedAfter[static_cast<std::size_t>(row.elem[2])] = 1;
            if (isZeroFixed(row.solver)) prog.m_solvedAfter[static_cast<std::size_t>(row.elem[0])] = prog.m_solvedAfter[static_cast<std::size_t>(row.elem[1])] = 1;
            prog.m_rows.push_back(row);
            prog.m_rowLeaf.push_back(static_cast<std::int64_t>(i));
        }
        prog.m_offsets.push_back(static_cast<std::int64_t>(prog.m_rows.size()));
    }
    for (std::size_t v = 0; v < constraints.size(); ++v)
        if (prog.m_valueIsAngle[v] && usedAsDistance[v])
            throw std::invalid_argument("SketchProgram::compile: constraint " + std::to_string(v) + " is read both as an angle and as a distance");
    prog.m_compileSeconds = std::chrono::duration<double>(Clock::now() - t0).count();
    prog.m_report.planSeconds = prog.m_compileSeconds;
    return prog;
}

SketchProgram::SketchProgram(SketchProgram&& o) noexcept { *this = std::move(o); }

SketchProgram& SketchProgram::operator=(SketchProgram&& o) noexcept
{
    if (this == &o) return *this;
    release();
    m_report = std::move(o.m_report);
    m_rows = std::move(o.m_rows), m_offsets = std::move(o.m_offsets), m_rowLeaf = std::move(o.m_rowLeaf);
    m_slotIsLine = std::move(o.m_slotIsLine), m_valueIsAngle = std::move(o.m_valueIsAngle), m_solvedAfter = std::move(o.m_solvedAfter);
    m_initial = std::move(o.m_initial);
    m_elements = std::move(o.m_elements), m_constraints = std::move(o.m_constraints);
    m_compileSeconds = o.m_compileSeconds;
    m_device = std::move(o.m_device);
    o.m_device.clear();
    m_stageValues = o.m_stageValues, m_stagePositions = o.m_stagePositions, m_stageCounts = o.m_stageCounts, m_stageK = o.m_stageK;
    o.m_stageValues = o.m_stagePositions = nullptr, o.m_stageCounts = nullptr, o.m_stageK = 0;
    m_stageDValues = o.m_stageDValues, m_stageDPositions = o.m_stageDPositions, m_stageKT = o.m_stageKT;
    o.m_stageDValues = o.m_stageDPositions = nullptr, o.m_stageKT = 0;
    m_recordedValues = std::move(o.m_recordedValues), m_recordedK = o.m_recordedK, m_recordedDevices = o.m_recordedDevices;
    o.m_recordedK = 0, o.m_recordedDevices = 0;
    return *this;
}

SketchProgram::~SketchProgram() { release(); }

void SketchProgram::release()
{
    for (gcs_b200_program* p : m_device) gcs_b200_program_destroy(p);
    m_device.clear();
    gcs_b200_host_free(m_stageValues), gcs_b200_host_free(m_stagePositions), gcs_b200_host_free(m_stageCounts);
    m_stageValues = m_stagePositions = nullptr, m_stageCounts = nullptr, m_stageK = 0;
    gcs_b200_host_free(m_stageDValues), gcs_b200_host_free(m_stageDPositions);
    m_stageDValues = m_stageDPositions = nullptr, m_stageKT = 0;
    m_recordedValues.clear(), m_recordedK = 0, m_recordedDevices = 0;
}

gcs_b200_program_desc SketchProgram::desc() const
{
    gcs_b200_program_desc d {};
    d.n_waves = static_cast<std::int32_t>(m_report.waves);
    d.n_slots = static_cast<std::int32_t>(nSlots());
    d.n_values = static_cast<std::int32_t>(nValues());
    d.n_rows = static_cast<std::int64_t>(m_rows.size());
    d.rows = m_rows.data(), d.offsets = m_offsets.data();
    d.slot_is_line = m_slotIsLine.data(), d.initial = m_initial.data(), d.value_is_angle = m_valueIsAngle.data();
    return d;
}

gcs_b200_program* SketchProgram::onDevice(int device)
{
    if (static_cast<std::size_t>(device) >= m_device.size()) m_device.resize(static_cast<std::size_t>(device) + 1, nullptr);
    gcs_b200_program*& p = m_device[static_cast<std::size_t>(device)];
    if (!p) {
        const gcs_b200_program_desc d = desc();
        const int rc = gcs_b200_program_create(&d, device, &p);
        if (rc != GCS_OK) cudaFailure("gcs_b200_program_create", rc);
    }
    return p;
}

ProgramRunStats SketchProgram::run(const double* values, std::int64_t K, double* positions, std::uint32_t* nonconverged, int nDevices)
{
    return runImpl(values, K, nullptr, 0, positions, nullptr, nonconverged, nDevices);
}

ProgramRunStats SketchProgram::runTangents(const double* values, std::int64_t K, const double* dvalues, int T, double* positions,
    double* dpositions, std::uint32_t* nonconverged, int nDevices)
{
    if (T < 1) throw std::invalid_argument("SketchProgram::runTangents: T must be >= 1 (got " + std::to_string(T) + ")");
    return runImpl(values, K, dvalues, T, positions, dpositions, nonconverged, nDevices);
}

ProgramRunStats SketchProgram::runFused(const double* values, std::int64_t K, const double* dvalues, int T, double* positions,
    double* dpositions, std::uint32_t* nonconverged, int nDevices)
{
    if (T < 0) throw std::invalid_argument("SketchProgram::runFused: T must be >= 0 (got " + std::to_string(T) + ")");
    return runImpl(values, K, dvalues, T, positions, dpositions, nonconverged, nDevices, RunKind::fused);
}

ProgramRunStats SketchProgram::record(const double* values, std::int64_t K, double* positions, std::uint32_t* nonconverged, int nDevices)
{
    m_recordedDevices = 0;  // a failed record() leaves nothing to sweep
    const ProgramRunStats st = runImpl(values, K, nullptr, 0, positions, nullptr, nonconverged, nDevices, RunKind::recorded);
    m_recordedValues.assign(values, values + static_cast<std::size_t>(K) * nValues());
    m_recordedK = K;
    // runImpl's split: instances in contiguous ranges over the first devicesFor(nDevices, K) devices
    m_recordedDevices = devicesFor(nDevices, K);
    return st;
}

ProgramRunStats SketchProgram::adjoints(const double* adjPositions, int T, double* adjValues)
{
    const auto t0 = Clock::now();
    if (m_recordedDevices < 1) throw std::logic_error("SketchProgram::adjoints: no recorded run; call record() first");
    if (T < 1) throw std::invalid_argument("SketchProgram::adjoints: T must be >= 1 (got " + std::to_string(T) + ")");
    const std::int64_t K = m_recordedK;
    const std::size_t nv = nValues(), table = nSlots() * 4;
    ProgramRunStats st = fanOut(K, m_recordedDevices, "gcs_b200_program_adjoints_host", [&](int g, std::int64_t lo, std::int64_t, float* ms) {
        return gcs_b200_program_adjoints_host(m_device[static_cast<std::size_t>(g)], T, adjPositions + lo * static_cast<std::int64_t>(table) * T,
            adjValues + lo * static_cast<std::int64_t>(nv) * T, ms);
    });
    // the device's adjoints of cos(v), to radians: adj = (-std::sin(v)) * adj_cos
    const long long n = static_cast<long long>(K) * static_cast<long long>(nv) * T;
    const std::uint8_t* angle = m_valueIsAngle.data();
    const double* rec = m_recordedValues.data();
#pragma omp parallel for schedule(static) if (n > 65536)
    for (long long q = 0; q < n; ++q) {
        const long long vq = q / T;
        if (angle[static_cast<std::size_t>(vq) % nv]) adjValues[q] = -std::sin(rec[vq]) * adjValues[q];
    }
    st.seconds = std::chrono::duration<double>(Clock::now() - t0).count();
    return st;
}

ProgramRunStats SketchProgram::fit(double* values, std::int64_t K, const FitSpec& spec, const double* targets, double* positions,
    gcs_b200_fit_result* results, std::uint32_t* nonconverged, int nDevices)
{
    const auto t0 = Clock::now();
    const auto bad = [](const std::string& what) { throw std::invalid_argument("SketchProgram::fit: " + what); };
    if (K < 1) bad("K must be >= 1");
    const std::size_t nf = spec.freeValues.size(), nobs = spec.obsSlots.size();
    if ((!spec.lower.empty() && spec.lower.size() != nf) || (!spec.upper.empty() && spec.upper.size() != nf))
        bad("lower and upper hold one bound per free value, or none");
    if (spec.obsCoords.size() != nobs || (!spec.weights.empty() && spec.weights.size() != nobs))
        bad("obsCoords (and weights, if any) hold one entry per observation");
    gcs_b200_fit_desc f {};
    f.n_free = static_cast<std::int32_t>(std::min<std::size_t>(nf, 1u << 30));
    f.n_obs = static_cast<std::int32_t>(std::min<std::size_t>(nobs, 1u << 30));
    f.free_values = spec.freeValues.data(), f.obs_slots = spec.obsSlots.data(), f.obs_coords = spec.obsCoords.data();
    f.lower = spec.lower.empty() ? nullptr : spec.lower.data();
    f.upper = spec.upper.empty() ? nullptr : spec.upper.data();
    f.weights = spec.weights.empty() ? nullptr : spec.weights.data();
    f.max_iterations = spec.maxIterations, f.lambda0 = spec.lambda0;
    f.cost_tol = spec.costTol, f.ftol = spec.ftol, f.xtol = spec.xtol, f.gtol = spec.gtol;
    const gcs_b200_program_desc d = desc();
    if (gcs_b200_fit_check(&d, &f) != GCS_OK) bad(gcs_b200_last_error());
    nDevices = devicesFor(nDevices, K);
    const std::size_t nv = nValues(), table = nSlots() * 4;
    stage(values, K, nullptr, 0);
    double* const cv = m_stageValues;
    for (int g = 0; g < nDevices; ++g) onDevice(g);
    const int variant = kernelVariant();
    ProgramRunStats st = fanOut(K, nDevices, "gcs_b200_program_fit_host", [&](int g, std::int64_t lo, std::int64_t hi, float* ms) {
        return gcs_b200_program_fit_host(m_device[static_cast<std::size_t>(g)], &f, hi - lo, cv + lo * static_cast<std::int64_t>(nv),
            targets + lo * static_cast<std::int64_t>(nobs), positions + lo * static_cast<std::int64_t>(table),
            nonconverged ? nonconverged + lo : nullptr, results + lo, variant, ms);
    });
    for (std::int64_t k = 0; k < K; ++k) {
        if (results[k].status == GCS_FIT_START_FAILED) continue;
        for (std::size_t i = 0; i < nf; ++i) {
            const std::size_t q = static_cast<std::size_t>(k) * nv + static_cast<std::size_t>(spec.freeValues[i]);
            values[q] = m_valueIsAngle[static_cast<std::size_t>(spec.freeValues[i])] ? std::copysign(std::acos(cv[q]), values[q]) : cv[q];
        }
    }
    st.seconds = std::chrono::duration<double>(Clock::now() - t0).count();
    return st;
}

// values [K][nValues()] and dvalues [K][nValues()][T] (radians) into the page-locked staging, in the C ABI's units
void SketchProgram::stage(const double* values, std::int64_t K, const double* dvalues, int T)
{
    const std::size_t nv = nValues(), table = nSlots() * 4;
    if (K > m_stageK) {
        gcs_b200_host_free(m_stageValues), gcs_b200_host_free(m_stagePositions), gcs_b200_host_free(m_stageCounts);
        m_stageK = 0;
        m_stageValues = static_cast<double*>(gcs_b200_host_alloc(std::max<std::size_t>(1, static_cast<std::size_t>(K) * nv) * sizeof(double)));
        m_stagePositions = static_cast<double*>(gcs_b200_host_alloc(std::max<std::size_t>(1, static_cast<std::size_t>(K) * table) * sizeof(double)));
        m_stageCounts = static_cast<std::uint32_t*>(gcs_b200_host_alloc(static_cast<std::size_t>(K) * sizeof(std::uint32_t)));
        if (!m_stageValues || !m_stagePositions || !m_stageCounts) throw std::bad_alloc();
        m_stageK = K;
    }
    const std::int64_t KT = K * T;
    if (KT > m_stageKT) {
        gcs_b200_host_free(m_stageDValues), gcs_b200_host_free(m_stageDPositions);
        m_stageKT = 0;
        m_stageDValues = static_cast<double*>(gcs_b200_host_alloc(std::max<std::size_t>(1, static_cast<std::size_t>(KT) * nv) * sizeof(double)));
        m_stageDPositions = static_cast<double*>(gcs_b200_host_alloc(std::max<std::size_t>(1, static_cast<std::size_t>(KT) * table) * sizeof(double)));
        if (!m_stageDValues || !m_stageDPositions) throw std::bad_alloc();
        m_stageKT = KT;
    }
    // angles go to the device as std::cos of the value: the host packer's rounding
    const long long nval = static_cast<long long>(K) * static_cast<long long>(nv);
    const std::uint8_t* angle = m_valueIsAngle.data();
    double* stage = m_stageValues;
#pragma omp parallel for schedule(static) if (nval > 65536)
    for (long long q = 0; q < nval; ++q) stage[q] = angle[static_cast<std::size_t>(q) % nv] ? std::cos(values[q]) : values[q];
    // and their directions as d(cos v) = -sin(v) dv
    double* dstage = m_stageDValues;
    const long long ndval = nval * T;
#pragma omp parallel for schedule(static) if (ndval > 65536)
    for (long long q = 0; q < ndval; ++q) {
        const long long vq = q / T;
        dstage[q] = angle[static_cast<std::size_t>(vq) % nv] ? -std::sin(values[vq]) * dvalues[q] : dvalues[q];
    }
}

// T = 0: run(), record() or a plain runFused(); T > 0: runTangents() or a tangent runFused()
ProgramRunStats SketchProgram::runImpl(const double* values, std::int64_t K, const double* dvalues, int T, double* positions,
    double* dpositions, std::uint32_t* nonconverged, int nDevices, RunKind how)
{
    const auto t0 = Clock::now();
    if (K < 1) throw std::invalid_argument("SketchProgram::run: K must be >= 1");
    nDevices = devicesFor(nDevices, K);
    const std::size_t nv = nValues(), table = nSlots() * 4;
    stage(values, K, dvalues, T);
    for (int g = 0; g < nDevices; ++g) onDevice(g);

    const int variant = kernelVariant();
    const char* entry = how == RunKind::fused ? "gcs_b200_program_run_fused_host"
        : how == RunKind::recorded            ? "gcs_b200_program_run_recorded_host"
        : T == 0                              ? "gcs_b200_program_run_host"
                                              : "gcs_b200_program_run_tangents_host";
    ProgramRunStats st = fanOut(K, nDevices, entry, [&](int g, std::int64_t lo, std::int64_t hi, float* ms) {
        gcs_b200_program* p = m_device[static_cast<std::size_t>(g)];
        const std::int64_t vo = lo * static_cast<std::int64_t>(nv), po = lo * static_cast<std::int64_t>(table);
        std::uint32_t* counts = nonconverged ? m_stageCounts + lo : nullptr;
        if (how == RunKind::fused)
            return gcs_b200_program_run_fused_host(p, hi - lo, m_stageValues + vo, m_stagePositions + po, counts, T, m_stageDValues + vo * T,
                m_stageDPositions + po * T, ms);
        return how == RunKind::recorded ? gcs_b200_program_run_recorded_host(p, hi - lo, m_stageValues + vo, m_stagePositions + po, counts, variant, ms)
            : T == 0 ? gcs_b200_program_run_host(p, hi - lo, m_stageValues + vo, m_stagePositions + po, counts, variant, ms)
            : gcs_b200_program_run_tangents_host(p, hi - lo, m_stageValues + vo, m_stagePositions + po, counts, T, m_stageDValues + vo * T,
                m_stageDPositions + po * T, variant, ms);
    });
    const long long npos = static_cast<long long>(K) * static_cast<long long>(table);
    const double* from = m_stagePositions;
#pragma omp parallel for schedule(static) if (npos > 65536)
    for (long long q = 0; q < npos; ++q) positions[q] = from[q];
    const long long ndpos = npos * T;
    const double* dfrom = m_stageDPositions;
#pragma omp parallel for schedule(static) if (ndpos > 65536)
    for (long long q = 0; q < ndpos; ++q) dpositions[q] = dfrom[q];
    if (nonconverged) std::memcpy(nonconverged, m_stageCounts, static_cast<std::size_t>(K) * sizeof(std::uint32_t));
    st.seconds = std::chrono::duration<double>(Clock::now() - t0).count();
    return st;
}

ProgramRunStats SketchProgram::solve()
{
    std::vector<double> values(nValues());
    for (std::size_t v = 0; v < values.size(); ++v) {
        const auto val = m_constraints[v]->getConstraintValue();  // value-less constraints are read by no row
        values[v] = val.has_value() ? val.value() : 0.0;
    }
    std::vector<double> pos(nSlots() * 4);
    const ProgramRunStats st = run(values.data(), 1, pos.data());
    // what a run writes: the target of every row and the anchors of the zero-fixed rows
    std::vector<std::uint8_t> written(nSlots(), 0);
    for (const auto& row : m_rows) {
        written[static_cast<std::size_t>(row.elem[2])] = 1;
        if (isZeroFixed(row.solver)) written[static_cast<std::size_t>(row.elem[0])] = written[static_cast<std::size_t>(row.elem[1])] = 1;
    }
    for (std::size_t s = 0; s < nSlots(); ++s) {
        if (!written[s]) continue;
        const double* p = pos.data() + 4 * s;
        if (m_slotIsLine[s])
            m_elements[s]->updateElementPosition(Eigen::Vector2d { p[0], p[1] }, Eigen::Vector2d { p[2], p[3] });
        else
            m_elements[s]->updateElementPosition(Eigen::Vector2d { p[0], p[1] });
    }
    return st;
}

}  // namespace Gcs::B200
