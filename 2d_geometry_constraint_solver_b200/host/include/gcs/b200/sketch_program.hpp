// sketch_program.hpp — a decomposed sketch planned once and solved on the device for many sets of
// constraint values (gcs_b200_program_* of include/gcs_b200.h).
//
// The wave plan of solveLeaves (which solver, which roles, which wave) depends on the topology, the
// solved flags and the canvas, not on the constraint values; so does the canvas half of every batch
// row (codes, canvas-side signs, canvas normals).  compile() does that work once on the host; run()
// hands the device the values of K instances, and every wave runs there as one gather launch, one
// launch per equation kind over rows x K sub-systems and one scatter launch, with no host round trip
// between waves.  Instance k's result equals what solveLeaves leaves in the elements when the
// constraints hold instance k's values, bit for bit.
#pragma once

#include <cstddef>
#include <cstdint>
#include <memory>
#include <vector>

#include <gcs/b200/leaf_batch.hpp>
#include <gcs/export.hpp>
#include <gcs/model/constraints.hpp>
#include <gcs/model/gcs_data_structures.hpp>

#include "gcs_b200.h"

namespace Gcs::B200 {

struct ProgramRunStats {
    std::int64_t launches = 0;              // kernel launches of the run (all devices)
    double uploadMs = 0, deviceMs = 0, downloadMs = 0;  // device time, summed over devices
    double seconds = 0;                     // host clock, call to return
};

class GCS_API SketchProgram {
public:
    // leaves: as decomposeConstraintGraph returns them.  elements / constraints: the slot order of
    // the position table and the value order of the value table; a constraint is identified by its
    // object (the decomposition shares the sketch's constraints with the leaves).  Uses the plan of
    // solveLeaves; throws what the reference's loop would throw for a leaf, and std::invalid_argument
    // when a leaf reads an element or constraint missing from the lists.  Unsupported leaves are
    // skipped and reported in report().  No device is needed.
    static SketchProgram compile(const std::vector<ConstraintGraph>& leaves, const std::vector<std::shared_ptr<Element>>& elements,
        const std::vector<std::shared_ptr<Constraint>>& constraints);

    SketchProgram(SketchProgram&&) noexcept;
    SketchProgram& operator=(SketchProgram&&) noexcept;
    SketchProgram(const SketchProgram&) = delete;
    SketchProgram& operator=(const SketchProgram&) = delete;
    ~SketchProgram();

    // K instances.  values: host [K][nValues()], angles in radians (converted with std::cos here, as
    // the packer does); positions: host [K][nSlots()][4] (point: x, y, then the initial contents);
    // nonconverged (may be null): per instance, the leaves whose chosen Newton run did not converge.
    // nDevices > 1: instances in contiguous ranges over device ordinals 0 .. nDevices-1, one program
    // copy per device, no collective.  Kernel class: kernelVariant().  Throws std::runtime_error when
    // the CUDA library fails (no device: there is no CPU path).
    ProgramRunStats run(const double* values, std::int64_t K, double* positions, std::uint32_t* nonconverged = nullptr, int nDevices = 1);

    // run(), plus the derivatives of the positions along T >= 1 directions in value space
    // (gcs_b200_program_run_tangents): dvalues host [K][nValues()][T], in radians for angles like the
    // values; dpositions host [K][nSlots()][4][T] receives sum_v dpositions/dvalues[v] * dvalues[v][t],
    // NaN downstream of a row whose chosen run did not converge.  Positions and counts are run()'s.
    // Throws std::invalid_argument for T < 1 before any device call.
    ProgramRunStats runTangents(const double* values, std::int64_t K, const double* dvalues, int T, double* positions, double* dpositions,
        std::uint32_t* nonconverged = nullptr, int nDevices = 1);

    // run(), also recording what adjoints() needs (gcs_b200_program_run_recorded): every wave's
    // batches stay on the device, about n_rows x K x 100 bytes.  Positions and counts are run()'s.
    ProgramRunStats record(const double* values, std::int64_t K, double* positions, std::uint32_t* nonconverged = nullptr,
        int nDevices = 1);

    // Reverse mode over the last record() (gcs_b200_program_adjoints), with its K and device split:
    // adjPositions host [K][nSlots()][4][T] (T >= 1 cotangents, weights on the position coordinates),
    // adjValues host [K][nValues()][T] receives sum_{s,c} adjPositions[k][s][c][t] * dpositions[k][s][c]
    // / dvalues[k][v], with respect to radians for angles: the device gives the adjoint with respect
    // to cos(v), and here adj = (-std::sin(v)) * adj_cos, v the recorded value.  NaN for every value
    // of (k, t) when the cotangent reaches a row whose chosen run did not converge.  Throws
    // std::logic_error before any device call when nothing was recorded, std::invalid_argument for
    // T < 1.
    ProgramRunStats adjoints(const double* adjPositions, int T, double* adjValues);

    // The edit loop: one instance with the constraints' current values, written into the elements -
    // the state solveLeaves leaves.
    ProgramRunStats solve();

    const BatchReport& report() const { return m_report; }  // per leaf: solver, wave, status (no timings but planSeconds)
    std::size_t nSlots() const { return m_slotIsLine.size(); }
    std::size_t nValues() const { return m_valueIsAngle.size(); }
    std::size_t waves() const { return m_report.waves; }
    const std::vector<gcs_b200_program_row>& rows() const { return m_rows; }
    const std::vector<std::int64_t>& offsets() const { return m_offsets; }  // [waves * GCS_KIND_COUNT + 1]
    const std::vector<std::int64_t>& rowLeaf() const { return m_rowLeaf; }  // leaf index of every row
    const std::vector<std::uint8_t>& solvedAfter() const { return m_solvedAfter; }  // per slot: solved after a run
    double compileSeconds() const { return m_compileSeconds; }
    int recordedDevices() const { return m_recordedDevices; }  // devices of the last record() (0: none)
    // the descriptor gcs_b200_program_create takes, pointing into this program's tables (valid while
    // the program lives and is not moved from)
    gcs_b200_program_desc desc() const;

private:
    SketchProgram() = default;
    gcs_b200_program* onDevice(int device);
    void release();
    ProgramRunStats runImpl(const double* values, std::int64_t K, const double* dvalues, int T, double* positions, double* dpositions,
        std::uint32_t* nonconverged, int nDevices, bool recorded = false);

    BatchReport m_report;
    std::vector<gcs_b200_program_row> m_rows;
    std::vector<std::int64_t> m_offsets, m_rowLeaf;
    std::vector<std::uint8_t> m_slotIsLine, m_valueIsAngle, m_solvedAfter;
    std::vector<double> m_initial;  // [nSlots][4]
    std::vector<std::shared_ptr<Element>> m_elements;
    std::vector<std::shared_ptr<Constraint>> m_constraints;
    double m_compileSeconds = 0;
    std::vector<gcs_b200_program*> m_device;  // uploaded lazily, by device ordinal
    // page-locked staging of run()
    double* m_stageValues = nullptr;
    double* m_stagePositions = nullptr;
    std::uint32_t* m_stageCounts = nullptr;
    std::int64_t m_stageK = 0;
    double* m_stageDValues = nullptr;
    double* m_stageDPositions = nullptr;
    std::int64_t m_stageKT = 0;  // instances x directions the tangent staging holds
    // the last record(): its values (radians) and device split; m_recordedDevices = 0: none
    std::vector<double> m_recordedValues;
    std::int64_t m_recordedK = 0;
    int m_recordedDevices = 0;
};

}  // namespace Gcs::B200
