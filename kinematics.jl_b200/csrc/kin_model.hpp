// kin_model.hpp -- host-side model tables and the compiler into a kin::Program.
#pragma once
#include <string>
#include <vector>

#include "kin_program.h"

namespace kin {

// Row-major 3x3 + translation, double precision, host side only.
struct Xf {
    double r[9];
    double p[3];
    static Xf identity();
    static Xf from_colmajor16(const double *m);
    Xf operator*(const Xf &b) const;
    void apply(const double *v, double *out) const;
};

// Copy of KinModelDesc with 0-based indices.
struct HostModel {
    int n_links = 0, n_joints = 0, with_base = 0;
    std::vector<int> parent;        // 0-based, -1 root
    std::vector<int> jtype, qidx;
    std::vector<Xf> pose;           // Joint.pose
    std::vector<double> axis;       // [L][3], normalised
    std::vector<double> defang;
    int n_sph = 0;
    std::vector<int> sph_link;      // 0-based
    std::vector<double> sph_c, sph_r;
    int n_box = 0;
    std::vector<Xf> box_inv;        // inv(pose)   (sdf.jl:58-61, transform.jl:62-65)
    std::vector<double> box_half;   // 0.5 * width (sdf.jl:68)
    std::vector<int> box_kind;      // row kind of the device table: 0 box, 1 rounded box (sphere), 2 cylinder (extension)
    std::vector<double> box_round;  // rounding radius of a kind-1 row (the sphere's radius)
    std::vector<unsigned long long> box_grid;   // device address of a kind-3 row's grid storage (KinGrid), else 0
    std::vector<int> topo;          // parents before children
    std::vector<unsigned> relmask;  // [L] bit c set <=> control column c moves link (rptable, mechanism.jl:117-139)

    int n_dof() const { return n_joints + (with_base ? 3 : 0); }
    bool finalize(std::string &err);  // validates, builds topo + relmask (control-joint bits only)
};

struct Program {
    ProgHeader h;
    std::vector<int32_t> ints;
    std::vector<double> reals;
};

// the box table of a program: n_box rows of BOX_REALS doubles (inverse pose, half extents, kind, rounding radius, pad)
void emit_box_rows(const HostModel &m, double *dst);
// the FP32 copy of n rows converted from the FP64 ones: puts back the grid addresses the conversion destroyed
void fix_grid_rows_f32(const double *rows64, float *rows32, int n);

// fk_links / jac_links are 0-based link indices in output order.
bool compile_program(const HostModel &m, const std::vector<int> &fk_links, const std::vector<int> &jac_links,
                     bool want_coll, bool want_stale, int jf_regs, Program &out, std::string &err);

}  // namespace kin
