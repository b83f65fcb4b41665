// kin_codegen.hpp -- model-specialised CUDA source for one compiled kinematic program (kin_program.h).
//
// The ahead-of-time kernels (kin_kernels.cuh) INTERPRET the program tables per configuration: node loop, table
// loads, flag tests, run-time relevance masks -- 71 % of their issued instructions are that interpretation, not
// arithmetic (profiles/r01c_fused_ws_sass_mix.txt).  For large batches the library instead generates the source of
// a kernel for THIS model and THESE requested outputs and compiles it with NVRTC for sm_100a (kin_jit.cpp):
//   * phase 1 (forward kinematics, joint frames, link transforms, Jacobians, sphere centres: algorithm.jl:1-114,
//     mechanism.jl:90-103, collision.jl:39-49) becomes straight-line code.  The generator evaluates the chain
//     SYMBOLICALLY: every transform entry is either a known constant or a named variable, multiplications by exact
//     0 / +-1 and additions of exact 0 disappear, constants fold on the host with the same correctly rounded
//     operations -- which leaves every remaining operation, and therefore every result, bit-identical to the
//     interpreting kernel (up to the sign of a zero);
//   * phase 2 (union SDF, truncation, gradient, chain rule: sdf.jl:34-41,108-119, collision.jl:67-94) is the same
//     C++ as the interpreting kernel, instantiated once per run of spheres with equal relevance mask, with the mask,
//     the column count and types, and the scratch / gradient / argmin switches as template constants.
// The generated text is compiled together with kin_device_math.cuh and kin_gen_skeleton.cuh (both embedded in the
// library).
#pragma once
#include <string>
#include <utility>
#include <vector>

#include "kin_model.hpp"

namespace kin {

struct GenOptions {
    int precision = 0;          // 0 = f64, 1 = f32
    int layout = 0;             // 0 = SoA, 1 = AoS (outputs staged per warp through shared memory), 2 = tiled
    bool want_T = false, want_J = false, coll = false;
    int with_rot = 0, rpy_jac = 0, keep_irrelevant = 0;
    bool want_grads = false, want_argmin = false, stale = false;
    int block = 128, min_blocks = 1;
    int qbatch = 0;             // > 0 (AoS): tiles per input batch (cp.async into shared memory behind a grid-wide barrier)
    int sched = 0;              // 1: FK / Jacobian only: tiles claimed from a counter, inputs prefetched into L2 one epoch at a time
    int epoch = 0;              //    sched: tiles per epoch
    int pf_dist = 0;            //    sched: epochs the L2 prefetch runs ahead (0: none)
    int warp = 0;               // 1: small-batch kernel, one WARP per configuration (lane = sphere in phase 2)
    int ik = 0;                 // 1: the batched Levenberg-Marquardt IK kernel around phase 1 (one link: T + rpy-Jacobian)
    unsigned ik_rot = 0;        //    ik with several links: bit l = link l has its rotation rows (KIKROT; unused for one link)
    int grad_mode = -1;         // >= 0: the gradient mode as a compile-time constant (only that code path is compiled in)
    int ksync = 0;              // 1: CTA-wide barrier after every node of phase 1 (the warps of a CTA then fetch the
                                //    straight-line code together: one instruction-cache fill serves all of them)
    int bulk = 0;               // 1: tiled layout, FK / Jacobian only: outputs staged per warp and written with cp.async.bulk (TMA)
    int prims = 0;              // 1: the SDF table holds rows other than boxes (sphere / cylinder): the row loops test the kind
    int es32 = 0;               // 1: SoA component stride held in 32 bits (ld < 2^32): one IMAD.WIDE per store address
    int const_fill = 0;         // 1: SoA, one thread per configuration: the outputs of GenSource::const_T / const_J are not
                                //    stored per thread; kin_const_fill_kernel writes those rows as contiguous runs (KCFILL)
    std::string key() const;    // cache key of the option set
};

struct GenSource {
    std::string config;         // "kin_gen_config.h": constants of the model + options
    std::string phase1;         // "kin_gen_phase1.inc": straight-line phase 1
    std::string phase2;         // "kin_gen_phase2.inc": the phase-2 run calls
    int n_ops = 0;              // arithmetic operations emitted in phase 1 (diagnostics)
    // outputs whose value does not depend on the configuration (links no control joint moves, zero / unit rotation
    // entries, Jacobian columns of joints that do not move the link): (component index, value).  kin_eval_host does
    // not move these rows over PCIe: the host fills them (SoA layout).
    std::vector<std::pair<int, double>> const_T, const_J;
    // the other outputs: (component index, expression) -- a variable of the generated code, possibly negated "(-tN)".
    // Two outputs with the same variable hold the same bits (rotation blocks shared by links joined through fixed
    // pure-translation joints, joint axes that are columns of a link rotation, ...): kin_eval_host moves one of them
    // over PCIe and lets the host copy the others.
    std::vector<std::pair<int, std::string>> expr_T, expr_J;
};

// Returns false (with err) when the program cannot be specialised (the caller then uses the interpreting kernel).
bool generate_source(const Program &p, const GenOptions &o, GenSource &out, std::string &err);

}  // namespace kin
