// kin_codegen.cpp -- see kin_codegen.hpp.  Load-time only.
#include "kin_codegen.hpp"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <sstream>
#include <vector>

namespace kin {

std::string GenOptions::key() const {
    char b[200];
    std::snprintf(b, sizeof b, "p%d l%d T%d J%d c%d r%d y%d k%d g%d a%d s%d b%d m%d q%d S%d.%d.%d y%d e%d G%d I%d W%d P%d B%d K%d Q%x", precision, layout, (int)want_T, (int)want_J,
                  (int)coll, with_rot, rpy_jac, keep_irrelevant, (int)want_grads, (int)want_argmin, (int)stale, block, min_blocks, qbatch, sched, epoch, pf_dist,
                  ksync, es32, grad_mode, ik, warp, prims, bulk, const_fill, ik_rot);
    return b;
}

namespace {

// A value of the symbolic evaluation: a constant known at generation time, or an expression (a variable name,
// possibly negated) of the generated code.
struct Val {
    bool c = true;
    double v = 0.0;
    std::string e;
};

class Emitter {
  public:
    explicit Emitter(bool f32) : f32_(f32) {}
    std::ostringstream os;
    int n_ops = 0;

    Val K(double x) const {
        Val r;
        r.c = true;
        r.v = f32_ ? (double)(float)x : x;
        return r;
    }
    static Val V(const std::string &name) {
        Val r;
        r.c = false;
        r.e = name;
        return r;
    }
    // hexadecimal floating literal: exact
    std::string lit(double x) const {
        char b[64];
        if (x == 0.0) return std::signbit(x) ? "real(-0.0)" : "real(0.0)";
        std::snprintf(b, sizeof b, "real(%a)", x);
        return b;
    }
    std::string str(const Val &a) const { return a.c ? lit(a.v) : a.e; }
    Val var(const std::string &expr) {
        const std::string name = "t" + std::to_string(next_++);
        os << "const real " << name << " = " << expr << ";\n";
        ++n_ops;
        return V(name);
    }
    Val neg(const Val &a) const {
        if (a.c) return K(-a.v);
        if (a.e.size() > 3 && a.e[0] == '(' && a.e[1] == '-') return V(a.e.substr(2, a.e.size() - 3));
        return V("(-" + a.e + ")");
    }
    // the folding rules below only remove operations whose result is exact (x * 0, x * +-1, x + 0) or evaluate
    // constants with the same correctly rounded operation the device would use: no result changes (except the sign
    // of a zero)
    Val mul(const Val &a, const Val &b) {
        if (a.c && b.c) return K(f32_ ? (double)((float)a.v * (float)b.v) : a.v * b.v);
        if (b.c) return mul(b, a);
        if (a.c) {
            if (a.v == 0.0) return K(0.0);
            if (a.v == 1.0) return b;
            if (a.v == -1.0) return neg(b);
        }
        return var("mul_(" + str(a) + ", " + str(b) + ")");
    }
    Val add(const Val &a, const Val &b) {
        if (a.c && b.c) return K(f32_ ? (double)((float)a.v + (float)b.v) : a.v + b.v);
        if (a.c && a.v == 0.0) return b;
        if (b.c && b.v == 0.0) return a;
        return var("add_(" + str(a) + ", " + str(b) + ")");
    }
    Val sub(const Val &a, const Val &b) {
        if (a.c && b.c) return K(f32_ ? (double)((float)a.v - (float)b.v) : a.v - b.v);
        if (b.c && b.v == 0.0) return a;
        if (a.c && a.v == 0.0) return neg(b);
        return var("sub_(" + str(a) + ", " + str(b) + ")");
    }
    Val fma(const Val &a, const Val &b, const Val &c) {
        if (a.c && b.c && c.c) return K(f32_ ? (double)std::fmaf((float)a.v, (float)b.v, (float)c.v) : std::fma(a.v, b.v, c.v));
        if ((a.c && a.v == 0.0) || (b.c && b.v == 0.0)) return c;
        if (a.c && a.v == 1.0) return add(b, c);
        if (b.c && b.v == 1.0) return add(a, c);
        if (a.c && a.v == -1.0) return sub(c, b);
        if (b.c && b.v == -1.0) return sub(c, a);
        if (c.c && c.v == 0.0) return mul(a, b);
        return var("fma_(" + str(a) + ", " + str(b) + ", " + str(c) + ")");
    }

  private:
    bool f32_;
    int next_ = 0;
};

struct TfV {
    Val r[9], p[3];
};

// out = a * C  (C: 9 rotation entries row-major, then 3 translation entries) -- tf_mul_const of kin_device_math.cuh
TfV tf_mul_const(Emitter &E, const TfV &a, const double *c, bool r_identity) {
    TfV o;
    const Val t0 = E.K(c[9]), t1 = E.K(c[10]), t2 = E.K(c[11]);
    for (int i = 0; i < 3; ++i)
        o.p[i] = E.fma(a.r[i * 3 + 0], t0, E.fma(a.r[i * 3 + 1], t1, E.fma(a.r[i * 3 + 2], t2, a.p[i])));
    if (r_identity) {
        for (int i = 0; i < 9; ++i) o.r[i] = a.r[i];
    } else {
        Val m[9];
        for (int i = 0; i < 9; ++i) m[i] = E.K(c[i]);
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j)
                o.r[i * 3 + j] = E.fma(a.r[i * 3 + 0], m[j], E.fma(a.r[i * 3 + 1], m[3 + j], E.mul(a.r[i * 3 + 2], m[6 + j])));
    }
    return o;
}

struct Frame {
    Val o[3], a[3];
    bool set = false;
};

}  // namespace

bool generate_source(const Program &p, const GenOptions &o, GenSource &out, std::string &err) {
    const ProgHeader &h = p.h;
    // AoS, one thread per configuration: the outputs of a warp are staged through shared memory in chunks of at most
    // AOS_CHUNK values per record (KPUT into a stage row, KFLUSH_* writes 32 records x chunk with the lanes running
    // along the records: whole sectors); get_jacobian! semantics (columns left untouched) cannot be staged
    // (the tiled layout with bulk stores, GenOptions::bulk, stages the same chunks: a chunk of a tile is one contiguous block)
    const bool aos = (o.layout == 1 || (o.layout == 2 && o.bulk)) && !o.warp && !o.ik;
    if (aos && o.want_J && o.keep_irrelevant) {
        err = "staged outputs with keep_irrelevant are not specialised";
        return false;
    }
    constexpr int AOS_CHUNK = 12;
    if (h.n_dof > 32) { err = "too many columns"; return false; }
    const bool f32 = o.precision == 1;
    out.const_T.clear();
    out.const_J.clear();
    out.expr_T.clear();
    out.expr_J.clear();
    Emitter E(f32);
    const int ND = h.n_dof, DC = h.n_joints, S = o.coll ? h.n_sph : 0;
    const int rows = o.with_rot ? 6 : 3;
    const int32_t *I = p.ints.data();
    const double *R = p.reals.data();
    std::vector<int> col_type(ND, 0);
    unsigned rev_mask = 0;
    for (int j = 0; j < ND; ++j) {
        col_type[j] = I[h.io_col_type + j];
        if (col_type[j] == 1) rev_mask |= 1u << j;
    }

    // ------------------------------------------------------------------ phase 1
    std::vector<bool> q_used(ND, false);
    for (int node = 0; node < h.n_nodes; ++node) {
        const int32_t *ni = I + h.io_node + node * NODE_INTS;
        if (ni[1] != NODE_ROOT) {
            if (ni[3] < 0 || ni[3] >= ND) { err = "node column out of range"; return false; }
            q_used[ni[3]] = true;
        }
    }
    for (int j = 0; j < ND; ++j)
        if (q_used[j]) E.os << "const real q" << j << " = KQ(" << j << ");\n";

    std::vector<Frame> frames(ND);
    std::vector<TfV> saved;
    std::vector<std::vector<Val>> centres(S, std::vector<Val>(3));
    TfV T;
    for (int node = 0; node < h.n_nodes; ++node) {
        const int32_t *ni = I + h.io_node + node * NODE_INTS;
        const double *nr = R + h.ro_node + node * NODE_REALS;
        const int jtype = ni[1];
        if (jtype == NODE_ROOT) {
            for (int i = 0; i < 9; ++i) T.r[i] = E.K(i % 4 == 0 ? 1.0 : 0.0);
            for (int i = 0; i < 3; ++i) T.p[i] = E.K(0.0);
        } else {
            const int psrc = ni[0], flags = ni[2], qcol = ni[3];
            if (psrc >= 0) {
                if (psrc >= (int)saved.size()) { err = "save slot read before it is written"; return false; }
                T = saved[psrc];
            }
            // A = T_parent * joint.pose : the joint frame (algorithm.jl:47-48)
            const TfV Aj = tf_mul_const(E, T, nr, flags & NF_OFF_R_IDENTITY);
            const int code = (flags >> NF_AXIS_SHIFT) & NF_AXIS_MASK;
            Frame f;
            f.set = true;
            for (int i = 0; i < 3; ++i) f.o[i] = Aj.p[i];
            if (code >= 1 && code <= 6) {
                const int k = (code - 1) % 3;
                for (int i = 0; i < 3; ++i) f.a[i] = code >= 4 ? E.mul(E.K(-1.0), Aj.r[i * 3 + k]) : Aj.r[i * 3 + k];
            } else {
                const Val x = E.K(nr[12]), y = E.K(nr[13]), z = E.K(nr[14]);
                for (int i = 0; i < 3; ++i) f.a[i] = E.fma(Aj.r[i * 3 + 0], x, E.fma(Aj.r[i * 3 + 1], y, E.mul(Aj.r[i * 3 + 2], z)));
            }
            frames[qcol] = f;
            const Val qa = Emitter::V("q" + std::to_string(qcol));
            T = Aj;
            if (jtype == 2) {          // prismatic: pose * Trans(axis * a), mechanism.jl:100-103
                for (int i = 0; i < 3; ++i) T.p[i] = E.fma(f.a[i], qa, Aj.p[i]);
            } else {                   // revolute: pose * R(axis, a), mechanism.jl:94-98
                const std::string sn = "sn" + std::to_string(node), cn = "cs" + std::to_string(node);
                E.os << "real " << sn << ", " << cn << "; sincos_(" << E.str(code >= 4 ? E.neg(qa) : qa) << ", &" << sn << ", &" << cn << ");\n";
                const Val s = Emitter::V(sn), c = Emitter::V(cn);
                if (code >= 1 && code <= 6) {
                    // rotation about a coordinate axis mixes the two other columns (GIVENS of the kernel)
                    const int k = (code - 1) % 3, u = (k + 1) % 3, v = (k + 2) % 3;
                    for (int i = 0; i < 3; ++i) {
                        const Val cu = Aj.r[i * 3 + u], cv = Aj.r[i * 3 + v];
                        T.r[i * 3 + u] = E.fma(c, cu, E.mul(s, cv));
                        T.r[i * 3 + v] = E.fma(c, cv, E.neg(E.mul(s, cu)));
                    }
                } else {
                    // Rodrigues form of the reference's quaternion rotation: Rot = c I + s [a]x + (1 - c) a a'
                    const Val x = E.K(nr[12]), y = E.K(nr[13]), z = E.K(nr[14]);
                    const Val t = E.sub(E.K(1.0), c);
                    const Val tx = E.mul(t, x), ty = E.mul(t, y), tz = E.mul(t, z);
                    Val m[9];
                    m[0] = E.fma(tx, x, c);                      m[1] = E.fma(tx, y, E.neg(E.mul(s, z))); m[2] = E.fma(tx, z, E.mul(s, y));
                    m[3] = E.fma(tx, y, E.mul(s, z));            m[4] = E.fma(ty, y, c);                  m[5] = E.fma(ty, z, E.neg(E.mul(s, x)));
                    m[6] = E.fma(tx, z, E.neg(E.mul(s, y)));     m[7] = E.fma(ty, z, E.mul(s, x));        m[8] = E.fma(tz, z, c);
                    for (int i = 0; i < 3; ++i)
                        for (int j = 0; j < 3; ++j)
                            T.r[i * 3 + j] = E.fma(Aj.r[i * 3 + 0], m[j], E.fma(Aj.r[i * 3 + 1], m[3 + j], E.mul(Aj.r[i * 3 + 2], m[6 + j])));
                }
            }
        }
        if (ni[4] >= 0) {
            if ((int)saved.size() <= ni[4]) saved.resize(ni[4] + 1);
            saved[ni[4]] = T;
        }
        if (o.ksync) E.os << "KSYNC();\n";

        // ---- requested links hanging from this node ----
        for (int a = ni[5]; a < ni[6]; ++a) {
            const int32_t *ai = I + h.io_att + a * ATT_INTS;
            const double *ar = R + h.ro_att + a * ATT_REALS;
            const bool do_T = ai[0] >= 0 && o.want_T, do_J = ai[2] >= 0 && o.want_J;
            if (!do_T && !do_J) continue;
            const TfV Tl = tf_mul_const(E, T, ar, ai[1] & AF_R_IDENTITY);
            if (do_T) {                        // get_transform, as 3x4 column-major
                const int base = 12 * ai[0];
                for (int c = 0; c < 3; ++c)
                    for (int r = 0; r < 3; ++r)
                        if (Tl.r[r * 3 + c].c) out.const_T.emplace_back(base + c * 3 + r, Tl.r[r * 3 + c].v);
                        else out.expr_T.emplace_back(base + c * 3 + r, Tl.r[r * 3 + c].e);
                for (int r = 0; r < 3; ++r)
                    if (Tl.p[r].c) out.const_T.emplace_back(base + 9 + r, Tl.p[r].v);
                    else out.expr_T.emplace_back(base + 9 + r, Tl.p[r].e);
                if (aos) {
                    for (int c = 0; c < 3; ++c)
                        for (int r = 0; r < 3; ++r) E.os << "KPUT(12, " << c * 3 + r << ", " << E.str(Tl.r[r * 3 + c]) << ");\n";
                    for (int r = 0; r < 3; ++r) E.os << "KPUT(12, " << 9 + r << ", " << E.str(Tl.p[r]) << ");\n";
                    E.os << "KFLUSH_T(" << base << ", 12);\n";
                } else {
                    for (int c = 0; c < 3; ++c)
                        for (int r = 0; r < 3; ++r) E.os << "KST_T(" << base + c * 3 + r << ", " << E.str(Tl.r[r * 3 + c]) << ");\n";
                    for (int r = 0; r < 3; ++r) E.os << "KST_T(" << base + 9 + r << ", " << E.str(Tl.p[r]) << ");\n";
                }
            }
            if (do_J) {                        // get_jacobian, algorithm.jl:83-114
                const int kbase = ai[2] * rows * ND;
                const unsigned mask = (unsigned)ai[3];
                std::string kk;
                if (o.with_rot && o.rpy_jac) {
                    kk = "kk" + std::to_string(a);
                    E.os << "real " << kk << "[6];\n{ Tf<real> TL;\n";
                    for (int i = 0; i < 9; ++i) E.os << "TL.r[" << i << "] = " << E.str(Tl.r[i]) << "; ";
                    E.os << "\nTL.p[0] = TL.p[1] = TL.p[2] = real(0);\nrpy_rate_coeffs(TL, " << kk << "); }\n";
                }
                // AoS: chunks of whole columns, at most AOS_CHUNK values, flushed after their last column
                const int cols_per_chunk = AOS_CHUNK / rows;
                int chunk_k0 = kbase, chunk_cnt = 0;
                auto stv = [&](int k, const Val &v) -> std::string {       // a value of the symbolic evaluation
                    if (v.c) out.const_J.emplace_back(k, v.v);
                    else out.expr_J.emplace_back(k, v.e);
                    return E.str(v);
                };
                auto stz = [&](int k) -> std::string { out.const_J.emplace_back(k, 0.0); return "real(0)"; };
                auto stj = [&](int k, const std::string &v) -> std::string {
                    if (aos) return "KPUT(" + std::to_string(chunk_cnt) + ", " + std::to_string(k - chunk_k0) + ", " + v + ");";
                    return "KST_J(" + std::to_string(k) + ", " + v + ");";
                };
                for (int j = 0; j < ND; ++j) {
                    const int kc = kbase + j * rows;
                    if (aos && j % cols_per_chunk == 0) { chunk_k0 = kc; chunk_cnt = std::min(cols_per_chunk, ND - j) * rows; }
                    if ((mask >> j) & 1u) {
                        const Frame &f = frames[j];
                        if (!f.set) { err = "Jacobian column of a joint that has not been visited"; return false; }
                        const bool rev = col_type[j] == 1;
                        Val cx, cy, cz;
                        if (rev) {             // joint_jacobian!, algorithm.jl:65-76
                            const Val dx = E.sub(Tl.p[0], f.o[0]), dy = E.sub(Tl.p[1], f.o[1]), dz = E.sub(Tl.p[2], f.o[2]);
                            cx = E.fma(f.a[1], dz, E.neg(E.mul(f.a[2], dy)));
                            cy = E.fma(f.a[2], dx, E.neg(E.mul(f.a[0], dz)));
                            cz = E.fma(f.a[0], dy, E.neg(E.mul(f.a[1], dx)));
                        } else { cx = f.a[0]; cy = f.a[1]; cz = f.a[2]; }
                        E.os << stj(kc, stv(kc, cx)) << " " << stj(kc + 1, stv(kc + 1, cy)) << " " << stj(kc + 2, stv(kc + 2, cz)) << "\n";
                        if (o.with_rot) {
                            if (rev) {
                                if (o.rpy_jac) {
                                    E.os << "{ real o3, o4, o5; rpy_rows(" << kk << ", " << E.str(f.a[0]) << ", " << E.str(f.a[1]) << ", "
                                         << E.str(f.a[2]) << ", o3, o4, o5); " << stj(kc + 3, "o3") << " " << stj(kc + 4, "o4") << " "
                                         << stj(kc + 5, "o5") << " }\n";
                                } else {
                                    for (int r = 0; r < 3; ++r) E.os << stj(kc + 3 + r, stv(kc + 3 + r, f.a[r])) << " ";
                                    E.os << "\n";
                                }
                            } else if (!o.keep_irrelevant || j >= DC) {
                                // prismatic: rows 4:6 untouched by the reference (algorithm.jl:78-81), except in the base
                                // block, which it always writes (algorithm.jl:102-104)
                                for (int r = 3; r < 6; ++r) E.os << stj(kc + r, stz(kc + r)) << " ";
                                E.os << "\n";
                            }
                        }
                    } else if (!o.keep_irrelevant) {
                        for (int r = 0; r < rows; ++r) E.os << stj(kc + r, stz(kc + r)) << " ";
                        E.os << "\n";
                    }
                    if (aos && ((j + 1) % cols_per_chunk == 0 || j + 1 == ND))
                        E.os << "KFLUSH_J(" << chunk_k0 << ", " << (kc + rows - chunk_k0) << ");\n";
                }
            }
        }

        // ---- collision-sphere centres on this node (collision.jl:54 / :80) ----
        if (o.coll)
            for (int k = ni[7]; k < ni[8]; ++k) {
                const int s = I[h.io_sph_order + k];
                const double *sr = R + h.ro_sph + s * SPH_REALS;
                const Val c0 = E.K(sr[0]), c1 = E.K(sr[1]), c2 = E.K(sr[2]);
                for (int i = 0; i < 3; ++i) {
                    centres[s][i] = E.fma(T.r[i * 3 + 0], c0, E.fma(T.r[i * 3 + 1], c1, E.fma(T.r[i * 3 + 2], c2, T.p[i])));
                    E.os << "KCEN_SET(" << s << ", " << i << ", " << E.str(centres[s][i]) << ");\n";
                }
            }
    }
    out.phase1 = E.os.str();
    out.n_ops = E.n_ops;

    // ------------------------------------------------------------------ phase 2: one call per run of equal masks
    std::ostringstream p2;
    if (o.coll) {
        // joint frames of the columns as the consumers of phase 2 see them
        p2 << "const JFrame<real> jfr[KND] = {\n";
        for (int j = 0; j < ND; ++j) {
            const Frame &f = frames[j];
            p2 << "  {{";
            for (int i = 0; i < 3; ++i) p2 << (f.set ? E.str(f.o[i]) : std::string("real(0)")) << (i < 2 ? ", " : "}, {");
            for (int i = 0; i < 3; ++i) p2 << (f.set ? E.str(f.a[i]) : std::string("real(0)")) << (i < 2 ? ", " : "}}");
            p2 << (j + 1 < ND ? ",\n" : "\n");
        }
        p2 << "};\n";
        // runs of consecutive spheres with equal relevance mask; groups of up to SPH_GROUP spheres inside a run
        struct Run { int sb, se; unsigned mask; };
        std::vector<Run> runs;
        for (int sb = 0; sb < S;) {
            const unsigned mask = (unsigned)I[h.io_sph_mask + sb];
            int se = sb + 1;
            while (se < S && (unsigned)I[h.io_sph_mask + se] == mask) ++se;
            runs.push_back({sb, se, mask});
            sb = se;
        }
        // distinct masks share one instantiation of phase 2b
        std::vector<unsigned> masks;
        for (const Run &r : runs) {
            bool seen = false;
            for (unsigned mk : masks) seen |= mk == r.mask;
            if (!seen) masks.push_back(r.mask);
        }
        p2 << "#if !KWARP\n#pragma unroll 1\nfor (int s0 = 0; s0 < KS;) {\n    int se, mi;\n";
        for (size_t r = 0; r < runs.size(); ++r) {
            size_t mi = 0;
            while (masks[mi] != runs[r].mask) ++mi;
            p2 << "    " << (r ? "else " : "") << (r + 1 < runs.size() ? "if (s0 < " + std::to_string(runs[r].se) + ") " : "") << "{ se = " << runs[r].se
               << "; mi = " << mi << "; }\n";
        }
        p2 << "    const int ge = min(s0 + SPH_GROUP, se);\n    phase2a_group<real>(s0, ge, KP2AARGS);\n";
        p2 << "    switch (mi) {\n";
        for (size_t mi = 0; mi < masks.size(); ++mi)
            p2 << "        case " << mi << ": phase2b_group<real, KND, 0x" << std::hex << masks[mi] << std::dec << "u>(s0, ge, KP2BARGS); break;\n";
        p2 << "        default: break;\n    }\n";
        p2 << "    s0 = ge;\n}\n#endif\n";
    }
    out.phase2 = p2.str();

    // ------------------------------------------------------------------ constants of the model + options
    std::ostringstream c;
    c << "#define KREAL " << (f32 ? "float" : "double") << "\n";
    c << "#define KPRIMS " << o.prims << "\n#define KBULK " << ((o.bulk && o.layout == 2 && !o.warp && !o.ik) ? 1 : 0) << "\n";
    c << "#define KWANT_T " << (o.want_T ? 1 : 0) << "\n#define KWANT_J " << (o.want_J ? 1 : 0) << "\n#define KCOLL " << (o.coll ? 1 : 0)
      << "\n#define KTILED " << (o.layout == 2 ? 1 : 0) << "\n#define KAOS " << (o.layout == 1 ? 1 : 0) << "\n";
    c << "#define KBS " << o.block << "\n#define KMINB " << o.min_blocks << "\n#define KWARP " << o.warp << "\n#define KIK " << o.ik << "\n#define KQB " << o.qbatch << "\n#define KSYNC_ON "
      << o.ksync << "\n#define KES32 " << o.es32 << "\n";
    const bool sched = o.sched && !o.coll && !o.warp && !o.ik;
    c << "#define KSCHED " << (sched ? 1 : 0) << "\n#define KEPOCH " << (sched ? std::max(1, o.epoch) : 1) << "\n#define KPFD " << (sched ? o.pf_dist : 0) << "\n";
    // the configuration-independent outputs as a table of rows (kin_gen_skeleton.cuh: kin_const_fill_kernel): component (T: k,
    // J: -1 - k) and value, written as the literals phase 1 stores -- the outputs keep their bits, sign of zero included
    // -- and, for the store macros, which components the table holds.  Phase 1 keeps every KST_* line (kin_eval_host and
    // the tests read the generated text); the skeleton drops the listed ones at compile time.
    const bool cfill = o.const_fill && o.layout == 0 && !o.warp && !o.ik && (!out.const_T.empty() || !out.const_J.empty());
    c << "#define KCFILL " << (cfill ? 1 : 0) << "\n";
    if (o.ik && h.n_fk > 1) c << "#define KIKROT 0x" << std::hex << o.ik_rot << std::dec << "u\n";
    c << "namespace kin {\n";
    for (int a = 0; a < 2; ++a) {
        const std::vector<std::pair<int, double>> &tab = a ? out.const_J : out.const_T;
        c << "__host__ __device__ constexpr bool " << (a ? "kcf_J" : "kcf_T") << "(int k) {";
        if (cfill && !tab.empty()) {
            c << "\n    switch (k) {";
            for (size_t i = 0; i < tab.size(); ++i) c << (i % 16 ? " " : "\n    ") << "case " << tab[i].first << ":";
            c << " return true;\n    default: return false;\n    }\n}\n";
        } else {
            c << " return false; }\n";
        }
    }
    if (cfill) {
        const size_t nT = out.const_T.size(), nc = nT + out.const_J.size();
        auto row = [&](size_t i) { return i < nT ? out.const_T[i] : std::make_pair(-1 - out.const_J[i - nT].first, out.const_J[i - nT].second); };
        c << "typedef KREAL real;\nconstexpr int KNCF = " << nc << ";\n__device__ const int KCF_ROW[KNCF] = {";
        for (size_t i = 0; i < nc; ++i) c << (i ? ", " : "") << (i % 16 ? "" : "\n    ") << row(i).first;
        c << "};\n__device__ const real KCF_VAL[KNCF] = {";
        for (size_t i = 0; i < nc; ++i) c << (i ? ", " : "") << (i % 6 ? "" : "\n    ") << E.lit(row(i).second);
        c << "};\n";
    }
    c << "constexpr int KND = " << ND << ", KDC = " << DC << ", KS = " << S << ", KNFK = " << (o.want_T ? h.n_fk : 0) << ", KNJAC = "
      << (o.want_J ? h.n_jac : 0) << ", KROWS = " << rows << ";\n";
    c << "constexpr int KGRADMODE = " << o.grad_mode << ";\n";
    c << "constexpr unsigned KREV = 0x" << std::hex << rev_mask << std::dec << "u;\n";
    c << "constexpr bool KSTALE = " << (o.stale ? "true" : "false") << ", KGRADS = " << (o.want_grads ? "true" : "false") << ", KARGMIN = "
      << (o.want_argmin ? "true" : "false") << ";\n";
    if (S > 0) {
        c << "__device__ const KREAL KRADIUS[KS] = {";
        for (int s = 0; s < S; ++s) {
            char b[64];
            const double r = f32 ? (double)(float)R[h.ro_sph + s * SPH_REALS + 3] : R[h.ro_sph + s * SPH_REALS + 3];
            std::snprintf(b, sizeof b, "%a", r);
            c << (s ? ", " : "") << "KREAL(" << b << ")";
        }
        c << "};\n";
        c << "__device__ const unsigned KSPHMASK[KS] = {";
        for (int s = 0; s < S; ++s) c << (s ? ", " : "") << "0x" << std::hex << (unsigned)I[h.io_sph_mask + s] << std::dec << "u";
        c << "};\n";
    }
    c << "}  // namespace kin\n";
    out.config = c.str();
    return true;
}

}  // namespace kin
