// kin_model.cpp -- host-side flattening of a mechanism into a kin::Program (see kin_program.h).
// Load-time only; nothing here runs per configuration.
#include "kin_model.hpp"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <functional>

namespace kin {

Xf Xf::identity() {
    Xf t;
    std::memset(&t, 0, sizeof t);
    t.r[0] = t.r[4] = t.r[8] = 1.0;
    return t;
}

Xf Xf::from_colmajor16(const double *m) {
    Xf t;
    for (int r = 0; r < 3; ++r) {
        for (int c = 0; c < 3; ++c) t.r[r * 3 + c] = m[c * 4 + r];
        t.p[r] = m[12 + r];
    }
    return t;
}

Xf Xf::operator*(const Xf &b) const {
    Xf o;
    for (int i = 0; i < 3; ++i) {
        for (int j = 0; j < 3; ++j)
            o.r[i * 3 + j] = r[i * 3 + 0] * b.r[0 * 3 + j] + r[i * 3 + 1] * b.r[1 * 3 + j] + r[i * 3 + 2] * b.r[2 * 3 + j];
        o.p[i] = r[i * 3 + 0] * b.p[0] + r[i * 3 + 1] * b.p[1] + r[i * 3 + 2] * b.p[2] + p[i];
    }
    return o;
}

void Xf::apply(const double *v, double *out) const {
    for (int i = 0; i < 3; ++i) out[i] = r[i * 3 + 0] * v[0] + r[i * 3 + 1] * v[1] + r[i * 3 + 2] * v[2] + p[i];
}

static bool is_identity3(const double *r) {
    static const double I[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    for (int i = 0; i < 9; ++i)
        if (r[i] != I[i]) return false;
    return true;
}

// joint_transform (mechanism.jl:90-103) of a joint that is NOT driven by the configuration:
// fixed -> pose; movable at a == 0.0 -> pose (the short-cut); otherwise pose * motion(a).
static Xf frozen_joint_transform(const HostModel &m, int l) {
    const Xf &pose = m.pose[l];
    double a = m.defang[l];
    if (m.jtype[l] == 0 || a == 0.0) return pose;
    Xf mot = Xf::identity();
    const double *ax = &m.axis[3 * l];
    if (m.jtype[l] == 1) {
        double w = std::cos(0.5 * a), s = std::sin(0.5 * a);
        double x = ax[0] * s, y = ax[1] * s, z = ax[2] * s;
        double inorm = 1.0 / std::sqrt(w * w + x * x + y * y + z * z);
        w *= inorm; x *= inorm; y *= inorm; z *= inorm;
        double xx = x * x, yy = y * y, zz = z * z, xy = x * y, zw = w * z, xz = x * z, yw = y * w, yz = y * z, xw = w * x;
        mot.r[0] = 1 - 2 * (yy + zz); mot.r[1] = 2 * (xy - zw);     mot.r[2] = 2 * (xz + yw);
        mot.r[3] = 2 * (xy + zw);     mot.r[4] = 1 - 2 * (xx + zz); mot.r[5] = 2 * (yz - xw);
        mot.r[6] = 2 * (xz - yw);     mot.r[7] = 2 * (yz + xw);     mot.r[8] = 1 - 2 * (xx + yy);
    } else {
        mot.p[0] = ax[0] * a; mot.p[1] = ax[1] * a; mot.p[2] = ax[2] * a;
    }
    return pose * mot;
}

bool HostModel::finalize(std::string &err) {
    if (n_links <= 0) { err = "n_links must be positive"; return false; }
    if (n_joints < 0 || n_joints + (with_base ? 3 : 0) > 32) { err = "n_joints (+3 base columns) exceeds KIN_MAX_JOINTS"; return false; }
    std::vector<int> seen(n_joints, 0);
    std::vector<std::vector<int>> kids(n_links);
    for (int l = 0; l < n_links; ++l) {
        if (parent[l] >= n_links || parent[l] == l || parent[l] < -1) { err = "parent_link out of range"; return false; }
        if (parent[l] < 0) { jtype[l] = 0; qidx[l] = -1; }
        else kids[parent[l]].push_back(l);
        if (jtype[l] < 0 || jtype[l] > 2) { err = "unknown joint type"; return false; }
        if (qidx[l] >= n_joints) { err = "q_index out of range"; return false; }
        if (jtype[l] == 0) qidx[l] = -1;
        if (qidx[l] >= 0) {
            if (seen[qidx[l]]++) { err = "two links share one q_index"; return false; }
        }
        if (jtype[l] != 0) {
            double *a = &axis[3 * l];
            double n = std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
            if (!(n > 0)) { err = "zero joint axis"; return false; }
            a[0] /= n; a[1] /= n; a[2] /= n;
        }
    }
    // parents before children (BFS from the roots); also detects cycles
    topo.clear();
    for (int l = 0; l < n_links; ++l)
        if (parent[l] < 0) topo.push_back(l);
    for (size_t k = 0; k < topo.size(); ++k)
        for (int c : kids[topo[k]]) topo.push_back(c);
    if ((int)topo.size() != n_links) { err = "link table is not a forest (cycle or dangling parent)"; return false; }
    relmask.assign(n_links, 0u);
    for (int l : topo) {
        unsigned mk = parent[l] >= 0 ? relmask[parent[l]] : 0u;
        if (qidx[l] >= 0) mk |= 1u << qidx[l];
        relmask[l] = mk;
    }
    for (int s = 0; s < n_sph; ++s)
        if (sph_link[s] < 0 || sph_link[s] >= n_links) { err = "sphere_link out of range"; return false; }
    return true;
}

void emit_box_rows(const HostModel &m, double *dst) {
    for (int b = 0; b < m.n_box; ++b) {
        double *br = dst + (size_t)b * BOX_REALS;
        std::memset(br, 0, sizeof(double) * BOX_REALS);
        std::memcpy(br, m.box_inv[b].r, sizeof(double) * 9);
        std::memcpy(br + 9, m.box_inv[b].p, sizeof(double) * 3);
        std::memcpy(br + 12, &m.box_half[3 * b], sizeof(double) * 3);
        br[15] = (size_t)b < m.box_kind.size() ? (double)m.box_kind[b] : 0.0;
        br[16] = (size_t)b < m.box_round.size() ? m.box_round[b] : 0.0;
        if (br[15] == 3.0) std::memcpy(br + 17, &m.box_grid[b], sizeof(double));     // the address as raw bits
    }
}

void fix_grid_rows_f32(const double *rows64, float *rows32, int n) {
    for (int b = 0; b < n; ++b)
        if (rows64[(size_t)b * BOX_REALS + 15] == 3.0)
            std::memcpy(rows32 + (size_t)b * BOX_REALS + 16, rows64 + (size_t)b * BOX_REALS + 17, sizeof(double));
}

namespace {
struct Node {
    int link;            // -1 for the virtual root
    int parent;          // node index (pre-compaction), -1 for root
    int jtype, qcol;
    Xf off;
    double axis[3];
    unsigned relmask;
    std::vector<int> kids;
    bool needed = false;
    // filled by the DFS
    int parent_src = PARENT_NONE, save_slot = -1;
};
struct Att {
    int node, fk, jac, flags;
    Xf C;
};
}  // namespace

bool compile_program(const HostModel &m, const std::vector<int> &fk_links, const std::vector<int> &jac_links,
                     bool want_coll, bool want_stale, int jf_regs, Program &out, std::string &err) {
    const int L = m.n_links;
    for (int l : fk_links) if (l < 0 || l >= L) { err = "fk link id out of range"; return false; }
    for (int l : jac_links) if (l < 0 || l >= L) { err = "jacobian link id out of range"; return false; }

    // ---- dynamic nodes and the constant offset of every link to its dynamic ancestor ----
    std::vector<Node> nodes(1);
    nodes[0].link = -1; nodes[0].parent = -1; nodes[0].jtype = NODE_ROOT; nodes[0].qcol = -1;
    nodes[0].off = Xf::identity(); nodes[0].relmask = 0;
    nodes[0].axis[0] = nodes[0].axis[1] = nodes[0].axis[2] = 0;
    // Planar base (transform.jl:33-37: Trans(x, y, 0) * Rz(theta)) = three ordinary nodes under the root:
    // prismatic x, prismatic y, revolute z, driven by columns D, D+1, D+2.  Their Jacobian columns are
    // exactly the reference's base block (algorithm.jl:98-105): (1,0,0), (0,1,0), z x (p - base).
    int root_node = 0;
    if (m.with_base) {
        const double ax[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
        for (int k = 0; k < 3; ++k) {
            Node n;
            n.link = -1; n.parent = root_node; n.jtype = k < 2 ? 2 : 1; n.qcol = m.n_joints + k;
            n.off = Xf::identity();
            std::memcpy(n.axis, ax[k], sizeof n.axis);
            n.relmask = nodes[root_node].relmask | (1u << n.qcol);
            nodes[root_node].kids.push_back((int)nodes.size());
            root_node = (int)nodes.size();
            nodes.push_back(n);
        }
    }
    const unsigned base_mask = nodes[root_node].relmask;
    std::vector<int> node_of(L, 0);     // dynamic node each link hangs from
    std::vector<Xf> C(L);               // link = T_node * C
    for (int l : m.topo) {
        int p = m.parent[l];
        if (p < 0) { node_of[l] = root_node; C[l] = Xf::identity(); continue; }
        if (m.qidx[l] >= 0) {
            Node n;
            n.link = l; n.parent = node_of[p]; n.jtype = m.jtype[l]; n.qcol = m.qidx[l];
            n.off = C[p] * m.pose[l];
            std::memcpy(n.axis, &m.axis[3 * l], sizeof n.axis);
            n.relmask = m.relmask[l] | base_mask;
            nodes[n.parent].kids.push_back((int)nodes.size());
            node_of[l] = (int)nodes.size();
            nodes.push_back(n);
            C[l] = Xf::identity();
        } else {
            node_of[l] = node_of[p];
            C[l] = C[p] * frozen_joint_transform(m, l);
        }
    }

    // ---- attachments (requested links) ----
    std::vector<Att> atts;
    for (size_t i = 0; i < fk_links.size(); ++i) {
        Att a; a.node = node_of[fk_links[i]]; a.fk = (int)i; a.jac = -1; a.C = C[fk_links[i]]; a.flags = 0;
        atts.push_back(a);
    }
    for (size_t k = 0; k < jac_links.size(); ++k) {
        bool merged = false;
        for (size_t i = 0; i < fk_links.size() && !merged; ++i)
            if (fk_links[i] == jac_links[k] && atts[i].jac < 0) { atts[i].jac = (int)k; merged = true; }
        if (!merged) {
            Att a; a.node = node_of[jac_links[k]]; a.fk = -1; a.jac = (int)k; a.C = C[jac_links[k]]; a.flags = 0;
            atts.push_back(a);
        }
    }
    for (Att &a : atts) {
        if (is_identity3(a.C.r)) a.flags |= AF_R_IDENTITY;
        if (a.C.p[0] == 0.0 && a.C.p[1] == 0.0 && a.C.p[2] == 0.0) a.flags |= AF_T_ZERO;
        nodes[a.node].needed = true;
    }
    const int S = want_coll ? m.n_sph : 0;
    std::vector<int> sph_node(S);
    std::vector<double> sph_c(3 * (size_t)S);
    for (int s = 0; s < S; ++s) {
        sph_node[s] = node_of[m.sph_link[s]];
        C[m.sph_link[s]].apply(&m.sph_c[3 * s], &sph_c[3 * s]);
        nodes[sph_node[s]].needed = true;
    }
    // a node is needed if anything below it is
    for (int i = (int)nodes.size() - 1; i > 0; --i)
        if (nodes[i].needed) nodes[nodes[i].parent].needed = true;
    nodes[0].needed = true;

    // ---- DFS pre-order with stack-disciplined save slots ----
    std::vector<int> order;
    int max_slots = 0;
    std::function<void(int, int)> dfs = [&](int n, int depth) {
        order.push_back(n);
        std::vector<int> kids;
        for (int k : nodes[n].kids) if (nodes[k].needed) kids.push_back(k);
        int next = depth;
        if (kids.size() >= 2) { nodes[n].save_slot = depth; next = depth + 1; max_slots = std::max(max_slots, next); }
        for (size_t i = 0; i < kids.size(); ++i) {
            nodes[kids[i]].parent_src = (i == 0) ? PARENT_CUR : nodes[n].save_slot;
            dfs(kids[i], next);
        }
    };
    dfs(0, 0);
    const int NN = (int)order.size();
    std::vector<int> pos(nodes.size(), -1);
    for (int i = 0; i < NN; ++i) pos[order[i]] = i;

    // attachments and spheres grouped by node position
    std::vector<int> att_idx(atts.size());
    for (size_t i = 0; i < atts.size(); ++i) att_idx[i] = (int)i;
    std::stable_sort(att_idx.begin(), att_idx.end(), [&](int a, int b) { return pos[atts[a].node] < pos[atts[b].node]; });
    std::vector<int> sph_order(S);
    for (int s = 0; s < S; ++s) sph_order[s] = s;
    std::stable_sort(sph_order.begin(), sph_order.end(), [&](int a, int b) { return pos[sph_node[a]] < pos[sph_node[b]]; });

    // ---- emit ----
    ProgHeader &h = out.h;
    std::memset(&h, 0, sizeof h);
    h.n_nodes = NN; h.n_att = (int)atts.size(); h.n_sph = S; h.n_box = want_coll ? m.n_box : 0;
    h.n_joints = m.n_joints; h.with_base = m.with_base; h.n_dof = m.n_dof();
    h.n_fk = (int)fk_links.size(); h.n_jac = (int)jac_links.size();

    std::vector<int32_t> &I = out.ints;
    I.clear();
    h.io_node = 0;
    I.resize((size_t)NN * NODE_INTS, 0);
    h.io_att = (int)I.size();          I.resize(I.size() + (size_t)h.n_att * ATT_INTS, 0);
    h.io_sph_order = (int)I.size();    I.resize(I.size() + S, 0);
    h.io_sph_mask = (int)I.size();     I.resize(I.size() + S, 0);
    h.io_col_type = (int)I.size();     I.resize(I.size() + m.n_dof(), 0);
    while (I.size() % 4) I.push_back(0);
    h.n_int = (int)I.size();

    std::vector<double> &R = out.reals;
    R.clear();
    h.ro_node = 0;                     R.resize((size_t)NN * NODE_REALS, 0.0);
    h.ro_att = (int)R.size();          R.resize(R.size() + (size_t)h.n_att * ATT_REALS, 0.0);
    h.ro_sph = (int)R.size();          R.resize(R.size() + (size_t)S * SPH_REALS, 0.0);
    h.ro_box = (int)R.size();          R.resize(R.size() + (size_t)h.n_box * BOX_REALS, 0.0);
    while (R.size() % 2) R.push_back(0.0);
    h.n_real = (int)R.size();

    size_t a_cursor = 0, s_cursor = 0;
    for (int i = 0; i < NN; ++i) {
        const Node &n = nodes[order[i]];
        int32_t *ni = &I[h.io_node + (size_t)i * NODE_INTS];
        double *nr = &R[h.ro_node + (size_t)i * NODE_REALS];
        int flags = 0;
        if (is_identity3(n.off.r)) flags |= NF_OFF_R_IDENTITY;
        int code = 0;
        for (int k = 0; k < 3 && n.jtype != NODE_ROOT; ++k) {
            int u = (k + 1) % 3, v = (k + 2) % 3;
            if (n.axis[u] == 0.0 && n.axis[v] == 0.0) {
                if (n.axis[k] == 1.0) code = 1 + k;
                if (n.axis[k] == -1.0) code = 4 + k;
            }
        }
        flags |= code << NF_AXIS_SHIFT;
        ni[0] = n.parent_src; ni[1] = n.jtype; ni[2] = flags; ni[3] = n.qcol; ni[4] = n.save_slot;
        ni[5] = (int)a_cursor;
        while (a_cursor < att_idx.size() && pos[atts[att_idx[a_cursor]].node] == i) ++a_cursor;
        ni[6] = (int)a_cursor;
        ni[7] = (int)s_cursor;
        while (s_cursor < (size_t)S && pos[sph_node[sph_order[s_cursor]]] == i) ++s_cursor;
        ni[8] = (int)s_cursor;
        ni[9] = (int)n.relmask;
        std::memcpy(nr, n.off.r, sizeof(double) * 9);
        std::memcpy(nr + 9, n.off.p, sizeof(double) * 3);
        std::memcpy(nr + 12, n.axis, sizeof(double) * 3);
    }
    for (int k = 0; k < h.n_att; ++k) {
        const Att &a = atts[att_idx[k]];
        int32_t *ai = &I[h.io_att + (size_t)k * ATT_INTS];
        ai[0] = a.fk; ai[1] = a.flags; ai[2] = a.jac; ai[3] = (int)nodes[a.node].relmask;
        double *ar = &R[h.ro_att + (size_t)k * ATT_REALS];
        std::memcpy(ar, a.C.r, sizeof(double) * 9);
        std::memcpy(ar + 9, a.C.p, sizeof(double) * 3);
    }
    for (int s = 0; s < S; ++s) {
        I[h.io_sph_order + s] = sph_order[s];
        I[h.io_sph_mask + s] = (int)nodes[sph_node[s]].relmask;
        double *sr = &R[h.ro_sph + (size_t)s * SPH_REALS];
        sr[0] = sph_c[3 * s]; sr[1] = sph_c[3 * s + 1]; sr[2] = sph_c[3 * s + 2]; sr[3] = m.sph_r[s];
    }
    for (int l = 0; l < L; ++l)
        if (m.qidx[l] >= 0) I[h.io_col_type + m.qidx[l]] = m.jtype[l];
    if (m.with_base) { I[h.io_col_type + m.n_joints] = 2; I[h.io_col_type + m.n_joints + 1] = 2; I[h.io_col_type + m.n_joints + 2] = 1; }
    if (h.n_box > 0) emit_box_rows(m, &R[h.ro_box]);

    // ---- per-thread scratch map ----
    // so_q doubles as the per-group (dmin, argmin) hand-over of the collision phase: 2 * SPH_GROUP slots
    int so = 0;
    const int q_slots = std::max(std::max(h.n_dof, 1), S > 0 ? 8 : 0);
    h.so_q = so;      so += q_slots;
    h.so_q2 = so;     so += q_slots;
    h.so_save = so;   so += 12 * max_slots;
    h.so_jf = so;     so += (want_coll && jf_regs > 0 && h.n_dof <= jf_regs) ? 0 : 6 * h.n_dof;   // frames in registers: no slots
    h.so_cent = so;   so += 3 * S;
    h.so_stale = so;  so += (want_coll && want_stale) ? 3 * h.n_dof : 0;
    h.n_slots = so;
    return true;
}

}  // namespace kin
