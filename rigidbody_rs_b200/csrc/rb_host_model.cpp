// rb_host_model.cpp -- see rb_host_model.h.  Plain C++17, no CUDA.
#include "rb_host_model.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>

namespace {

// ------------------------------------------------------------------ a very small XML reader
// Enough for URDF: elements, attributes, comments, declarations.  No entities, no CDATA.
struct XmlNode {
    std::string tag;
    std::map<std::string, std::string> attr;
    std::vector<XmlNode> kids;
    const XmlNode* child(const char* t) const {
        for (const auto& k : kids) if (k.tag == t) return &k;
        return nullptr;
    }
    const char* get(const char* a) const {
        auto it = attr.find(a);
        return it == attr.end() ? nullptr : it->second.c_str();
    }
};

struct XmlParser {
    const std::string& s;
    size_t i = 0;
    std::string err;
    explicit XmlParser(const std::string& src) : s(src) {}

    void skip_ws() { while (i < s.size() && isspace((unsigned char)s[i])) ++i; }
    bool starts(const char* lit) const { return s.compare(i, strlen(lit), lit) == 0; }

    // Skips text, comments, <? ?> and <! > until the next real tag.  Returns false at end of input.
    bool next_tag() {
        while (i < s.size()) {
            size_t lt = s.find('<', i);
            if (lt == std::string::npos) { i = s.size(); return false; }
            i = lt;
            if (starts("<!--")) {
                size_t e = s.find("-->", i + 4);
                if (e == std::string::npos) { err = "unterminated comment"; return false; }
                i = e + 3;
            } else if (starts("<?")) {
                size_t e = s.find("?>", i + 2);
                if (e == std::string::npos) { err = "unterminated declaration"; return false; }
                i = e + 2;
            } else if (starts("<!")) {
                size_t e = s.find('>', i + 2);
                if (e == std::string::npos) { err = "unterminated <!"; return false; }
                i = e + 1;
            } else {
                return true;
            }
        }
        return false;
    }

    static bool name_char(char c) { return isalnum((unsigned char)c) || c == '_' || c == '-' || c == ':' || c == '.'; }

    // Parses the element starting at s[i] == '<'.  On return i is just past its end tag.
    bool element(XmlNode& out) {
        ++i;  // '<'
        size_t b = i;
        while (i < s.size() && name_char(s[i])) ++i;
        out.tag = s.substr(b, i - b);
        if (out.tag.empty()) { err = "empty tag name"; return false; }
        for (;;) {
            skip_ws();
            if (i >= s.size()) { err = "unterminated tag <" + out.tag; return false; }
            if (s[i] == '/') {
                if (i + 1 < s.size() && s[i + 1] == '>') { i += 2; return true; }
                err = "stray '/' in <" + out.tag; return false;
            }
            if (s[i] == '>') { ++i; break; }
            size_t ab = i;
            while (i < s.size() && name_char(s[i])) ++i;
            std::string an = s.substr(ab, i - ab);
            skip_ws();
            if (an.empty() || i >= s.size() || s[i] != '=') { err = "bad attribute in <" + out.tag; return false; }
            ++i; skip_ws();
            if (i >= s.size() || (s[i] != '"' && s[i] != '\'')) { err = "unquoted attribute in <" + out.tag; return false; }
            char qc = s[i++];
            size_t vb = i;
            while (i < s.size() && s[i] != qc) ++i;
            if (i >= s.size()) { err = "unterminated attribute value in <" + out.tag; return false; }
            out.attr[an] = s.substr(vb, i - vb);
            ++i;
        }
        // children until </tag>
        for (;;) {
            if (!next_tag()) { if (err.empty()) err = "missing </" + out.tag + ">"; return false; }
            if (s[i + 1] == '/') {
                size_t e = s.find('>', i);
                if (e == std::string::npos) { err = "unterminated end tag"; return false; }
                std::string en = s.substr(i + 2, e - i - 2);
                while (!en.empty() && isspace((unsigned char)en.back())) en.pop_back();
                if (en != out.tag) { err = "mismatched </" + en + "> for <" + out.tag + ">"; return false; }
                i = e + 1;
                return true;
            }
            XmlNode k;
            if (!element(k)) return false;
            out.kids.push_back(std::move(k));
        }
    }
};

bool parse_floats(const char* s, int n, double* out) {
    if (!s) { for (int k = 0; k < n; ++k) out[k] = 0.0; return true; }   // xurdf: missing attribute -> zeros
    const char* p = s;
    for (int k = 0; k < n; ++k) {
        char* e = nullptr;
        out[k] = strtod(p, &e);
        if (e == p) return false;
        p = e;
    }
    while (*p && isspace((unsigned char)*p)) ++p;
    return *p == 0;
}

double snap(double x) {
    // A roll of +-pi/2 in fp64 leaves cos = 6.1e-17 instead of 0 (and the reference's quaternion round trip
    // leaves ~2e-16): treat entries within 2^-50 of 0 / +-1 as exact so the specialised kernels can drop them.
    const double eps = 8.881784197001252e-16;
    if (std::fabs(x) < eps) return 0.0;
    if (std::fabs(x - 1.0) < eps) return 1.0;
    if (std::fabs(x + 1.0) < eps) return -1.0;
    return x;
}

void finish_model(RbHostModel& m) {
    // composite (sub-tree) masses, leaves to base (multibody.rs:157,170: masses only ever add)
    m.serial = true;
    for (int i = 0; i < m.n; ++i) { m.jt[i].mc = m.jt[i].m; m.serial = m.serial && (int)m.jt[i].parent == i - 1; }
    for (int i = m.n - 1; i >= 0; --i) {
        const int p = (int)m.jt[i].parent;
        if (p >= 0) m.jt[p].mc += m.jt[i].mc;
    }
}

// I_o = I_c + m [c]x [c]x^T  (inertia.rs:31-32), six unique entries
void origin_inertia(double mass, const double c[3], const double Ic[9], double I6[6]) {
    const double cx = c[0], cy = c[1], cz = c[2];
    // [c]x [c]x^T = (c.c) Id - c c^T
    const double cc = cx * cx + cy * cy + cz * cz;
    I6[0] = Ic[0] + mass * (cc - cx * cx);
    I6[1] = Ic[1] + mass * (-cx * cy);
    I6[2] = Ic[2] + mass * (-cx * cz);
    I6[3] = Ic[4] + mass * (cc - cy * cy);
    I6[4] = Ic[5] + mass * (-cy * cz);
    I6[5] = Ic[8] + mass * (cc - cz * cz);
}

using RawJoint = RbRawJoint;

void mat3_mul(const double A[9], const double B[9], double C[9]) {
    double T[9];
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) T[3 * r + c] = A[3 * r] * B[c] + A[3 * r + 1] * B[3 + c] + A[3 * r + 2] * B[6 + c];
    memcpy(C, T, sizeof T);
}
void mat3_t(const double A[9], double T[9]) {
    const double B[9] = {A[0], A[3], A[6], A[1], A[4], A[7], A[2], A[5], A[8]};
    memcpy(T, B, sizeof B);
}
void mat3_vec(const double A[9], const double v[3], double o[3]) {
    const double x = A[0] * v[0] + A[1] * v[1] + A[2] * v[2], y = A[3] * v[0] + A[4] * v[1] + A[5] * v[2],
                 z = A[6] * v[0] + A[7] * v[1] + A[8] * v[2];
    o[0] = x; o[1] = y; o[2] = z;
}

// The kernels rotate every joint about its frame's z axis, as the reference's rnea / crba do (multibody.rs:29,130).
// A joint whose axis a is not +z (the reference would silently mis-handle it: joint_transform uses the axis,
// joint.rs:48-50, the dynamics do not) is re-based: its frame is rotated by Q with Q z = a, so Rot(a, q) = Q Rz(q) Q^T
// and everything attached to that frame (link inertia, the next joint's placement) is re-expressed in the rotated
// frame.  tau, qdd, H and the tip position are invariant; the tip-frame Jacobian needs the last Q back (model.tip).
int build_model(const std::vector<RawJoint>& raw, RbHostModel& out, std::string& err) {
    out.raw = raw;
    std::vector<double> Qs(raw.size() * 9);
    std::vector<char> Qid(raw.size());
    for (size_t i = 0; i < raw.size(); ++i) {
        const RawJoint& j = raw[i];
        if (j.parent < -1 || j.parent >= (int)i) { err = "parent[i] must be -1 (base) or an earlier joint (topological order)"; return RB_ERR_ARG; }
        const double Id[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        const double* Qprev = j.parent >= 0 ? &Qs[(size_t)j.parent * 9] : Id;
        const bool prev_identity = j.parent >= 0 ? (bool)Qid[j.parent] : true;
        const double an = std::sqrt(j.axis[0] * j.axis[0] + j.axis[1] * j.axis[1] + j.axis[2] * j.axis[2]);
        if (!(an > 0.0) || !std::isfinite(an)) { err = "joint axis must be a non-zero finite vector"; return RB_ERR_ARG; }
        const double a[3] = {j.axis[0] / an, j.axis[1] / an, j.axis[2] / an};       // UnitVector3::new_normalize (joint.rs:56)
        double Q[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
        const bool identity = std::fabs(a[0]) < 1e-12 && std::fabs(a[1]) < 1e-12 && a[2] > 0.0;
        if (!identity) {
            if (a[2] < -1.0 + 1e-12) {
                const double F[9] = {1, 0, 0, 0, -1, 0, 0, 0, -1};                   // z -> -z: half turn about x
                memcpy(Q, F, sizeof F);
            } else {
                // minimal rotation taking z to a:  Q = I + [v]x + [v]x^2 / (1 + c),  v = z x a,  c = z . a
                const double vx = -a[1], vy = a[0], c = a[2], k = 1.0 / (1.0 + c);
                const double F[9] = {1.0 - k * vy * vy, k * vx * vy,       vy,
                                     k * vx * vy,       1.0 - k * vx * vx, -vx,
                                     -vy,               vx,                1.0 - k * (vx * vx + vy * vy)};
                memcpy(Q, F, sizeof F);
            }
        }
        RbJointK r{};
        double R[9], t[3], com[3], Ic[9];
        memcpy(R, j.R, sizeof R); memcpy(t, j.t, sizeof t); memcpy(com, j.com, sizeof com); memcpy(Ic, j.Ic, sizeof Ic);
        if (!prev_identity) {                       // placement re-expressed in the re-based parent frame
            double Qt[9]; mat3_t(Qprev, Qt);
            mat3_mul(Qt, R, R);
            mat3_vec(Qt, t, t);
        }
        if (!identity) {                            // child frame re-based: link inertia follows
            double Qt[9]; mat3_t(Q, Qt);
            mat3_mul(R, Q, R);
            mat3_vec(Qt, com, com);
            mat3_mul(Qt, Ic, Ic); mat3_mul(Ic, Q, Ic);
        }
        for (int e = 0; e < 9; ++e) r.R[e] = snap(R[e]);
        for (int e = 0; e < 3; ++e) r.t[e] = t[e];
        r.m = j.mass;
        for (int e = 0; e < 3; ++e) r.h[e] = j.mass * com[e];
        origin_inertia(j.mass, com, Ic, r.I);                                        // joint.rs:66
        r.parent = (double)j.parent;
        out.jt.push_back(r);
        memcpy(&Qs[i * 9], Q, sizeof Q);
        Qid[i] = identity;
    }
    out.link_rot.assign(raw.size() * 9, 0.0);       // the original frames seen from the re-based ones
    for (size_t i = 0; i < raw.size(); ++i) {
        mat3_t(&Qs[i * 9], &out.link_rot[i * 9]);
        for (int e = 0; e < 9; ++e) out.link_rot[i * 9 + e] = snap(out.link_rot[i * 9 + e]);
    }
    memcpy(out.tip, &out.link_rot[(raw.size() - 1) * 9], sizeof out.tip);
    out.n = (int)raw.size();
    finish_model(out);
    return RB_OK;
}

}  // namespace

int rb_model_from_urdf(const char* path, RbHostModel& out, std::string& err) {
    if (!path) { err = "urdf path is NULL"; return RB_ERR_NULL; }
    std::ifstream f(path, std::ios::binary);
    if (!f) { err = std::string("cannot open URDF '") + path + "'"; return RB_ERR_URDF; }
    std::stringstream ss; ss << f.rdbuf();
    const std::string src = ss.str();
    XmlParser xp(src);
    XmlNode robot;
    bool found = false;
    while (xp.next_tag()) {
        XmlNode n;
        if (!xp.element(n)) { err = "URDF parse error: " + xp.err; return RB_ERR_URDF; }
        if (n.tag == "robot") { robot = std::move(n); found = true; break; }
    }
    if (!found) { err = xp.err.empty() ? "no <robot> element" : "URDF parse error: " + xp.err; return RB_ERR_URDF; }

    // xurdf: `links` and `joints` are the <robot>'s direct children in document order
    struct L { double mass = 0.0, com[3] = {0, 0, 0}, six[6] = {0, 0, 0, 0, 0, 0}; };
    struct J { std::string name, type; double xyz[3], rpy[3], axis[3], lim[4]; };
    std::vector<L> links; std::vector<J> joints;
    for (const auto& el : robot.kids) {
        if (el.tag == "link") {
            L l;
            if (const XmlNode* in = el.child("inertial")) {
                const XmlNode* o = in->child("origin");
                const XmlNode* ms = in->child("mass");
                const XmlNode* ie = in->child("inertia");
                if (!parse_floats(o ? o->get("xyz") : nullptr, 3, l.com)) { err = "bad inertial origin"; return RB_ERR_URDF; }
                if (!ms || !ms->get("value") || !parse_floats(ms->get("value"), 1, &l.mass)) { err = "bad <mass>"; return RB_ERR_URDF; }
                static const char* keys[6] = {"ixx", "ixy", "ixz", "iyy", "iyz", "izz"};
                for (int k = 0; k < 6; ++k)
                    if (!ie || !ie->get(keys[k]) || !parse_floats(ie->get(keys[k]), 1, &l.six[k])) { err = "bad <inertia>"; return RB_ERR_URDF; }
            }
            links.push_back(l);
        } else if (el.tag == "joint") {
            J j;
            j.name = el.get("name") ? el.get("name") : "";
            j.type = el.get("type") ? el.get("type") : "";
            const XmlNode* o = el.child("origin");
            const XmlNode* a = el.child("axis");
            const XmlNode* lm = el.child("limit");
            if (!parse_floats(o ? o->get("xyz") : nullptr, 3, j.xyz) || !parse_floats(o ? o->get("rpy") : nullptr, 3, j.rpy)) {
                err = "bad joint origin in '" + j.name + "'"; return RB_ERR_URDF;
            }
            j.axis[0] = 1.0; j.axis[1] = 0.0; j.axis[2] = 0.0;
            if (a && a->get("xyz") && !parse_floats(a->get("xyz"), 3, j.axis)) { err = "bad joint axis in '" + j.name + "'"; return RB_ERR_URDF; }
            static const char* lk[4] = {"lower", "upper", "velocity", "effort"};
            for (int k = 0; k < 4; ++k) { j.lim[k] = 0.0; if (lm && lm->get(lk[k])) parse_floats(lm->get(lk[k]), 1, &j.lim[k]); }
            joints.push_back(j);
        }
    }

    out = RbHostModel();
    std::vector<RawJoint> raw;
    const size_t pairs = std::min(links.size(), joints.size());          // zip (multibody.rs:70)
    for (size_t k = 0; k < pairs; ++k) {
        const J& j = joints[k];
        const L& l = links[k];
        if (j.type.find("fixed") != std::string::npos) continue;          // multibody.rs:71
        if (raw.size() >= RB_MAX_JOINTS) { err = "more than RB_MAX_JOINTS movable joints"; return RB_ERR_UNSUPPORTED; }
        RawJoint r{};
        memcpy(r.axis, j.axis, sizeof r.axis);
        r.parent = (int)raw.size() - 1;                                   // serial: f[i-1] (multibody.rs:148)
        // Rotation3::from_euler_angles(roll, pitch, yaw) = Rz(yaw) Ry(pitch) Rx(roll)   (joint.rs:59-63)
        const double sr = std::sin(j.rpy[0]), cr = std::cos(j.rpy[0]);
        const double sp = std::sin(j.rpy[1]), cp = std::cos(j.rpy[1]);
        const double sy = std::sin(j.rpy[2]), cy = std::cos(j.rpy[2]);
        const double R[9] = {cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr,
                             sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr,
                             -sp,     cp * sr,                cp * cr};
        memcpy(r.R, R, sizeof R);
        memcpy(r.t, j.xyz, sizeof r.t);
        r.mass = l.mass;
        memcpy(r.com, l.com, sizeof r.com);
        const double Ic[9] = {l.six[0], l.six[1], l.six[2], l.six[1], l.six[3], l.six[4], l.six[2], l.six[4], l.six[5]};
        memcpy(r.Ic, Ic, sizeof Ic);
        raw.push_back(r);
        const int i = (int)raw.size() - 1;
        out.lim.lower[i] = j.lim[0]; out.lim.upper[i] = j.lim[1];
        out.lim.velocity[i] = j.lim[2]; out.lim.effort[i] = j.lim[3];
        out.names.push_back(j.name);
    }
    if (raw.empty()) { err = "URDF holds no movable joint"; return RB_ERR_URDF; }
    return build_model(raw, out, err);
}

int rb_model_from_desc(const RbChainDesc* d, RbHostModel& out, std::string& err) {
    if (!d) { err = "descriptor is NULL"; return RB_ERR_NULL; }
    if (d->n_joints < 1) { err = "n_joints must be >= 1"; return RB_ERR_ARG; }
    if (d->n_joints > RB_MAX_JOINTS) { err = "n_joints exceeds RB_MAX_JOINTS"; return RB_ERR_UNSUPPORTED; }
    if (!d->parent_rot || !d->parent_trans || !d->mass || !d->com || !d->inertia_com) {
        err = "descriptor array is NULL"; return RB_ERR_NULL;
    }
    out = RbHostModel();
    std::vector<RawJoint> raw;
    for (int i = 0; i < d->n_joints; ++i) {
        RawJoint r{};
        r.parent = d->parent ? d->parent[i] : i - 1;
        r.axis[0] = 0.0; r.axis[1] = 0.0; r.axis[2] = 1.0;
        if (d->axis) memcpy(r.axis, d->axis + 3 * i, sizeof r.axis);
        const double* R = d->parent_rot + 9 * i;
        // must be a rotation: R R^T = Id within 1e-9
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) {
                double dot = 0.0;
                for (int k = 0; k < 3; ++k) dot += R[3 * a + k] * R[3 * b + k];
                if (!(std::fabs(dot - (a == b ? 1.0 : 0.0)) < 1e-9)) { err = "parent_rot is not a rotation matrix"; return RB_ERR_ARG; }
            }
        memcpy(r.R, R, sizeof r.R);
        memcpy(r.t, d->parent_trans + 3 * i, sizeof r.t);
        r.mass = d->mass[i];
        if (!(r.mass > 0.0) || !std::isfinite(r.mass)) { err = "link mass must be positive and finite"; return RB_ERR_ARG; }
        memcpy(r.com, d->com + 3 * i, sizeof r.com);
        memcpy(r.Ic, d->inertia_com + 9 * i, sizeof r.Ic);
        raw.push_back(r);
        out.lim.lower[i] = -3.141592653589793; out.lim.upper[i] = 3.141592653589793;
        out.lim.velocity[i] = 2.0; out.lim.effort[i] = 50.0;
        out.names.push_back("joint" + std::to_string(i + 1));
    }
    for (int k = 0; k < 3; ++k) {
        if (!std::isfinite(d->gravity[k])) { err = "gravity must be finite"; return RB_ERR_ARG; }
        out.g[k] = d->gravity[k];
    }
    return build_model(raw, out, err);
}

std::vector<double> rb_model_flat(const RbHostModel& m) {
    std::vector<double> v((size_t)RB_MODEL_DOUBLES(m.n));
    static_assert(sizeof(RbJointK) == 24 * sizeof(double), "RbJointK must be 24 doubles");
    memcpy(v.data(), m.jt.data(), (size_t)m.n * sizeof(RbJointK));
    for (int k = 0; k < 3; ++k) v[(size_t)m.n * 24 + k] = m.g[k];
    for (int k = 0; k < 9; ++k) v[(size_t)m.n * 24 + 3 + k] = m.tip[k];
    return v;
}

std::string rb_model_emit_header(const RbHostModel& m, const char* tab_name) {
    std::vector<double> flat = rb_model_flat(m);
    std::string o;
    char buf[96];
    o += "// generated by rb_modelgen -- do not edit\n#pragma once\n";
    o += std::string("struct ") + tab_name + " {\n";
    snprintf(buf, sizeof buf, "    static constexpr int N = %d;\n", m.n); o += buf;
    o += "    static constexpr double T[N][24] = {\n";
    for (int i = 0; i < m.n; ++i) {
        o += "        {";
        for (int k = 0; k < 24; ++k) {
            snprintf(buf, sizeof buf, "%a%s", flat[(size_t)i * 24 + k], k == 23 ? "" : ", "); o += buf;
        }
        o += "},\n";
    }
    o += "    };\n";
    snprintf(buf, sizeof buf, "    static constexpr double G[3] = {%a, %a, %a};\n", m.g[0], m.g[1], m.g[2]); o += buf;
    o += "    static constexpr double TIP[9] = {";
    for (int k = 0; k < 9; ++k) { snprintf(buf, sizeof buf, "%a%s", m.tip[k], k == 8 ? "};\n" : ", "); o += buf; }
    o += "};\n";
    return o;
}
