// Per-instance physical parameters (trepb_*_varied_batch*): the override map and its expansion.
//
// A call varies n entries of the description (TREPB_PAR_* table, flat index); row r of `values` holds instance
// (or trajectory) r's numbers for them.  The kernels see the system through one vector of doubles per instance:
//   * specialised kernels: the kNPAR run-time parameter slots in trepb::param_map order (the Gravity sum re-formed);
//   * table-driven kernels: the numeric region of the packed blob (frame_value ... dpool, byte offsets as in the blob)
//     followed by grav[3].
// VariedMap says where each element of that vector comes from - the base description, a column of the row, or a
// Gravity sum - so that element i is a pure function of (map, row, i).  The specialised kernels evaluate it with
// compile-time i straight into sys.par (no run-time-indexed register array), the table-driven kernels into a
// per-thread slot of global scratch, and the host into a vector that must equal re-packing the description
// rebuilt with the row's numbers, byte for byte (tests/test_varied_params.py).
#pragma once
#include <stdint.h>
#include "trepb_sys.h"

namespace trepb {

struct VariedMap {
    int n_out;             // elements of the expanded vector
    int n;                 // columns of a row (varied entries)
    int ngp;               // Gravity potentials
    int toff[8];           // table-driven: offsets (doubles) of frame_value, frame_se3, frame_mass, pot_d, force_d,
                           // con_d, dpool and grav in the expanded vector
    const int* src;        // [n_out] >= 0: row column; -1: base[i]; -2 - j: Gravity sum component j
    const double* base;    // [n_out]
    const int* gcol;       // [ngp][3] row column of that Gravity potential's component, or -1: gbase
    const double* gbase;   // [ngp][3]
};

// What a varied launch hands the kernels besides their usual parameters.
struct VariedArgs {
    VariedMap map;
    const double* values;  // [rows][map.n]
    double* slots;         // table-driven: [threads of the grid][map.n_out] scratch; specialised: unused
};

// Element i of the expanded vector for one row.  The Gravity sum is formed in potential order from 0, as
// pack_system forms grav[].
TREPB_HD double varied_value(const VariedMap& m, const double* row, int i) {
    const int s = m.src[i];
    if (s >= 0) return row[s];
    if (s == -1) return m.base[i];
    const int j = -2 - s;
    double g = 0.0;
    for (int k = 0; k < m.ngp; ++k) {
        const int c = m.gcol[3 * k + j];
        g += c >= 0 ? row[c] : m.gbase[3 * k + j];
    }
    return g;
}

// Element i of the expanded vector for one row, as a function object (the cooperative kernels' plan evaluation,
// trepb_coop_sys.h, reads the elements it needs without expanding the whole vector).
struct VariedX {
    VariedMap m;
    const double* row;
    TREPB_HD double operator()(int i) const { return varied_value(m, row, i); }
};

// Table-driven: expand one row into `slot` and point the numeric tables of `sys` at it (the integer tables stay
// where they are, e.g. in the CTA's shared-memory copy of the blob).
TREPB_HD void varied_point(RtSys& sys, const VariedMap& m, const double* row, double* slot) {
    for (int i = 0; i < m.n_out; ++i) slot[i] = varied_value(m, row, i);
    sys.frame_value = slot + m.toff[0];
    sys.frame_se3 = slot + m.toff[1];
    sys.frame_mass = slot + m.toff[2];
    sys.pot_d_ = slot + m.toff[3];
    sys.force_d_ = slot + m.toff[4];
    sys.con_d_ = slot + m.toff[5];
    sys.dpool_ = slot + m.toff[6];
    for (int j = 0; j < 3; ++j) sys.grav[j] = slot[m.toff[7] + j];
}

}  // namespace trepb

#include <string>
#include <vector>
#include "trepb_codegen.h"

namespace trepb {

// Host side of a map: arrays behind VariedMap's pointers.
struct VariedHost {
    int n_out = 0, n = 0, ngp = 0;
    int toff[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    std::vector<int> src, gcol;
    std::vector<double> base, gbase;
    VariedMap view(const int* dsrc, const double* dbase, const int* dgcol, const double* dgbase) const {
        VariedMap m;
        m.n_out = n_out; m.n = n; m.ngp = ngp;
        for (int k = 0; k < 8; ++k) m.toff[k] = toff[k];
        m.src = dsrc; m.base = dbase; m.gcol = dgcol; m.gbase = dgbase;
        return m;
    }
    VariedMap host_view() const { return view(src.data(), base.data(), gcol.data(), gbase.data()); }
};

inline const char* varied_table_name(int t) {
    static const char* names[7] = {"FRAME_VALUE", "FRAME_SE3", "FRAME_MASS", "POT_D", "FORCE_D", "CON_D", "DPOOL"};
    return t >= 0 && t < 7 ? names[t] : "?";
}

// Which entries may vary: the run-time parameter slots of param_map (non-zero, and not +-1 in frame_se3), minus the
// spline x-points of a NonlinearConfigSpring (they must increase) and the components of Gravity potentials whose sum
// over all Gravity potentials is exactly 0 (that sum is structure).  No entry may be named twice.
inline bool varied_check(const PackedSys& P, int n, const int32_t* table, const int32_t* index, std::string* err) {
    auto fail = [&](int k, const std::string& why) {
        *err = "varied entry " + std::to_string(k) + " (" + varied_table_name(table[k]) + "[" +
               std::to_string(index[k]) + "]): " + why;
        return false;
    };
    if (n < 0) { *err = "varied: n must be >= 0"; return false; }
    if (n > 0 && (!table || !index)) { *err = "varied: table and index are required"; return false; }
    const RtSys s = P.view(P.blob.data());
    const ParamMap M = param_map(P);
    std::vector<std::vector<char>> seen(7);
    for (int t = 0; t < 7; ++t) seen[t].assign(M.slot[t].size(), 0);
    for (int k = 0; k < n; ++k) {
        const int t = table[k], i = index[k];
        if (t < 0 || t > 6) return fail(k, "unknown table (TREPB_PAR_FRAME_VALUE ... TREPB_PAR_DPOOL)");
        if (i < 0 || i >= (int)M.slot[t].size())
            return fail(k, "index out of range (the table has " + std::to_string(M.slot[t].size()) + " entries)");
        if (seen[t][i]) return fail(k, "named more than once");
        seen[t][i] = 1;
        const int sl = M.slot[t][i];
        if (sl == -1) return fail(k, "the description's value is 0, which is structure (it folds away in the specialised kernels and in trepb_struct_hash); only non-zero entries can vary");
        if (sl < -1) return fail(k, "the description's value is +-1 in a CONST_SE3 transform, which is structure; only other entries can vary");
        if (t == TREPB_PAR_DPOOL)
            for (int p = 0; p < s.npot; ++p)
                if (s.pot_kind(p) == P_NONLINEAR_CONFIG_SPRING && i >= s.pot_i(p, 1) && i < s.pot_i(p, 1) + s.pot_i(p, 2))
                    return fail(k, "a spline x-point of a NonlinearConfigSpring (they must increase); its coefficients can vary");
        if (t == TREPB_PAR_POT_D && s.pot_kind(i / 4) == P_GRAVITY && i % 4 < 3 && M.slot[PT_GRAV][i % 4] < 0)
            return fail(k, "a Gravity component whose sum over all Gravity potentials is 0, which is structure");
    }
    return true;
}

// Builds the map for a checked entry list.  slots = true: the specialised kernels' parameter vector; false: the
// table-driven kernels' numeric region + grav.
inline void varied_map(const PackedSys& P, int n, const int32_t* table, const int32_t* index, bool slots, VariedHost* out) {
    VariedHost& H = *out;
    const RtSys s = P.view(P.blob.data());
    const ParamMap M = param_map(P);
    H.n = n;
    int gpos[3];
    if (slots) {
        H.n_out = (int)M.values.size();
        H.base = M.values;
        for (int j = 0; j < 3; ++j) gpos[j] = M.slot[PT_GRAV][j];
    } else {
        const size_t o0 = P.off[11];
        const int nnum = (int)((P.off[18] - o0) / sizeof(double));
        for (int t = 0; t < 7; ++t) H.toff[t] = (int)((P.off[11 + t] - o0) / sizeof(double));
        H.toff[7] = nnum;
        H.n_out = nnum + 3;
        H.base.resize(H.n_out);
        for (int i = 0; i < nnum; ++i) H.base[i] = ((const double*)(P.blob.data() + o0))[i];
        for (int j = 0; j < 3; ++j) { H.base[nnum + j] = s.grav[j]; gpos[j] = nnum + j; }
    }
    H.src.assign(H.n_out, -1);
    bool grav_varied = false;
    for (int k = 0; k < n; ++k) {
        const int t = table[k], i = index[k];
        H.src[slots ? M.slot[t][i] : H.toff[t] + i] = k;
        if (t == TREPB_PAR_POT_D && s.pot_kind(i / 4) == P_GRAVITY && i % 4 < 3) grav_varied = true;
    }
    H.ngp = 0;
    H.gcol.clear(); H.gbase.clear();
    if (!grav_varied) return;
    for (int p = 0; p < s.npot; ++p) {
        if (s.pot_kind(p) != P_GRAVITY) continue;
        ++H.ngp;
        for (int j = 0; j < 3; ++j) {
            int c = -1;
            for (int k = 0; k < n; ++k)
                if (table[k] == TREPB_PAR_POT_D && index[k] == 4 * p + j) c = k;
            H.gcol.push_back(c);
            H.gbase.push_back(s.pot_d(p, j));
        }
    }
    for (int j = 0; j < 3; ++j)
        if (gpos[j] >= 0) H.src[gpos[j]] = -2 - j;
}

}  // namespace trepb
