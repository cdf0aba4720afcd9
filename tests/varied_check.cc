// TEST INFRASTRUCTURE: g++ build of the per-instance parameter expansion (trep_b200/csrc/trepb_varied.h), so that
// the map from (description, varied entries, row) to what the kernels read is pinned on a machine without a GPU.
#include "../trep_b200/csrc/trepb_varied.h"

using namespace trepb;

extern "C" {

// The expansion of one row: the specialised kernels' parameter slots (slots = 1) or the table-driven kernels' numeric
// region + grav (slots = 0).  Returns its length (-1: invalid description or entries), writes up to cap doubles.
int vc_expand(const trepb_sysdesc* d, int n, const int32_t* table, const int32_t* index, int slots, const double* row,
              double* out, int cap) {
    PackedSys P;
    std::string err;
    if (!pack_system(d, &P, &err) || !varied_check(P, n, table, index, &err)) return -1;
    VariedHost H;
    varied_map(P, n, table, index, slots != 0, &H);
    const VariedMap m = H.host_view();
    for (int i = 0; i < m.n_out && i < cap; ++i) out[i] = varied_value(m, row, i);
    return m.n_out;
}

// What packing a description gives: param_map(pack(d)).values (slots = 1), or the numeric region of pack(d).blob
// followed by grav (slots = 0).
int vc_packed(const trepb_sysdesc* d, int slots, double* out, int cap) {
    PackedSys P;
    std::string err;
    if (!pack_system(d, &P, &err)) return -1;
    std::vector<double> v;
    if (slots) {
        v = param_map(P).values;
    } else {
        const double* p = (const double*)(P.blob.data() + P.off[11]);
        v.assign(p, p + (P.off[18] - P.off[11]) / sizeof(double));
        for (int j = 0; j < 3; ++j) v.push_back(P.proto.grav[j]);
    }
    for (size_t i = 0; i < v.size() && (int)i < cap; ++i) out[i] = v[i];
    return (int)v.size();
}

}  // extern "C"
