// lattice.cuh -- device-side view of a finished pnp_lattice, shared by lattice.cu and crf.cu.
#pragma once
#include "common.cuh"

namespace pnp {

struct LatticeView {
    const int32_t *offset;   // [n_lp, D+1]
    const float *bary;       // [n_lp, D+1]
    const int32_t *nbr;      // [D+1, vertex_stride, 2]
    const int32_t *row_ptr;  // [M+1]
    const int32_t *csr_pix;  // [n_entries]
    const float *csr_w;      // [n_entries]
    const float *csr_norm;   // [n_entries] norm[csr_pix[k]]
    const float *norm;       // [n_lp]
    int Dp1;                 // d + 1
    int M;                   // vertices
    int vertex_stride;
    int shared;              // 1: one image's lattice applied to every image
    int N;                   // pixels per image
    float alpha;             // 1 / (1 + 2^-d)
    int vp;                  // floats between consecutive rows of a vertex-value buffer (= Cp; set per call by view_for)
};

static inline LatticeView make_view(const pnp_lattice *lat) {
    LatticeView v;
    v.offset = lat->offset;
    v.bary = lat->bary;
    v.nbr = lat->nbr;
    v.row_ptr = lat->row_ptr;
    v.csr_pix = lat->csr_pix;
    v.csr_w = lat->csr_w;
    v.csr_norm = lat->csr_norm;
    v.norm = lat->norm;
    v.Dp1 = lat->d + 1;
    v.M = lat->n_vertices;
    v.vertex_stride = lat->vertex_stride;
    v.shared = lat->shared;
    v.N = lat->n_pixels;
    v.alpha = 1.0f / (1 + powf(2, -lat->d));
    v.vp = 0;
    return v;
}

}  // namespace pnp
