// Workspace layout + internal declarations of the fusion head (forward_tri_modal fwd/bwd).
// See DESIGN.md section 3 for the algorithm (tests/factorised_model.py is its executable spec).
#pragma once
#include "common.cuh"
#include "gemm.cuh"

namespace team {

struct HeadDims {
    int B;      // samples
    int B2;     // own rows = image rows [0,B) + text rows [B,2B)
    int C;      // classes (prototype rows)
    int P;      // prompt rows
    int M;      // shared key rows = C + P
    int Ns;     // step rows = M + 10 state-table rows
    int Nsp;    // Ns rounded up to 16 (leading dimension of all [.,Ns] matrices)
    int Rt;     // table-query rows = C + 10
    int Tc;     // text-class rows for the classification logits (0 = none)
    int nctas;  // CTAs of the per-sample reduction kernels (size of the partial buffers)
};

constexpr int OWN_PARTIAL_LEN = 3 * D;   // dgamma, dbeta, dbfc of the own rows
constexpr int NRM_MAX_PARTIALS = 64;     // per-segment column-sum partials of nrm_bwd (bias gradients)

// Every GEMM operand of the head is a Mat (gemm.cuh).
struct HeadWS {
    // ---- step level
    Mat Wsum[3];                      // [D][D] summed projections img/text/state
    float* bsum[3];
    Mat Wqkv;                         // [3D][D] packed {Wq;Wk;Wv}
    Mat Wfc;                          // f = caller's w_fc
    Mat protos, E, img, txt, tcls;    // caller's inputs (f) + bf16 shadows
    float* Zc;                        // [Tc][D] encode_text(text_cls), pre-normalisation
    float* Ztab;                      // [Rt][D] pre-normalisation proto/state rows
    Mat S;                            // [Nsp][D] step rows
    float* invS;                      // [Nsp] inverse norms (proto + state rows)
    Mat QKVs;                         // [Nsp][3D]
    Mat VFs;                          // [Nsp + 64][D]: VF rows of the step, then the table rows s and n of the Gram formulation
    float* TT;                        // [Nsp][Nsp]
    float *mt, *Zt;                   // [Nsp]
    Mat Pt;                           // [Nsp][Nsp]
    float* NFt;                       // [Nsp][D]
    // ---- per sample
    Mat Xo;                           // [B2][D]
    float* invo;                      // [B2]
    Mat QKVo;                         // [B2][3D]
    Mat VFo;                          // [B2][D]
    Mat SQ;                           // [B2][Nsp]  scores of own queries; backward: dA then dS in place
    float* SK;                        // [B2][Nsp]
    Mat Aext;                         // [B2][Nsp]
    float* aown;                      // [B2][2]
    float* Ybo;                       // [B2][D]
    // ---- backward scratch
    Mat dYo;                          // [B2][D]
    float* rowdot;                    // [B2]
    float* dsown;                     // [B2][2]
    Mat dSK;                          // [B2][Nsp]
    Mat dVFo;                         // [B2][D]
    float* dVFo_own;                  // [B2][D]   own-row part (ln_own_bwd), summed into dVFo by add_rows_kernel
    Mat dQKVo;                        // [B2][3D]
    Mat dXo;                          // [B2][D]   du_o, then + dQKV Wqkv, then dz in place
    float* Rfull;                     // [Nsp][D]  residual gradient of the step rows, then + dQKVs Wqkv
    Mat Gfull;                        // [Nsp][D]
    float* hfull;                     // [Nsp]
    Mat dTT;                          // [Nsp][Nsp]
    float* tmpNN;                     // [Nsp][Nsp]
    Mat dVFs;                         // [Nsp][D]
    Mat dQKVs;                        // [Nsp][3D]
    Mat dZtab;                        // [Rt][D]
    Mat GG;                           // [B2][D]   table-row cotangents .* gamma: rows [0,B) g_proto/C, rows [B,2B) g_state
    Mat A1, A23;                      // [B2][ldA] coefficient matrices of the R/G GEMM (see table_rows_bwd_kernel)
    float* RG;                        // [ldA][D]  A1^T GG + A23^T VFo
    float* dVFs_a;                    // [Nsp][D]  Aext^T dYo
    float* dbfc_parts;                // [8][D]
    int ldA;                          // 2 * round_up(Rt, 64)
    float* tab_partials;              // [nctas][table_partial_len]
    float* tab_reduced;               // [table_partial_len]
    float* own_partials;              // [nctas][OWN_PARTIAL_LEN]
    float* own_reduced;               // [OWN_PARTIAL_LEN]
    float* nrm_partials;              // [4][NRM_MAX_PARTIALS][D]
    float* W0;                        // [B2][Nsp + 64] sample x table dot products of the table-query rows (head_table_gram.cuh)
    float *xs, *xst;                  // [B][D] sum_{k<C} xhat_k and xhat of the state row (forward -> backward)
    float* RS;                        // [B][8][32] per (sample, row) scalars of the forward (lane = row)
    float* GT;                        // [832] step-level dot products of the table rows (table_gram_prep_kernel)
    void* gemm_ws;                    // split-K scratch
    size_t gemm_ws_bytes;
    size_t total_bytes;
};

HeadDims head_dims(int64_t B, int C, int P, int Tc);
// carve `base` (may be null: sizing only) into the HeadWS pointers
void head_plan(const HeadDims& d, int mode, void* base, HeadWS* ws);

int peer_allreduce_range(cudaStream_t st, const team_peer_comm* c, int64_t offset, int64_t n, int channel);
int cosine_logits_launch(cudaStream_t st, const float* x, int64_t n_rows, const float* w, int64_t num_classes,
                         const float* sigma_dev, float* logits, int64_t* argmax);

}  // namespace team
