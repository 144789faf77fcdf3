/*
 * chgnet_b200.h — C ABI of the B200-native CHGNet hot path (libchgnet_b200.so).
 *
 * The reference (CederGroupHub/chgnet) has NO native interface for this path:
 * it is pure PyTorch (SURVEY.md §2b).  This header is therefore the boundary a
 * reference maintainer would bind with ctypes from chgnet/model/model.py; each
 * entry point names the reference lines it replaces.  See INTEGRATION.md for
 * the binding stub.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into caller-allocated memory unless it
 *     says "host"; no entry point allocates or frees device memory;
 *   - features are fp32 rows of width 64 (CHGNet atom/bond/angle_fea_dim = 64),
 *     indices are int32 (reference chgnet/graph/crystalgraph.py:12,
 *     converter.py:143-159);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*);
 *   - return value: 0 on success, negative on error; chg_last_error() then
 *     returns a static, thread-local message;
 *   - weight matrices are passed pre-packed; "…_t" means transposed to
 *     [in_features][out_features] (k-major), otherwise the PyTorch layout
 *     [out_features][in_features].  chgnet_b200/weights.py does the packing.
 *
 * Row layouts used throughout
 *   P rows of width 128 = [core(64) | gate(64)] pre-activations of a GatedMLP
 *   (reference chgnet/model/functions.py:168-183).
 */
#ifndef CHGNET_B200_H
#define CHGNET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CHG_FEA 64
#define CHG_MAX_CONV 8
#define CHG_MAX_Z 94 /* rows of the atom embedding / AtomRef tables (encoders.py:22-32) */
#define CHG_OK 0
#define CHG_ERR_ARG (-1)
#define CHG_ERR_CUDA (-2)

const char* chg_last_error(void);
int chg_abi_version(void);
/* number of kernel launches issued by this library since load (host counter) */
int64_t chg_launch_count(void);
/* run-time option (returns CHG_ERR_ARG for any other name):
 *   "ws_min_rows": AtomConv / BondConv inference calls with at least this many rows (default 4096) run the
 *                  warp-specialised tcgen05 kernels, smaller ones the FFMA kernels (launch-bound regime: the
 *                  persistent tcgen05 kernels' fixed cost loses on a few tiles).  Tests set 0 to run the tcgen05
 *                  kernels on small graphs.
 * (env CHG_PACK_THREADS = worker threads of the host packers / many-structure builder, default min(16, cores)). */
int chg_set_option(const char* name, int32_t value);

/* ---- K0: atom embedding.  x[i] = emb[z[i]-1]   (model.py:432-434, encoders.py:32) */
int chg_embed_atoms(const int32_t* z, const float* emb, int32_t n_atoms, float* x, void* stream);

/* ---- K1a: bond geometry per directed edge (model.py:840, encoders.py:98-102)
 * cart = frac @ L[g];  r = x_c - (x_n + img @ L[g]);  d = |r|;  rhat = r/d        */
int chg_edge_geometry(const float* frac, const float* lattice, const int32_t* atom_owner,
                      const int32_t* center, const int32_t* nbr, const float* image,
                      int32_t n_edges, float* rvec, float* dist, float* rhat, void* stream);

/* ---- K1b: radial Bessel basis (ag + bg) fused with the three 31->64 embeddings
 * (encoders.py:106-110, basis.py:108-116,188-205, model.py:435-437).
 * w3t = [3][n_radial][64] : bond_embedding^T, bond_weights_ag^T, bond_weights_bg^T */
int chg_bond_basis_embed(const float* dist, const int32_t* u2d, int32_t n_bonds,
                         const float* freq_ag, const float* freq_bg, int32_t n_radial,
                         float rc_ag, float rc_bg, int32_t p, const float* w3t,
                         float* e0, float* wag, float* wbg,
                         float* basis_out /* training: [Eu][64] = ag basis | bg basis, or NULL */,
                         void* stream);
/* reverse of K1b: g_dist[u] = d(E)/d(d_u).  w3 = [3][64][n_radial] (PyTorch layout) */
int chg_bond_basis_bwd(const float* dist, const int32_t* u2d, int32_t n_bonds,
                       const float* freq_ag, const float* freq_bg, int32_t n_radial,
                       float rc_ag, float rc_bg, int32_t p, const float* w3,
                       const float* g_e0, const float* g_wag, const float* g_wbg,
                       float* g_dist,
                       double* g_freq /* training: [2][n_radial] += dL/d(freq_ag, freq_bg), or NULL */,
                       void* stream);

/* ---- K2: Fourier angle basis fused with angle_embedding
 * (model.py:864-870, encoders.py:144-146, basis.py:35-40, model.py:439).
 * n_basis = 2*n_freq+1; wt = [n_basis][64]                                        */
int chg_angle_basis_embed(const float* rhat, const int32_t* ang_di, const int32_t* ang_dj,
                          int32_t n_angles, const float* freq, int32_t n_freq,
                          const float* wt, float* a0,
                          float* basis_out /* training: [A][64], basis in columns 0..2*n_freq, or NULL */,
                          void* stream);
/* reverse of K2: g_rhat[e] += dE/d rhat_e (fp64 atomics); w = [64][n_basis]        */
int chg_angle_basis_bwd(const float* rhat, const int32_t* ang_di, const int32_t* ang_dj,
                        int32_t n_angles, const float* freq, int32_t n_freq,
                        const float* w, const float* g_a0, double* g_rhat /* may be NULL if g_freq */,
                        double* g_freq /* training: [n_freq] += dL/d(freq), or NULL */, void* stream);

/* ---- dense feature mixing: y[yr(r)] = x[xr(r)] @ wt (+ bias) (+ residual[yr(r)]), r < m
 * x [.][k], wt [k][n_out], k in {64,128,256}, n_out multiple of 64; xr = x_rows ?
 * x_rows[r] : r (fused gather), yr likewise (fused scatter, rows must be unique).
 * Used for the per-atom / per-bond halves of every GatedMLP first layer, for
 * mlp_out + residual (layers.py:129-132, 256-260) and for their transposes.
 * BondConv / AngleUpdate only touch the bonds of the bond graph (d < 3 A, about 1/8
 * of all bonds): x_rows / y_rows carry that compaction.                            */
int chg_linear(const float* x, const int32_t* x_rows, int32_t m, int32_t k, const float* wt,
               const float* bias, const float* residual, const int32_t* y_rows, int32_t n_out,
               float* y, void* stream);
/* row movers for the same compaction: dst[i] = src[idx[i]]  /  dst[idx[i]] = src[i]   */
int chg_gather_rows(const float* src, const int32_t* idx, int32_t n, int32_t width, float* dst,
                    void* stream);
int chg_scatter_rows(const float* src, const int32_t* idx, int32_t n, int32_t width, float* dst,
                     void* stream);

/* ---- K4: AtomConv message (layers.py:113-121, functions.py:168-183)
 * pre = pcn[c][0:128] + pe[u] + pcn[n][128:256];  p = W2.silu(pre)+b2;
 * msg = silu(LN1(p_core)) * sigmoid(LN2(p_gate)) * wag[u].
 * pcn [N][256], pe [Eu][128] (first-layer bias folded in), w2t [64][128] block
 * diagonal halves (core|gate), ln = [4][64] (g1,b1,g2,b2) or NULL.               */
int chg_atom_conv_fwd(const float* pcn, const float* pe, const float* wag,
                      const int32_t* center, const int32_t* nbr, const int32_t* d2u,
                      int32_t n_edges, const float* w2t, const float* b2, const float* ln,
                      float* msg, float* save_p, float* save_pre /* training: [Ed][128] or NULL */,
                      void* stream);
/* reverse: g_pre[e][128] = dE/dpre, g_w[e][64] = dE/d wag row contribution        */
int chg_atom_conv_bwd(const float* pcn, const float* pe, const float* wag,
                      const int32_t* center, const int32_t* nbr, const int32_t* d2u,
                      int32_t n_edges, const float* save_p, const float* g_agg,
                      const float* w2, const float* ln, float* g_pre, float* g_w,
                      float* g_p /* training: [Ed][128] dL/dp, or NULL */,
                      double* g_ln /* training: [4][64] += dL/d(ln), or NULL */, void* stream);

/* ---- K4s/K5s: segmented gather-reduce (functions.py:25-37 without atomics)
 * out[r] (+)= sum_{k in [ptr[r],ptr[r+1])} data[perm ? perm[k] : k], width 64|128 */
int chg_segment_sum(const float* data, int32_t width, const int32_t* perm,
                    const int32_t* ptr, int32_t n_rows,
                    int32_t n_items /* ptr[n_rows]; scheduling hint only */, int32_t accumulate,
                    float* out, int32_t out_ld /* row stride of out, in floats */, void* stream);

/* ---- K4f / K5f: message + aggregation fused (the default inference path; layers.py:113-126, 238-254)
 * agg[s] = sum over the rows r of segment s of  G(pre_r) * w_r,  rows sorted by segment:
 *   AtomConv: rows = directed edges sorted by centre, segment = centre atom (ptr_c [N+1]), w = wag[d2u];
 *   BondConv: rows = angles sorted by bond slot i, segment = slot i (ptr_i [Es+1]), w = wbg[i] * wbg[j].
 * One warp-specialised tcgen05 kernel (csrc/gated_ws.cu): gather + add of the first-layer rows, the two 64x64
 * second-layer products as 3xTF32 on the tensor cores, LayerNorm / SiLU x sigmoid, and the segmented sum inside the
 * CTA (the [rows][64] message never reaches HBM), followed by a small stitch kernel for segments that span
 * 16-row strips (fixed order: deterministic).  save_p / save_pre [rows][128] may be NULL (no reverse pass).
 * `work`: caller scratch of chg_gated_fused_workspace_floats(rows) floats.  Calls with fewer rows than
 * "ws_min_rows" (chg_set_option) run the unfused FFMA pair chg_*_conv_fwd -> chg_segment_sum instead.         */
int64_t chg_gated_fused_workspace_floats(int32_t n_rows);
int chg_atom_conv_fused(const float* pcn, const float* pe, const float* wag, const int32_t* center,
                        const int32_t* nbr, const int32_t* d2u, const int32_t* ptr_c, int32_t n_edges,
                        int32_t n_atoms, const float* w2t, const float* b2, const float* ln, float* agg,
                        float* save_p, float* work, void* stream);
int chg_bond_conv_fused(const float* pij, const float* px, const float* pa, const float* wbg,
                        const int32_t* ang_atom, const int32_t* ang_i, const int32_t* ang_j,
                        const int32_t* ptr_i, int32_t n_angles, int32_t n_slots, const float* w2t,
                        const float* b2, const float* ln, float* agg, float* save_pre, float* save_p,
                        float* work, void* stream);

/* ---- K5: BondConv message (layers.py:238-249)
 * pre = pij[i][0:128] + pij[j][128:256] + px[c] + pa[a], pa = ang @ W1a (chg_linear);
 * upd = G(pre) * wbg[i] * wbg[j].  save_pre/save_p may be NULL (no backward).
 * i, j index the rows of pij / wbg (compact bond-graph slots).                      */
int chg_bond_conv_fwd(const float* pij, const float* px, const float* pa, const float* wbg,
                      const int32_t* ang_atom, const int32_t* ang_i, const int32_t* ang_j,
                      int32_t n_angles, const float* w2t, const float* b2, const float* ln,
                      float* upd, float* save_pre, float* save_p, void* stream);
/* g_pre[a][128] = dE/dpre; gw_i / gw_j [a][64] = dE/d wbg row contributions.
 * dE/d ang = g_pre @ W1a is a chg_linear call on g_pre.                             */
int chg_bond_conv_bwd(const float* save_pre, const float* save_p, const float* wbg,
                      const int32_t* ang_i, const int32_t* ang_j, int32_t n_angles,
                      const float* g_agg, const float* w2, const float* ln, float* g_pre,
                      float* gw_i, float* gw_j, float* g_p /* training, or NULL */,
                      double* g_ln /* training, or NULL */, void* stream);

/* ---- K6: AngleUpdate (layers.py:348-360): ang_new = ang + G0(pre), no hidden layer    */
int chg_angle_update_fwd(const float* pij, const float* px, const float* pa, const float* ang,
                         const int32_t* ang_atom, const int32_t* ang_i, const int32_t* ang_j,
                         int32_t n_angles, const float* ln, float* ang_new, float* save_p,
                         void* stream);
/* g_ang_in may be NULL (zero).  g_pre = dE/dpre; dE/d ang = g_ang_in + g_pre @ W1a
 * (chg_linear with residual).                                                       */
int chg_angle_update_bwd(const float* save_p, const float* g_ang_in, int32_t n_angles,
                         const float* ln, float* g_pre, double* g_ln /* training, or NULL */,
                         void* stream);

/* ---- K7: readout (model.py:497-509) + AtomRef sum (composition_model.py:175-205)
 * h = LN(x); site_e = MLP(h); e_graph[owner] += site_e (fp64); e_ref[owner] +=
 * atom_ref[z-1] (fp64).  mlp_wt [n_hidden][64][64] (k-major), mlp_w same in
 * PyTorch layout (needed only when g_x != NULL), mlp_b [n_hidden][64],
 * w_last [64], b_last host scalar.  Optional outputs (NULL to skip): h_out [N][64]
 * (for crystal_fea), g_x [N][64] = d(sum E)/dx.                                   */
int chg_readout(const float* x, const int32_t* z, const int32_t* atom_owner, int32_t n_atoms,
                const float* ln, const float* mlp_wt, const float* mlp_w, const float* mlp_b,
                int32_t n_hidden, const float* w_last, float b_last, const float* atom_ref,
                float* site_e, float* h_out, double* e_graph, double* e_ref, float* g_x,
                void* stream);
/* ---- K7a: magmom head (model.py:483-487): m = |w.x + b|                         */
int chg_magmom(const float* x, int32_t n_atoms, const float* w, float b, float* m, void* stream);

/* ---- K1c: force + virial (model.py:517-535 as ONE reverse pass)
 * g_r[e] = (g_rhat[e] - rhat (rhat.g_rhat))/d + [e == u2d[d2u[e]]] g_dist[d2u[e]] rhat
 * force[c] -= g_r; force[n] += g_r; virial[owner[c]] += rvec (x) g_r   (fp64)       */
int chg_force_virial(const float* rvec, const float* dist, const float* rhat,
                     const double* g_rhat, const float* g_dist, const int32_t* d2u,
                     const int32_t* u2d, const int32_t* center, const int32_t* nbr,
                     const int32_t* atom_owner, int32_t n_edges, double* force,
                     double* virial, void* stream);

/* ======================= whole-path entry points =======================
 * One call for CHGNet._compute + the two autograd.grad calls (reference model.py:389-542): the kernel
 * schedule of chgnet_b200/engine.py run natively on a caller-provided workspace.  This is what a
 * non-Python host, or model.py through a single ctypes call, binds; the per-kernel entry points above
 * stay available for unit parity tests and ncu isolation.                                           */
typedef struct {
  int32_t num_radial;        /* 31 (0.3.0) / 9 (0.2.0), <= 32                                       */
  int32_t num_angular;       /* 2*n_freq+1: 31 / 9, odd, <= 31                                      */
  int32_t n_conv;            /* AtomConv layers (4); BondConv = n_conv-1, live AngleUpdate = n_conv-2 */
  int32_t cutoff_coeff;      /* envelope exponent p (8 / 5), 0 = no envelope                        */
  int32_t n_readout_hidden;  /* hidden 64x64 layers of the readout MLP (3 / 2)                      */
  int32_t use_ln;            /* LayerNorm inside the GatedMLPs (gMLP_norm="layer")                  */
  int32_t readout_ln;        /* readout_norm="layer"                                                */
  int32_t has_mlp_out_bias;  /* 0.2.0 checkpoints                                                   */
  float atom_graph_cutoff;   /* 6 A */
  float bond_graph_cutoff;   /* 3 A */
  float b_last;              /* bias of the last readout layer  (set by chg_pack_weights_host)      */
  float b_mag;               /* bias of the site_wise head      (set by chg_pack_weights_host)      */
} chg_hparams;

/* one GatedMLP (+ mlp_out) of the reference state_dict, PyTorch layout [out][in], HOST pointers      */
typedef struct {
  const float* core_w1; const float* core_b1; const float* gate_w1; const float* gate_b1; /* [64][192|256], [64] */
  const float* core_w2; const float* core_b2; const float* gate_w2; const float* gate_b2; /* [64][64]; NULL for angle layers */
  const float* ln1_w; const float* ln1_b; const float* ln2_w; const float* ln2_b;         /* bn1 / bn2, NULL without LayerNorm */
  const float* out_w; const float* out_b;   /* mlp_out.layers.1 [64][64] (+ bias or NULL); NULL for angle layers */
} chg_gated_sd;
typedef struct {
  const float* atom_embedding;                                  /* [94][64] */
  const float* freq_ag; const float* freq_bg; const float* freq_ang;
  const float* bond_embedding; const float* bond_weights_ag; const float* bond_weights_bg; /* [64][num_radial] */
  const float* angle_embedding;                                 /* [64][num_angular] */
  chg_gated_sd atom[CHG_MAX_CONV];   /* atom_conv_layers.{t}.twoBody_atom + mlp_out */
  chg_gated_sd bond[CHG_MAX_CONV];   /* bond_conv_layers.{t}.twoBody_bond + mlp_out */
  chg_gated_sd angle[CHG_MAX_CONV];  /* angle_layers.{t}.twoBody_bond               */
  const float* readout_ln_w; const float* readout_ln_b;
  const float* mlp_w[4]; const float* mlp_b[4];                 /* hidden readout layers */
  const float* mlp_last_w; float mlp_last_b;                    /* [64], scalar */
  const float* site_wise_w; float site_wise_b;
  const float* atom_ref;                                        /* composition_model.fc.weight [94] or NULL */
} chg_state_dict;
/* number of floats of the packed weight blob; pack on the HOST (weights.py::pack_weights restated),
 * then copy the blob to the device (64-byte aligned) and hand it to chg_forward                      */
int64_t chg_packed_floats(const chg_hparams* hp);
int chg_pack_weights_host(chg_hparams* hp, const chg_state_dict* sd, float* packed_host);

/* the SoA batch descriptor (chgnet_b200/batch.py::DeviceBatch): device pointers, int32 indices.
 * Directed edges are sorted by centre atom, angles by bond i; ptr_* are CSR row pointers and perm_* the
 * grouping permutations (by neighbour atom, by undirected bond, by bond j, by centre atom of the
 * angle); short_ids / ang_is / ang_js address the compact slots of the bond-graph bonds.              */
typedef struct {
  int32_t n_atoms, n_edges, n_bonds, n_angles, n_graphs, n_short;
  const int32_t* z; const float* frac; const int32_t* owner; const float* lattice;   /* [N], [N][3], [N], [B][9] */
  const int32_t* center; const int32_t* nbr; const float* image;                     /* [Ed], [Ed], [Ed][3] */
  const int32_t* d2u; const int32_t* u2d;                                            /* [Ed], [Eu] */
  const int32_t* ptr_c; const int32_t* perm_n; const int32_t* ptr_n; const int32_t* perm_u; const int32_t* ptr_u;
  const int32_t* ang_atom; const int32_t* ang_di; const int32_t* ang_dj; const int32_t* ang_is; const int32_t* ang_js;
  const int32_t* ptr_is; const int32_t* perm_js; const int32_t* ptr_js; const int32_t* perm_x; const int32_t* ptr_x;
  const int32_t* short_ids;   /* [Es] */
  const int32_t* graph_ptr;   /* [B+1] atoms of each graph (only for crystal_fea) */
} chg_batch;
/* caller-allocated outputs; NULL = not wanted (energy, e_ref, site_e are required).  force / virial
 * non-NULL runs the reverse pass.  energy / e_ref are EXTENSIVE (eV): e = (energy + e_ref) / n_atoms. */
typedef struct {
  double* energy; double* e_ref; float* site_e;      /* [B], [B], [N] */
  float* magmom; float* atom_fea; float* crystal_fea;  /* [N], [N][64], [B][64] */
  double* force; double* virial;                     /* [N][3], [B][9] = sum_e r (x) dE/dr (stress = 160.21766208 / V * virial) */
} chg_outputs;
/* workspace size for these sizes / wanted outputs (pointers of `sizes` may be NULL; of `wanted` only
 * NULL-ness matters); `trace` (optional) receives the newline-separated list of kernel calls         */
int chg_forward_plan(const chg_hparams* hp, const chg_batch* sizes, const chg_outputs* wanted,
                     size_t* workspace_bytes, char* trace, size_t trace_cap);
int chg_forward(const chg_hparams* hp, const float* packed_weights, const chg_batch* batch,
                const chg_outputs* out, void* workspace /* 256-byte aligned */, size_t workspace_bytes,
                void* stream);

/* ======================= host-native graph construction (row f1, host stage) =======================
 * The reference's only native component on this path is its C graph builder
 * (chgnet/graph/cygraph.pyx:69-175 -> create_graph.c:100-107, called from converter.py:257-266 after
 * pymatgen's neighbour list, converter.py:132).  chg_graph_build does both steps in C++ on the HOST
 * (no device work): periodic neighbour list (1e-8 < d <= r_atom, sorted by centre, neighbour, image),
 * undirected-bond pairing (numbered by first appearance) and the bond graph (d < r_bond), with the row
 * order of chgnet_b200/graphgen.py (pinned against the reference's Graph class).  frac [n][3] and
 * lattice [3][3] (rows = lattice vectors) are fp64 HOST arrays; the graph object owns host memory
 * until chg_graph_free.                                                                             */
typedef struct chg_graph chg_graph;
int chg_graph_build(const double* frac, const double* lattice, int32_t n_atoms, double r_atom, double r_bond,
                    chg_graph** out);
void chg_graph_sizes(const chg_graph* g, int64_t* n_edges, int64_t* n_bonds, int64_t* n_angles);
/* copies into caller arrays (NULL = skip): atom_graph [Ed][2], image [Ed][3], d2u [Ed], u2d [Eu],
 * bond_graph [A][5] = (centre atom, undirected i, directed i, undirected j, directed j)               */
int chg_graph_export(const chg_graph* g, int32_t* atom_graph, float* image, int32_t* d2u, int32_t* u2d,
                     int32_t* bond_graph);
void chg_graph_free(chg_graph* g);

/* Many structures at once (the converter loop of the reference's predict_structure, model.py:578-583): chg_graph_build
 * for n structures on the library's persistent worker threads; out[i] is always a handle to free; returns the first
 * failure's code (message in chg_last_error).  chg_graph_views: counts [n][3] = directed edges, bonds, angles; ptrs
 * [n][5] = host pointers to atom_graph, image, d2u, u2d, bond_graph inside the handles (valid until freed; exactly what
 * chg_pack_batch_wire / chg_pack_batch_host take); n_isolated [n] (or NULL) = atoms without a neighbour.         */
int chg_graph_build_many(int32_t n, const double* const* frac, const double* const* lattice, const int32_t* n_atoms,
                         double r_atom, double r_bond, chg_graph** out);
int chg_graph_views(int32_t n, chg_graph* const* graphs, int64_t* counts, uint64_t* ptrs, int32_t* n_isolated);
void chg_graph_free_many(int32_t n, chg_graph** graphs);

/* ---- device graph builder (one structure): fractional coordinates -> the edge / angle arrays of chg_batch, on the device
 * (csrc/graph_device.cu).  Replaces the host-side neighbour list + create_graph.c / cygraph.pyx + line graph
 * (converter.py:102-190, graph.py:132-328, fast_converter_libraries/create_graph.c:100-219) that the reference
 * runs on the CPU every MD step (dynamics.py:156-157).  Integer outputs are bit-identical to chg_graph_build.
 * frac [N][3] fp64 on the DEVICE; lattice [9] fp64 on the host (rows = lattice vectors).  Outputs (device,
 * caller-allocated): center / nbr / d2u [cap_edges], image [cap_edges][3] fp32, u2d [cap_edges / 2], ptr_c [N + 1],
 * ang_atom / ang_i / ang_di / ang_j / ang_dj [cap_angles] (undirected / directed indices as in bond_graph).
 * sizes_out (host) = {n_edges, n_bonds, n_angles, 0}; synchronises the stream twice (one int32 each).
 * CHG_ERR_ARG + "capacity" in chg_last_error() when a capacity is too small (sizes_out holds what is needed).      */
int64_t chg_graph_device_scratch_bytes(int32_t n_atoms, int32_t cap_edges);
int chg_graph_build_device(const double* frac, const double* lattice, int32_t n_atoms, double r_atom, double r_bond,
                           int32_t cap_edges, int32_t cap_angles, int32_t* center, int32_t* nbr, float* image,
                           int32_t* d2u, int32_t* u2d, int32_t* ptr_c, int32_t* ang_atom, int32_t* ang_i,
                           int32_t* ang_di, int32_t* ang_j, int32_t* ang_dj, void* scratch, int32_t* sizes_out,
                           void* stream);

/* ---- device-resident MD / relaxation updates (csrc/md.cu; the reference integrates on the host through ASE,
 * dynamics.py:129-181, 190-204).  x, v, f [N][3] fp64 on the device; inv_mass [N]; inv_lattice [9] on the HOST
 * (frac = x @ inv_lattice).  frac64 feeds chg_graph_build_device, frac32 is chg_batch.frac.
 *   chg_md_kick_drift: v += dt/2 f/m; x += dt v; frac; max_disp2 (device double, may be NULL) = max |x - x_ref|^2
 *   chg_md_kick      : v += dt/2 f/m; *e_kin (device double, may be NULL) += kinetic energy
 *   chg_fire_step    : one FIRE update with its state in device memory (12 doubles: dt, alpha, n_pos, sums, ...)   */
int chg_md_kick_drift(double* x, double* v, const double* f, const double* inv_mass, int32_t n_atoms, double dt,
                      const double* inv_lattice, double* frac64, float* frac32, const double* x_ref,
                      double* max_disp2, void* stream);
int chg_md_kick(double* v, const double* f, const double* inv_mass, int32_t n_atoms, double dt, double* e_kin,
                void* stream);
int chg_fire_step(double* x, double* v, const double* f, int32_t n_atoms, double* state, const double* inv_lattice,
                  double* frac64, float* frac32, double dt_max, double max_step, void* stream);

/* ---- Berendsen NVT / NPT with the cell in device memory (csrc/md.cu).  Replaces ASE's NVTBerendsen,
 * Inhomogeneous_NPTBerendsen and NPTBerendsen that the reference's MolecularDynamics drives on the host
 * (dynamics.py:595-609, 671-715; one CHGNetCalculator.calculate per step, dynamics.py:129-181).  Everything a
 * captured step reads is device memory, so one CUDA graph serves every step until the lists are rebuilt.
 * cell_state: 64 doubles = L [0..8] (rows = lattice vectors), L^-1 [9..17], L_old^-1 [18..26], L_ref [27..35] and
 * L_ref^-1 [36..44] (the cell of the last list build), V [45], lambda [46], T [47], max_i |(s_i - s_ref,i) L_ref|^2
 * [52], ||L_ref^-1 L - I||_F [53].  params: 8 doubles = T0 (K), P0 (eV/A^3), dt/tau_t, dt beta/(3 tau_p), mask [3],
 * k_B (eV/K).  flags: 1 thermostat, 2 isotropic barostat, 4 per-axis barostat, 8 remove the mean momentum.
 * mom_part [blocks][3], k_part [blocks][4] = per-block partials (blocks = chg_md_partial_blocks(n_atoms)), summed
 * in a fixed order: the trajectory does not depend on the scheduling.  virial [9] fp64 (chg_forward's output;
 * sigma = virial / V); lattice32 [9] is what chg_batch.lattice points at.
 *   chg_md_cell_step      : one block: K from k_part -> lambda -> P_a = -sigma_aa + lambda^2 K_aa / V -> mu -> L, L^-1,
 *                           V, lattice32, strain; resets the displacement maximum
 *   chg_md_kick_drift_cell: v *= lambda; x = (x L_old^-1) L (barostat); v += dt/2 f/m; v -= mean(m v)/m (flag 8);
 *                           x += dt v; frac64 / frac32 = x L^-1; displacement maximum against s_ref (may be NULL)
 *   chg_md_kick_partials  : v += dt/2 f/m (f may be NULL: no kick); k_part = partials of K_aa = sum m v_a^2 and K_tr */
int chg_md_partial_blocks(int32_t n_atoms);
int chg_md_cell_step(const double* params, double* cell_state, const double* k_part, int32_t n_atoms,
                     const double* virial, float* lattice32, int32_t flags, void* stream);
int chg_md_kick_drift_cell(double* x, double* v, const double* f, const double* inv_mass, int32_t n_atoms, double dt,
                           double* cell_state, double* mom_part, double* frac64, float* frac32, const double* s_ref,
                           int32_t flags, void* stream);
int chg_md_kick_partials(double* v, const double* f, const double* inv_mass, int32_t n_atoms, double dt,
                         double* k_part, void* stream);

/* ---- device CSR build: the segment structures of chg_batch from the packed index arrays
 * (replaces the torch sorts / searchsorted / nonzero of BatchedGraph-side preprocessing; csrc/batch_csr.cu).
 * Inputs: directed edges sorted by centre, angles sorted by bond i (chg_pack_batch_host reports both).
 * Outputs (caller-allocated int32): ptr_c [N+1]; perm_n [Ed], ptr_n [N+1] (edges by neighbour); perm_u [Ed],
 * ptr_u [Eu+1] (the 2 directed edges of every bond); ptr_i [Eu+1]; perm_j [A], ptr_j [Eu+1] (angles by bond j);
 * perm_x [A], ptr_x [N+1] (angles by atom); and, when n_short >= 0 (= the number of distinct bonds that occur in
 * angles, counted by chg_pack_batch_host): short_ids [Es], ang_is / ang_js [A], ptr_is [Es+1], ptr_js [Es+1]
 * (perm_js == perm_j).  Inside every segment the permutations are ascending (== a stable sort by key).
 * with_reverse = 0 skips the transposed groupings.  scratch: chg_build_csr_scratch_ints(...) int32.           */
typedef struct chg_csr_in {
  int32_t n_atoms, n_edges, n_bonds, n_angles, n_short, with_reverse;
  const int32_t *center, *nbr, *d2u, *ang_atom, *ang_i, *ang_j;
} chg_csr_in;
typedef struct chg_csr_out {
  int32_t *ptr_c, *perm_n, *ptr_n, *perm_u, *ptr_u, *ptr_i, *perm_j, *ptr_j, *perm_x, *ptr_x;
  int32_t *short_ids, *ang_is, *ang_js, *ptr_is, *ptr_js;
} chg_csr_out;
int64_t chg_build_csr_scratch_ints(int32_t n_atoms, int32_t n_edges, int32_t n_bonds, int32_t n_angles);
int chg_build_csr(const chg_csr_in* in, const chg_csr_out* out, int32_t* scratch, void* stream);
/* n_short for index arrays that live on the device (device graph builder): one int32 to the host, synchronises.
 * scratch: 2 * (n_bonds + 1) + 4096 int32.                                                                  */
int chg_bond_graph_count(const int32_t* ang_i, const int32_t* ang_j, int32_t n_angles, int32_t n_bonds,
                         int32_t* scratch, int32_t* count_out, void* stream);

/* host batch packer: B CrystalGraphs (HOST arrays, int32 / fp32, contiguous) -> the concatenated,
 * offset-adjusted SoA of chg_batch in one pass (BatchedGraph.from_graphs, model.py:820-899, without
 * per-graph tensor ops).  counts [B][4] = atoms, directed edges, undirected bonds, angles; ptrs [B][8] =
 * atomic_number, atom_frac_coord, atom_graph, neighbor_image, directed2undirected, undirected2directed,
 * bond_graph, lattice.  ibuf (int32) = z[N] owner[N] center[Ed] nbr[Ed] d2u[Ed] u2d[Eu] ang_atom[A]
 * ang_i[A] ang_di[A] ang_j[A] ang_dj[A]; fbuf (fp32) = frac[N*3] image[Ed*3] lattice[B*9];
 * flags_out[0/1] = edges sorted by centre / angles sorted by bond i within every graph;
 * flags_out[2] = index (in the batch) of the first atom whose atomic number is outside [1, CHG_MAX_Z],
 * or -1 (the caller raises IndexError like the reference's nn.Embedding, tests/test_encoders.py:25-28);
 * flags_out[3] = number of distinct bonds that occur in angles (n_short of chg_build_csr: no device sync). */
int chg_pack_batch_host(int32_t n_graphs, const int64_t* counts, const void* const* ptrs, int32_t* ibuf,
                        float* fbuf, int32_t* flags_out);

/* Pinned staging memory for the two packers (cudaHostAlloc; write_combined != 0: write-combined - written by the
 * packer's threads with streaming stores and read only by the copy engine; never read it on the CPU). */
int chg_host_alloc(int64_t bytes, int32_t write_combined, void** out);
int chg_host_free(void* p);

/* The same batch over a COMPACT wire format, packed by persistent worker threads and shipped in two phases whose
 * copies overlap the packing (csrc/batch_wire.cu): the bond-graph columns that are functions of the two directed-edge
 * columns (ang_atom = center[ang_di], ang_i = d2u[ang_di], ang_j = d2u[ang_dj]; graph.py:233-277) and the fp32 images
 * (shipped as int8) are re-created on the device.  Both properties are VERIFIED per angle / image while packing:
 * flags_out[4] != 0 (1 image not an integer in [-127, 127], 2 columns not derivable, 3 edge index out of range) means
 * nothing usable was produced and the caller uses chg_pack_batch_host.  counts / ptrs / flags_out[0..3] as above.
 *   host staging (pinned): ibuf_host [2N + 3Ed + Eu + 2A] = z owner center nbr d2u u2d ang_di ang_dj;
 *                          fbuf_host [3N + 9B] = frac lattice;  img_host [3Ed] int8
 *   device:                ibuf_dev [2N + 3Ed + Eu + 5A] = the host layout followed by ang_atom ang_i ang_j;
 *                          fbuf_dev [3N + 9B + 3Ed] = frac lattice image;  img_dev [3Ed] scratch
 * All three device pointers NULL: pack only (no CUDA call).  Copies and the two expansion kernels are enqueued on
 * `stream`; the host buffers may be reused once an event recorded after the call has completed.                 */
int chg_pack_batch_wire(int32_t n_graphs, const int64_t* counts, const void* const* ptrs, int32_t* ibuf_host,
                        float* fbuf_host, int8_t* img_host, int32_t* ibuf_dev, float* fbuf_dev, int8_t* img_dev,
                        int32_t* flags_out, void* stream);

/* ======================= training (reference trainer.py:398-411, 779-869) =======================
 * The reverse pass over activations is the one above (seeded with the loss instead of 1); these
 * entry points add the parameter gradients, the loss terms and the optimizer step for losses on
 * energies and magnetic moments; losses on forces / stresses additionally use the second-order
 * entry points further down (DESIGN.md §10).                                                    */

/* dL/dW^T: out[k][j] = sum_r act(x[xr(r)][k]) * g[gr(r)][j],  k < 64, j < n_out (multiple of 64);
 * colsum[j] = sum_r g[gr(r)][j] (bias gradient) or NULL.  x_silu != 0 applies SiLU to x (second
 * GatedMLP layer: the hidden activations are recomputed from the saved pre-activations).
 * ldx / ldg / ldo are row strides in floats (column-slice views are allowed).  Deterministic:
 * per-CTA partials in `workspace` (>= chg_wgrad_workspace_floats(n_out) floats), summed in fp64. */
int64_t chg_wgrad_workspace_floats(int32_t n_out);
int chg_wgrad(const float* x, const float* x2 /* non-NULL: act = silu'(x) * x2 (tangent of the hidden layer) */,
              int32_t ldx, const int32_t* x_rows, int32_t x_silu, const float* g,
              int32_t ldg, const int32_t* g_rows, int32_t m, int32_t n_out, float* out, int32_t ldo,
              float* colsum, float* workspace, void* stream);
/* out[c] += sum_r a[r][c] * (bmul ? bmul[r][c] : 1) * (rowscale ? rowscale[r] : 1), n in {64,128,256} */
int chg_colsum(const float* a, int32_t lda, const float* bmul, int32_t ldb, const float* rowscale,
               int32_t m, int32_t n, double* out, void* stream);
/* reverse of the readout MLP with seed[i] = dL/d(site energy i); returns g_x = dL/dx and, for the
 * parameter gradients, h_all [n_hidden+1][N][64] (input of every linear), gz_all [n_hidden][N][64]
 * (dL/d pre-activation), g_h0 [N][64] (dL/d LayerNorm output), xhat [N][64]                       */
int chg_readout_bwd(const float* x, int32_t n_atoms, const float* ln, const float* mlp_wt,
                    const float* mlp_w, const float* mlp_b, int32_t n_hidden, const float* w_last,
                    const float* seed, float* g_x, float* h_all, float* gz_all, float* g_h0,
                    float* xhat, void* stream);
/* m = |x.w + b|: g_lin[i] = sign(x_i.w + b) g_m[i];  g_x[i] += g_lin[i] w                          */
int chg_magmom_bwd(const float* x, int32_t n_atoms, const float* w, float b, const float* g_m,
                   float* g_x, float* g_lin, void* stream);
/* one CombinedLoss term (trainer.py:797-867) over a flat vector, NaN targets masked:
 * sums[0..2] += (sum loss_i, sum |err_i|, count); g_pred[i] = d loss_i / d pred_i.
 * kind 0 MSE, 1 MAE, 2 Huber(delta)                                                               */
int chg_loss_terms(const float* pred, const float* target, int32_t n, int32_t kind, float delta,
                   float* g_pred, double* sums, void* stream);
/* torch.optim.Adam (trainer.py:178-189) on one flat fp32 buffer; step counts from 1               */
int chg_adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int32_t step, void* stream);

/* ======================= second order: losses on forces and stresses =======================
 * F = -dE/dcart and sigma = (c/V) dE/d(strain) come from the reverse pass, so their parameter
 * gradient is d/dtheta of  T = sum_e <dE/dr_e, rdot_e>  with the loss-weighted direction
 * rdot_e = -(gF[c] - gF[n]) + r_e . (gS c/V) held fixed (reference model.py:518-535 create_graph=True,
 * trainer.py:409).  T is evaluated by a TANGENT pass along rdot (the *_tan / *_tangent kernels mirror
 * the forward kernels), then one more reverse pass over (primal, tangent) (the *_bwd2 kernels) gives
 * dT/dtheta together with the energy / magmom part of the loss.  "lam" arguments are adjoints
 * dE/d(.) recorded by the force pass; "bar" arguments are the adjoints of the primal intermediates in
 * this second reverse pass.                                                                        */
int chg_edge_tangent(const float* rvec, const float* dist, const float* rhat, const int32_t* center,
                     const int32_t* nbr, const int32_t* atom_owner, const float* u_atom /* [N][3] */,
                     const float* w_graph /* [B][9] */, int32_t n_edges, float* ddist, float* drhat,
                     void* stream);
/* tangent of K1b along ddist; tbasis [Eu][64] = (dB/dd ddist) for the ag | bg bases              */
int chg_bond_basis_tangent(const float* dist, const float* ddist, const int32_t* u2d, int32_t n_bonds,
                           const float* freq_ag, const float* freq_bg, int32_t n_radial, float rc_ag,
                           float rc_bg, int32_t p, const float* w3t, float* e0d, float* wagd, float* wbgd,
                           float* tbasis, void* stream);
/* g_freq [2][n_radial] += d/dfreq < lam, (dB/dd ddist) W >                                          */
int chg_bond_basis_bwd2(const float* dist, const float* ddist, const int32_t* u2d, int32_t n_bonds,
                        const float* freq_ag, const float* freq_bg, int32_t n_radial, float rc_ag,
                        float rc_bg, int32_t p, const float* w3, const float* lam_e0, const float* lam_wag,
                        const float* lam_wbg, double* g_freq, void* stream);
int chg_angle_basis_tangent(const float* rhat, const float* drhat, const int32_t* ang_di,
                            const int32_t* ang_dj, int32_t n_angles, const float* freq, int32_t n_freq,
                            const float* wt, float* a0d, float* tbasis, void* stream);
int chg_angle_basis_bwd2(const float* rhat, const float* drhat, const int32_t* ang_di, const int32_t* ang_dj,
                         int32_t n_angles, const float* freq, int32_t n_freq, const float* w,
                         const float* lam_a0, double* g_freq, void* stream);
/* tangent of K4: msg' = o' wag[u] + o wag'[u]; also returns pre' and p' [Ed][128] for the reverse    */
int chg_atom_conv_tan(const float* pcn_d, const float* pe_d, const float* wag, const float* wag_d,
                      const int32_t* center, const int32_t* nbr, const int32_t* d2u, int32_t n_edges,
                      const float* save_pre, const float* save_p, const float* w2t, const float* ln,
                      float* msg_d, float* pre_d, float* p_d, void* stream);
/* reverse of (K4, its tangent): bar_pre = adjoint of pre, bar_w [Ed][64] = adjoint of the wag rows,
 * u_out [Ed][128] = adjoint of p (for the second-layer weight gradient), g_ln accumulated        */
int chg_atom_conv_bwd2(const float* save_pre, const float* save_p, const float* pre_d, const float* p_d,
                       const float* g_p_lam, const float* wag, const float* wag_d, const int32_t* center,
                       const int32_t* d2u, int32_t n_edges, const float* lam_agg, const float* bar_agg,
                       const float* w2, const float* ln, float* bar_pre, float* bar_w, float* u_out,
                       double* g_ln, void* stream);
int chg_bond_conv_tan(const float* pij_d, const float* px_d, const float* pa_d, const float* wbg,
                      const float* wbg_d, const int32_t* ang_atom, const int32_t* ang_i, const int32_t* ang_j,
                      int32_t n_angles, const float* save_pre, const float* save_p, const float* w2t,
                      const float* ln, float* upd_d, float* pre_d, float* p_d, void* stream);
int chg_bond_conv_bwd2(const float* save_pre, const float* save_p, const float* pre_d, const float* p_d,
                       const float* g_p_lam, const float* wbg, const float* wbg_d, const int32_t* ang_i,
                       const int32_t* ang_j, int32_t n_angles, const float* lam_agg, const float* bar_agg,
                       const float* w2, const float* ln, float* bar_pre, float* bar_wi, float* bar_wj,
                       float* u_out, double* g_ln, void* stream);
int chg_angle_update_tan(const float* pij_d, const float* px_d, const float* pa_d, const float* ang_d,
                         const int32_t* ang_atom, const int32_t* ang_i, const int32_t* ang_j,
                         int32_t n_angles, const float* save_p, const float* ln, float* ang_new_d, float* p_d,
                         void* stream);
/* lam_ang / bar_ang: adjoints of ang_new (NULL = zero)                                              */
int chg_angle_update_bwd2(const float* save_p, const float* p_d, const float* lam_ang, const float* bar_ang,
                          int32_t n_angles, const float* ln, float* bar_pre, double* g_ln, void* stream);
/* reverse of (readout, its tangent along xd) for  sum_i seed_i site_e_i + <d site_e_i/dx_i, xd_i>:
 * bar_x = adjoint of x; h_all / hd_all [n_hidden+1][N][64] inputs of every linear and their tangents;
 * gz_all / zbar_all [n_hidden][N][64] adjoints of the tangent / primal pre-activations; g_h0 / hbar0
 * adjoints of the tangent / primal LayerNorm output; xhat, xhatd                                      */
int chg_readout_bwd2(const float* x, const float* xd, int32_t n_atoms, const float* ln, const float* mlp_wt,
                     const float* mlp_w, const float* mlp_b, int32_t n_hidden, const float* w_last,
                     const float* seed, float* bar_x, float* h_all, float* hd_all, float* gz_all,
                     float* zbar_all, float* g_h0, float* hbar0, float* xhat, float* xhatd, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CHGNET_B200_H */
