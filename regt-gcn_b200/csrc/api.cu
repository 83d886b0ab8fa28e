// C-ABI entry points of the cell + head (include/regt_b200.h), the choice of their kernels and the workspace layout.
#include <stdlib.h>

#include "common.cuh"

namespace regt {

constexpr int F = REGT_F;

Route route_of(const regt_args* a) {
  const char* e = getenv("REGT_UNFUSED");
  const bool unfused = e && e[0] == '1';
  const bool tf32x3 = a->precision == REGT_PREC_TF32X3, bf16 = a->precision == REGT_PREC_BF16;
  const bool fused_step = a->fuse_head && a->y && a->d_out && a->loss;   // forward, loss and head gradients in one step
  Route r{};
  // bf16: the fused H = 64 cell where it is built for the shape (REGT_UNFUSED does not apply: it names the tf32x3 cells),
  // else the GEMM-by-GEMM cell on the single-pass bf16 GEMMs
  // head_only: no cell, so none of the cell couplings below applies (k_head_tc, tiled G, out_hidden partials)
  r.cell = a->head_only ? CellPath::None
         : bf16 ? (cell_tc_fits(a) ? CellPath::Bf16 : CellPath::Bf16Gemm)
                : !tf32x3 ? CellPath::Fp32 : (!unfused && cell_f_fits(a)) ? CellPath::Tf32x3Fused : CellPath::Tf32x3Unfused;
  if (r.cell == CellPath::Bf16 && fused_step && head_tc_fits(a->H, a->O))   // k_head_tc's partials are summed by the fused cell backward
    r.head = HeadPath::Bf16;
  else if (tf32x3 && a->H % 32 == 0 && head_f_fits(a->O) && (long long)a->B * a->N >= 128 && a->out)
    r.head = HeadPath::Tf32x3;
  else if (fused_step && head_fused_fits(a->H, a->O))
    r.head = HeadPath::FusedFfma;
  else
    r.head = HeadPath::Rows;
  r.g_tiled = r.cell == CellPath::Tf32x3Fused || r.cell == CellPath::Bf16;
  r.hid_partials = r.cell == CellPath::Bf16 && (r.head == HeadPath::Bf16 || r.head == HeadPath::FusedFfma);
  return r;
}

// head_only: what the head and the loss need, no cell planes.  G comes first, so that a caller (the period-sharing
// combine backward) finds the gradient wrt out_hidden at the start of the workspace
static Layout make_head_layout(const regt_args* a, Layout L, Carver& c) {
  const size_t H = a->H, O = a->O, BN = (size_t)a->B * a->N, BNp = (BN + 127) / 128 * 128;
  L.G = c.take<float>(BNp * H);
  if (a->precision == REGT_PREC_TF32X3) {   // tensor-core head (head_f.cu)
    L.hf_rh = c.take<float>(BN * H);
    L.hf_do32 = c.take<float>(BN * 32);
    L.hf_split = c.take<float>(max(gemm_nt_scratch_floats(HEAD_HID, (int)H, GemmKind::Tf32x3), gemm_nt_scratch_floats((int)H, HEAD_HID, GemmKind::Tf32x3)));
    L.hf_loss_floats = BN / 8 + 2;
    L.hf_loss = c.take<float>(L.hf_loss_floats);
    // ones column of the row head's dW1 / db1 contraction.  Taken whichever head the route picks: the head calls of a
    // pass (training, evaluation, the final window alone) route differently, and one workspace sized for the largest
    // of them must hold every one
    L.Feat = c.take<float>(BNp * 32);
  }
  L.a1 = c.take<float>(BN * HEAD_HID);
  L.d_a1 = c.take<float>(BN * HEAD_HID);
  size_t pf = (size_t)128 * (O * HEAD_HID + HEAD_HID * H);          // head split-K partials (<= 128 splits)
  pf = max(pf, (size_t)152 * HEAD_HID * (H + 32));                   // head dW1 on the tensor cores (+ the 32-wide second operand)
  pf = max(pf, BN / 64 + 2);                                         // loss partials
  pf += H * HEAD_HID + HEAD_HID * O + 64;                            // transposed head weights (tail)
  L.hpart = c.take<float>((size_t)148 * (HEAD_HID * H + O * HEAD_HID + HEAD_HID + O + 8));
  L.part = c.take<float>(pf);
  L.part_floats = pf;
  if (a->y) {
    L.inv_c = c.take<float>(a->B);
    L.lc_part = c.take<unsigned int>((size_t)a->B * LC_CHUNKS);
  }
  L.total = align_up(c.off, 256);
  return L;
}

Layout make_layout(const regt_args* a, void* base) {
  Layout L{};
  L.route = route_of(a);
  Carver c(base);
  if (L.route.cell == CellPath::None) return make_head_layout(a, L, c);
  const size_t H = a->H, T = a->T, R = a->plan.R > 0 ? a->plan.R : 1, O = a->O;
  const size_t BN = (size_t)a->B * a->N, rows = BN * T;
  const size_t nseg = a->plan.nseg;
  L.Wzr = c.take<float>((F + H) * 2 * H);
  L.Wc = c.take<float>((F + H) * H);
  L.czr = c.take<float>(2 * H);
  L.cc = c.take<float>(H);
  L.M0t = c.take<float>(F * H);
  L.M1t = c.take<float>(R * F * H);
  L.c0 = c.take<float>(H);
  L.Lsum = c.take<float>(H * H);
  L.probs = c.take<float>(T);
  L.S = c.take<float>(BN * F * T);
  L.U = c.take<float>((size_t)a->B * (nseg ? nseg : 1) * F * T);
  if (L.route.cell == CellPath::Tf32x3Fused) {
    // fused 3xTF32 cell (cell_f.cu): three saved planes in tile layout; the backward kernel writes the gate-gradient
    // blocks D and h, h*R as TRANSPOSED tiles [T*nqt][cols][128 rows] for the weight-gradient contraction (gemm_kt)
    const size_t nqt = (BN + 127) / 128, rowsP = T * nqt * 128;
    const bool inf = a->inference != 0;     // forward only: one Z tile per CTA (re-read by its own epilogue), nothing else saved
    L.tc_img_f = c.take<unsigned char>(F_IMG_BYTES);
    L.tc_img_b = c.take<unsigned char>(F_IMG_BYTES);
    L.Zp = c.take<float>(inf ? (size_t)TC_MAX_CTAS * 128 * H : rowsP * H);
    L.Rp = c.take<float>(inf ? 4 : rowsP * H);
    L.Hcp = c.take<float>(inf ? 4 : rowsP * H);
    L.Xt = c.take<float>(BN * F * T);
    L.h = c.take<float>(inf ? 4 : rowsP * H);
    L.hR = c.take<float>(inf ? 4 : rowsP * H);
    L.D = c.take<float>(inf ? 4 : rowsP * 4 * H);
    L.Feat = c.take<float>(inf ? 4 : nqt * 128 * 32);      // the head's ones column (row major, BNp rows)
    L.FeatT = c.take<float>(inf ? 4 : rowsP * 32);
    L.tc_dpp = c.take<float>(2 * (T * TC_MAX_CTAS + 64));   // fp64 attention-gradient partials
  } else if (L.route.cell != CellPath::Bf16) {   // fp32 and the GEMM-by-GEMM cells (tf32x3, bf16): row-major planes
    const bool gemm_cell = L.route.cell != CellPath::Fp32;
    L.h = c.take<float>(rows * H);
    L.Z = c.take<float>(rows * H);
    L.Rg = c.take<float>(rows * H);
    L.Hc = c.take<float>(rows * H);
    L.hR = c.take<float>(rows * H);
    L.Hn = c.take<float>(rows * H);
    L.D = c.take<float>(rows * 4 * H);
    L.Feat = c.take<float>(gemm_cell ? rows * 32 : 4);
    L.bsplit = c.take<float>(L.route.cell == CellPath::Tf32x3Unfused ? gemm_nt_scratch_floats((int)H, 2 * (int)H, GemmKind::Tf32x3)
                             : L.route.cell == CellPath::Bf16Gemm  ? gemm_nt_scratch_floats((int)H, 2 * (int)H, GemmKind::Bf16)
                                                                   : 4);
  } else {   // bf16 fused tcgen05 kernels: tile-layout planes
    const size_t nqt = (BN + 127) / 128, plane = T * nqt * 128 * H;
    L.tc_img_f = c.take<unsigned char>(TC_IMG_BYTES);
    L.tc_img_b = c.take<unsigned char>(TC_IMG_BYTES);
    L.Zp = c.take<float>(plane);
    L.Rp = c.take<float>(plane);
    L.Hcp = c.take<float>(plane);
    L.dhp_p = c.take<float>(a->mode == REGT_MODE_REGIONAL ? plane : 4);
    L.Xt = c.take<float>(BN * F * T);
    L.hid_part = c.take<float>(T * nqt * 128 * H);
    L.tc_wpart = c.take<float>((size_t)TC_MAX_CTAS * 128 * 192);
    L.tc_dpp = c.take<float>(T * TC_MAX_CTAS + 64);   // one attention-gradient partial per (CTA, period)
  }
  if (a->precision == REGT_PREC_TF32X3) {   // tensor-core head (head_f.cu)
    L.hf_rh = c.take<float>(BN * H);
    L.hf_do32 = c.take<float>(BN * 32);
    L.hf_split = c.take<float>(max(gemm_nt_scratch_floats(HEAD_HID, (int)H, GemmKind::Tf32x3), gemm_nt_scratch_floats((int)H, HEAD_HID, GemmKind::Tf32x3)));
    L.hf_loss_floats = BN / 8 + 2;
    L.hf_loss = c.take<float>(L.hf_loss_floats);
  }
  L.a1 = c.take<float>(BN * HEAD_HID);
  L.G = c.take<float>(((BN + 127) / 128) * 128 * H);   // padded: the tensor-core backward reads whole 128-row tiles
  L.d_a1 = c.take<float>(BN * HEAD_HID);
  L.dB = c.take<float>(3 * H * H);
  L.dP = c.take<float>(3 * H * F);
  L.dcg = c.take<float>(3 * H);
  L.dM0 = c.take<float>(H * F);
  L.dM1 = c.take<float>(R * H * F);
  L.dc0 = c.take<float>(H);
  L.dprobs = c.take<float>(T);
  size_t pf = (size_t)3 * WGRAD_SPLITS * H * H;                    // H x H split-K partials
  pf = max(pf, (size_t)WGRAD_SPLITS * 4 * H * 32);                  // F-wide partials ([4H][F+1] fp32 path, [4H][32] tf32x3 GEMM)
  pf = max(pf, (size_t)3 * H * H + 2 * 1024 * 64);                     // tf32x3: packed B^T operands + attention partials
  pf = max(pf, (size_t)WGRAD_SPLITS * (3 * H * H + 4 * H * 32));    // tf32x3: H x H and F-wide weight-gradient partials side by side
  pf = max(pf, (size_t)(2048 + R + 2) * H * F);                     // per-region dM1 partials: <= 2048 + R chunks (cell.cu)
  pf = max(pf, (size_t)128 * T);                                    // attention partials
  pf = max(pf, (size_t)128 * (O * HEAD_HID + HEAD_HID * H));        // head split-K partials (<= 128 splits)
  pf = max(pf, (size_t)152 * HEAD_HID * (H + 32));                  // head dW1 on the tensor cores (+ the 32-wide second operand, tf32x3)
  pf = max(pf, BN / 64 + 2);                                        // loss partials
  pf += H * HEAD_HID + HEAD_HID * O + 64;                           // transposed head weights (tail)
  L.hpart = c.take<float>((size_t)148 * (HEAD_HID * H + O * HEAD_HID + HEAD_HID + O + 8));
  L.part = c.take<float>(pf);
  L.part_floats = pf;
  if (feat_in(a) < F && (L.route.cell == CellPath::Fp32 || L.route.cell == CellPath::Tf32x3Unfused || L.route.cell == CellPath::Bf16Gemm))
    L.xw = c.take<float>((size_t)a->B * (a->x_rows > 0 ? a->x_rows : a->N) * F * T);
  // whenever y is set, masked or not: changing a step's loss never grows (and so never re-allocates) its workspace
  if (a->y) {
    L.inv_c = c.take<float>(a->B);
    L.lc_part = c.take<unsigned int>((size_t)a->B * LC_CHUNKS);
  }
  L.m1cp = c.take<int32_t>(R + 2);   // last: tests locate it from the end of the workspace
  L.total = align_up(c.off, 256);
  return L;
}

static int check_features(const regt_args* a, const char* who) {
  REGT_CHECK(a->F >= 0 && a->F <= REGT_F, "%s: F=%d node features; the kernels take 1..%d (0 means %d)", who, a->F, REGT_F,
             REGT_F);
  return 0;
}

// the GEMM-by-GEMM tensor-core cells run the H x H contractions in 32-column boxes
static int check_tc_width(const regt_args* a) {
  if (a->precision == REGT_PREC_TF32X3)
    REGT_CHECK(a->H % 32 == 0, "precision tf32x3 needs hidden %% 32 == 0 (got %d); use precision fp32", a->H);
  if (a->precision == REGT_PREC_BF16)
    REGT_CHECK(a->H % 32 == 0, "precision bf16 needs hidden %% 32 == 0 (got %d); use precision fp32", a->H);
  return 0;
}

static int validate(const regt_args* a, const char* who) {
  REGT_CHECK(a != nullptr, "%s: args is NULL", who);
  if (check_features(a, who)) return -1;
  REGT_CHECK(a->B > 0 && a->N > 0 && a->T > 0 && a->O > 0, "%s: bad dims B=%d N=%d T=%d O=%d", who, a->B, a->N, a->T, a->O);
  REGT_CHECK(a->H >= 8 && a->H % 8 == 0 && a->H <= 1024, "%s: H=%d must be a multiple of 8 in [8,1024]", who, a->H);
  REGT_CHECK(a->mode >= 0 && a->mode <= 2, "%s: bad mode %d", who, a->mode);
  REGT_CHECK(a->loss_kind == REGT_LOSS_MSE || a->loss_kind == REGT_LOSS_MAE, "%s: bad loss_kind %d (0 = MSE, 1 = MAE)", who,
             a->loss_kind);
  REGT_CHECK(!a->loss_masked || a->y, "%s: loss_masked needs y (the mask is read from the targets)", who);
  REGT_CHECK(a->x_rows == 0 || a->x_rows >= a->N, "%s: x_rows=%d must be 0 or >= N=%d", who, a->x_rows, a->N);
  REGT_CHECK(a->plan.N == a->N, "%s: plan built for %d nodes, args say %d", who, a->plan.N, a->N);
  REGT_CHECK((long long)a->B * a->N * a->T < (1ll << 31), "%s: B*N*T overflows int32 rows", who);
  REGT_CHECK(a->workspace && a->workspace_bytes >= regt_workspace_bytes(a), "%s: workspace missing or too small", who);
  REGT_CHECK(a->precision >= 0 && a->precision <= 2, "%s: bad precision %d", who, a->precision);
  REGT_CHECK(a->head_only == 0 || a->head_only == 1, "%s: head_only must be 0 or 1 (got %d)", who, a->head_only);
  return 0;
}

}  // namespace regt

using namespace regt;

extern "C" size_t regt_workspace_bytes(const regt_args* a) {
  if (!a || check_features(a, "regt_workspace_bytes")) return 0;
  return make_layout(a, nullptr).total;
}

extern "C" int regt_cell_forward(const regt_args* a) {
  if (validate(a, "regt_cell_forward")) return -1;
  REGT_CHECK(!a->head_only, "regt_cell_forward: head_only args run no cell (their workspace holds no cell planes)");
  REGT_CHECK(a->x && a->out_hidden, "regt_cell_forward: x / out_hidden is NULL");
  if (check_tc_width(a)) return -1;
  Layout L = make_layout(a, a->workspace);
  cudaStream_t st = (cudaStream_t)a->stream;
  prof_mark("<begin>", st);
  switch (L.route.cell) {
    case CellPath::Fp32: return cell_forward_fp32(a, L, st);
    case CellPath::Tf32x3Unfused: return cell_forward_g(a, L, st);
    case CellPath::Tf32x3Fused: return cell_forward_f(a, L, st);
    case CellPath::Bf16: return cell_forward_tc(a, L, st);
    case CellPath::Bf16Gemm: return cell_forward_g(a, L, st);
  }
  return -1;
}

extern "C" int regt_cell_backward(const regt_args* a) {
  if (validate(a, "regt_cell_backward")) return -1;
  REGT_CHECK(!a->head_only, "regt_cell_backward: head_only args run no cell (their workspace holds no cell planes)");
  REGT_CHECK(!a->inference, "regt_cell_backward: the forward ran with inference=1 (no activations were saved)");
  if (check_tc_width(a)) return -1;
  Layout L = make_layout(a, a->workspace);
  cudaStream_t st = (cudaStream_t)a->stream;
  prof_mark("<begin>", st);
  switch (L.route.cell) {
    case CellPath::Fp32: return cell_backward_fp32(a, L, st);
    case CellPath::Tf32x3Unfused: return cell_backward_g(a, L, st);
    case CellPath::Tf32x3Fused: return cell_backward_f(a, L, st);
    case CellPath::Bf16: return cell_backward_tc(a, L, st);
    case CellPath::Bf16Gemm: return cell_backward_g(a, L, st);
  }
  return -1;
}

static int validate_x(const regt_args* a, const regt_xgrad_plan* xp, const char* who) {
  REGT_CHECK(a != nullptr, "%s: args is NULL", who);
  if (check_features(a, who)) return -1;
  REGT_CHECK(a->precision != REGT_PREC_BF16, "%s: precision bf16 keeps no gate-gradient plane; use fp32 or tf32x3", who);
  REGT_CHECK(a->x_rows == 0 || a->x_rows == a->N,
             "%s: region shards (x_rows=%d != N=%d) are not supported: their halo rows belong to other ranks", who, a->x_rows, a->N);
  REGT_CHECK(!a->inference, "%s: the forward ran with inference=1 (no activations were saved)", who);
  REGT_CHECK(!a->head_only, "%s: head_only args run no cell (their workspace holds no cell planes)", who);
  if (validate(a, who)) return -1;
  REGT_CHECK(xp && xp->N == a->N && xp->n_src == 2 * a->N + a->plan.nseg && xp->rowptr && xp->col && xp->val,
             "%s: transposed plan missing or built for another graph", who);
  return 0;
}

extern "C" size_t regt_cell_backward_x_scratch_bytes(const regt_args* a, const regt_xgrad_plan* xp) {
  if (!a || !xp) return 0;
  return cell_backward_x_scratch_bytes(a, xp);
}

extern "C" int regt_cell_backward_x(const regt_args* a, const regt_xgrad_plan* xp, float* d_x, void* scratch,
                                    size_t scratch_bytes) {
  if (validate_x(a, xp, "regt_cell_backward_x")) return -1;
  REGT_CHECK(d_x, "regt_cell_backward_x: d_x is NULL");
  REGT_CHECK(scratch && scratch_bytes >= cell_backward_x_scratch_bytes(a, xp), "regt_cell_backward_x: scratch missing or too small");
  if (a->precision == REGT_PREC_TF32X3)
    REGT_CHECK(a->H % 32 == 0, "precision tf32x3 needs hidden %% 32 == 0 (got %d); use precision fp32", a->H);
  Layout L = make_layout(a, a->workspace);
  cudaStream_t st = (cudaStream_t)a->stream;
  prof_mark("<begin>", st);
  return cell_backward_x(a, L, xp, d_x, scratch, st);
}

extern "C" int regt_head_forward(const regt_args* a) {
  if (validate(a, "regt_head_forward")) return -1;
  REGT_CHECK(a->out_hidden && a->out, "regt_head_forward: out_hidden / out is NULL");
  Layout L = make_layout(a, a->workspace);
  prof_mark("<begin>", (cudaStream_t)a->stream);
  return head_forward(a, L, (cudaStream_t)a->stream);
}

extern "C" int regt_head_backward(const regt_args* a) {
  if (validate(a, "regt_head_backward")) return -1;
  REGT_CHECK(!a->inference, "regt_head_backward: the forward ran with inference=1 (no activations were saved)");
  Layout L = make_layout(a, a->workspace);
  prof_mark("<begin>", (cudaStream_t)a->stream);
  return head_backward(a, L, (cudaStream_t)a->stream);
}

// TEST HOOK: the kernels route_of picks for these arguments, out = {cell, head, g_tiled, hid_partials} (CellPath, HeadPath;
// cell 5 = none: head_only)
extern "C" int regt_debug_route(const regt_args* a, int32_t* out) {
  REGT_CHECK(a && out, "regt_debug_route: args and out must be non-NULL");
  const Route r = route_of(a);
  out[0] = (int32_t)r.cell;
  out[1] = (int32_t)r.head;
  out[2] = r.g_tiled;
  out[3] = r.hid_partials;
  return 0;
}
