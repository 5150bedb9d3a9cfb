// K2 orchestration: a validated, pre-encoded list of ops (conv / maxpool / avgpool / stem im2col) executed
// back to back on one stream.  The host (pd_fusion_b200/backbone.py) builds the list from a torchvision-layout
// state_dict; this file replaces the Python-side `for i in range(0, L, batch_size): model(batch)` loop of
// data/openneuro_features.py:257-261 with one call over all slices of all subjects in the batch.
#include <vector>

#include "common.cuh"
#include "ops.cuh"

struct pdf_plan {
  std::vector<pdf_op> ops;
  std::vector<pdf::TcConv> tc;   // parallel to ops (only meaningful for bf16 convs)
  double flops = 0.0;
};

using namespace pdf;

static int validate_op(const pdf_op& op, int i) {
  PDF_REQUIRE(op.kind >= PDF_OP_CONV && op.kind <= PDF_OP_STEM_FUSED, "op %d: unknown kind %d", i, op.kind);
  PDF_REQUIRE(op.precision == PDF_PREC_F32 || op.precision == PDF_PREC_BF16, "op %d: bad precision", i);
  PDF_REQUIRE(op.n > 0 && op.h > 0 && op.w > 0 && op.c > 0, "op %d: bad input shape", i);
  PDF_REQUIRE(op.d_in && op.d_out, "op %d: null in/out pointer", i);
  if (op.kind == PDF_OP_CONV) {
    PDF_REQUIRE(op.k > 0 && op.r > 0 && op.s > 0 && op.stride > 0 && op.pad >= 0 && op.ho > 0 && op.wo > 0 && op.d_weight,
                "op %d: bad conv description", i);
    PDF_REQUIRE(op.ho == (op.h + 2 * op.pad - op.r) / op.stride + 1 && op.wo == (op.w + 2 * op.pad - op.s) / op.stride + 1,
                "op %d: inconsistent conv output size", i);
  }
  if (op.sc_c || op.sc_hw) {          // shortcut segment: x at stride 1 when its size equals the output's, else at stride 2
    const int sc_h = op.sc_hw >> 16, sc_w = op.sc_hw & 0xffff;
    PDF_REQUIRE(op.kind == PDF_OP_CONV && op.precision == PDF_PREC_BF16 && op.r == 1 && op.s == 1 && op.stride == 1 && op.pad == 0 &&
                !op.out_f32 && op.sc_c > 0 && op.sc_c % 64 == 0 && op.c % 64 == 0 && op.d_residual && sc_h > 0 && sc_w > 0,
                "op %d: a shortcut segment needs a bf16 1x1 stride-1 conv with bf16 output, c and sc_c multiples of 64, d_residual = x", i);
    PDF_REQUIRE((sc_h == op.ho && sc_w == op.wo) || (op.ho == (sc_h - 1) / 2 + 1 && op.wo == (sc_w - 1) / 2 + 1),
                "op %d: shortcut input %dx%d is neither the output size %dx%d nor its stride-2 source", i, sc_h, sc_w, op.ho, op.wo);
  }
  if (op.kind == PDF_OP_MAXPOOL)
    PDF_REQUIRE(op.ho == (op.h + 2 - 3) / 2 + 1 && op.wo == (op.w + 2 - 3) / 2 + 1, "op %d: maxpool is 3x3 s2 p1", i);
  if (op.kind == PDF_OP_STEM_IM2COL)
    PDF_REQUIRE(op.precision == PDF_PREC_BF16 && op.c == 1 && op.k % 8 == 0 && op.k >= 56 && op.ho == (op.h + 6 - 7) / 2 + 1 &&
                op.wo == (op.w + 6 - 7) / 2 + 1, "op %d: stem im2col is 7x7 s2 p3 on one bf16 channel, kpad multiple of 8", i);
  if (op.kind == PDF_OP_STEM_FUSED) {
    const int h1 = (op.h + 6 - 7) / 2 + 1;
    PDF_REQUIRE(op.precision == PDF_PREC_BF16 && op.c == 1 && op.k == 64 && op.h == op.w && op.ho == op.wo &&
                op.ho == (h1 + 2 - 3) / 2 + 1 && op.d_weight && op.d_bias, "op %d: fused stem is 7x7 s2 p3 (1 -> 64 ch) + maxpool 3x3 s2 p1", i);
  }
  return PDF_OK;
}

extern "C" int pdf_plan_create(pdf_plan** out, const pdf_op* ops, int n_ops) {
  PDF_REQUIRE(out && ops && n_ops > 0, "pdf_plan_create: bad arguments");
  int ndev = 0;
  PDF_CHECK_CUDA(cudaGetDeviceCount(&ndev));
  PDF_REQUIRE(ndev > 0, "pdf_plan_create: no CUDA device");
  pdf_plan* plan = new pdf_plan();
  plan->ops.assign(ops, ops + n_ops);
  plan->tc.resize(n_ops);
  for (int i = 0; i < n_ops; ++i) {
    const pdf_op& op = plan->ops[i];
    int rc = validate_op(op, i);
    if (rc == PDF_OK && op.kind == PDF_OP_STEM_FUSED) rc = prepare_stem_tc(op, &plan->tc[i]);
    if (rc == PDF_OK && op.kind == PDF_OP_STEM_FUSED) plan->flops += 2.0 * op.n * ((op.h - 1) / 2 + 1) * ((op.w - 1) / 2 + 1) * 64.0 * 49.0;
    if (rc == PDF_OK && op.kind == PDF_OP_CONV) {
      plan->flops += 2.0 * op.n * op.ho * op.wo * (double)op.k * op.r * op.s * (op.c + op.sc_c);   // (+ the shortcut segment's K)
      if (op.d_weight2) {
        plan->flops += 2.0 * op.n * op.ho * op.wo * (double)op.k * op.c;
        if (op.precision != PDF_PREC_BF16) {
          set_error("op %d: a fused 1x1 convolution exists on the bf16 path only", i);
          rc = PDF_ERR_ARG;
        }
      }
      if (op.d_weight3) {
        plan->flops += 2.0 * op.n * op.ho * op.wo * (double)op.k3 * op.k;
        if (op.precision != PDF_PREC_BF16) {
          set_error("op %d: a chained 1x1 convolution exists on the bf16 path only", i);
          rc = PDF_ERR_ARG;
        }
      }
      if (rc == PDF_OK && op.precision == PDF_PREC_BF16) rc = prepare_conv_tc(op, &plan->tc[i]);
    }
    if (rc != PDF_OK) { delete plan; return rc; }
  }
  *out = plan;
  return PDF_OK;
}

extern "C" int pdf_plan_run_range(const pdf_plan* plan, int first, int count, pdf_stream_t stream) {
  PDF_REQUIRE(plan && first >= 0 && count >= 0 && first + count <= (int)plan->ops.size(), "pdf_plan_run_range: bad range");
  cudaStream_t s = as_stream(stream);
  for (int i = first; i < first + count; ++i) {
    const pdf_op& op = plan->ops[i];
    int rc = PDF_OK;
    switch (op.kind) {
      case PDF_OP_CONV: rc = (op.precision == PDF_PREC_BF16) ? launch_conv_tc(plan->tc[i], s) : launch_conv_f32(op, s); break;
      case PDF_OP_MAXPOOL: rc = launch_maxpool(op, s); break;
      case PDF_OP_AVGPOOL: rc = launch_avgpool(op, s); break;
      case PDF_OP_STEM_IM2COL: rc = launch_stem_im2col(op, s); break;
      case PDF_OP_STEM_FUSED: rc = launch_stem_fused(op, plan->tc[i].tmap_b, plan->tc[i].tmap_a, s); break;
    }
    if (rc != PDF_OK) return rc;
  }
  return PDF_OK;
}

extern "C" int pdf_plan_run(const pdf_plan* plan, pdf_stream_t stream) {
  PDF_REQUIRE(plan, "pdf_plan_run: null plan");
  return pdf_plan_run_range(plan, 0, (int)plan->ops.size(), stream);
}

extern "C" void pdf_plan_destroy(pdf_plan* plan) { delete plan; }
extern "C" double pdf_plan_flops(const pdf_plan* plan) { return plan ? plan->flops : 0.0; }
