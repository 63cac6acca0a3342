/*
 * The GPU twin of train_cnn.c: the reference's demo CNN trained on the device through the flat C ABI only — no Python, no PyTorch:
 *   GXExecutorSimpleBindEx(dev_type 2)   device arrays + the device executor (sm_100a kernels)
 *   GXNDArraySyncCopyFromCPU             Xavier initialisation on the host, copied to the device
 *   GXImperativeInvokeByName("sgd_update", out = weight)   the update on the device, in place
 *   GXNDArraySave                        checkpoint from the device arrays, served with the host GXPredCreate(dev_type 1)
 *
 *   gcc -O2 -I geomx_b200/include examples/c_api/train_cnn_gpu.c -L geomx_b200/lib -lgeomx_capi -Wl,-rpath,$PWD/geomx_b200/lib -lm -o train_cnn_gpu
 *   ./train_cnn_gpu [steps] [prefix] [device]
 * Exit codes as train_cnn.c: 0 trained and served, 1 a C API call failed, 2 checkpoint unreadable, 3 predictor disagrees, 4 the loss did not halve.
 */
#define _POSIX_C_SOURCE 199309L
#include <time.h>

#include "cnn_common.h"

static double now_ms(void) { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return t.tv_sec * 1e3 + t.tv_nsec / 1e6; }

int main(int argc, char** argv) {
  const int steps = argc > 1 ? atoi(argv[1]) : 60;
  const char* prefix = argc > 2 ? argv[2] : "/tmp/geomx_capi_cnn_gpu";
  const int dev = argc > 3 ? atoi(argv[3]) : 0;
  SymbolHandle net = build();
  uint32_t nargs, naux, i, nout;
  const char** names;
  const char* shape_keys[] = {"data"};
  const uint32_t ind[] = {0, 4}, dims[] = {B, 1, 28, 28};
  const char* no_grad[] = {"data", "softmax_label"};
  const char* sgd_keys[] = {"lr"};
  const char* sgd_vals[] = {"0.1"};
  ExecutorHandle ex;
  NDArrayHandle *args, *grads, *aux, *outs;
  NDArrayHandle arg_copy[16], grad_copy[16];
  char arg_names[16][64];
  static float X[B * 784], y[B], prob[B * 10], host_w[256 * 512];
  float first = 0, last = 0;
  int step, data_i = -1, label_i = -1, timed = 0;
  double t0 = 0;

  CK(GXExecutorSimpleBindEx(net, 2, dev, 1, shape_keys, ind, dims, "write", 2, no_grad, &ex, &nargs, &args, &grads, &naux, &aux));
  memcpy(arg_copy, args, nargs * sizeof(NDArrayHandle)); memcpy(grad_copy, grads, nargs * sizeof(NDArrayHandle));     /* the lists are thread-local returns */
  CK(GXSymbolListArguments(net, &nargs, &names));
  for (i = 0; i < nargs; ++i) { strncpy(arg_names[i], names[i], 63); arg_names[i][63] = 0; }
  for (i = 0; i < nargs; ++i) {
    size_t n = numel(arg_copy[i]), k;
    if (!strcmp(arg_names[i], "data")) { data_i = (int)i; continue; }
    if (!strcmp(arg_names[i], "softmax_label")) { label_i = (int)i; continue; }
    if (n > sizeof host_w / sizeof host_w[0]) { fprintf(stderr, "parameter %s too large\n", arg_names[i]); return 1; }
    if (strstr(arg_names[i], "weight")) {                       /* uniform Xavier over fan-in, drawn on the host */
      uint32_t nd; const uint32_t* s; float scale;
      CK(GXNDArrayGetShape(arg_copy[i], &nd, &s));
      scale = sqrtf(3.0f / (float)(n / s[0]));
      for (k = 0; k < n; ++k) host_w[k] = (2.0f * frand() - 1.0f) * scale;
    } else for (k = 0; k < n; ++k) host_w[k] = 0.0f;
    CK(GXNDArraySyncCopyFromCPU(arg_copy[i], host_w, n));
  }
  for (step = 0; step < steps; ++step) {
    float loss = 0; int b;
    if (step == 2) { CK(GXNDArrayWaitAll()); t0 = now_ms(); }   /* two warm-up steps */
    make_batch(X, y);
    CK(GXNDArraySyncCopyFromCPU(arg_copy[data_i], X, B * 784));
    CK(GXNDArraySyncCopyFromCPU(arg_copy[label_i], y, B));
    CK(GXExecutorForward(ex, 1));
    CK(GXExecutorBackward(ex, 0, NULL));
    CK(GXExecutorOutputs(ex, &nout, &outs));
    CK(GXNDArraySyncCopyToCPU(outs[0], prob, B * 10));
    for (b = 0; b < B; ++b) loss -= logf(prob[b * 10 + (int)y[b]] + 1e-12f) / B;
    if (step == 0) first = loss;
    last = loss;
    for (i = 0; i < nargs; ++i) {                              /* SGD, lr 0.1, on the device: weight = sgd_update(weight, grad) */
      NDArrayHandle in[2]; NDArrayHandle* out; int nout_upd = 1;
      if ((int)i == data_i || (int)i == label_i) continue;
      in[0] = arg_copy[i]; in[1] = grad_copy[i]; out = &arg_copy[i];
      CK(GXImperativeInvokeByName("sgd_update", 2, in, &nout_upd, &out, 1, sgd_keys, sgd_vals));
    }
    if (step >= 2) ++timed;
    if (step % 10 == 0 || step + 1 == steps) printf("step %d loss %.4f\n", step, loss);
  }
  CK(GXNDArrayWaitAll());
  if (timed > 0) printf("%.3f ms/step over %d steps (host clock, device synchronised)\n", (now_ms() - t0) / timed, timed);
  /* checkpoint from the device arrays in the reference's format, then serve it through the host predict API */
  {
    char fsym[512], fpar[512], keys[16][80];
    const char* kp[16]; NDArrayHandle hp[16]; uint32_t n = 0;
    PredictorHandle pred; FILE* f; long sz; char* json; char* blob; long psz;
    const char* in_keys[] = {"data"};
    uint32_t agree = 0; int b, c;
    static float pprob[B * 10];
    snprintf(fsym, sizeof fsym, "%s-symbol.json", prefix); snprintf(fpar, sizeof fpar, "%s-0001.params", prefix);
    CK(GXSymbolSaveToFile(net, fsym));
    for (i = 0; i < nargs; ++i) {
      if ((int)i == data_i || (int)i == label_i) continue;
      snprintf(keys[n], 80, "arg:%.70s", arg_names[i]); kp[n] = keys[n]; hp[n] = arg_copy[i]; ++n;
    }
    CK(GXNDArraySave(fpar, n, hp, kp));
    f = fopen(fsym, "rb"); fseek(f, 0, SEEK_END); sz = ftell(f); fseek(f, 0, SEEK_SET); json = (char*)calloc((size_t)sz + 1, 1); if (fread(json, 1, (size_t)sz, f) != (size_t)sz) return 2; fclose(f);
    f = fopen(fpar, "rb"); fseek(f, 0, SEEK_END); psz = ftell(f); fseek(f, 0, SEEK_SET); blob = (char*)malloc((size_t)psz); if (fread(blob, 1, (size_t)psz, f) != (size_t)psz) return 2; fclose(f);
    CK(GXPredCreate(json, blob, (int)psz, 1, 0, 1, in_keys, ind, dims, &pred));
    CK(GXPredSetInput(pred, "data", X, B * 784));
    CK(GXPredForward(pred));
    CK(GXPredGetOutput(pred, 0, pprob, B * 10));
    CK(GXNDArraySyncCopyFromCPU(arg_copy[data_i], X, B * 784));
    CK(GXExecutorForward(ex, 0));
    CK(GXExecutorOutputs(ex, &nout, &outs));
    CK(GXNDArraySyncCopyToCPU(outs[0], prob, B * 10));
    for (b = 0; b < B; ++b) {
      int pa = 0, pb = 0;
      for (c = 1; c < 10; ++c) { if (prob[b * 10 + c] > prob[b * 10 + pa]) pa = c; if (pprob[b * 10 + c] > pprob[b * 10 + pb]) pb = c; }
      agree += pa == pb && fabsf(prob[b * 10 + pa] - pprob[b * 10 + pb]) < 1e-4f;
    }
    printf("loss %.4f -> %.4f; predictor agrees with the device executor on %u/%d examples\n", first, last, agree, B);
    CK(GXPredFree(pred)); free(json); free(blob);
    if (agree != B) return 3;
  }
  CK(GXExecutorFree(ex)); CK(GXSymbolFree(net));
  return last < 0.5f * first ? 0 : 4;
}
