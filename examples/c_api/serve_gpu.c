/*
 * Serving a checkpoint on the GPU through the C predict API only — no Python, no PyTorch:
 *   GXPredCreate(dev_type 1)   the host predictor
 *   GXPredCreate(dev_type 2)   the same graph and parameters on a GPU (sm_100a kernels; the second Forward on is one CUDA graph launch)
 * Both serve one seeded batch; the program prints the max relative difference max|gpu - cpu| / max|cpu| of every output.
 *
 *   gcc -O2 -I geomx_b200/include examples/c_api/serve_gpu.c -L geomx_b200/lib -lgeomx_capi -Wl,-rpath,$PWD/geomx_b200/lib -lm -o serve_gpu
 *   ./serve_gpu model-symbol.json model-0000.params [batch C H W] [device]
 * Exit codes: 0 the two agree within 1e-4, 1 a C API call failed, 2 a file is unreadable, 3 the two disagree.
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include "geomx/c_api.h"

#define CK(x)                                                                     \
  do {                                                                            \
    if ((x) != 0) {                                                               \
      fprintf(stderr, "%s:%d %s failed: %s\n", __FILE__, __LINE__, #x, GXRTGetLastError()); \
      exit(1);                                                                    \
    }                                                                             \
  } while (0)

static char* slurp(const char* path, long* size) {
  FILE* f = fopen(path, "rb");
  char* buf;
  if (!f) return NULL;
  fseek(f, 0, SEEK_END);
  *size = ftell(f);
  fseek(f, 0, SEEK_SET);
  buf = (char*)malloc((size_t)*size + 1);
  if (buf && fread(buf, 1, (size_t)*size, f) != (size_t)*size) { free(buf); buf = NULL; }
  if (buf) buf[*size] = '\0';
  fclose(f);
  return buf;
}

static float* serve(int dev_type, int dev, const char* json, const char* params, long psize, const uint32_t* dims, const float* x, uint32_t n, uint32_t index,
                    uint32_t* out_size) {
  const char* keys[] = {"data"};
  const uint32_t ind[] = {0, 4};
  PredictorHandle h;
  uint32_t *shape, ndim, i, size = 1;
  float* y;
  int engine, rep;
  CK(GXPredCreate(json, params, (int)psize, dev_type, dev, 1, keys, ind, dims, &h));
  CK(GXPredGetEngine(h, &engine));
  CK(GXPredSetInput(h, "data", x, n));
  for (rep = 0; rep < 3; ++rep) CK(GXPredForward(h));      /* eager, captured, replayed */
  CK(GXPredGetOutputShape(h, index, &shape, &ndim));
  for (i = 0; i < ndim; ++i) size *= shape[i];
  y = (float*)malloc(size * sizeof(float));
  CK(GXPredGetOutput(h, index, y, size));
  printf("dev_type %d: engine %d, output %u: %u values\n", dev_type, engine, index, size);
  CK(GXPredFree(h));
  *out_size = size;
  return y;
}

int main(int argc, char** argv) {
  long jsize, psize;
  char *json, *params;
  uint32_t dims[4] = {8, 3, 224, 224}, n, i, index, nout, cs, gs;
  int dev = argc > 7 ? atoi(argv[7]) : 0, worst_bad = 0;
  float* x;
  double worst = 0;
  PredictorHandle probe;
  const char* keys[] = {"data"};
  const uint32_t ind[] = {0, 4};
  uint64_t seed = 12345;
  if (argc < 3) { fprintf(stderr, "usage: %s model-symbol.json model.params [batch C H W] [device]\n", argv[0]); return 2; }
  for (i = 0; i < 4 && (int)(3 + i) < argc; ++i) dims[i] = (uint32_t)atoi(argv[3 + i]);
  json = slurp(argv[1], &jsize);
  params = slurp(argv[2], &psize);
  if (!json || !params) { fprintf(stderr, "cannot read %s or %s\n", argv[1], argv[2]); return 2; }
  n = dims[0] * dims[1] * dims[2] * dims[3];
  x = (float*)malloc(n * sizeof(float));
  for (i = 0; i < n; ++i) {                                 /* seeded uniform [-1, 1) */
    seed = seed * 6364136223846793005ULL + 1442695040888963407ULL;
    x[i] = (float)((seed >> 40) / 8388608.0 - 1.0);
  }
  CK(GXPredCreate(json, params, (int)psize, 1, 0, 1, keys, ind, dims, &probe));
  CK(GXPredGetNumOutputs(probe, &nout));
  CK(GXPredFree(probe));
  for (index = 0; index < nout; ++index) {
    float* c = serve(1, dev, json, params, psize, dims, x, n, index, &cs);
    float* g = serve(2, dev, json, params, psize, dims, x, n, index, &gs);
    double num = 0, den = 0, r;
    if (cs != gs) { fprintf(stderr, "output %u: %u values on the host, %u on the GPU\n", index, cs, gs); return 3; }
    for (i = 0; i < cs; ++i) {
      const double d = fabs((double)g[i] - (double)c[i]), m = fabs((double)c[i]);
      if (d > num || d != d) num = d;
      if (m > den) den = m;
    }
    r = num / (den > 1e-30 ? den : 1e-30);
    printf("output %u: max relative difference %.3g\n", index, r);
    if (r > worst || r != r) worst = r;
    if (!(r <= 1e-4)) worst_bad = 1;
    free(c); free(g);
  }
  printf("max relative difference over %u output(s): %.3g (bound 1e-4)\n", nout, worst);
  free(x); free(json); free(params);
  return worst_bad ? 3 : 0;
}
