/*
 * The GPU twin of dist_train_cnn.c: data-parallel training of the demo CNN over the HiPS parameter server, every process a plain C program,
 * the workers computing on the device:
 *   GXExecutorSimpleBindEx(dev_type 2)   device arrays + the device executor (sm_100a kernels)
 *   GXKVStoreInitND / PullND             rank 0's initial weights, copied into the device arrays of every worker
 *   GXKVStorePushND                      ONE call with every gradient per step; with two visible GPUs a second executor on device 1 lists the
 *                                        same keys, so the push first sums both devices' gradients on device 0, then sends one message per key
 *   GXKVStorePullND                      ONE call with every weight per step: all round trips at once, then copies into both devices' arrays
 * The server sums the workers' pushes and applies SGD natively (the spec travels as server command 7; rescale_grad averages over workers and
 * devices); the scheduler does rendezvous and barriers.
 *
 *   gcc -O2 -I geomx_b200/include examples/c_api/dist_train_cnn_gpu.c -L geomx_b200/lib -lgeomx_capi -Wl,-rpath,$PWD/geomx_b200/lib -lm -o dist_train_cnn_gpu
 *   export DMLC_PS_ROOT_URI=127.0.0.1 DMLC_PS_ROOT_PORT=9092 DMLC_NUM_SERVER=1 DMLC_NUM_WORKER=2 DMLC_NUM_ALL_WORKER=2
 *   DMLC_ROLE=scheduler ./dist_train_cnn_gpu & DMLC_ROLE=server ./dist_train_cnn_gpu & DMLC_ROLE=worker ./dist_train_cnn_gpu 40 & DMLC_ROLE=worker ./dist_train_cnn_gpu 40
 */
#define BATCH 16
#include "cnn_common.h"

#define KCK(call) do { if ((call) != 0) { fprintf(stderr, "%s:%d: %s\n", __FILE__, __LINE__, GXGetLastError()); exit(1); } } while (0)
#define MAXP 16

int main(int argc, char** argv) {
  const int steps = argc > 1 ? atoi(argv[1]) : 40;
  KVStoreHandle kv;
  int is_worker = 0, rank = 0, nworkers = 1, ngpu = 0, ndev, d;
  KCK(GXKVStoreIsWorkerNode(&is_worker));
  KCK(GXKVStoreCreate("dist_sync", &kv));
  if (!is_worker) {                                        /* scheduler / server: serve until the workers end the job */
    KCK(GXKVStoreRunServer(kv));
    KCK(GXKVStoreFree(kv));
    return 0;
  }
  KCK(GXKVStoreGetRank(kv, &rank)); KCK(GXKVStoreGetGroupSize(kv, &nworkers));
  CK(GXGetGPUCount(&ngpu));
  if (ngpu < 1) { fprintf(stderr, "no CUDA device\n"); return 1; }
  ndev = ngpu >= 2 ? 2 : 1;
  if (rank == 0) {
    char spec[160];
    snprintf(spec, sizeof spec, "name=sgd;lr=0.1;wd=0.0;rescale_grad=%.9g;clip_gradient=-1.0;momentum=0.0", 1.0 / (nworkers * ndev));
    KCK(GXKVStoreSendCommmandToServers(kv, 7, spec));
  }
  {
    SymbolHandle net = build();
    uint32_t nargs, naux, i, nout, np = 0;
    const char** names;
    const char* shape_keys[] = {"data"};
    const uint32_t ind[] = {0, 4}, dims[] = {B, 1, 28, 28};
    const char* no_grad[] = {"data", "softmax_label"};
    ExecutorHandle ex[2];
    NDArrayHandle *args, *grads, *aux, *outs;
    NDArrayHandle arg_copy[2][MAXP], grad_copy[2][MAXP];
    NDArrayHandle push_vals[2 * MAXP], pull_outs[2 * MAXP];
    int keys[2 * MAXP], pidx[MAXP], data_i = -1, label_i = -1, step;
    static float X[B * 784], y[B], prob[B * 10], host_w[256 * 512];
    float first = 0, last = 0;
    double checksum = 0;

    for (d = 0; d < ndev; ++d) {
      CK(GXExecutorSimpleBindEx(net, 2, d, 1, shape_keys, ind, dims, "write", 2, no_grad, &ex[d], &nargs, &args, &grads, &naux, &aux));
      memcpy(arg_copy[d], args, nargs * sizeof(NDArrayHandle)); memcpy(grad_copy[d], grads, nargs * sizeof(NDArrayHandle));
    }
    CK(GXSymbolListArguments(net, &nargs, &names));
    for (i = 0; i < nargs; ++i) {
      if (!strcmp(names[i], "data")) data_i = (int)i;
      else if (!strcmp(names[i], "softmax_label")) label_i = (int)i;
      else pidx[np++] = (int)i;
    }
    /* every worker draws its own initial values on the host; Init keeps rank 0's, the pull makes every device of every worker start there */
    rng_state = 777u + 1000u * (uint32_t)rank;
    for (i = 0; i < np; ++i) {
      const int a = pidx[i];
      size_t n = numel(arg_copy[0][a]), k;
      uint32_t nd; const uint32_t* s;
      if (n > sizeof host_w / sizeof host_w[0]) { fprintf(stderr, "parameter %s too large\n", names[a]); return 1; }
      CK(GXNDArrayGetShape(arg_copy[0][a], &nd, &s));
      for (k = 0; k < n; ++k) host_w[k] = nd > 1 ? (2.0f * frand() - 1.0f) * sqrtf(3.0f / (float)(n / s[0])) : 0.0f;
      CK(GXNDArraySyncCopyFromCPU(arg_copy[0][a], host_w, n));
      keys[i] = a; push_vals[i] = arg_copy[0][a];
    }
    KCK(GXKVStoreInitND(kv, np, keys, push_vals));
    for (d = 0; d < ndev; ++d)
      for (i = 0; i < np; ++i) { keys[d * np + i] = pidx[i]; pull_outs[d * np + i] = arg_copy[d][pidx[i]]; push_vals[d * np + i] = grad_copy[d][pidx[i]]; }
    KCK(GXKVStorePullND(kv, np * ndev, keys, pull_outs, 0));
    rng_state = 4242u + 99u * (uint32_t)rank;                /* different data on every worker and device */
    for (step = 0; step < steps; ++step) {
      float loss = 0; int b;
      for (d = 0; d < ndev; ++d) {
        make_batch(X, y);
        CK(GXNDArraySyncCopyFromCPU(arg_copy[d][data_i], X, B * 784)); CK(GXNDArraySyncCopyFromCPU(arg_copy[d][label_i], y, B));
        CK(GXExecutorForward(ex[d], 1)); CK(GXExecutorBackward(ex[d], 0, NULL));
        if (d == 0) {
          CK(GXExecutorOutputs(ex[0], &nout, &outs)); CK(GXNDArraySyncCopyToCPU(outs[0], prob, B * 10));
          for (b = 0; b < B; ++b) loss -= logf(prob[b * 10 + (int)y[b]] + 1e-12f) / B;
        }
      }
      if (step == 0) first = loss;
      last = loss;
      KCK(GXKVStorePushND(kv, np * ndev, keys, push_vals, 0));
      KCK(GXKVStorePullND(kv, np * ndev, keys, pull_outs, 0));
      if (step % 10 == 0) printf("rank %d step %d loss %.4f (%d device%s)\n", rank, step, loss, ndev, ndev > 1 ? "s" : "");
    }
    for (i = 0; i < np; ++i) {
      const int a = pidx[i];
      size_t n = numel(arg_copy[0][a]), k;
      CK(GXNDArraySyncCopyToCPU(arg_copy[0][a], host_w, n));
      for (k = 0; k < n; ++k) checksum += (double)host_w[k] * (double)(1 + (k + (size_t)a) % 7);
    }
    printf("FINAL rank %d of %d loss %.4f -> %.4f checksum %.6f\n", rank, nworkers, first, last, checksum);
    for (d = 0; d < ndev; ++d) CK(GXExecutorFree(ex[d]));
    CK(GXSymbolFree(net));
  }
  KCK(GXKVStoreFree(kv));
  return 0;
}
