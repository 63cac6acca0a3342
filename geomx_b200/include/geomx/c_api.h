/*
 * geomx_b200 — flat C ABI (lib/libgeomx_capi.so; the same symbols are exported by the Python extension lib/_C*.so).
 *
 * Role of the reference's include/mxnet/c_api.h + c_predict_api.h for front ends that link no Python: function names and argument order
 * follow the reference with the prefix GX instead of MX.  Every function returns 0 on success and -1 on failure; the message of the last
 * failure of the calling thread is GXRTGetLastError() (KVStore group: GXGetLastError()).  Returned string / array pointers live in
 * thread-local storage of the library and stay valid until the next call of the same function group on the same thread.
 *
 * What executes where: an NDArray handle owns HOST memory (GXNDArrayCreate, GXNDArrayCreateEx with dev_type 1) or float32 DEVICE memory
 * (GXNDArrayCreateEx with dev_type 2, from the native pool).  Executors bound to host arrays compute in float32 on the host
 * (csrc/runtime/train_exec.h); executors bound to device arrays (GXExecutorSimpleBindEx / GXExecutorBind with dev_type 2) and imperative
 * calls on device arrays run sm_100a kernels of libgeomx_kernels.so (csrc/runtime/device_exec.h), which this library loads at the first
 * device request from its own directory — it has no link-time dependency on CUDA.  Device work is ordered on one stream per device in call
 * order; SyncCopyToCPU and the Wait* functions synchronise it.  Functions that read host bytes (Slice / At / Reshape / Detach, autograd,
 * the raw-buffer GXKVStoreInit / Push / Pull, and GXPred* on host predictors) refuse device arrays.  Predictors created with dev_type 2 run
 * on the GPU (csrc/runtime/predict_device.h) and take host or device buffers.  GXKVStoreInitND / PushND / PullND take host or device
 * NDArrays on every store type: `local` reduces on the host, `device` on each key's GPU with peer copies and sm_100a kernels, and the dist
 * stores reduce device values on the GPU before they go on the wire (csrc/runtime/kvstore_nd.h).  The NVLink fabric and mixed precision
 * are driven from the Python package; the dist GXKVStore* types are the TCP parameter-server plane both share.
 *
 * dtype flags: 0 float32, 1 float64, 2 float16, 3 uint8, 4 int32, 5 int8, 6 int64.  grad_req: 0 null, 1 write, 3 add.
 */
#ifndef GEOMX_C_API_H_
#define GEOMX_C_API_H_

#include <stddef.h>
#include <stdbool.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* NDArrayHandle;
typedef void* SymbolHandle;
typedef void* AtomicSymbolCreator;
typedef void* ExecutorHandle;
typedef void* KVStoreHandle;
typedef void* RecordIOHandle;
typedef void* DataIterHandle;
typedef void* DataIterCreator;
typedef void* PredictorHandle;
typedef void* NDListHandle;

const char* GXRTGetLastError(void);
const char* GXGetLastError(void);                       /* KVStore group */
int GXGetVersion(int* out);
int GXRandomSeed(int seed);

/* ---- NDArray ------------------------------------------------------------------------------------------------------------------------- */
int GXNDArrayCreate(const uint32_t* shape, uint32_t ndim, int dtype, NDArrayHandle* out);                                       /* host */
/* dev_type 1 CPU (= GXNDArrayCreate), 2 GPU: float32 device memory on dev_id (zero-filled); GetData then returns the device pointer,
 * GetContext (2, dev_id), SyncCopy* copy host <-> device, Save / SaveRawBytes copy to the host first */
int GXNDArrayCreateEx(const uint32_t* shape, uint32_t ndim, int dev_type, int dev_id, int delay_alloc, int dtype, NDArrayHandle* out);
int GXNDArrayFree(NDArrayHandle h);
int GXNDArrayGetShape(NDArrayHandle h, uint32_t* out_ndim, const uint32_t** out_shape);
int GXNDArrayGetDType(NDArrayHandle h, int* out);
int GXNDArrayGetData(NDArrayHandle h, void** out);
int GXNDArraySyncCopyFromCPU(NDArrayHandle h, const void* data, size_t size_elems);
int GXNDArraySyncCopyToCPU(NDArrayHandle h, void* data, size_t size_elems);
int GXNDArraySave(const char* fname, uint32_t num, NDArrayHandle* handles, const char** keys);      /* byte-compatible .params */
int GXNDArrayLoad(const char* fname, uint32_t* out_size, NDArrayHandle** out_handles, uint32_t* out_name_size, const char*** out_names);
int GXNDArrayCreateNone(NDArrayHandle* out);
int GXNDArraySlice(NDArrayHandle h, uint32_t begin, uint32_t end, NDArrayHandle* out);            /* copies (host arrays do not alias) */
int GXNDArrayAt(NDArrayHandle h, uint32_t idx, NDArrayHandle* out);
int GXNDArrayReshape(NDArrayHandle h, int ndim, const int* dims, NDArrayHandle* out);
int GXNDArrayGetContext(NDArrayHandle h, int* out_dev_type, int* out_dev_id);
int GXNDArrayGetStorageType(NDArrayHandle h, int* out);
int GXNDArrayWaitToRead(NDArrayHandle h);
int GXNDArrayWaitToWrite(NDArrayHandle h);
int GXNDArrayWaitAll(void);
int GXNDArraySaveRawBytes(NDArrayHandle h, size_t* out_size, const char** out_buf);
int GXNDArrayLoadFromRawBytes(const void* buf, size_t size, NDArrayHandle* out);
int GXNDArrayGetGrad(NDArrayHandle h, NDArrayHandle* out);
int GXNDArrayDetach(NDArrayHandle h, NDArrayHandle* out);

/* ---- Symbol -------------------------------------------------------------------------------------------------------------------------- */
int GXListAllOpNames(uint32_t* out_size, const char*** out_array);
int GXSymbolListAtomicSymbolCreators(uint32_t* out_size, AtomicSymbolCreator** out_array);
int GXSymbolGetAtomicSymbolName(AtomicSymbolCreator creator, const char** name);
int GXSymbolGetAtomicSymbolInfo(AtomicSymbolCreator creator, const char** name, const char** description, uint32_t* num_args, const char*** arg_names,
                                const char*** arg_type_infos, const char*** arg_descriptions, const char** key_var_num_args, const char** return_type);
int GXSymbolCreateAtomicSymbol(AtomicSymbolCreator creator, uint32_t num_param, const char** keys, const char** vals, SymbolHandle* out);
int GXSymbolCreateAtomicSymbolByName(const char* op, uint32_t num_param, const char** keys, const char** vals, SymbolHandle* out);
int GXSymbolCreateVariable(const char* name, SymbolHandle* out);
int GXSymbolCreateGroup(uint32_t num, SymbolHandle* symbols, SymbolHandle* out);
int GXSymbolCreateFromJSON(const char* json, SymbolHandle* out);              /* the reference's nnvm dialect or geomx_b200-symbol-1 */
int GXSymbolCreateFromFile(const char* fname, SymbolHandle* out);
int GXSymbolSaveToJSON(SymbolHandle sym, const char** out_json);              /* nnvm dialect */
int GXSymbolSaveToFile(SymbolHandle sym, const char* fname);
int GXSymbolFree(SymbolHandle sym);
int GXSymbolCopy(SymbolHandle sym, SymbolHandle* out);
int GXSymbolPrint(SymbolHandle sym, const char** out_str);
int GXSymbolGetName(SymbolHandle sym, const char** out, int* success);
int GXSymbolGetAttr(SymbolHandle sym, const char* key, const char** out, int* success);
int GXSymbolSetAttr(SymbolHandle sym, const char* key, const char* value);
int GXSymbolListAttr(SymbolHandle sym, uint32_t* out_size, const char*** out);           /* out_size pairs ("node$key", value) */
int GXSymbolListAttrShallow(SymbolHandle sym, uint32_t* out_size, const char*** out);    /* out_size pairs (key, value) */
int GXSymbolListArguments(SymbolHandle sym, uint32_t* out_size, const char*** out);
int GXSymbolListOutputs(SymbolHandle sym, uint32_t* out_size, const char*** out);
int GXSymbolListAuxiliaryStates(SymbolHandle sym, uint32_t* out_size, const char*** out);
int GXSymbolGetNumOutputs(SymbolHandle sym, uint32_t* out);
int GXSymbolGetInternals(SymbolHandle sym, SymbolHandle* out);
int GXSymbolGetChildren(SymbolHandle sym, SymbolHandle* out);
int GXSymbolGetOutput(SymbolHandle sym, uint32_t index, SymbolHandle* out);
int GXSymbolCompose(SymbolHandle sym, const char* name, uint32_t num_args, const char** keys, SymbolHandle* args);   /* keys == NULL: positional */
/* shapes are CSR-packed: argument i has dims shape_data[ind_ptr[i] .. ind_ptr[i+1]); keys == NULL: positional in ListArguments order */
int GXSymbolInferShape(SymbolHandle sym, uint32_t num_args, const char** keys, const uint32_t* ind_ptr, const uint32_t* shape_data, uint32_t* in_shape_size,
                       const uint32_t** in_shape_ndim, const uint32_t*** in_shape_data, uint32_t* out_shape_size, const uint32_t** out_shape_ndim,
                       const uint32_t*** out_shape_data, uint32_t* aux_shape_size, const uint32_t** aux_shape_ndim, const uint32_t*** aux_shape_data, int* complete);
int GXSymbolInferShapePartial(SymbolHandle sym, uint32_t num_args, const char** keys, const uint32_t* ind_ptr, const uint32_t* shape_data, uint32_t* in_shape_size,
                              const uint32_t** in_shape_ndim, const uint32_t*** in_shape_data, uint32_t* out_shape_size, const uint32_t** out_shape_ndim,
                              const uint32_t*** out_shape_data, uint32_t* aux_shape_size, const uint32_t** aux_shape_ndim, const uint32_t*** aux_shape_data, int* complete);
int GXSymbolInferType(SymbolHandle sym, uint32_t num_args, const char** keys, const int* arg_type_data, uint32_t* in_type_size, const int** in_type_data,
                      uint32_t* out_type_size, const int** out_type_data, uint32_t* aux_type_size, const int** aux_type_data, int* complete);

/* ---- Executor (float32; host arrays: host executor, device arrays: device executor) --------------------------------------------------- */
int GXExecutorBind(SymbolHandle sym, int dev_type, int dev_id, uint32_t len, NDArrayHandle* in_args, NDArrayHandle* arg_grad_store, const uint32_t* grad_req_type,
                   uint32_t aux_states_len, NDArrayHandle* aux_states, ExecutorHandle* out);
/* allocates arguments / gradients / auxiliary states from the given input shapes; grad_req "null" | "write" | "add" for every argument
 * except those named in no_grad_keys; the arrays belong to the executor and come back in ListArguments / ListAuxiliaryStates order */
int GXExecutorSimpleBind(SymbolHandle sym, uint32_t num_shapes, const char** keys, const uint32_t* ind_ptr, const uint32_t* shape_data, const char* grad_req,
                         uint32_t num_no_grad, const char** no_grad_keys, ExecutorHandle* out, uint32_t* num_args, NDArrayHandle** in_args, NDArrayHandle** arg_grads,
                         uint32_t* num_aux, NDArrayHandle** aux_states);
/* the same with a device: dev_type 1 = GXExecutorSimpleBind; dev_type 2 allocates device arrays on dev_id and binds the device executor,
 * whose Outputs are device arrays.  Operators outside the device set are refused here with the node's name. */
int GXExecutorSimpleBindEx(SymbolHandle sym, int dev_type, int dev_id, uint32_t num_shapes, const char** keys, const uint32_t* ind_ptr, const uint32_t* shape_data,
                           const char* grad_req, uint32_t num_no_grad, const char** no_grad_keys, ExecutorHandle* out, uint32_t* num_args, NDArrayHandle** in_args,
                           NDArrayHandle** arg_grads, uint32_t* num_aux, NDArrayHandle** aux_states);
int GXExecutorForward(ExecutorHandle h, int is_train);
int GXExecutorBackward(ExecutorHandle h, uint32_t len, NDArrayHandle* head_grads);       /* len 0 for loss heads */
int GXExecutorBackwardEx(ExecutorHandle h, uint32_t len, NDArrayHandle* head_grads, int is_train);
int GXExecutorOutputs(ExecutorHandle h, uint32_t* out_size, NDArrayHandle** out);         /* valid until Free, refreshed by every Forward */
int GXExecutorPrint(ExecutorHandle h, const char** out_str);
int GXExecutorFree(ExecutorHandle h);

/* ---- imperative invoke + autograd ----------------------------------------------------------------------------------------------------
 * Device inputs run the operator on their device (outputs: device arrays on the same device, which may alias an input); sgd_update,
 * sgd_mom_update and adam_update take the optimizer states as trailing inputs and update them in place.  Autograd records host arrays only. */
int GXImperativeInvoke(AtomicSymbolCreator creator, int num_inputs, NDArrayHandle* inputs, int* num_outputs, NDArrayHandle** outputs, int num_params,
                       const char** param_keys, const char** param_vals);
int GXImperativeInvokeByName(const char* op, int num_inputs, NDArrayHandle* inputs, int* num_outputs, NDArrayHandle** outputs, int num_params,
                             const char** param_keys, const char** param_vals);
int GXAutogradSetIsRecording(int is_recording, int* prev);
int GXAutogradSetIsTraining(int is_training, int* prev);
int GXAutogradIsRecording(bool* curr);
int GXAutogradIsTraining(bool* curr);
int GXAutogradMarkVariables(uint32_t num_var, NDArrayHandle* var_handles, const uint32_t* reqs_array, NDArrayHandle* grad_handles);
int GXAutogradBackward(uint32_t num_output, NDArrayHandle* output_handles, NDArrayHandle* ograd_handles, int retain_graph);
int GXAutogradBackwardEx(uint32_t num_output, NDArrayHandle* output_handles, NDArrayHandle* ograd_handles, int retain_graph, int is_train);
int GXAutogradComputeGradient(uint32_t num_output, NDArrayHandle* output_handles);
int GXAutogradGetSymbol(NDArrayHandle handle, SymbolHandle* out);

/* ---- RecordIO ------------------------------------------------------------------------------------------------------------------------ */
int GXRecordIOWriterCreate(const char* uri, RecordIOHandle* out);
int GXRecordIOWriterFree(RecordIOHandle h);
int GXRecordIOWriterWriteRecord(RecordIOHandle h, const char* buf, size_t size);
int GXRecordIOWriterTell(RecordIOHandle h, size_t* pos);
int GXRecordIOReaderCreate(const char* uri, RecordIOHandle* out);
int GXRecordIOReaderFree(RecordIOHandle h);
int GXRecordIOReaderReadRecord(RecordIOHandle h, const char** buf, size_t* size);         /* *buf == NULL at end of file */
int GXRecordIOReaderSeek(RecordIOHandle h, size_t pos);
int GXRecordIOReaderTell(RecordIOHandle h, size_t* pos);

/* ---- data iterators (MNISTIter, CSVIter) ---------------------------------------------------------------------------------------------- */
int GXListDataIters(uint32_t* out_size, DataIterCreator** out_array);
int GXDataIterGetIterInfo(DataIterCreator creator, const char** name, const char** description, uint32_t* num_args, const char*** arg_names,
                          const char*** arg_type_infos, const char*** arg_descriptions);
int GXDataIterCreateIter(DataIterCreator creator, uint32_t num_param, const char** keys, const char** vals, DataIterHandle* out);
int GXDataIterFree(DataIterHandle h);
int GXDataIterBeforeFirst(DataIterHandle h);
int GXDataIterNext(DataIterHandle h, int* out);
int GXDataIterGetData(DataIterHandle h, NDArrayHandle* out);                              /* owned by the iterator */
int GXDataIterGetLabel(DataIterHandle h, NDArrayHandle* out);
int GXDataIterGetIndex(DataIterHandle h, uint64_t** out_index, uint64_t* out_size);
int GXDataIterGetPadNum(DataIterHandle h, int* pad);

/* ---- KVStore --------------------------------------------------------------------------------------------------------------------------
 * GXKVStoreCreate types: "local", "local_update_cpu", "local_allreduce_cpu" — in-process, values reduced and kept on the host;
 * "device", "local_allreduce_device" — in-process, each key kept and reduced on its home GPU (the device of the value given to Init);
 * any other type (dist_sync, dist_async, ...) — a worker of the HiPS TCP parameter-server plane (two tiers).
 * In-process stores: GetRank 0, GroupSize 1, Barrier / Wait* do nothing, SetGradientCompression("2bit") on device stores only; the raw-buffer
 * Init / Push / Pull, the row-sparse forms and RunServer are refused (use the ND forms). */
int GXInitPSEnv(int num, const char** keys, const char** vals);
int GXKVStoreIsWorkerNode(int* out);
int GXKVStoreIsServerNode(int* out);
int GXKVStoreIsSchedulerNode(int* out);
int GXKVStoreCreate(const char* type, KVStoreHandle* out);
int GXKVStoreFree(KVStoreHandle h);
int GXKVStoreGetRank(KVStoreHandle h, int* out);
int GXKVStoreGetGroupSize(KVStoreHandle h, int* out);
int GXKVStoreGetNumAllWorkers(KVStoreHandle h, int* out);
int GXKVStoreIsMasterWorker(KVStoreHandle h, int* out);
int GXKVStoreInit(KVStoreHandle h, int key, const void* data, size_t elems, int dtype);
int GXKVStorePush(KVStoreHandle h, int key, const void* data, size_t elems, int dtype, int priority, int* handle);
int GXKVStorePull(KVStoreHandle h, int key, void* out, size_t elems, int dtype, int priority, int* handle);
int GXKVStorePushRowSparse(KVStoreHandle h, int key, const int64_t* row_ids, size_t nrows, const float* rows, size_t row_len, int priority, int* handle);
int GXKVStorePullRowSparse(KVStoreHandle h, int key, const int64_t* row_ids, size_t nrows, float* out, size_t row_len, int priority, int* handle);
/* NDArray forms, host or device arrays (device arrays: float32).  Push: a key listed k times is k values, summed left to right in the
 * order given, then stored (or handed to the updater) or sent once.  Pull: a key listed k times fills k outputs.  Init: a key may appear
 * once and be initialised once.  The values of one key in one call are all host or all device arrays.  Local / device stores never block
 * on device arrays: copies and sums are ordered on the devices' streams, so later work issued on any device sees the result.  Dist stores:
 * PushND reduces device values on their GPU (and quantises them there under 2-bit compression), synchronises that GPU once and sends
 * asynchronously; PullND requests every key of the call, waits for all replies (the keys of one call share their round trips), then
 * enqueues the copies to the device outputs and returns. */
int GXKVStoreInitND(KVStoreHandle h, uint32_t num, const int* keys, NDArrayHandle* vals);
int GXKVStorePushND(KVStoreHandle h, uint32_t num, const int* keys, NDArrayHandle* vals, int priority);
int GXKVStorePullND(KVStoreHandle h, uint32_t num, const int* keys, NDArrayHandle* vals, int priority);
/* local / device stores: updater(key, recv, local, arg) replaces the assignment of a push; recv holds the reduced sum and local the stored
 * value, both on the key's home (device arrays for a device key, so GXImperativeInvokeByName("sgd_update", ...) on them runs on the GPU).
 * The handles belong to the store.  Dist stores update on their servers (command 7, or GXKVStoreRunServerEx) and refuse this call. */
typedef void (*GXKVStoreUpdater)(int key, NDArrayHandle recv, NDArrayHandle local, void* arg);
int GXKVStoreSetUpdater(KVStoreHandle h, GXKVStoreUpdater updater, void* arg);
int GXKVStoreWait(KVStoreHandle h, int handle);
int GXKVStoreWaitAll(KVStoreHandle h);
int GXKVStoreBarrier(KVStoreHandle h);
int GXKVStoreSendCommmandToServers(KVStoreHandle h, int head, const char* body);
int GXKVStoreSetGradientCompression(KVStoreHandle h, const char* type, float threshold);
int GXKVStoreGetNumDeadNode(KVStoreHandle h, int node_id, int timeout_sec, int* out);
int GXKVStoreGetType(KVStoreHandle h, const char** out);
typedef void (*GXKVController)(int head, const char* body, void* arg);
typedef void (*GXKVUpdater)(int key, const float* grad, float* weight, size_t n, void* arg);
int GXKVStoreRunServer(KVStoreHandle h);
int GXKVStoreRunServerEx(KVStoreHandle h, GXKVController controller, void* controller_arg, GXKVUpdater updater, void* updater_arg);
int GXKVStoreShutdown(KVStoreHandle h);

/* ---- profiler / engine / storage ------------------------------------------------------------------------------------------------------ */
int GXSetProfilerConfig(int num, const char* const* keys, const char* const* vals);
int GXSetProfilerState(int state);
int GXProfilePause(int paused);
int GXDumpProfile(int finished);
int GXProfileSetMarker(const char* name, const char* category);
int GXProfileAddDuration(const char* name, const char* category, double start_us, double dur_us);
double GXProfileNowUs(void);
typedef void* ProfileHandle;
int GXProfileCreateDomain(const char* domain, ProfileHandle* out);
int GXProfileCreateTask(ProfileHandle domain, const char* name, ProfileHandle* out);
int GXProfileCreateFrame(ProfileHandle domain, const char* name, ProfileHandle* out);
int GXProfileCreateEvent(const char* name, ProfileHandle* out);
int GXProfileCreateCounter(ProfileHandle domain, const char* name, ProfileHandle* out);
int GXProfileDestroyHandle(ProfileHandle h);
int GXProfileDurationStart(ProfileHandle h);
int GXProfileDurationStop(ProfileHandle h);
int GXProfileSetCounter(ProfileHandle h, uint64_t value);
int GXProfileAdjustCounter(ProfileHandle h, int64_t delta);
int GXSetNumOMPThreads(int n);
int GXGetNumOMPThreads(int* out);
int GXEngineSetBulkSize(int size, int* prev);
int GXGetGPUCount(int* out);
int GXNotifyShutdown(void);
typedef void (*GXEngineFn)(void* arg);
int GXEngineNewVariable(int* out);
int GXEnginePushAsync(GXEngineFn fn, void* arg, const int* const_vars, int num_const, const int* mutable_vars, int num_mutable, int priority, const char* name);
int GXEnginePushAsyncEx(GXEngineFn fn, void* arg, const int* const_vars, int num_const, const int* mutable_vars, int num_mutable, int priority, const char* name,
                        int device, int prop);
int GXEngineDeleteVariable(int var);
int GXEngineWaitForVar(int var);
int GXEngineWaitAll(void);
int GXStorageAlloc(size_t nbytes, void** out);
int GXStorageFree(void* p);

/* ---- predict API (include/mxnet/c_predict_api.h) --------------------------------------------------------------------------------------- */
/* dev_type 1: the host (the planned predictor, or the general executor for operators outside its set).  dev_type 2: the planned predictor
 * on GPU dev_id with sm_100a kernels; create refuses a graph it cannot serve (the error names the node).  A device handle owns a stream,
 * an arena and its input buffers, shares the parameters with its MultiThread / Reshape siblings, and may be driven from its own thread.
 * SetInput copies in (host or device memory) and returns when the source has been read; Forward is asynchronous, the first one runs
 * eagerly and every later one replays a CUDA graph; GetOutput waits and copies out (host or device memory); Free waits for the stream. */
int GXPredCreate(const char* symbol_json, const void* param_bytes, int param_size, int dev_type, int dev_id, uint32_t num_input_nodes, const char** input_keys,
                 const uint32_t* input_shape_indptr, const uint32_t* input_shape_data, PredictorHandle* out);
int GXPredCreatePartialOut(const char* symbol_json, const void* param_bytes, int param_size, int dev_type, int dev_id, uint32_t num_input_nodes,
                           const char** input_keys, const uint32_t* input_shape_indptr, const uint32_t* input_shape_data, uint32_t num_output_nodes,
                           const char** output_keys, PredictorHandle* out);
int GXPredCreateMultiThread(const char* symbol_json, const void* param_bytes, int param_size, int dev_type, int dev_id, uint32_t num_input_nodes,
                            const char** input_keys, const uint32_t* input_shape_indptr, const uint32_t* input_shape_data, int num_threads, PredictorHandle* out);
int GXPredReshape(uint32_t num_input_nodes, const char** input_keys, const uint32_t* input_shape_indptr, const uint32_t* input_shape_data, PredictorHandle handle,
                  PredictorHandle* out);
int GXPredGetOutputShape(PredictorHandle handle, uint32_t index, uint32_t** shape_data, uint32_t* shape_ndim);
int GXPredGetNumOutputs(PredictorHandle handle, uint32_t* out);
int GXPredSetInput(PredictorHandle handle, const char* key, const float* data, uint32_t size);
int GXPredForward(PredictorHandle handle);
int GXPredPartialForward(PredictorHandle handle, int step, int* step_left);
int GXPredGetOutput(PredictorHandle handle, uint32_t index, float* data, uint32_t size);
int GXPredGetPlan(PredictorHandle handle, uint64_t* arena_bytes, uint32_t* num_ops);
int GXPredGetEngine(PredictorHandle handle, int* out);        /* 1 planned predictor, 2 general executor (operators outside the planned set), 3 planned predictor on a GPU */
int GXPredFree(PredictorHandle handle);
int GXNDListCreate(const char* nd_file_bytes, int nd_file_size, NDListHandle* out, uint32_t* out_length);
int GXNDListGet(NDListHandle handle, uint32_t index, const char** out_key, const float** out_data, const uint32_t** out_shape, uint32_t* out_ndim);
int GXNDListFree(NDListHandle handle);

#ifdef __cplusplus
}
#endif
#endif  /* GEOMX_C_API_H_ */
