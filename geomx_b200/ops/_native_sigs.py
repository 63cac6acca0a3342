"""ctypes signatures of ``libgeomx_kernels.so`` (flat C ABI; see ``csrc/kernels/*.cu`` ``GX_API`` functions)."""
import ctypes as C

P, I, L, F, U = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_uint32

SIGS = {
    # gemm_tcgen05.cu
    "gx_gemm_tf32": [P, L, I, P, L, I, I, I, I, P, L, P, P, L, P, I, I, I, I, F, I, P],
    "gx_gemm_tf32_pool": [P, L, I, P, L, I, I, I, I, P, P, I, I, I, P, F, P],
    "gx_mlp_chain_fwd_bwd": [P] * 17 + [I] * 5 + [P],
    "gx_cnn_fwd": [P] * 11 + [I, P, I, P],
    "gx_cnn_bwd": [P] * 9 + [I, P],
    "gx_cnn_wgrad1": [P] * 6 + [I, P],
    "gx_cnn_bwd_all": [P] * 11 + [I, P],
    "gx_cnn_bwd_exchange": [P] * 11 + [I, P, P, I, P],
    "gx_depthwise_fwd": [P, P, P, P] + [I] * 11 + [P],
    "gx_depthwise_dgrad": [P, P, P] + [I] * 10 + [P],
    "gx_depthwise_wgrad": [P, P, P, P] + [I] * 10 + [P],
    "gx_cnn_set_debug": [P],
    "gx_mlp_chain_smem_bytes": [],
    "gx_mlp_chain_set_debug": [P],
    "gx_gemm_set_debug": [P],
    "gx_gemm_set_precision": [I],
    "gx_gemm_get_precision": [],
    "gx_gemm_simt": [P, L, I, P, L, I, I, I, I, P, L, P, P, L, P, I, I, I, I, F, P],
    # conv_pool.cu
    "gx_im2col": [P, P, I, I, I, I, I, I, I, I, I, I, I, P],
    "gx_col2im": [P, P, I, I, I, I, I, I, I, I, I, I, I, P],
    "gx_nchw_to_rows": [P, P, I, I, I, P],
    "gx_colsum": [P, P, L, I, L, I, P],
    "gx_chansum_nchw": [P, P, I, I, I, P],
    "gx_relu_fwd": [P, P, L, P],
    "gx_relu_bwd": [P, P, P, L, P],
    "gx_maxpool2x2_fwd": [P, P, P, L, I, I, P],
    "gx_maxpool2x2_bwd": [P, P, P, L, I, I, P],
    "gx_pool_relu_bwd_rows": [P, P, P, P, P, I, I, I, I, P],
    "gx_conv_relu_pool_fwd": [P, P, P, P, P, I, I, I, I, I, I, I, P],
    "gx_conv_relu_pool_wgrad": [P, P, P, P, P, P, I, I, I, I, I, I, I, P],
    "gx_conv_relu_pool_im2col_fwd": [P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, P],
    "gx_conv_relu_pool_wgrad_col2im": [P, P, P, P, P, P, I, I, I, I, I, I, I, I, I, I, P],
    # loss_head.cu
    "gx_softmax_ce_fwd": [P, P, P, I, I, P],
    "gx_softmax_ce_bwd": [P, P, P, P, I, I, P],
    "gx_head_fwd_bwd": [P, P, P, P, P, P, P, P, P, P, I, I, I, I, P],
    # optim.cu
    "gx_arena_opt": [I, P, P, P, P, L, P, F, F, F, F, F, F, F, F, F, P, P, P],
    "gx_multi_tensor_opt": [I, P, I, L, F, F, F, F, F, F, F, F, F, P],
    "gx_single_opt": [I, P, P, P, P, L, F, F, F, F, F, F, F, F, F, P],
    "gx_nary_sum": [P, P, I, L, P],
    "gx_scale_cast": [P, I, P, I, F, L, P],
    # compress.cu
    "gx_quantize_2bit": [P, P, P, L, F, P],
    "gx_dequantize_2bit": [P, P, L, F, I, P],
    "gx_bsc_compress_batch": [P, I, I, F, P],
    "gx_bsc_pull_compress_batch": [P, I, P],
    "gx_bsc_decompress": [P, P, L, I, I, P],
    "gx_fp8_block_quantize": [P, P, P, P, L, P],
    "gx_fp8_block_dequantize": [P, P, P, L, I, P],
    "gx_dgt_contrib": [P, P, L, I, F, I, P],
    "gx_bsc_seg_size": [],
    # batchnorm.cu
    "gx_bn_fwd": [P, P, P, P, P, P, P, P, I, I, I, I, F, F, P],
    "gx_bn_bwd": [P, P, P, P, P, P, P, P, I, I, I, P],
    # predict_ops.cu
    "gx_map_fwd": [I, P, P, L, F, F, P],
    "gx_channel_affine": [P, P, P, P, L, I, L, P],
    "gx_transpose": [P, P, I, P, P, P],
    "gx_embedding_fwd": [P, P, P, L, L, L, P],
    "gx_im2col_dilated": [P, P] + [I] * 13 + [P],
    # kv_comm.cu
    "gx_kv_sum_quantize": [P, P, I, L, P, P, F, P],
    "gx_kv_dequant_sum": [P, P, I, L, F, I, P],
    # graph_ops.cu (runtime calls of the C API)
    "gx_rt_memcpy_peer": [P, I, P, I, C.c_ulonglong, P],
    "gx_rt_stream_join": [P, P, I],
    "gx_rt_host_alloc": [C.c_ulonglong, P],
    "gx_rt_host_free": [P],
    # hips_fabric.cu
    "gx_fabric_params_size": [],
    "gx_hips_fsa_step": [P, I, P],
    "gx_hips_fsa_ll_step": [P, I, P],
    "gx_hips_fsa_direct_step": [P, I, P],
    "gx_hips_max_grid": [],
    "gx_hips_async_step": [P, P, P, P, I, I, I, P],
    "gx_hips_party_allreduce": [P, P, P, F, I, I, I, P],
    "gx_fabric_barrier": [P, I, I, I, P, P],
    "gx_fabric_probe": [P, P, P, P, P, I, I, P],
    "gx_unique_i64": [P, I, P, P, P, P, C.c_longlong, P],
    "gx_gather_rows": [P, P, P, I, I, P],
    "gx_scatter_rows": [P, P, P, I, I, I, P],
}


def declare(lib):
    for name, args in SIGS.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    # storage_gpu.cu (device memory pool): pointer / 64-bit returns
    U64 = C.c_uint64
    for name, args, res in (("gx_gpu_pool_create_sim", [I, U64, I, U64, I, I], I), ("gx_gpu_pool_destroy", [I], I), ("gx_gpu_pool_alloc", [I, U64, P], P),
                            ("gx_gpu_pool_free", [I, P, P], I), ("gx_gpu_pool_release_all", [I], I), ("gx_gpu_pool_round_size", [I, U64], U64),
                            ("gx_gpu_pool_stats", [I, C.POINTER(U64)], I)):
        fn = getattr(lib, name); fn.argtypes = args; fn.restype = res
    lib.gx_unique_i64_workspace.argtypes = [C.c_int]
    lib.gx_unique_i64_workspace.restype = C.c_longlong
