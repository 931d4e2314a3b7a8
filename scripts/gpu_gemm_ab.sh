# GEMM / conv kernel tests
timeout 900 python -m pytest tests/test_kernels_gpu.py tests/test_unet_gpu.py -x -q -m gpu -p no:cacheprovider 2>&1 | tail -4
