# attention kernel tests (under a timeout: a protocol bug traps after the watchdog)
timeout 600 python -m pytest tests/test_kernels_gpu.py -x -q -m gpu -p no:cacheprovider -k "attention" 2>&1 | tail -5
