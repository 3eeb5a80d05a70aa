python -m pytest tests/test_gpu_parity.py tests/test_jar_vectors.py tests/test_gpu_fuzz.py -m gpu -x -q -k "long or random_case_against or tie" 2>&1 | tail -4
PLAAC_LONG_TIES=1 python -m pytest tests/test_gpu_parity.py -m gpu -q -k "long_sequences or mixed_batch" 2>&1 | tail -2
