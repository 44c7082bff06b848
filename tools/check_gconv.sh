#!/bin/bash
timeout 600 python -m pytest tests/test_gpu_1_kernels.py -m gpu -x -q -k gconv 2>&1 | tail -4
