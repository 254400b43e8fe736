#!/bin/bash
# k_step_lean variants (scripts/build_variant.sh <tag> -D...) timed side by side in one visit: fp64, L=4096, 24 iterations.
t() { python scripts/prof_fp64.py 4096 24 2>&1 | tail -1 | python -c "import json,sys; d=json.loads(sys.stdin.read()); print('   ', round(d['us_per_iteration'],1), d['path'][9:45])"; }
echo "main"; t
echo "b4"; SPGG_B200_LIB=$PWD/build/libspgg_b4.so t   # -DSPGG_LEAN_BATCH=4
echo "tr8 8x128thr"; SPGG_B200_LIB=$PWD/build/libspgg_tr8.so SPGG_GEN_TR=8 SPGG_GEN_THREADS=128 t
echo "tr8 8x256thr"; SPGG_B200_LIB=$PWD/build/libspgg_tr8.so SPGG_GEN_TR=8 SPGG_GEN_THREADS=256 t
echo "main 16x128thr(tr16 layout)"; SPGG_GEN_TR=16 SPGG_GEN_THREADS=128 t
echo "main again"; t
