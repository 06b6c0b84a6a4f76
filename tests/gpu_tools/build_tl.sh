#!/bin/bash
# Developer tool: lib/libmlstm_b200_tl.so = the regular objects with the fused backward rebuilt under -DMLSTM_TIMELINE
set -e
cd "$(dirname "$0")/../../xlstm_yolo_b200"
python -m xlstm_yolo_b200.build >/dev/null 2>&1 || (cd .. && python -m xlstm_yolo_b200.build >/dev/null)
nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo --expt-relaxed-constexpr -Xcompiler -fPIC -DMLSTM_TIMELINE \
  -c csrc/mlstm_tc_bwd_fused.cu -o lib/mlstm_tc_bwd_fused_tl.o
OBJS=$(ls lib/*.o | grep -v "_tl.o" | grep -v "mlstm_tc_bwd_fused.o")
nvcc -shared -o lib/libmlstm_b200_tl.so $OBJS lib/mlstm_tc_bwd_fused_tl.o -lcudart_static -ldl -lrt -lpthread
ls -la lib/libmlstm_b200_tl.so
