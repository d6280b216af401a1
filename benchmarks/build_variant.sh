#!/bin/bash
# build_variant.sh NAME [-D...]: libmmr_b200 with extra defines -> <package>/build/libmmr_NAME.so (experiments; MMR_LIB_PATH selects it)
set -e
NAME=$1; shift
P=$(dirname "$0")/../multimodal-rag-for-image-text-search_b200
mkdir -p $P/build/v_$NAME
F="-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC"
nvcc $F "$@" -c -o $P/build/v_$NAME/mmr_b200.o $P/csrc/mmr_b200.cu &
nvcc $F "$@" -c -o $P/build/v_$NAME/mmr_encoder.o $P/csrc/mmr_encoder.cu &
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $P/build/libmmr_$NAME.so $P/build/v_$NAME/mmr_b200.o $P/build/v_$NAME/mmr_encoder.o
echo built $NAME
