#!/bin/bash
# Builds libmmlst.so in-tree for sm_100a (B200).  nvcc cross-compiles without a GPU.
set -e
cd "$(dirname "$0")"
NVCC=${NVCC:-/usr/local/cuda/bin/nvcc}
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-O3,-Wall -Xptxas -v"
SRCS="api.cu select.cu score.cu score_runs.cu coverage.cu pileup_atomic.cu pileup_bitsliced.cu consensus.cu contig_stats.cu hamming.cu hamming_exact.cu hamming_tc.cu st_match.cu ingest.cu de.cu allreduce.cu exchange.cu"
OBJS=""
for s in $SRCS; do
  o="${s%.cu}.o"
  if [ ! -f "$o" ] || [ "$s" -nt "$o" ] || [ common.cuh -nt "$o" ] || [ pileup.cuh -nt "$o" ] || [ score_runs_kernels.cuh -nt "$o" ] || [ ingest_core.cuh -nt "$o" ] || [ bgzf_crc.cuh -nt "$o" ] || [ de.h -nt "$o" ] || [ ../../include/mmlst.h -nt "$o" ]; then
    $NVCC $FLAGS -c "$s" -o "$o" 2> "${s%.cu}.ptxas.log" || { cat "${s%.cu}.ptxas.log"; exit 1; }
  fi
  OBJS="$OBJS $o"
done
EXTRA=""
if [ -f bam_unpack.cpp ]; then
  g++ -O3 -std=c++17 -fPIC -Wall -pthread -c bam_unpack.cpp -o bam_unpack.o
  g++ -O3 -std=c++17 -fPIC -Wall -c inflate_fast.cpp -o inflate_fast.o
  OBJS="$OBJS bam_unpack.o inflate_fast.o"; EXTRA="-lz -lpthread -ldl"
fi
$NVCC -gencode arch=compute_100a,code=sm_100a -shared -o ../libmmlst.so $OBJS $EXTRA
echo "built $(cd .. && pwd)/libmmlst.so"
