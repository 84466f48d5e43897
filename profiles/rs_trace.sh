#!/bin/bash
# phase breakdown of k_rs_score (prologue / scoring / flush / ticket / column sums / selection) from %globaltimer stamps
# usage: bash profiles/rs_trace.sh TAG
TAG=${1:-r2}
O=gpurun_out
mkdir -p $O
APC_RS_TRACE=1 python -m autodriver_pointcloud_preprocessor_b200._build --force > /dev/null 2>&1
python profiles/rs_trace.py > $O/rs_trace_$TAG.txt 2>&1; echo "trace rc=$?"
python -m autodriver_pointcloud_preprocessor_b200._build --force > /dev/null 2>&1
cat $O/rs_trace_$TAG.txt | tail -12
