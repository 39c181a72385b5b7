#!/bin/bash
# device timeline (ELECTOR_TRACE=2) of single-chunk pipelined calls through the C driver, for the current library and,
# when elector_b200/libelector_poa_old.so exists, for that older build (A/B of scheduling changes)
python tools/dump_csr.py ${1:-10000} 1 /tmp/tr_c1 > /dev/null
export ELECTOR_PIPELINE_CHUNKS=1 ELECTOR_PIPELINE_WORKERS=1 ELECTOR_TRACE=2
run() { echo "=== $1"; shift; env "$@" elector_b200/bin/pipe_driver /tmp/tr_c1 4 2>&1 | grep -v "^call 0" | tail -${TAILN:-14}; }
run "current"  X=1
if [ -f elector_b200/libelector_poa_old.so ]; then mkdir -p /tmp/oldlib; cp elector_b200/libelector_poa_old.so /tmp/oldlib/libelector_poa.so; TAILN=40 run "old build" LD_LIBRARY_PATH=/tmp/oldlib; fi
