#!/bin/bash
# A/B of two builds of the ranking kernel on one box: alternating processes, config 3 at 100k queries.
for i in 1 2 3; do
  for lib in "$@"; do
    HOLE_B200_LIB=$lib PROBE_Q3=100000 PROBE_ENV=$(basename $lib) python tools/rank_probe.py 2>&1 | grep "^rank "
  done
done
