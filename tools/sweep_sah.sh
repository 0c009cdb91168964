#!/bin/bash
# Sweep the own-tree build knobs (env) over a few workloads; each run in its own process with a timeout.
cd "$(dirname "$0")/.."
for scene in ${SCENES:-c2_spot c3_renault}; do
  for leaf in ${LEAFS:-2 4 6}; do
    for ct in ${CTS:-50 100 200}; do
      for st in ${STACKS:-24}; do
        echo -n "leaf=$leaf ct=$ct stack=$st  "
        MFX_SAH_TRAV_COST_PCT=$ct MFX_STACK_SMEM=$st timeout 120 python tools/ab_env.py MFX_SAH_MAX_LEAF $leaf $scene ${SPP:-8} 3 rebuild 2>&1 | tail -1
      done
    done
  done
done
