#!/bin/bash
# A/B of the symmetric Chamfer scan launch forms on the GPU box (tools/variants/symp = nn_variants.cu built in-tree):
#   grid (one CTA per work item) vs balanced (2 CTAs/SM, equal unit ranges).
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
export GENPC_CHAMFER_MODE=sym
for form in grid balanced; do
  case $form in
    grid) export GENPC_SYM_BALANCED=0 ;;
    balanced) export GENPC_SYM_BALANCED=1 ;;
  esac
  ./tools/variants/symp | sed "s/\"variant\": \"/\"variant\": \"SYM $form /"
done
