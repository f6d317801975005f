#!/bin/bash
# two-layer [64,64] PFN: parity tests of the streaming two-layer kernel, phase stamps, A/B timing against the general kernel
timeout 900 python -m pytest tests -m gpu -x -q -k "two_layer or general_kernel or full_size or golden" 2>&1 | tail -3
for wl in cfg2_nuscenes32_b16_pillar0.2_bev512 cfg4_waymo64_pillar0.1_bev1024 cfg3_10sweep_p32_b8; do
  timeout 300 python profiles/scripts/phase_times_stack.py $wl 2>&1 | tail -7
  timeout 300 python profiles/scripts/stack_times.py $wl 2>&1 | tail -1
  [ -n "$AB" ] && timeout 300 python profiles/scripts/stack_times.py --generic $wl 2>&1 | tail -1
done
