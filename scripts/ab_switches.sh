#!/bin/bash
# Every documented A/B switch still yields a correct library: the parity tests of the path it touches, once per switch.
run() {  # run VAR=value "k expression" files...
  local setting=$1 kexpr=$2; shift 2
  echo "== $setting"
  if [ -n "$kexpr" ]; then env "$setting" python -m pytest -q -m gpu -x "$@" -k "$kexpr" 2>&1 | tail -1
  else env "$setting" python -m pytest -q -m gpu -x "$@" 2>&1 | tail -1; fi
}
run PSGLA_CONV_FUSE2=0 "dncnn_forward or psgla_replay or reference_fixture or fused_layer" tests/test_image_gpu.py
