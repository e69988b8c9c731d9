#!/bin/bash
# streaming NHWC 3x3: CTA shape sweep (variant libraries from tools/build_variant.sh)
P=knowledge-distillation-by-replacing-cheap-conv_b200
for lib in libkdcc.so libkdcc_w4o3.so libkdcc_w8o1.so; do
  [ -f $P/$lib ] || continue
  echo "== $lib: $(KDCC_LIB=$PWD/$P/$lib timeout -s KILL 120 python tools/time_dw_nhwc.py 2>&1 | tail -3 | tr '\n' '|')"
done
