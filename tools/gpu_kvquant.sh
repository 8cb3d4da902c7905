#!/bin/bash
# Quantized-KV decode: its GPU tests, the attention kernel benchmark and the end-to-end decode with --kv-bits none / 8 / 4,
# in one call on a GPU host.  Usage: OUT_DIR=DIR bash tools/gpu_kvquant.sh TAG [tests|kernel|decode|all|suite]
# (suite: the whole GPU suite, smoke and the default bench line); results go to DIR (default kvquant_out/).
TAG=${1:-kvq}
WHAT=${2:-all}
O=${OUT_DIR:-kvquant_out}; mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/${TAG}_gpu.txt 2>&1
if [[ $WHAT == tests || $WHAT == all ]]; then
  timeout 900 python -m pytest tests/test_gpu_kv_quant.py -m gpu -q > $O/${TAG}_pytest_kvquant.log 2>&1
  echo "pytest rc=$?" >> $O/${TAG}_pytest_kvquant.log; tail -4 $O/${TAG}_pytest_kvquant.log
fi
if [[ $WHAT == kernel || $WHAT == all ]]; then
  timeout 600 python tools/kvbench.py --out $O/${TAG}_kvbench.json > $O/${TAG}_kvbench.txt 2>&1; echo "kvbench rc=$?"
  grep -E "^#|keys   32768" $O/${TAG}_kvbench.txt
fi
if [[ $WHAT == decode || $WHAT == all ]]; then
  timeout 900 python tools/decode_bench.py --model llama-3-8b --prompt 8000 --quantized-kv-start 7999 --kv-bits none,8,4 \
    --repeat 1 > $O/${TAG}_decode_llama-3-8b_p8000.json 2> $O/${TAG}_decode_8b.err; echo "decode 8b rc=$?"
  cat $O/${TAG}_decode_llama-3-8b_p8000.json
  timeout 1200 python tools/decode_bench.py --model llama-3.2-3b --prompt 32768 --quantized-kv-start 32767 --kv-bits none,8,4 \
    --repeat 1 > $O/${TAG}_decode_llama-3.2-3b_p32768.json 2> $O/${TAG}_decode_3b.err; echo "decode 3b rc=$?"
  cat $O/${TAG}_decode_llama-3.2-3b_p32768.json
fi
if [[ $WHAT == suite ]]; then
  timeout 900 python -m pytest tests -m gpu -q > $O/${TAG}_pytest.log 2>&1; echo "pytest rc=$?" >> $O/${TAG}_pytest.log; tail -3 $O/${TAG}_pytest.log
  timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > $O/${TAG}_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $O/${TAG}_smoke.log
  timeout 400 python bench.py --gpus 1 > $O/${TAG}_bench.json 2> $O/${TAG}_bench.err; cat $O/${TAG}_bench.json
fi
