#!/bin/bash
# Rotating KV cache (max_kv_size): its GPU tests and the end-to-end decode with a ring against the flat cache, in one
# call on a GPU host.  Usage: OUT_DIR=DIR bash tools/gpu_ring.sh TAG [tests|decode|all|suite]
# (suite: the whole GPU suite, smoke and the default bench line); results go to DIR (default ring_out/).
TAG=${1:-ring}
WHAT=${2:-all}
O=${OUT_DIR:-ring_out}; mkdir -p $O
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/${TAG}_gpu.txt 2>&1
if [[ $WHAT == suite ]]; then
  timeout 1500 python -m pytest tests -m gpu -q > $O/${TAG}_pytest.log 2>&1; echo "pytest rc=$?" >> $O/${TAG}_pytest.log; tail -3 $O/${TAG}_pytest.log
  timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > $O/${TAG}_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $O/${TAG}_smoke.log
  timeout 400 python bench.py --gpus 1 > $O/${TAG}_bench.json 2> $O/${TAG}_bench.err; cat $O/${TAG}_bench.json
fi
if [[ $WHAT == tests || $WHAT == all ]]; then
  timeout 900 python -m pytest tests/test_gpu_rotating_cache.py -m gpu -q > $O/${TAG}_pytest_ring.log 2>&1
  echo "pytest rc=$?" >> $O/${TAG}_pytest_ring.log; tail -4 $O/${TAG}_pytest_ring.log
fi
if [[ $WHAT == decode || $WHAT == all || $WHAT == suite ]]; then
  # 3B at a 32 768-token prompt: the flat cache against a 4096-position ring, bf16 / 8-bit / 4-bit
  timeout 1500 python tools/decode_bench.py --model llama-3.2-3b --prompt 32768 --quantized-kv-start 32767 \
    --kv-bits none,8,4 --max-kv-size none,4096 --repeat 1 \
    > $O/${TAG}_decode_llama-3.2-3b_p32768.json 2> $O/${TAG}_decode_3b.err; echo "decode 3b rc=$?"
  cat $O/${TAG}_decode_llama-3.2-3b_p32768.json
  # 8B, 1000-token prompt, 4000 generated tokens on a 2048-position ring (wraps at token 1048) against the flat cache:
  # the captured step at positions before and after the wrap, device tokens against host tokens
  timeout 1500 python tools/decode_bench.py --model llama-3-8b --prompt 1000 --tokens 4000 --max-kv-size none,2048 \
    --graph-positions 2047,2048,3000,4000,4999 --repeat 1 \
    > $O/${TAG}_decode_llama-3-8b_p1000_t4000.json 2> $O/${TAG}_decode_8b.err; echo "decode 8b rc=$?"
  cat $O/${TAG}_decode_llama-3-8b_p1000_t4000.json
fi
