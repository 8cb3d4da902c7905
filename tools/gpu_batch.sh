#!/bin/bash
# Batched generation with per-row prompt lengths: the whole GPU suite, smoke, the default bench line, batch_generate on
# the 8B checkpoint at B = 1 / 4 / 16 / 32 (equal and ragged prompt lengths, bf16 and 4-bit caches) and the batch-1
# 8B decode line of r07, in one call on a GPU host.
# Usage: OUT_DIR=DIR [PARENT_TREE=DIR] bash tools/gpu_batch.sh TAG [all|decode]  (decode: the benchmarks of
# batch_generate and the batch-1 line only)
# PARENT_TREE: a built checkout of the parent commit; its bench line and batch-1 decode line are run in the same call,
# alternating with this tree's, so that the two are compared at one state of the machine.
TAG=${1:-batch}
WHAT=${2:-all}
O=${OUT_DIR:-batch_out}; mkdir -p $O
P=${PARENT_TREE:-}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/${TAG}_gpu.txt 2>&1; cat $O/${TAG}_gpu.txt
if [[ $WHAT == all ]]; then
timeout 1800 python -m pytest tests -m gpu -q > $O/${TAG}_pytest.log 2>&1; echo "pytest rc=$?" >> $O/${TAG}_pytest.log
tail -3 $O/${TAG}_pytest.log; grep -E "^(FAILED|ERROR)" $O/${TAG}_pytest.log | head -20
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > $O/${TAG}_smoke.log 2>&1; echo "smoke rc=$?"; tail -1 $O/${TAG}_smoke.log
for i in 1 2; do
  timeout 400 python bench.py --gpus 1 > $O/${TAG}_bench_$i.json 2> $O/${TAG}_bench_$i.err; echo "bench $i rc=$?"
  cut -c1-220 $O/${TAG}_bench_$i.json
  if [[ -n $P ]]; then
    (cd $P && timeout 400 python bench.py --gpus 1) > $O/${TAG}_bench_parent_$i.json 2> $O/${TAG}_bench_parent_$i.err
    echo "parent bench $i rc=$?"; cut -c1-220 $O/${TAG}_bench_parent_$i.json
  fi
done
fi
# batch_generate: 8B bpw-4.0, 512-token prompts (ragged: 256 .. 512), 128 tokens per row
for R in "" "--ragged"; do
  N=$([[ -n $R ]] && echo ragged || echo equal)
  timeout 1500 python tools/decode_bench.py --model llama-3-8b --prompt 512 --tokens 128 --batch 1,4,16,32 $R \
    --kv-bits none,4 --repeat 2 > $O/${TAG}_batch_llama-3-8b_p512_t128_$N.json 2> $O/${TAG}_batch_$N.err
  echo "batch $N rc=$?"; cut -c1-400 $O/${TAG}_batch_llama-3-8b_p512_t128_$N.json
done
# the batch-1 line of r07 (8B, 1000-token prompt, 4000 tokens, flat and 2048-position ring): the glue kernels it runs
# read their position through the per-row path now
timeout 1500 python tools/decode_bench.py --model llama-3-8b --prompt 1000 --tokens 4000 --max-kv-size none,2048 \
  --graph-positions 2047,2048,3000,4000,4999 --repeat 1 \
  > $O/${TAG}_decode_llama-3-8b_p1000_t4000.json 2> $O/${TAG}_decode_8b.err; echo "decode 8b rc=$?"
cut -c1-700 $O/${TAG}_decode_llama-3-8b_p1000_t4000.json
if [[ -n $P ]]; then
  (cd $P && timeout 1500 python tools/decode_bench.py --model llama-3-8b --prompt 1000 --tokens 4000 --max-kv-size none \
    --graph-positions 2047,3000 --repeat 1) > $O/${TAG}_decode_parent_llama-3-8b_p1000_t4000.json 2> $O/${TAG}_decode_parent_8b.err
  echo "parent decode 8b rc=$?"; cut -c1-700 $O/${TAG}_decode_parent_llama-3-8b_p1000_t4000.json
fi
