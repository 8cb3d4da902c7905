#!/bin/bash
# Speculative decoding on a GPU host: the whole GPU suite and smoke; the single-token decode-step ops bit for bit
# against the parent build; the default bench line and the batch-1 8B decode line (this tree and the parent,
# alternating); tools/spec_bench.py.  The GPU's name and power limit go next to the numbers.
# Usage: OUT_DIR=DIR [PARENT_TREE=DIR] bash tools/gpu_spec.sh TAG [all|ab|bench]
#   all: suite, smoke, bitwise comparison, bench and decode lines; ab: the bitwise comparison only; bench: spec_bench.py
# PARENT_TREE: a built checkout of the parent commit.
TAG=${1:-spec}
WHAT=${2:-all}
O=${OUT_DIR:-spec_out}; mkdir -p $O
P=${PARENT_TREE:-}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $O/${TAG}_gpu.txt 2>&1; cat $O/${TAG}_gpu.txt
if [[ $WHAT == all ]]; then
  timeout 1800 python -m pytest tests -m gpu -q -s > $O/${TAG}_pytest.log 2>&1; echo "pytest rc=$?" >> $O/${TAG}_pytest.log
  tail -3 $O/${TAG}_pytest.log; grep -E "^(FAILED|ERROR)" $O/${TAG}_pytest.log | head -20
  grep -E "acceptance:|llama-3.2-1b k=" $O/${TAG}_pytest.log | head -12
  timeout 120 python -c "import __graft_entry__ as g; g.smoke()" > $O/${TAG}_smoke.log 2>&1; echo "smoke rc=$?"
  tail -1 $O/${TAG}_smoke.log
fi
if [[ ($WHAT == all || $WHAT == ab) && -n $P ]]; then
  timeout 600 python tools/decode_step_ab.py > $O/${TAG}_decode_step_digests.json 2> $O/${TAG}_ab.err
  cp tools/decode_step_ab.py $P/tools/ && (cd $P && timeout 600 python tools/decode_step_ab.py) \
    > $O/${TAG}_decode_step_digests_parent_commit.json 2>> $O/${TAG}_ab.err
  if [[ -s $O/${TAG}_decode_step_digests.json ]] \
      && cmp $O/${TAG}_decode_step_digests.json $O/${TAG}_decode_step_digests_parent_commit.json; then
    echo "single-token decode-step ops: bitwise equal to the parent commit" | tee $O/${TAG}_decode_step_ab.txt
  else
    echo "single-token decode-step ops: NOT shown equal to the parent commit (differ, or a run failed)" \
      | tee $O/${TAG}_decode_step_ab.txt
  fi
fi
if [[ $WHAT == all ]]; then
  for i in 1 2; do
    timeout 400 python bench.py --gpus 1 > $O/${TAG}_bench_$i.json 2> $O/${TAG}_bench_$i.err; echo "bench $i rc=$?"
    cut -c1-220 $O/${TAG}_bench_$i.json
    if [[ -n $P ]]; then
      (cd $P && timeout 400 python bench.py --gpus 1) > $O/${TAG}_bench_parent_commit_$i.json 2> $O/${TAG}_bench_parent_$i.err
      echo "parent bench $i rc=$?"; cut -c1-220 $O/${TAG}_bench_parent_commit_$i.json
    fi
  done
  # the batch-1 8B decode line (flat cache, 1000-token prompt), this tree and the parent
  for T in this parent; do
    D=.; N=decode; [[ $T == parent ]] && { [[ -n $P ]] || continue; D=$P; N=decode_parent_commit; }
    (cd $D && timeout 1500 python tools/decode_bench.py --model llama-3-8b --prompt 1000 --tokens 1000 \
      --max-kv-size none --graph-positions 1000,1999 --repeat 1) > $O/${TAG}_${N}_llama-3-8b_p1000_t1000.json \
      2> $O/${TAG}_${N}.err
    echo "$N rc=$?"; cut -c1-500 $O/${TAG}_${N}_llama-3-8b_p1000_t1000.json
  done
fi
if [[ $WHAT == bench ]]; then
  timeout 1100 python tools/spec_bench.py > $O/${TAG}_spec_llama-3-8b.json 2> $O/${TAG}_spec.err
  echo "spec_bench rc=$?"; cut -c1-600 $O/${TAG}_spec_llama-3-8b.json; tail -5 $O/${TAG}_spec.err
fi
