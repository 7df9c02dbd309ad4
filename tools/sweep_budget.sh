#!/bin/bash
# SM budget sweep of the bench step (pipelined schedule, 3 groups). usage: bash tools/sweep_budget.sh
for budget in 0 100 116 132 148; do
  line=$(FPCC_SM_BUDGET=$budget python bench.py --steps 3 --warmup 2 --no-cpu-baseline --groups 3 2>&1 >/dev/null | grep "step_device\|Error\|error" | tr '\n' ' ')
  echo "budget=$budget: $line"
done
