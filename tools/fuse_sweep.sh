#!/bin/bash
# Which map sizes should apply their AdaGN inside the consumer conv?  (development helper; default: H >= 64 only)
cd "${GRAFT_REPO_ROOT:-/root/repo}"
run() { timeout 300 python bench.py --steps 3 --warmup 3 --no-extras --no-train --no-cpu-baseline "$@" 2>/dev/null | tail -1 | python -c "import sys,json; d=json.loads(sys.stdin.read()); print(round(d['value'],1), 'img/s', {k: round(v['ms_per_unet_eval'],2) for k,v in d['kernel_breakdown'].items() if k in ('conv_igemm','conv_igemm_xf','adagn','adagn_coef')})"; }
echo -n "default (H>=64): "; run
echo -n "every layer: "; run --fuse-adagn
echo -n "none: "; run --no-fuse-adagn
echo -n "default again: "; run
