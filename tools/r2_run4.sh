#!/bin/bash
cd "$GRAFT_REPO_ROOT" 2>/dev/null || cd /root/repo
mkdir -p gpurun_out
( timeout 1200 python -m pytest tests -m gpu -x -q -p no:cacheprovider 2>&1 | grep -v Warning | tail -30 ) > gpurun_out/r2h_pytest.log
( timeout 900 python bench.py --config c3 --steps 1 --warmup 0 --machines 32 --cpu-seconds 8 ) > gpurun_out/r2h_c3_m32.json 2> gpurun_out/r2h_c3_m32.err
bash tools/r2_profile.sh
