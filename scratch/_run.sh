#!/bin/bash
python -c "import __graft_entry__ as g; g.build()" > /tmp/build.log 2>&1 || { tail -30 /tmp/build.log; exit 1; }
timeout 200 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
timeout 300 python -m pytest -p no:cacheprovider -q -s -m gpu tests/test_dropout.py 2>&1 | grep -E "passed|failed|FAILED|measured|Error" | tail -15
timeout 60 python -m pytest -p no:cacheprovider -q -m gpu tests/test_bench.py tests/test_cabi.py 2>&1 | tail -1
timeout 150 python bench.py --gpus 1 --steps 5 --warmup 2 --no-cpu-baseline --no-e2e 2>/dev/null | grep '^{' | python -c "import json,sys; d=json.loads(sys.stdin.read()); print('rmg34', round(d['value']), d['gpu_launches'])"
