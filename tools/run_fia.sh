# sweep of the iteration at which long-running QPs switch to the explicit operator (FCCQP_FULL_INVERSE_AT; default 6, 8 for n + m <= 32)
for v in 4 6 8; do
  export FCCQP_FULL_INVERSE_AT=$v
  echo "== full_inverse_at $v"
  timeout 200 python tools/prof_shape.py humanoid 32768 3 cold 2>&1 | tail -1
  timeout 200 python tools/prof_shape.py multicontact 16384 3 cold 2>&1 | tail -1
  timeout 200 python tools/prof_run.py 65536 4 cold 2>&1 | tail -1
done
