# window_steps N: the --steps to give bench.py at N envs per GPU. bench.py times exactly --steps steps, so a fixed
# small K would time one launch (launch latency, not throughput): 2^28 env-steps (about 135 ms at 4,096 envs on
# one B200), at least 256 and at most 65,536 steps.
window_steps() {
  k=$(( (1 << 28) / $1 ))
  [ "$k" -gt 65536 ] && k=65536
  [ "$k" -lt 256 ] && k=256
  echo "$k"
}
