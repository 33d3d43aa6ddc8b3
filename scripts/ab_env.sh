# A/B of an environment switch on the train step (run under gpurun):  bash scripts/ab_env.sh MOBODY_PDL 0 1
#                                                                     bash scripts/ab_env.sh MOBODY_TRAIN_SIDE 0 1
var=$1; shift
for v in "$@"; do
  export $var=$v
  echo "=== $var=$v" >> gpurun_out/ab_env.log
  python - >> gpurun_out/ab_env.log 2>&1 <<'PY'
import bench, torch
import mobody_b200 as mb
dev = torch.device("cuda:0")
for batch, s, a in ((128, None, None), (4096, 27, 8)):
    print(batch, bench.gpu_train_rate(mb, dev, batch, steps=300 if batch == 128 else 100, s_dim=s, a_dim=a))
PY
done
