set +e
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_train.py -q -m gpu --timeout 600 -p no:cacheprovider -s > gpurun_out/train.log 2>&1; echo "train exit $?"; grep -E "per-tensor|passed|failed" gpurun_out/train.log | tail -7
timeout 600 python scripts/train_profile.py --batch 128 > gpurun_out/train_profile_b128_r02c.log 2>&1; head -12 gpurun_out/train_profile_b128_r02c.log
