cd $GRAFT_REPO_ROOT
python -m pytest tests/test_gpu_concurrent.py tests/test_gpu_api.py -x -q -m gpu > gpurun_out/pytest_new.log 2>&1; echo "pytest rc=$?"; tail -4 gpurun_out/pytest_new.log
bash scripts/gpu_sweep_libs.sh 4k10_n15
echo "--- 3 windows"; bash scripts/gpu_sweep_libs.sh 4k10_n15 --concurrent 3 2>&1 | grep "eo_filt6\|base"
