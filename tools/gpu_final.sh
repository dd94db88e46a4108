# final pass of a round: GPU tests, default bench (+ reference arm, smoke).  Usage: bash tools/gpu_final.sh TAG
TAG=${1:-final}
python -m pytest tests -m gpu -x -q > gpurun_out/test_gpu_$TAG.log 2>&1; tail -3 gpurun_out/test_gpu_$TAG.log
( time timeout 900 python bench.py > gpurun_out/bench_$TAG.json 2> gpurun_out/bench_$TAG.err ) 2>&1 | grep real; grep '^\[bench\]' gpurun_out/bench_$TAG.err | cut -c1-420
( time timeout 900 python bench.py --impl reference --steps 20 --warmup 3 > gpurun_out/bench_${TAG}_ref.json 2> gpurun_out/bench_${TAG}_ref.err ) 2>&1 | grep real; cut -c1-200 gpurun_out/bench_${TAG}_ref.json
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1 | cut -c1-200
