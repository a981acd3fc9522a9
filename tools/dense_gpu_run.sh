# The GPU runs behind profiles/r3_*: the whole GPU suite (including tests/test_gpu_dense.py), smoke, one bench.py line
# and the dense-matrix measurements. Run from the repository root after a build: bash tools/dense_gpu_run.sh OUTDIR
set -x
O="${1:?usage: dense_gpu_run.sh OUTDIR}"
mkdir -p "$O"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$O"/card.csv 2>&1
python -m pytest tests/test_gpu_dense.py -q > "$O"/pytest_gpu_dense.log 2>&1; echo "pytest rc=$?" >> "$O"/pytest_gpu_dense.log
python -m pytest tests -m gpu -q --ignore=tests/test_gpu_dense.py > "$O"/pytest_gpu_rest.log 2>&1; echo "pytest rc=$?" >> "$O"/pytest_gpu_rest.log
python -c "import __graft_entry__ as g; g.smoke()" > "$O"/smoke.log 2>&1; echo "smoke rc=$?" >> "$O"/smoke.log
python bench.py --gpus 1 --steps 5 --warmup 2 > "$O"/bench_default.json 2> "$O"/bench_default.err
python benchmarks/dense_matrix.py --cases C5,C2,C3 --reps 2 > "$O"/dense_matrix.jsonl 2> "$O"/dense_matrix.err
echo done
