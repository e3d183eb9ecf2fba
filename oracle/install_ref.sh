#!/bin/bash
# Copies the UNMODIFIED reference sources of the hot path into oracle/_ref/ (git-ignored, made by build() where a checkout of the
# reference exists and kept beside the built library) so that bench.py can time the reference's own PyTorch-eager path on the B200
# (`gpu_eager_baseline`, SURVEY.md section 8(d) "Reference GPU baseline") and scripts/bench_train_ref.py its training step.
# The reference is not an installable package (no setup.py / pyproject.toml), hence a file copy instead of pip.
#   oracle/install_ref.sh <reference checkout>
set -e
REF=$1
DST="$(cd "$(dirname "$0")" && pwd)/_ref"
rm -rf "$DST"
mkdir -p "$DST/autoregressive/models" "$DST/tokenizer/tokenizer_image" "$DST/utils"
for f in generate.py gpt_t2i.py gpt.py dinov2_adapter.py vit_adapter.py; do cp "$REF/autoregressive/models/$f" "$DST/autoregressive/models/$f"; done
cp "$REF/tokenizer/tokenizer_image/vq_model.py" "$DST/tokenizer/tokenizer_image/vq_model.py"
cp "$REF/utils/drop_path.py" "$DST/utils/drop_path.py"
( cd "$DST" && find . -type f | sort | xargs sha256sum ) > "$DST/SHA256SUMS"
echo "reference hot-path sources installed into $DST:"; cat "$DST/SHA256SUMS"
