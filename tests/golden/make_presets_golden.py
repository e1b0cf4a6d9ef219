"""Dumps the reference's hparam_presets dict to presets_golden.json (SPARSE_VAE_REFERENCE names the reference checkout)."""
import importlib.util
import json
import sys
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[2]))
from oracle.reference_harness import require_reference  # noqa: E402

spec = importlib.util.spec_from_file_location('ref_presets', require_reference() / 'hparam_presets.py')
mod = importlib.util.module_from_spec(spec)
spec.loader.exec_module(mod)
Path(__file__).with_name('presets_golden.json').write_text(json.dumps(mod.hparam_presets, indent=1, sort_keys=True))
