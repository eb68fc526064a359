#!/usr/bin/env python
"""TEST INFRASTRUCTURE ONLY -- golden vectors for the SURVEY.md section 8f "next" rows, frozen from
the UNMODIFIED reference in the build container (needs /root/reference):

    PYTHONDONTWRITEBYTECODE=1 python oracle/gen_golden_next.py

* app_post.npz   -- omega4_main.py:992-1056 (P98 normalise, frequency compensation, mel band mean
  -> sqrt -> clamp, per-band smoothing).  That block is inline code of the 1800-line pygame
  application method ``ProfessionalLiveAudioAnalyzer.process_audio_spectrum``; the application
  class cannot be constructed headless, so the script imports ``omega4_main`` behind a permissive
  pygame stub, cuts exactly those source lines out of the method with ``inspect`` and executes
  them, unmodified, against a stand-in ``self`` that carries the attributes the block reads
  (the real ``apply_frequency_compensation`` method and the real ``PrecomputedFrequencyMapper``
  band table included).
* meters_weighting.npz -- ProfessionalMetering.apply_a_weighting / apply_c_weighting / Z mode and
  calculate_lufs in those modes (professional_meters.py:74-127, 155-229).
* bass_zoom.npz -- BassZoomPanel._process_bass_detail_internal bar values (omega4/panels/bass_zoom.py:141-214).
"""
import inspect
import os
import sys
import textwrap
import types
from unittest import mock

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("OMEGA4_REFERENCE", "/root/reference")
OUT = os.path.join(ROOT, "tests", "golden")
sys.dont_write_bytecode = True


class _Stub(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        m = mock.MagicMock(name=f"{self.__name__}.{name}")
        setattr(self, name, m)
        return m


pg = _Stub("pygame")
pg.Surface = object
pg.Rect = object
pg.font = types.SimpleNamespace(Font=object, SysFont=mock.MagicMock(), init=mock.MagicMock())
sys.modules["pygame"] = pg
for sub in ("gfxdraw", "locals"):
    sys.modules["pygame." + sub] = _Stub("pygame." + sub)
sys.path.insert(0, REF)
sys.path.insert(0, os.path.join(ROOT, "audio-analyzer-omega_b200"))

import omega4_main  # noqa: E402
from omega4.audio.multi_resolution_fft import MultiResolutionFFT, FFTConfig, WindowType  # noqa: E402
from omega4.optimization.freq_mapper import PrecomputedFrequencyMapper  # noqa: E402
from omega4.panels.professional_meters import ProfessionalMetering  # noqa: E402
from omega4.panels.bass_zoom import BassZoomPanel  # noqa: E402
from omega4_b200.batch.synth import synth_channel  # noqa: E402

HOP, W = 512, 2048
BASELINE = [((20, 200), 8192, 1024, 1.5), ((200, 1000), 4096, 512, 1.2),
            ((1000, 5000), 2048, 256, 1.0), ((5000, 20000), 1024, 256, 1.5)]


def _post_block_source():
    """The source lines of process_audio_spectrum from the P98 normalisation to the smoothing carry."""
    src = inspect.getsource(omega4_main.ProfessionalLiveAudioAnalyzer.process_audio_spectrum).splitlines()
    start = next(i for i, l in enumerate(src) if "Apply initial normalization to prevent overflow" in l)
    end = next(i for i, l in enumerate(src) if "self.prev_band_values = band_values.copy()" in l)
    return textwrap.dedent("\n".join(src[start:end + 1]))


def gen_app_post():
    cls = omega4_main.ProfessionalLiveAudioAnalyzer
    code = compile(_post_block_source(), "omega4_main.py:process_audio_spectrum[992:1056]", "exec")
    sr, bars = omega4_main.SAMPLE_RATE, 512
    mr = MultiResolutionFFT(sample_rate=sr)
    mr.configs = [FFTConfig(fr, n, h, w, WindowType.BLACKMAN) for fr, n, h, w in BASELINE]
    mr._setup_windows(); mr._setup_buffers(); mr._setup_frequency_arrays(); mr._setup_working_arrays()
    x = synth_channel(5, 0, 80 * HOP, sr)
    x[40 * HOP:44 * HOP] = 0.0                        # silence: max == 0 branch, smoothing decay
    x[60 * HOP:] *= 30.0                              # hot: bars clamp at 1 (python-int elements, float64 frames)
    out = {}
    for variant, attrs in (("default", {}),
                           ("normalized", {"normalization_enabled": True}),
                           ("vocal", {"current_content_type": "vocal", "vocal_suppression": 0.5}),
                           ("plain", {"freq_compensation_enabled": False, "smoothing_enabled": False})):
        me = types.SimpleNamespace(
            freq_compensation_enabled=True, normalization_enabled=False, smoothing_enabled=True,
            current_content_type="instrumental", vocal_suppression=0.0, bars=bars,
            freqs=np.fft.rfftfreq(omega4_main.FFT_SIZE_BASE, 1 / sr),
            band_indices=PrecomputedFrequencyMapper(sr, omega4_main.FFT_SIZE_BASE, bars).mapping.band_indices)
        for k, v in attrs.items():
            setattr(me, k, v)
        me.apply_frequency_compensation = types.MethodType(cls.apply_frequency_compensation, me)
        for r in mr.buffers if hasattr(mr, "buffers") else []:
            r.reset() if hasattr(r, "reset") else None
        mr.reset_all_buffers()
        rows_in, rows_band, rows_peak, dts = [], [], [], []
        for k in range(len(x) // HOP):
            res = mr.process_audio_chunk(x[k * HOP:(k + 1) * HOP])
            if not res:
                continue
            spectrum = mr.combine_results_optimized(res, target_bins=bars)[0]
            ns = {"self": me, "spectrum": spectrum, "np": np,
                  "SAMPLE_RATE": sr, "FFT_SIZE_BASE": omega4_main.FFT_SIZE_BASE}
            exec(code, ns)
            rows_in.append(spectrum)
            rows_band.append(np.asarray(ns["band_values"], dtype=np.float64))
            rows_peak.append(np.asarray(ns["peak_values"], dtype=np.float64))
            dts.append(str(np.asarray(ns["band_values"]).dtype))
        if variant == "default":
            out["combined"] = np.stack(rows_in)
        out[f"band_{variant}"] = np.stack(rows_band)
        out[f"peak_{variant}"] = np.stack(rows_peak)
        out[f"dtypes_{variant}"] = np.array(dts)
    # every row (the smoothing state runs through them), the expected values at 3 of every 4 bands: all 437 would take
    # the file past 1 MB
    cols = np.flatnonzero(np.arange(out["band_default"].shape[1]) % 4 != 3).astype(np.int32)
    out = {k: v[:, cols] if k.startswith(("band_", "peak_")) else v for k, v in out.items()}
    out["band_cols"] = cols
    out["bands"] = np.array(PrecomputedFrequencyMapper(sr, omega4_main.FFT_SIZE_BASE, bars).mapping.band_indices, dtype=np.int32)
    np.savez_compressed(os.path.join(OUT, "app_post.npz"), **out)


def gen_meter_weighting():
    sr = 48000
    x = synth_channel(9, 1, 40 * HOP, sr)
    x[20 * HOP:22 * HOP] *= 1e-7                      # below the rms gate
    out = {"x": x}
    for mode in ("A", "C", "Z"):
        m = ProfessionalMetering(sr)
        m.weighting_mode = mode
        ws, li, rows = [], [], []
        for k in range(3, len(x) // HOP):
            fr = x[(k + 1) * HOP - W:(k + 1) * HOP] * np.hanning(W)
            if k in (3, 10, 20, 39):
                ws.append(np.asarray(m.apply_weighting(fr), dtype=np.float64))
            d = m.calculate_lufs(fr)
            li.append(m.lufs_momentary_history[-1])
            rows.append([d["momentary"], d["short_term"], d["integrated"], d["range"], d["true_peak"]])
        out[f"weighted_{mode}"] = np.stack(ws)
        out[f"lufs_inst_{mode}"] = np.array(li)
        out[f"meters_{mode}"] = np.array(rows)
        if mode == "A":
            for name, (b, a) in ((n, m.a_weighting_filter[n]) for n in ("hp1", "hp2", "lp1", "lp2")):
                out[f"A_{name}_b"], out[f"A_{name}_a"] = np.asarray(b), np.asarray(a)
        if mode == "C":
            for name, (b, a) in ((n, m.c_weighting_filter[n]) for n in ("hp", "lp")):
                out[f"C_{name}_b"], out[f"C_{name}_a"] = np.asarray(b), np.asarray(a)
    out["weighted_hops"] = np.array([3, 10, 20, 39])
    np.savez_compressed(os.path.join(OUT, "meters_weighting.npz"), **out)


def gen_bass_zoom():
    """BassZoomPanel._process_bass_detail_internal on the app's Hann-windowed 2048-sample frames
    (omega4_main.py:1197), bar values only (the peak hold is wall-clock driven)."""
    sr = 48000
    x = synth_channel(2, 0, 60 * HOP, sr)
    x[30 * HOP:34 * HOP] = 0.0
    panel = BassZoomPanel(sr)
    panel.bass_thread_running = False                      # the worker thread is not used
    frames, bars = [], []
    for k in range(3, 60):
        fr = x[(k + 1) * HOP - W:(k + 1) * HOP] * np.hanning(W)
        res = panel._process_bass_detail_internal(fr)
        panel.bass_bar_values = res["bar_values"]
        frames.append(fr.astype(np.float32))
        bars.append(np.array(res["bar_values"], dtype=np.float64))
    # the reference computes on the float64 frame; the fixture stores float32 frames (what the GPU path is fed)
    # and re-runs the reference on exactly those so that input and output belong together
    panel2 = BassZoomPanel(sr)
    panel2.bass_thread_running = False
    bars32 = []
    for fr in frames:
        res = panel2._process_bass_detail_internal(fr.astype(np.float64))
        panel2.bass_bar_values = res["bar_values"]
        bars32.append(np.array(res["bar_values"], dtype=np.float64))
    np.savez_compressed(os.path.join(OUT, "bass_zoom.npz"), frames=np.stack(frames), bars=np.stack(bars32),
                        n_bars=panel.bass_detail_bars,
                        bin_first=np.array([g[0] for g in panel.bass_bin_mapping], dtype=np.int32),
                        bin_count=np.array([len(g) for g in panel.bass_bin_mapping], dtype=np.int32),
                        ranges=np.array(panel.bass_freq_ranges, dtype=np.float64))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    which = sys.argv[1:] or ["app_post", "meter_weighting", "bass_zoom"]
    if "app_post" in which:
        gen_app_post()
    if "meter_weighting" in which:
        gen_meter_weighting()
    if "bass_zoom" in which:
        gen_bass_zoom()
    for f in ("app_post.npz", "meters_weighting.npz", "bass_zoom.npz"):
        pth = os.path.join(OUT, f)
        if os.path.exists(pth):
            print(f, os.path.getsize(pth))
