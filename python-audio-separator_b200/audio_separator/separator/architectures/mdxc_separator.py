"""B200 MDXC architecture plugin (non-Roformer TFC_TDF_net models, e.g. MDX23C-8KFFT-InstVoc_HQ).

Plugin contract of the reference's MDXCSeparator (audio_separator/separator/architectures/mdxc_separator.py:19-228):
ctor `(common_config, arch_config)` with arch keys segment_size / override_model_segment_size / batch_size / overlap /
pitch_shift, `separate(path, custom_output_names)`, `demix(mix) -> {instrument: (2, N)}`.  The chunk loop runs on the GPU
through libb200sep.so (MdxcEngine for TFC_TDF_net checkpoints, RoformerEngine for BS-Roformer and Mel-Band Roformer checkpoints -- the Roformer branch of
demix, mdxc_separator.py:272-343).  Pitch shifting is not part of this path.

arch key `b200_sharded` (default False): one process per GPU in an initialised torch.distributed process group (backend nccl); every rank calls
separate(path) on the same file, each computes the chunks of its part of the track (b200/sharded.py), rank 0 gathers the stems, writes the files and
returns their names, the other ranks return [].
"""
import os

import numpy as np
import torch

from ..b200.engine import MdxcEngine, TfcNet
from ..b200.roformer import BSRoformerConfig, BSRoformerNet, MelBandRoformerConfig, RoformerEngine
from ..common_separator import CommonSeparator, normalize


class MDXCSeparator(CommonSeparator):
    def __init__(self, common_config, arch_config):
        super().__init__(config=common_config)
        self.model_data_cfgdict = self.model_data  # the model's YAML as a dict (mdxc_separator.py:60)
        self.segment_size = arch_config.get("segment_size", 256)
        self.override_model_segment_size = arch_config.get("override_model_segment_size", False)
        self.overlap = arch_config.get("overlap", 8)
        self.batch_size = arch_config.get("batch_size", 1)
        self.pitch_shift = arch_config.get("pitch_shift", 0)
        self.process_all_stems = arch_config.get("process_all_stems", True)
        self.sharded = bool(arch_config.get("b200_sharded", False))
        self.is_roformer = bool(self.is_roformer_model)
        if self.pitch_shift:
            raise NotImplementedError("pitch_shift is not part of the accelerated path")
        if not torch.cuda.is_available():
            raise RuntimeError("MDXCSeparator (B200 build) needs a CUDA device: there is no CPU path in this package")
        self.torch_device = torch.device("cuda", torch.cuda.current_device())
        self._dist = {}
        if self.sharded:
            import torch.distributed as dist

            if not dist.is_initialized():
                raise RuntimeError("mdxc_params['b200_sharded'] needs an initialised torch.distributed process group (backend nccl, one process per GPU)")
            self._dist = {"dist": dist}
        self.is_primary_stem_main_target = bool(self.model_data_cfgdict["training"].get("target_instrument"))  # :69, both model families
        self._engines = {}  # dim_t -> engine: the chunk length is fixed per engine, and separate() switches it for clips shorter than 10 s (:137-143)
        self.load_model()

    def load_model(self):
        """Replaces TFC_TDF_net(config).load_state_dict(torch.load(ckpt)) (mdxc_separator.py:76-116)."""
        cfg = self.model_data_cfgdict
        audio, model, training = cfg["audio"], cfg["model"], cfg["training"]
        if self.is_roformer:
            return self._load_roformer(cfg)
        if model.get("norm") != "InstanceNorm" or model.get("act", "gelu") != "gelu" or list(model.get("scale", [2, 2])) != [2, 2]:
            raise ValueError("the B200 TFC_TDF_net supports norm=InstanceNorm, act=gelu, scale=[2,2] (the MDX23C configuration)")
        path = self.model_path
        if path.lower().endswith(".npz"):
            with np.load(path) as z:
                state = {k: z[k] for k in z.files}
        else:
            sd = torch.load(path, map_location="cpu", weights_only=True)
            state = {k: v.float().numpy() for k, v in (sd.get("state_dict", sd)).items()}
        self._state = state
        self._select_engine()

    def _select_engine(self):
        """The engine for the current `override_model_segment_size` (dim_t = segment_size or the model's inference.dim_t, :281-286 / :355-360); built once per dim_t."""
        cfg = self.model_data_cfgdict
        audio, model, training = cfg["audio"], cfg["model"], cfg["training"]
        dim_t = int(self.segment_size if self.override_model_segment_size else cfg["inference"]["dim_t"])
        if dim_t not in self._engines:
            if self.is_roformer:
                eng = RoformerEngine(self.net, dim_t, self.overlap, audio.get("sample_rate", 44100), len(training["instruments"]), max(1, int(self.batch_size)), **self._dist)
                self._engines[dim_t] = (self.net, eng, self.net.forward)
            else:
                targets = 1 if training.get("target_instrument") else len(training["instruments"])
                net = TfcNet(self._state, audio["dim_f"], dim_t, model["num_subbands"], audio.get("num_channels", 2), model["num_scales"], model["num_blocks_per_scale"],
                             model["num_channels"], model["growth"], model["bottleneck_factor"], targets, max_batch=max(1, int(self.batch_size)))
                eng = MdxcEngine(net, audio["n_fft"], audio["hop_length"], audio["dim_f"], dim_t, self.overlap, **self._dist)
                self._engines[dim_t] = (net, eng, eng.model_run)
        self.net, self.engine, self.model_run = self._engines[dim_t]

    def _load_roformer(self, cfg):
        """RoformerLoader.load_model (roformer/roformer_loader.py:82-195): BSRoformer(**model section) + load_state_dict."""
        model, training = cfg["model"], cfg["training"]
        if "num_bands" in model:  # roformer_loader.py:_create_mel_band_roformer
            rcfg = MelBandRoformerConfig.from_model_section(model)
        elif "freqs_per_bands" in model:
            rcfg = BSRoformerConfig.from_model_section(model)
        else:
            raise ValueError("Unknown Roformer model type in configuration (neither num_bands nor freqs_per_bands)")
        path = self.model_path
        if path.lower().endswith(".npz"):
            with np.load(path) as z:
                state = {k: z[k] for k in z.files}
        else:
            sd = torch.load(path, map_location="cpu", weights_only=True)
            state = {k: v.float().numpy() for k, v in (sd.get("state_dict", sd)).items()}
        self.net = BSRoformerNet(rcfg, state, device=self.torch_device)
        self._select_engine()

    def _demix_engine(self, orig):
        """(S, 2, N) ndarray of the engine's stems; None on the ranks other than 0 of a sharded run (they hold only their slice)."""
        out = self.engine.gather(self.engine.demix_device(torch.as_tensor(orig).to(self.torch_device)), orig.shape[1])
        return None if out is None else out.cpu().numpy()

    def _demix_roformer(self, mix):
        """Roformer branch of demix + the stem dictionary (mdxc_separator.py:272-343, :406-468)."""
        training = self.model_data_cfgdict["training"]
        orig = np.ascontiguousarray(mix, dtype=np.float32)
        out = self._demix_engine(orig)
        if out is None:
            return None
        if self.net.cfg.num_stems > 1:
            return {k: v for k, v in zip(training["instruments"], out)}
        primary = out[0]
        if self.is_primary_stem_main_target:  # single-target models also return the residual as the secondary stem
            return {self.primary_stem_name: primary, self.secondary_stem_name: orig - primary}
        return primary

    def demix(self, mix):
        """(2, N) ndarray -> {instrument: (2, N) ndarray} (mdxc_separator.py:406-434) or the single target's array; None on a sharded rank other than 0."""
        if self.is_roformer:
            return self._demix_roformer(mix)
        orig = np.ascontiguousarray(mix, dtype=np.float32)
        out = self._demix_engine(orig)
        if out is None:
            return None
        training = self.model_data_cfgdict["training"]
        if self.net.num_targets > 1:
            return {k: v for k, v in zip(training["instruments"], out)}
        primary = out[0]
        if self.is_primary_stem_main_target:  # single-target models also return the residual as the secondary stem (:452-461)
            return {self.primary_stem_name: primary, self.secondary_stem_name: orig - primary}
        return primary

    def separate(self, audio_file_path, custom_output_names=None):
        self.audio_file_path = audio_file_path
        self.audio_file_base = os.path.splitext(os.path.basename(audio_file_path))[0]
        mix = self.prepare_mix(self.audio_file_path)
        if mix.shape[1] / self.sample_rate < 10.0 and not self.override_model_segment_size:  # :137-143 (the switch is sticky in the reference too)
            self.override_model_segment_size = True
            self.logger.warning(f"Audio duration ({mix.shape[1] / self.sample_rate:.2f}s) is less than 10 seconds.")
            self.logger.warning("Automatically enabling override_model_segment_size for better processing of short audio.")
            self._select_engine()
        mix = normalize(wave=np.array(mix, dtype=np.float32), max_peak=self.normalization_threshold, min_peak=self.amplification_threshold)  # :149
        source = self.demix(mix)
        if source is None:  # a sharded rank other than 0: rank 0 writes the files
            return []
        output_files = []
        if isinstance(source, dict):  # (:156-214)
            training = self.model_data_cfgdict["training"]
            stem_list = [training["target_instrument"]] if training.get("target_instrument") else list(training["instruments"])
            norm = lambda w: normalize(wave=w, max_peak=self.normalization_threshold, min_peak=self.amplification_threshold).T  # noqa: E731
            if self.process_all_stems and len(stem_list) > 2:  # every stem of a multi-stem model, in the model's order
                for stem_name in stem_list:
                    if self.output_single_stem and self.output_single_stem.lower() != stem_name.lower():
                        continue
                    path = self.get_stem_output_path(stem_name, custom_output_names)
                    self.final_process(path, norm(source[stem_name]), stem_name)
                    output_files.append(path)
                return output_files
            self.primary_source, self.secondary_source = norm(source[self.primary_stem_name]), norm(source[self.secondary_stem_name])
            for name, src in ((self.secondary_stem_name, self.secondary_source), (self.primary_stem_name, self.primary_source)):  # secondary file first
                if self.output_single_stem and self.output_single_stem.lower() != name.lower():
                    continue
                path = self.get_stem_output_path(name, custom_output_names)
                self.final_process(path, src, name)
                output_files.append(path)
            return output_files
        # a bare array = a single-source model without a target instrument: only the primary stem is written, as it is (:216-226)
        if not self.output_single_stem or self.output_single_stem.lower() == self.primary_stem_name.lower():
            self.primary_source = source.T
            path = self.get_stem_output_path(self.primary_stem_name, custom_output_names)
            self.final_process(path, self.primary_source, self.primary_stem_name)
            output_files.append(path)
        return output_files
