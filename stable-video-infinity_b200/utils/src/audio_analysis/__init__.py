"""wav2vec2 audio encoder of SVI-Talk (reference utils/src/audio_analysis)."""
