"""gr_lora_b200 -- B200-native LoRa PHY demodulator behind the gr-lora block API.

Only what the hot path needs: the CUDA library + C ABI (csrc/, ../include/lora_b200.h), the
host-side mirrors of the reference blocks (decoder, lora_receiver) and the synthetic
transmitter used to produce inputs (tx)."""
from .decoder import decoder, dissect_frame, split_tables, tables_build_host  # noqa: F401
from .channelizer import channelizer  # noqa: F401
from .gateway import gateway  # noqa: F401
from .lora_receiver import lora_receiver  # noqa: F401
from .message_socket_sink import message_socket_sink  # noqa: F401
from .loraconfig import LoRaConfig  # noqa: F401

__all__ = ["decoder", "channelizer", "gateway", "message_socket_sink", "lora_receiver", "LoRaConfig", "dissect_frame", "split_tables", "tables_build_host"]
