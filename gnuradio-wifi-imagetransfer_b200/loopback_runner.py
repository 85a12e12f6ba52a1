"""GNU-Radio-free runner that speaks the reference applications' UDP contract (SURVEY.md 8f row 1).

It stands where the `IRS_tranceiver` loopback flowgraph stands (gnu_radio/IRS_tranceiver.py):

    UDP :50010  (network.socket_pdu 'UDP_SERVER', :248)         <- upload_image_udp.py / upload_featuremap_udp.py
      -> ieee802_11.mac (:271,313-314) -> wifi_phy_hier TX (:178-184) -> x0.6 (:295) -> packet_pad2 100/1000 (:277)
      -> x sqrt(10^(snr/10)) (:294) -> channel_model(noise_voltage 1, CFO, taps [1]) (:282-288)
      -> RX chain (:268-273) -> "Extract Pics": data[24:][4:] (IRS_tranceiver_epy_block_2.py:31-38)
    UDP -> localhost:10010                                       -> download_image_udp.py / download_featuremap_udp.py

so the reference's sender and viewer scripts run unchanged against it.  All PHY work happens in
libwifi_b200.so on the GPU (TX, Philox channel, RX); this file only moves datagrams.

    python -c "import wifi_b200; wifi_b200.loopback_runner.main()" --encoding 3 --snr 27
"""
import argparse
import math
import socket
import threading

import numpy as np

from .wifi_phy_hier import mac, wifi_phy_hier


class IrsTransceiver:
    """Defaults are the flowgraph's variables (IRS_tranceiver.py:80-92)."""

    def __init__(self, in_port=50010, out_addr=("localhost", 10010), snr=22.0, epsilon=0.0, encoding=3, chan_est=0,
                 freq=5.89e9, samp_rate=20e6, device=0, mtu=1024, idle_flush_s=0.2, seed=0, doppler_hz=None, k_factor=None):
        self.snr, self.epsilon, self.freq, self.samp_rate = float(snr), float(epsilon), float(freq), float(samp_rate)
        # doppler_hz / k_factor (either one) replace the flowgraph's fixed tap [1] with one flat Rayleigh/Rician tap of unit
        # power that fades continuously across datagrams: one realisation, sample n of the link at time n
        self.fading = None
        if doppler_hz is not None or k_factor is not None:
            self.fading = dict(taps=((0, 1.0),), doppler=float(doppler_hz or 0.0) / self.samp_rate, k_factor=float(k_factor or 0.0), seed=seed)
        self.mtu, self.idle_flush_s, self.seed = mtu, idle_flush_s, seed
        self.phy = wifi_phy_hier(bandwidth=samp_rate, chan_est=chan_est, encoding=encoding, frequency=freq, sensitivity=0.56,
                                 device=device, max_samples=1 << 20)
        self.mac = mac([0x23] * 6, [0x42] * 6, [0xff] * 6)
        self.rx_sock = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
        self.rx_sock.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
        self.rx_sock.bind(("", in_port))
        self.in_port = self.rx_sock.getsockname()[1]
        self.rx_sock.settimeout(idle_flush_s)
        self.tx_sock = socket.socket(socket.AF_INET, socket.SOCK_DGRAM)
        self.out_addr = out_addr
        self._stop = threading.Event()
        self._n0 = 0
        self.stats = {"datagrams_in": 0, "pdus_out": 0, "dropped_oversize": 0}

    # GRC-style setters of the flowgraph (IRS_tranceiver.py:355-450)
    def set_snr(self, snr):
        self.snr = float(snr)

    def set_epsilon(self, epsilon):
        self.epsilon = float(epsilon)

    def set_encoding(self, encoding):
        self.phy.set_encoding(encoding)

    def set_chan_est(self, chan_est):
        self.phy.set_chan_est(chan_est)

    def _through_channel(self, burst):
        # x0.6, 100 zeros before / 1000 after, x sqrt(10^(snr/10)), then channel_model(noise_voltage=1):
        # complex noise with unit variance per component = sigma^2 of 2 in the library's convention
        gain = 0.6 * math.sqrt(10 ** (self.snr / 10.0))
        n_out = 100 + burst.size + 1000
        x = np.concatenate([np.zeros(100, np.complex64), burst, np.zeros(1000, np.complex64)]).astype(np.complex64)
        # channel_model(frequency_offset = epsilon * freq / 10e6) (IRS_tranceiver.py:284,425,434): GNU Radio reads that
        # value as normalised cycles per sample, i.e. a phase step of 2 pi frequency_offset; the library's cfo is rad/sample
        cfo = 2 * math.pi * self.epsilon * self.freq / 10e6
        fading = None if self.fading is None else dict(self.fading, t0=self._n0)
        y = self.phy.handle.channel(x, n_out=n_out, n0=self._n0, gain=gain, cfo=cfo, noise_sigma=math.sqrt(2.0), seed=self.seed,
                                    fading=fading)
        self._n0 += n_out
        return y

    def _emit(self, pdus):
        for _meta, mpdu in pdus:
            self.tx_sock.sendto(bytes(mpdu[24:][4:]), self.out_addr)     # "Extract Pics"
            self.stats["pdus_out"] += 1

    def handle_datagram(self, data):
        data = data[:self.mtu]
        self.stats["datagrams_in"] += 1
        try:
            pdu = self.mac.app_in(data)
        except ValueError:
            self.stats["dropped_oversize"] += 1      # upstream throws, catch_exceptions=True swallows it
            return
        burst = self.phy.mac_in(pdu)
        self.phy.samp_out.clear()
        # one datagram = one padded burst (100 zeros, frame, 1000 zeros): it is complete, so the stream is flushed
        # behind it and the patch reaches the viewer now instead of when the next one arrives
        self._emit(self.phy.samp_in(self._through_channel(burst), flush=True))

    def serve(self, max_datagrams=None):
        n = 0
        while not self._stop.is_set() and (max_datagrams is None or n < max_datagrams):
            try:
                data, _ = self.rx_sock.recvfrom(65536)
            except socket.timeout:
                continue
            self.handle_datagram(data)
            n += 1

    def stop(self):
        self._stop.set()

    def close(self):
        self.rx_sock.close()
        self.tx_sock.close()
        self.phy.handle.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--in-port", type=int, default=50010)
    ap.add_argument("--out-host", default="localhost")
    ap.add_argument("--out-port", type=int, default=10010)
    ap.add_argument("--snr", type=float, default=22.0)
    ap.add_argument("--epsilon", type=float, default=0.0)
    ap.add_argument("--encoding", type=int, default=3)
    ap.add_argument("--chan-est", type=int, default=0)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--doppler-hz", type=float, default=None, help="maximum Doppler shift of a flat fading channel (Hz)")
    ap.add_argument("--k-factor", type=float, default=None, help="Rician K of the flat fading channel (linear, 0: Rayleigh)")
    a = ap.parse_args()
    t = IrsTransceiver(a.in_port, (a.out_host, a.out_port), a.snr, a.epsilon, a.encoding, a.chan_est, device=a.device,
                       doppler_hz=a.doppler_hz, k_factor=a.k_factor)
    print("listening on UDP :%d, forwarding decoded patches to %s:%d" % (t.in_port, a.out_host, a.out_port))
    try:
        t.serve()
    finally:
        t.close()


if __name__ == "__main__":
    main()
