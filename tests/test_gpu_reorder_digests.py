"""The device reordering code computes what it computed at commit 8a44053 ("Multilevel k-way graph partitioning on
the device"): SHA-256 digests of its outputs on seeded graphs, recorded with that commit on an NVIDIA B200 by
profiles/tools/reorder_digests.py (device RCM permutations, ttg_kway_symmetrise's weighted CSR, device k-way labels
for seeds 0-2 and k = 2, 7, 125 with their stats, permute_graph's relabelled CSR), and the workspace sizes the C ABI
reports on both sides of its node and edge limits (0: refused)."""
import importlib.util
import os

import pytest

pytestmark = pytest.mark.gpu
TOOL = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "profiles", "tools",
                    "reorder_digests.py")

DIGESTS = {
    "cliques/input": "9ad8c3495b7c9c15437e70f9df8c46c79d4b9ef09ee480226f9e2388de853363",
    "cliques/kway": "50140ec876ae9514fb459a53da67171b4be6801c0a3ae558ee1729e4836af96f",
    "cliques/kway_symmetrise": "cc170ab0e8e752478ad9574b695a932c5628601cea3f248428aff8776edd1eab",
    "cliques/permute": "13116eb8da6ef6d98fee1868e8e06f3ac06ddf2f8df03856d23cc25623de1859",
    "cliques/rcm": "3cded67b3066f68a9aa5a948c63081ce61391fb34ad299f8cc9e290a99f13e37",
    "community/input": "588c7f45e54ea0afbedf8154208d51f8a13a92123d58fc62092fd03e9739ca34",
    "community/kway": "39ae15cf08059a651ab87fdcfe84f2b6dd04d5e6356799cc3acfc80b52381d30",
    "community/kway_symmetrise": "2219e16a64518e027fb499d426c175c475ea99a23079244db5480667aba5ab45",
    "community/permute": "c24b7657ec5b707b805406fb4bd5cb8ea4da08508ab53bd0cada34998ac05d45",
    "community/rcm": "bcffb1e32e730fa481d52dc52980b7479aac6c6a90b02b589ae270b1eabd7b9d",
    "edgeless/input": "34443b0adb62be8f33a3c12b4438205996e80aaf1a51c4b39c62345bea9b5f99",
    "edgeless/kway": "e1f8dce29ca24d9cda6041db6b433276ccc1def6bfd9c8e4a3cca0ba71a30eb1",
    "edgeless/kway_symmetrise": "808d341c4385a0e4bbb26d4ffa68f0a5266d4dee1078f90ec88c54c1178b55e9",
    "edgeless/permute": "883a709e3f198d36fa6cd6a24535e580837f1eef92ceca5ee8bddbf1eae066db",
    "edgeless/rcm": "29b1a23373031f1fee3c0a06035e0faa7542c420811417c827df91f1b0d4939a",
    "families/input": "5ee4e6bcae451e512cb2b27273db80eebe522ab14e092392b54df5c06a3d7ede",
    "families/kway": "ccbae77fcfd3c30ecce6c456de929fc7c3d5c1b98e9d8663492ba5908319d741",
    "families/kway_symmetrise": "85d19cedf63bc3c7171b69d40322e95fcec25d59429ed4142a4399cdc2c4255c",
    "families/permute": "0667d9a16a75650fda4754d0e1ff403dc4dee01f2973677a4bf3ec345252e5d5",
    "families/rcm": "4d73ca779ce504a981cd992fda9468a1f7689cbd453767c54404d271e3d6a384",
    "grid64/input": "ae9b990274842f5767b258509011832fdefae67f914a69c5eb09447cdec35f01",
    "grid64/kway": "29e015ffafcc76664621eaf74b8821d0765c3ab35ea0ef0b84584c7687fbba32",
    "grid64/kway_symmetrise": "e56b4bdb9ceb00560c0aab25dde865efdbfa6291140f79166becbdc9ceb3d70c",
    "grid64/permute": "91355f3acfaaf4263cfdd13d2d354ff9cb97ca952d679c96302df1c48f2b9a05",
    "grid64/rcm": "0b22c77b7e3c05caa9bc2ddaa25183e20c7495596694d643525089403c90ef62",
    "isolated_hub/input": "b5102f1740231399934c3996b18af63a4f330196500a3b669b05de40698bc0bd",
    "isolated_hub/kway": "04fa704e3d1e79f044172c41ee40ab54741c26b4ca094bf314932cb63dcab291",
    "isolated_hub/kway_symmetrise": "f881c3e13b531db57d408648b33d8d64118a8d5676eef6f90ba6df477a4ee89d",
    "isolated_hub/permute": "d850eacd1339f46dbb1bc1edb83868af65edd12300075078d359e102b52203b1",
    "isolated_hub/rcm": "df8cb277b9bc15b10b7071284bcc27fa5496afdb760856e313281b1e94bc5181",
    "one_node/input": "a670e0911933b02fc8abf646ebaf0aa9f6168186fc3e18c3ac7996ceb6cae4f5",
    "one_node/kway": "e3b0c44298fc1c149afbf4c8996fb92427ae41e4649b934ca495991b7852b855",
    "one_node/kway_symmetrise": "25933619c6acbe9b573b2d571deb078e0d7bb3b277ad7981a96035a7a5999a1a",
    "one_node/permute": "639a49fc8977e683bbbd5633f79ff3e809f1c4c24be31e14482cc2b26c1f1036",
    "one_node/rcm": "ba553f9413e2fef99c0d1c2ad6c5d34ab435aef491a26c047ef48231c1631b75",
    "planted/input": "d71e391ec3943a2b25b0276a90a1a33b557ea9946060fee8cb968248e883b6e7",
    "planted/kway": "ac71ce2c30f26803803c7764811c67263872560d17d7c0878e63fee14e636930",
    "planted/kway_symmetrise": "eb0a581e2d7f611dda8272feab590742a1c36fb21fde1a6da39934c307d34cac",
    "planted/permute": "d07b000c125d58b9b7ca09dac44c5449050604b64e57e612bc59702b908fd56f",
    "planted/rcm": "e77b05def9ed5d3b1fe70cb955228e732dc5678c5d4c056c1a96da8bcdeaee23",
    "powerlaw/input": "ceca68a06a54c095cc45a9e373165d2c8bcd61dd78e7b91128cbbedc097259af",
    "powerlaw/kway": "5b804e74a72d4bc2a98bdbfa860b81e8ad135f71d742ebf2c3268c58fe6ee09c",
    "powerlaw/kway_symmetrise": "f29a6ea98fb37481a0c4ec2e9266e0b563a86cdcdb3b58bc80c1053152e71df6",
    "powerlaw/permute": "d98d629ed0b8e263dd3bf1190cc7f609d9ea42e0f7157161a743e56be11d0ab2",
    "powerlaw/rcm": "d9c21ffe38f926a4dd8f5ecc832df116edfb6e4889b6029d3bca7930b3afe7a2",
    "unsorted/input": "3213d65ac173750f612c2d581eb80b841914879332262b9e98f5872f3a4c59ce",
    "unsorted/kway": "a1d2502f6033099c69d4e4e0c22d6c019579b6d5a12128b49d000152ba0906a8",
    "unsorted/kway_symmetrise": "4a106f2e962770425550b13a1263e66f8d8beda259679cbc8f6ed3c142ae80c2",
    "unsorted/permute": "427bb5fd16ee8518a90c97f60b3b2b0437240877f58309d38b659af31402cb62",
    "unsorted/rcm": "2e0683b4d56e80d3cdcb75f58d73c3c86186ca1543278d1f86284db868d7477c",
}

WORKSPACE_BYTES = {
    "ttg_kway_coarsen_workspace_bytes(1000, 1099511627776)": 35189369906944,
    "ttg_kway_coarsen_workspace_bytes(1000, 1099511627777)": 0,
    "ttg_kway_coarsen_workspace_bytes(2147483646, 0)": 77357282560,
    "ttg_kway_coarsen_workspace_bytes(2147483647, 0)": 0,
    "ttg_kway_coarsen_workspace_bytes(2147483648, 0)": 0,
    "ttg_kway_refine_workspace_bytes(2147483646, 2)": 152519211008,
    "ttg_kway_refine_workspace_bytes(2147483647, 2)": 0,
    "ttg_kway_refine_workspace_bytes(2147483648, 2)": 0,
    "ttg_kway_symmetrise_workspace_bytes(1000, 1099511627776)": 52786553694976,
    "ttg_kway_symmetrise_workspace_bytes(1000, 1099511627777)": 0,
    "ttg_kway_symmetrise_workspace_bytes(2147483646, 0)": 2304,
    "ttg_kway_symmetrise_workspace_bytes(2147483647, 0)": 0,
    "ttg_kway_symmetrise_workspace_bytes(2147483648, 0)": 0,
    "ttg_permute_csr_workspace_bytes(2147483646)": 34367248128,
    "ttg_permute_csr_workspace_bytes(2147483647)": 34367248128,
    "ttg_permute_csr_workspace_bytes(2147483648)": 0,
    "ttg_rcm_order_workspace_bytes(2147483646)": 131044372480,
    "ttg_rcm_order_workspace_bytes(2147483647)": 131044372480,
    "ttg_rcm_order_workspace_bytes(2147483648)": 0,
    "ttg_rcm_symmetrise_workspace_bytes(1000, 1099511627776)": 52785720731648,
    "ttg_rcm_symmetrise_workspace_bytes(1000, 1099511627777)": 0,
    "ttg_rcm_symmetrise_workspace_bytes(2147483646, 0)": 2560,
    "ttg_rcm_symmetrise_workspace_bytes(2147483647, 0)": 2560,
    "ttg_rcm_symmetrise_workspace_bytes(2147483648, 0)": 0,
}


def _tool():
    spec = importlib.util.spec_from_file_location("reorder_digests", TOOL)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_outputs_match_the_recorded_digests(ttg_lib):
    got = _tool().digests()
    assert sorted(got) == sorted(DIGESTS)
    assert [k for k in DIGESTS if got[k] != DIGESTS[k]] == []


def test_workspace_sizes_at_the_limits(ttg_lib):
    assert _tool().workspace_sizes() == WORKSPACE_BYTES
