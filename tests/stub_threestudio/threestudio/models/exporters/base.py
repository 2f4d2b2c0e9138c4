"""models/exporters/base.py of the reference, interface only: ExporterOutput (save_name, save_type, params) and
Exporter(BaseObject), whose configure(geometry, material, background) keeps the three modules without registering them."""
from dataclasses import dataclass
from typing import Any, Dict, List

from threestudio.utils.base import BaseObject


@dataclass
class ExporterOutput:
    save_name: str
    save_type: str
    params: Dict[str, Any]


class Exporter(BaseObject):
    @dataclass
    class Config(BaseObject.Config):
        save_video: bool = False

    cfg: Config

    def configure(self, geometry, material, background) -> None:
        @dataclass
        class SubModules:
            geometry: Any
            material: Any
            background: Any

        self.sub_modules = SubModules(geometry, material, background)

    @property
    def geometry(self):
        return self.sub_modules.geometry

    @property
    def material(self):
        return self.sub_modules.material

    @property
    def background(self):
        return self.sub_modules.background

    def __call__(self, *args, **kwargs) -> List[ExporterOutput]:
        raise NotImplementedError
